/*
 * fastobj.c -- CPython extension `structuredetector_b200._fastobj`: the object-assembly loop of the decoder.
 *
 * Replaces the Python loops of the reference decoder that turn the packed top-K tensors into
 * ImageAnnotation / Object / Keypoint instances (src/sdnet/data/decoders.py:103-139 for Decoder,
 * :142-159 for raw_parts, :345-423 for KeypointDecoder): the reference reads every scalar with .item();
 * here the packed result arrives in ONE device->host copy and this module walks it in C.
 *
 * Keypoint and Object declare __slots__, so an instance is one tp_alloc plus direct stores at the slot
 * offsets (no __init__ call, no attribute protocol): ~0.1 us per object instead of ~0.4 us.  The arithmetic
 * is the reference's: coordinates are float32 values widened to double and multiplied by in/out in double
 * (utils.py:19-26 via decoders.py:139), `score > conf` for objects and `not score < conf` for raw parts in
 * double (decoders.py:116,153).  `conf` is one threshold, or a sequence of thresholds indexed by the slot's class
 * (anchor classes for assemble / json_text, part kinds for keypoints).
 *
 * Host-only C (gcc); built by structuredetector_b200/build.py next to the CUDA library.
 */
#define PY_SSIZE_T_CLEAN
#include <Python.h>
#include <descrobject.h>
#include <stdint.h>
#include <string.h>
#include <structmember.h>

typedef struct {
  PyTypeObject* type;
  Py_ssize_t off[4];
  int n;
} SlotClass;

/* Offsets of the named __slots__ members of a class; fails if one of them is not a slot. */
static int slot_class_init(SlotClass* sc, PyObject* type, const char* const* names, int n) {
  if (!PyType_Check(type)) {
    PyErr_SetString(PyExc_TypeError, "expected a class");
    return -1;
  }
  sc->type = (PyTypeObject*)type;
  sc->n = n;
  for (int i = 0; i < n; ++i) {
    PyObject* d = PyObject_GetAttrString(type, names[i]);
    if (!d) return -1;
    if (Py_TYPE(d) != &PyMemberDescr_Type || ((PyMemberDescrObject*)d)->d_member->type != T_OBJECT_EX) {
      Py_DECREF(d);
      PyErr_Format(PyExc_TypeError, "%s.%s is not a __slots__ member", sc->type->tp_name, names[i]);
      return -1;
    }
    sc->off[i] = ((PyMemberDescrObject*)d)->d_member->offset;
    Py_DECREF(d);
  }
  return 0;
}

#define SLOT(obj, sc, i) (*(PyObject**)((char*)(obj) + (sc)->off[i]))

/* Keypoint(kind, x, y, score) without running __init__; steals nothing, returns a new reference. */
static PyObject* new_keypoint(const SlotClass* kc, PyObject* kind, double x, double y, double score) {
  PyObject* o = kc->type->tp_alloc(kc->type, 0);
  if (!o) return NULL;
  PyObject *px = PyFloat_FromDouble(x), *py = PyFloat_FromDouble(y), *ps = PyFloat_FromDouble(score);
  if (!px || !py || !ps) {
    Py_XDECREF(px); Py_XDECREF(py); Py_XDECREF(ps); Py_DECREF(o);
    return NULL;
  }
  Py_INCREF(kind);
  SLOT(o, kc, 0) = kind;
  SLOT(o, kc, 1) = px;
  SLOT(o, kc, 2) = py;
  SLOT(o, kc, 3) = ps;
  return o;
}

typedef struct {
  Py_buffer anchor, part, assign;
} Views;

/* The threshold of a slot: one number for every class, or one per class index.  A class index the table does not
 * cover compares against -inf, so the slot is always kept and name_at reports the missing name. */
typedef struct {
  double scalar;
  double* table; /* NULL: scalar for every class */
  Py_ssize_t n;
} Conf;

static int conf_parse(PyObject* obj, Conf* c) {
  c->table = NULL;
  c->n = 0;
  c->scalar = 0.0;
  if (!PySequence_Check(obj)) {
    c->scalar = PyFloat_AsDouble(obj);
    return (c->scalar == -1.0 && PyErr_Occurred()) ? -1 : 0;
  }
  PyObject* seq = PySequence_Fast(obj, "conf must be a number or a sequence of per-class thresholds");
  if (!seq) return -1;
  c->n = PySequence_Fast_GET_SIZE(seq);
  c->table = (double*)PyMem_Malloc((size_t)(c->n > 0 ? c->n : 1) * sizeof(double));
  if (!c->table) { Py_DECREF(seq); PyErr_NoMemory(); return -1; }
  for (Py_ssize_t i = 0; i < c->n; ++i) {
    c->table[i] = PyFloat_AsDouble(PySequence_Fast_GET_ITEM(seq, i));
    if (c->table[i] == -1.0 && PyErr_Occurred()) { Py_DECREF(seq); PyMem_Free(c->table); c->table = NULL; return -1; }
  }
  Py_DECREF(seq);
  return 0;
}

static void conf_release(Conf* c) {
  if (c->table) PyMem_Free(c->table);
  c->table = NULL;
}

static inline double conf_of(const Conf* c, float cls) {
  if (!c->table) return c->scalar;
  const long idx = (long)cls;
  return (idx >= 0 && idx < c->n) ? c->table[idx] : -1.0 / 0.0;
}

static void views_release(Views* v) {
  if (v->anchor.obj) PyBuffer_Release(&v->anchor);
  if (v->part.obj) PyBuffer_Release(&v->part);
  if (v->assign.obj) PyBuffer_Release(&v->assign);
}

static PyObject* name_at(PyObject* names, long idx) {
  if (idx < 0 || idx >= PyList_GET_SIZE(names)) {
    PyErr_Format(PyExc_IndexError, "class index %ld outside the label map (%zd names)", idx, PyList_GET_SIZE(names));
    return NULL;
  }
  PyObject* n = PyList_GET_ITEM(names, idx);
  if (n == Py_None) {
    PyErr_Format(PyExc_KeyError, "class index %ld has no name in the label map", idx);
    return NULL;
  }
  return n;
}

/* assemble(anchor_out, part_out, assign, B, K, P, conf, sx, sy, labels, kinds, anchor_name, Keypoint, Object, ImageAnnotation)
 *   -> list[ImageAnnotation]       (decoders.py:103-139); conf: a number or one threshold per anchor class */
static PyObject* assemble(PyObject* self, PyObject* args) {
  PyObject *a_obj, *p_obj, *s_obj, *c_obj, *labels, *kinds, *anchor_name, *kp_type, *obj_type, *ann_type;
  Py_ssize_t B, K, P;
  double sx, sy;
  if (!PyArg_ParseTuple(args, "OOOnnnOddO!O!UOOO", &a_obj, &p_obj, &s_obj, &B, &K, &P, &c_obj, &sx, &sy, &PyList_Type, &labels,
                        &PyList_Type, &kinds, &anchor_name, &kp_type, &obj_type, &ann_type))
    return NULL;
  static const char* const kp_names[] = {"kind", "x", "y", "score"};
  static const char* const ob_names[] = {"name", "anchor", "parts", "box"};
  SlotClass kc, oc;
  if (slot_class_init(&kc, kp_type, kp_names, 4) < 0 || slot_class_init(&oc, obj_type, ob_names, 4) < 0) return NULL;
  Conf conf;
  if (conf_parse(c_obj, &conf) < 0) return NULL;
  Views v = {{0}, {0}, {0}};
  PyObject* result = NULL;
  PyObject** buckets = NULL;
  Py_ssize_t* fill = NULL;
  if (PyObject_GetBuffer(a_obj, &v.anchor, PyBUF_SIMPLE) < 0 || PyObject_GetBuffer(p_obj, &v.part, PyBUF_SIMPLE) < 0 ||
      PyObject_GetBuffer(s_obj, &v.assign, PyBUF_SIMPLE) < 0)
    goto done;
  if (B < 0 || K <= 0 || P <= 0 || v.anchor.len < B * K * 16 || v.part.len < B * P * 24 || v.assign.len < B * P * 4) {
    PyErr_SetString(PyExc_ValueError, "packed buffers are smaller than (B, K, 4) / (B, P, 6) / (B, P)");
    goto done;
  }
  buckets = (PyObject**)PyMem_Calloc((size_t)K, sizeof(PyObject*));
  fill = (Py_ssize_t*)PyMem_Calloc((size_t)K, 2 * sizeof(Py_ssize_t)); /* [0, K): parts per slot, [K, 2K): filled so far */
  result = PyList_New(B);
  if (!buckets || !fill || !result) { Py_CLEAR(result); PyErr_NoMemory(); goto done; }
  const float* A = (const float*)v.anchor.buf;
  const float* Pt = (const float*)v.part.buf;
  const int32_t* S = (const int32_t*)v.assign.buf;
  for (Py_ssize_t b = 0; b < B; ++b) {
    const float* a = A + b * K * 4;
    const float* p = Pt + b * P * 6;
    const int32_t* s = S + b * P;
    int failed = 0;
    /* parts of each anchor slot, in part-slot (= score) order; only slots that will be emitted get a list.
     * Two sweeps, so that every list is allocated once at its final size. */
    Py_ssize_t n_objects = 0;
    for (Py_ssize_t k = 0; k < K; ++k) {
      fill[k] = fill[K + k] = 0;
      n_objects += (double)a[k * 4 + 2] > conf_of(&conf, a[k * 4 + 3]); /* decoders.py:116: score <= conf_thresh -> skip */
    }
    for (Py_ssize_t i = 0; i < P; ++i) {
      const int32_t slot = s[i];
      /* grouped onto an anchor that is not emitted (score == float32(conf) > conf): dropped, as in the reference */
      if (slot >= 0 && slot < K && (double)a[slot * 4 + 2] > conf_of(&conf, a[slot * 4 + 3])) ++fill[slot];
    }
    for (Py_ssize_t i = 0; i < P && !failed; ++i) {
      const int32_t slot = s[i];
      if (slot < 0 || slot >= K || !((double)a[slot * 4 + 2] > conf_of(&conf, a[slot * 4 + 3]))) continue;
      PyObject* kind = name_at(kinds, (long)p[i * 6 + 3]);
      PyObject* kp = kind ? new_keypoint(&kc, kind, (double)p[i * 6] * sx, (double)p[i * 6 + 1] * sy, (double)p[i * 6 + 2]) : NULL;
      if (!kp) { failed = 1; break; }
      if (!buckets[slot] && !(buckets[slot] = PyList_New(fill[slot]))) { Py_DECREF(kp); failed = 1; break; }
      PyList_SET_ITEM(buckets[slot], fill[K + slot]++, kp);
    }
    if (failed) /* a list with unset items must not be seen by anyone: fill the holes before it is released */
      for (Py_ssize_t k = 0; k < K; ++k)
        if (buckets[k])
          for (Py_ssize_t q = fill[K + k]; q < fill[k]; ++q) { Py_INCREF(Py_None); PyList_SET_ITEM(buckets[k], q, Py_None); }
    PyObject* objects = failed ? NULL : PyList_New(n_objects);
    if (!objects) failed = 1;
    Py_ssize_t n_out = 0;
    for (Py_ssize_t k = 0; k < K && !failed; ++k) {
      if (!((double)a[k * 4 + 2] > conf_of(&conf, a[k * 4 + 3]))) continue;
      PyObject* label = name_at(labels, (long)a[k * 4 + 3]);
      PyObject* anchor = label ? new_keypoint(&kc, anchor_name, (double)a[k * 4] * sx, (double)a[k * 4 + 1] * sy, (double)a[k * 4 + 2]) : NULL;
      PyObject* parts = buckets[k] ? buckets[k] : (anchor ? PyList_New(0) : NULL);
      buckets[k] = NULL;
      PyObject* o = (anchor && parts) ? oc.type->tp_alloc(oc.type, 0) : NULL;
      if (!o) { Py_XDECREF(anchor); Py_XDECREF(parts); failed = 1; break; }
      Py_INCREF(label);
      SLOT(o, &oc, 0) = label;
      SLOT(o, &oc, 1) = anchor;
      SLOT(o, &oc, 2) = parts;
      Py_INCREF(Py_None);
      SLOT(o, &oc, 3) = Py_None;
      PyList_SET_ITEM(objects, n_out++, o);
    }
    if (objects && failed)
      for (Py_ssize_t q = n_out; q < n_objects; ++q) { Py_INCREF(Py_None); PyList_SET_ITEM(objects, q, Py_None); }
    for (Py_ssize_t k = 0; k < K; ++k) Py_CLEAR(buckets[k]);
    PyObject* ann = NULL;
    if (!failed) {
      PyObject* path = PyUnicode_FromFormat("batch_%zd", b);
      if (path) {
        ann = PyObject_CallFunctionObjArgs(ann_type, path, objects, NULL);
        Py_DECREF(path);
      }
    }
    Py_XDECREF(objects);
    if (!ann) { Py_CLEAR(result); goto done; }
    PyList_SET_ITEM(result, b, ann);
  }
done:
  if (buckets) PyMem_Free(buckets);
  if (fill) PyMem_Free(fill);
  views_release(&v);
  conf_release(&conf);
  return result;
}

/* keypoints(rows, B, n, width, conf, sx, sy, names, Keypoint) -> list[list[Keypoint]]
 * Every slot of a (B, n, width) float32 array (x, y, score, class, ...) whose score is not below conf (a number or one
 * threshold per class), in slot order: raw_parts of Decoder (decoders.py:142-159; double arithmetic). */
static PyObject* keypoints(PyObject* self, PyObject* args) {
  PyObject *r_obj, *c_obj, *names, *kp_type;
  Py_ssize_t B, n, width;
  double sx, sy;
  if (!PyArg_ParseTuple(args, "OnnnOddO!O", &r_obj, &B, &n, &width, &c_obj, &sx, &sy, &PyList_Type, &names, &kp_type)) return NULL;
  static const char* const kp_names[] = {"kind", "x", "y", "score"};
  SlotClass kc;
  if (slot_class_init(&kc, kp_type, kp_names, 4) < 0) return NULL;
  Conf conf;
  if (conf_parse(c_obj, &conf) < 0) return NULL;
  Py_buffer rows;
  if (PyObject_GetBuffer(r_obj, &rows, PyBUF_SIMPLE) < 0) { conf_release(&conf); return NULL; }
  PyObject* result = NULL;
  if (B < 0 || n <= 0 || width < 4 || rows.len < B * n * width * 4) {
    PyErr_SetString(PyExc_ValueError, "packed buffer is smaller than (B, n, width)");
    goto done;
  }
  result = PyList_New(B);
  if (!result) goto done;
  const float* R = (const float*)rows.buf;
  for (Py_ssize_t b = 0; b < B; ++b) {
    PyObject* out = PyList_New(0);
    if (!out) { Py_CLEAR(result); goto done; }
    PyList_SET_ITEM(result, b, out);
    for (Py_ssize_t i = 0; i < n; ++i) {
      const float* r = R + (b * n + i) * width;
      if ((double)r[2] < conf_of(&conf, r[3])) continue; /* decoders.py:153 */
      PyObject* kind = name_at(names, (long)r[3]);
      PyObject* kp = kind ? new_keypoint(&kc, kind, (double)r[0] * sx, (double)r[1] * sy, (double)r[2]) : NULL;
      if (!kp || PyList_Append(out, kp) < 0) { Py_XDECREF(kp); Py_CLEAR(result); goto done; }
      Py_DECREF(kp);
    }
  }
done:
  PyBuffer_Release(&rows);
  conf_release(&conf);
  return result;
}

/* ---- packed detections -> JSON text, without building a single annotation object ---------------------------
 * json_text(anchor_out, part_out, assign, B, K, P, conf, sx, sy, resize, labels_json, kinds_json, anchor_json,
 *           paths_json, sizes_json) -> list[str]
 * One string per image, byte-identical to json.dumps(annotation.json_repr(), indent=2) of the annotation the decoder
 * would have returned (utils.py:275-286; Keypoint / Object json_repr :52-57, 205-212), optionally after
 * annotation.resize(net_size, img_size) as `detect` does (cli/detect.py:42-53): resize[b] = (rx, ry) or None.
 * Names, paths and image sizes arrive already JSON-encoded (json.dumps on the Python side); floats are written with
 * float.__repr__'s shortest round-trip form, which is what json.dumps uses. */
typedef struct {
  char* data;
  size_t len, cap;
} Buf;

static int buf_reserve(Buf* b, size_t extra) {
  if (b->len + extra <= b->cap) return 0;
  size_t cap = b->cap ? b->cap : 4096;
  while (cap < b->len + extra) cap *= 2;
  char* d = (char*)PyMem_Realloc(b->data, cap);
  if (!d) { PyErr_NoMemory(); return -1; }
  b->data = d;
  b->cap = cap;
  return 0;
}
static int buf_put(Buf* b, const char* s, size_t n) {
  if (buf_reserve(b, n) < 0) return -1;
  memcpy(b->data + b->len, s, n);
  b->len += n;
  return 0;
}
#define PUT(b, lit) buf_put((b), (lit), sizeof(lit) - 1)
static int buf_put_obj(Buf* b, PyObject* str) {
  Py_ssize_t n;
  const char* s = PyUnicode_AsUTF8AndSize(str, &n);
  return s ? buf_put(b, s, (size_t)n) : -1;
}
static int buf_put_double(Buf* b, double v) {
  if (v != v) return PUT(b, "NaN");
  if (v > 1.7976931348623157e308) return PUT(b, "Infinity");
  if (v < -1.7976931348623157e308) return PUT(b, "-Infinity");
  char* s = PyOS_double_to_string(v, 'r', 0, Py_DTSF_ADD_DOT_0, NULL);
  if (!s) return -1;
  const int rc = buf_put(b, s, strlen(s));
  PyMem_Free(s);
  return rc;
}
/* one keypoint of an object's "parts" list (8 spaces deep) */
static int put_keypoint(Buf* b, PyObject* kind_json, double x, double y, double score) {
  if (PUT(b, "        {\n          \"kind\": ") < 0 || buf_put_obj(b, kind_json) < 0 ||
      PUT(b, ",\n          \"location\": {\n            \"x\": ") < 0 || buf_put_double(b, x) < 0 ||
      PUT(b, ",\n            \"y\": ") < 0 || buf_put_double(b, y) < 0 || PUT(b, "\n          },\n          \"score\": ") < 0 ||
      buf_put_double(b, score) < 0 || PUT(b, "\n        }") < 0)
    return -1;
  return 0;
}

static PyObject* json_text(PyObject* self, PyObject* args) {
  PyObject *a_obj, *p_obj, *s_obj, *c_obj, *resize, *labels, *kinds, *anchor_json, *paths, *sizes;
  Py_ssize_t B, K, P;
  double sx, sy;
  if (!PyArg_ParseTuple(args, "OOOnnnOddO!O!O!UO!O!", &a_obj, &p_obj, &s_obj, &B, &K, &P, &c_obj, &sx, &sy, &PyList_Type, &resize,
                        &PyList_Type, &labels, &PyList_Type, &kinds, &anchor_json, &PyList_Type, &paths, &PyList_Type, &sizes))
    return NULL;
  if (PyList_GET_SIZE(resize) != B || PyList_GET_SIZE(paths) != B || PyList_GET_SIZE(sizes) != B) {
    PyErr_SetString(PyExc_ValueError, "resize, paths and sizes need one entry per image");
    return NULL;
  }
  Conf conf;
  if (conf_parse(c_obj, &conf) < 0) return NULL;
  Views v = {{0}, {0}, {0}};
  PyObject* result = NULL;
  Buf buf = {NULL, 0, 0};
  if (PyObject_GetBuffer(a_obj, &v.anchor, PyBUF_SIMPLE) < 0 || PyObject_GetBuffer(p_obj, &v.part, PyBUF_SIMPLE) < 0 ||
      PyObject_GetBuffer(s_obj, &v.assign, PyBUF_SIMPLE) < 0)
    goto done;
  if (B < 0 || K <= 0 || P <= 0 || v.anchor.len < B * K * 16 || v.part.len < B * P * 24 || v.assign.len < B * P * 4) {
    PyErr_SetString(PyExc_ValueError, "packed buffers are smaller than (B, K, 4) / (B, P, 6) / (B, P)");
    goto done;
  }
  result = PyList_New(B);
  if (!result) goto done;
  const float* A = (const float*)v.anchor.buf;
  const float* Pt = (const float*)v.part.buf;
  const int32_t* S = (const int32_t*)v.assign.buf;
  for (Py_ssize_t b = 0; b < B; ++b) {
    const float* a = A + b * K * 4;
    const float* p = Pt + b * P * 6;
    const int32_t* s = S + b * P;
    double rx = 1.0, ry = 1.0;
    int resized = 0;
    PyObject* r = PyList_GET_ITEM(resize, b);
    if (r != Py_None) {
      if (!PyArg_ParseTuple(r, "dd", &rx, &ry)) { Py_CLEAR(result); goto done; }
      resized = 1;
    }
    buf.len = 0;
    int bad = PUT(&buf, "{\n  \"image_path\": ") < 0 || buf_put_obj(&buf, PyList_GET_ITEM(paths, b)) < 0 ||
              PUT(&buf, ",\n  \"img_size\": ") < 0 || buf_put_obj(&buf, PyList_GET_ITEM(sizes, b)) < 0 ||
              PUT(&buf, ",\n  \"objects\": [") < 0;
    Py_ssize_t n_out = 0;
    for (Py_ssize_t k = 0; k < K && !bad; ++k) {
      if (!((double)a[k * 4 + 2] > conf_of(&conf, a[k * 4 + 3]))) continue;
      PyObject* label = name_at(labels, (long)a[k * 4 + 3]);
      if (!label) { bad = 1; break; }
      bad = (n_out && PUT(&buf, ",") < 0) || PUT(&buf, "\n    {\n      \"label\": ") < 0 || buf_put_obj(&buf, label) < 0 ||
            PUT(&buf, ",\n      \"box\": null,\n      \"parts\": [\n") < 0;
      double x = (double)a[k * 4] * sx, y = (double)a[k * 4 + 1] * sy;
      if (resized) { x *= rx; y *= ry; }
      bad = bad || put_keypoint(&buf, anchor_json, x, y, (double)a[k * 4 + 2]) < 0;
      for (Py_ssize_t i = 0; i < P && !bad; ++i) {
        if (s[i] != k) continue;
        PyObject* kind = name_at(kinds, (long)p[i * 6 + 3]);
        if (!kind) { bad = 1; break; }
        double px = (double)p[i * 6] * sx, py = (double)p[i * 6 + 1] * sy;
        if (resized) { px *= rx; py *= ry; }
        bad = PUT(&buf, ",\n") < 0 || put_keypoint(&buf, kind, px, py, (double)p[i * 6 + 2]) < 0;
      }
      bad = bad || PUT(&buf, "\n      ]\n    }") < 0;
      ++n_out;
    }
    bad = bad || (n_out && PUT(&buf, "\n  ") < 0) || PUT(&buf, "]\n}") < 0;
    PyObject* text = bad ? NULL : PyUnicode_DecodeUTF8(buf.data, (Py_ssize_t)buf.len, "strict");
    if (!text) { Py_CLEAR(result); goto done; }
    PyList_SET_ITEM(result, b, text);
  }
done:
  if (buf.data) PyMem_Free(buf.data);
  views_release(&v);
  conf_release(&conf);
  return result;
}

static PyMethodDef methods[] = {
    {"assemble", assemble, METH_VARARGS, "packed detections -> list[ImageAnnotation] (decoders.py:103-139)"},
    {"keypoints", keypoints, METH_VARARGS, "packed part rows -> list[list[Keypoint]] (decoders.py:142-159)"},
    {"json_text", json_text, METH_VARARGS, "packed detections -> list[str], one JSON document per image (utils.py:275-286)"},
    {NULL, NULL, 0, NULL}};

static struct PyModuleDef module = {PyModuleDef_HEAD_INIT, "_fastobj", "C object assembly of the SDNet decoding path", -1, methods};

PyMODINIT_FUNC PyInit__fastobj(void) { return PyModule_Create(&module); }
