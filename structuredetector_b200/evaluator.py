"""The reference evaluator's metrics, computed on the device from the packed detections.

Mirrors ``Evaluation`` / ``Evaluations`` / ``Evaluator`` of the reference (reference:
src/sdnet/model/evaluator.py:13-120, 123-206, 209-646): same attribute and property names, same
formulas, so tables and CSV code written against them keep working.  What moves to the GPU is the matching:
``eval_anchor`` (:244-284) and ``eval_part`` (:286-334) -- per image and label, detections in score order
against their nearest ground truth -- through ``sdnet_match_launch``; ``eval_csi`` with ``compute_csi``
(:380-420, 539-581) and ``eval_classif`` (:429-474) -- predicted objects (anchor + grouped parts) against
ground-truth objects -- through ``sdnet_match_objects_launch``; both straight on the tensors
``sdnet_decode_launch`` wrote: no Python object is built for a prediction.  ``ThresholdSweep`` runs both at many
confidence thresholds, and optionally grouping distances, from one decode (``sdnet_sweep_launch``): the precision /
recall / F1 curve over the threshold, or its surface over (threshold, grouping distance).
"""
from __future__ import annotations

import ctypes
import math
from functools import reduce
from pathlib import Path

import numpy as np
import torch

from . import _native, ops

__all__ = ["Evaluation", "Evaluations", "Evaluator", "ThresholdSweep"]


class Evaluation:
    """tp / npos / ndet counters plus the localisation errors of the true positives."""

    def __init__(self, tp=0, npos=0, ndet=0, acc=None, counts=None):
        assert tp >= 0 and ndet >= 0 and npos >= 0, "tp, npos and ndet should be positive"
        assert tp <= ndet, "tp must be lower than or equal to ndet"
        assert tp <= npos, "tp must be lower than or equal to npos"
        self.tp, self.npos, self.ndet = tp, npos, ndet
        self.acc = acc or []
        self.count_errors = counts or []

    def reset(self):
        self.__init__()

    def __iadd__(self, other):
        self.tp += other.tp
        self.npos += other.npos
        self.ndet += other.ndet
        self.acc += other.acc
        self.count_errors += other.count_errors
        return self

    def __add__(self, other):
        total = Evaluation(self.tp, self.npos, self.ndet, list(self.acc), list(self.count_errors))
        total += other
        return total

    fp = property(lambda self: self.ndet - self.tp)
    fn = property(lambda self: self.npos - self.tp)

    @property
    def csi(self):
        union = self.npos + self.ndet - self.tp
        return self.tp / union if union != 0 else 1

    @property
    def precision(self):
        return self.tp / self.ndet if self.ndet != 0 else 1 if self.npos == 0 else 0

    @property
    def recall(self):
        return self.tp / self.npos if self.npos != 0 else 1 if self.ndet == 0 else 0

    @property
    def f1_score(self):
        total = self.npos + self.ndet
        return 2 * self.tp / total if total != 0 else 1

    @property
    def avg_acc(self):
        return np.mean(self.acc) if len(self.acc) != 0 else float("nan")

    @property
    def acc_err(self):
        return np.std(self.acc) / np.sqrt(len(self.acc)) if len(self.acc) != 0 else float("nan")

    def stats(self):
        return (f"{self.npos}", f"{self.ndet}", f"{self.recall:.2%}", f"{self.precision:.2%}", f"{self.f1_score:.2%}",
                f"{self.avg_acc:.4%}", f"{self.acc_err:.4%}")

    COLUMNS = ("Gts.", "Preds.", "Rec.", "Prec.", "F1 Score", "L. Acc.", "L. Err.")

    @staticmethod
    def columns():
        """Column headers of ``stats()`` (evaluator.py:88-98; ``rich`` Column objects when rich is installed)."""
        try:
            from rich.table import Column
        except ImportError:
            return Evaluation.COLUMNS
        return tuple(Column(name, justify="right", **({"style": "green"} if name == "F1 Score" else {}))
                     for name in Evaluation.COLUMNS)

    def pretty_print(self):
        single = Evaluations()
        single.evals = {"": self}
        _print_table(None, single)

    def save_conf_matrix(self):
        """One 10 x 10 (expected parts, predicted parts) count matrix per label, as ``conf_mat_<label>.npy``
        (evaluator.py:107-113)."""
        by_label = {}
        for label, predicted, expected in self.count_errors:
            by_label.setdefault(label, []).append((predicted, expected))
        for label, pairs in by_label.items():
            mat = np.zeros((10, 10))
            for predicted, expected in pairs:
                mat[expected, predicted] += 1
            np.save(f"conf_mat_{label}.npy", mat)

    def __repr__(self):
        return (f"f1: {self.f1_score:.2%}, rec: {self.recall:.2%}, prec: {self.precision:.2%}, npos: {self.npos}, "
                f"ndet: {self.ndet}, tp/fp/fn: {self.tp}/{self.fp}/{self.fn}, avg_acc: {self.avg_acc:.2}")


def _print_table(title, evaluations):
    """A ``rich`` table like the reference prints (evaluator.py:190-196, 583-604); plain text without rich."""
    rows = [(label, *evaluation.stats()) for label, evaluation in evaluations.items()]
    total = ("Total", *evaluations.reduce().stats()) if len(evaluations) > 1 else None
    try:
        from rich import print as rprint
        from rich.table import Column, Table
    except ImportError:
        if title:
            print(title)
        for row in rows + ([total] if total else []):
            print(" ", *row)
        return
    table = Table(Column("Label", style="bold"), *Evaluation.columns(), title=title)
    for row in rows:
        table.add_row(*row)
    if total:
        table.add_row(*total, style="bold")
    rprint(table)


class Evaluations:
    """One ``Evaluation`` per label."""

    def __init__(self, labels=None):
        self.evals = {label: Evaluation() for label in labels} if labels else {}

    def reset(self):
        for evaluation in self.evals.values():
            evaluation.reset()

    labels = property(lambda self: self.evals.keys())

    def items(self):
        return self.evals.items()

    def __getitem__(self, label):
        return self.evals[label]

    def __setitem__(self, label, evaluation):
        self.evals[label] = evaluation

    def __len__(self):
        return len(self.evals)

    def __iadd__(self, other):
        assert self.labels == other.labels, "The Evaluations should have the same labels"
        for label, evaluation in other.items():
            self.evals[label] += evaluation
        return self

    def __add__(self, other):
        assert self.labels == other.labels, "The Evaluations should have the same labels"
        total = Evaluations()
        total.evals = {label: self.evals[label] + evaluation for label, evaluation in other.items()}
        return total

    def __or__(self, other):
        merged = Evaluations()
        merged.evals = {label: self[label] + other[label] for label in self.labels & other.labels}
        merged.evals.update({label: self[label] for label in self.labels - other.labels})
        merged.evals.update({label: other[label] for label in other.labels - self.labels})
        return merged

    def __ior__(self, other):
        """In-place union (evaluator.py:180-185; the reference's version recurses into itself -- this does what it
        is written to mean): labels only ``other`` has are adopted, shared labels are summed."""
        for label, evaluation in other.items():
            self.evals[label] = self.evals[label] + evaluation if label in self.evals else evaluation
        return self

    def reduce(self):
        return reduce(Evaluation.__iadd__, self.evals.values(), Evaluation())

    def pretty_print(self, table_name=None):
        _print_table(table_name, self)

    def __repr__(self):
        lines = [f"total: {self.reduce()}"] if len(self) > 1 else []
        return "\n".join(lines + [f"{label}: {evaluation}" for label, evaluation in self.items()])


class Evaluator:
    """``Evaluator(args)`` reads ``args.labels`` / ``args.parts`` (name -> class index, args.py),
    ``args.width`` / ``args.height`` (network input size), ``args.dist_threshold``, and for the decoder
    side ``args.conf_threshold`` and ``args.down_ratio`` -- the reference evaluator's fields
    (evaluator.py:210-213,245-250) plus the two the decoder applied before it."""

    def __init__(self, args):
        self.args = args
        self.labels = args.labels.keys()
        self.kp_labels = args.parts.keys()
        self._label_index = dict(args.labels)
        self._part_index = dict(args.parts)
        self._label_names = {index: name for name, index in args.labels.items()}
        self._part_names = {index: name for name, index in args.parts.items()}
        self.lib = _native.load()
        self.reset()

    def reset(self):
        self.anchor_eval = Evaluations(self.labels)
        self.part_eval = Evaluations(self.kp_labels)
        self.csi_eval = Evaluations(self.labels)
        self.classification_eval = Evaluations(Evaluator.get_classification_labels())

    @property
    def kps_eval(self):
        return self.anchor_eval | self.part_eval

    @staticmethod
    def get_classification_labels():
        """The reference's hard-coded (label, number of parts) classes (evaluator.py:422-427)."""
        return [f"bean_{index}" for index in range(10)] + [f"maize_{index}" for index in range(10)]

    # -- ground truth -> tensors -------------------------------------------------------------
    def _pack_ground_truth(self, annotations, device):
        rows_a = [[(obj.anchor.x, obj.anchor.y, self._label_index.get(obj.name, -1)) for obj in ann.objects]
                  for ann in annotations]
        rows_p = [[(kp.x, kp.y, self._part_index.get(kp.kind, -1)) for obj in ann.objects for kp in obj.parts]
                  for ann in annotations]

        owners = [[j for j, obj in enumerate(ann.objects) for _ in obj.parts] for ann in annotations]
        if any(len(obj.parts) > 64 for ann in annotations for obj in ann.objects):
            raise ValueError("a ground-truth object has more than 64 parts; the object matcher tracks them in a 64-bit mask")

        def pack(rows):
            width = max(1, max((len(r) for r in rows), default=0))
            if width > _native.MAX_GT:
                raise ValueError(f"{width} ground-truth points in one image; the matcher takes at most {_native.MAX_GT}")
            data = np.zeros((len(rows), width, 3), dtype=np.float64)
            for b, row in enumerate(rows):
                if row:
                    data[b, : len(row)] = row
            counts = np.array([len(r) for r in rows], dtype=np.int32)
            return torch.from_numpy(data).to(device), torch.from_numpy(counts).to(device), width

        scale = np.empty((len(annotations), 4), dtype=np.float64)
        for b, ann in enumerate(annotations):
            img_w, img_h = ann.img_size
            scale[b] = (img_w / self.args.width, img_h / self.args.height, min(ann.img_size) * self.args.dist_threshold,
                        min(ann.img_size))
        owner = np.zeros((len(annotations), max(1, max((len(o) for o in owners), default=0))), dtype=np.int32)
        for b, row in enumerate(owners):
            owner[b, : len(row)] = row
        return pack(rows_a), pack(rows_p), torch.from_numpy(scale).to(device), torch.from_numpy(owner).to(device)

    # -- the batched equivalent of accumulate(prediction, annotation, raw_parts) -------------------
    def accumulate_packed(self, packed: ops.PackedDetections, annotations, out_size, conf_thresh=None, eval_csi=False,
                          eval_classif=False):
        """Add one decoded batch.  ``packed`` = ``ops.decode_packed(...)`` (device tensors),
        ``annotations`` = the batch's ground truth (``ImageAnnotation`` with ``img_size``, coordinates in the
        network-input frame, as the reference's dataset yields them), ``out_size`` = (W, H) of the heat maps.
        Equivalent to ``accumulate(prediction, annotation, raw_parts, eval_csi, eval_classif)`` of the reference per
        image (evaluator.py:226-242; ``evaluate`` passes True, True: cli/evaluate.py:43-45).

        ``conf_thresh`` may be a mapping from label or part name to threshold, as ``Decoder`` takes it (the one the
        batch was decoded with): detections are then counted against their own label's threshold, and a name the
        mapping leaves out takes ``args.conf_threshold``."""
        default = self.args.conf_threshold
        conf = ops.class_thresholds(default if conf_thresh is None else conf_thresh, self._index_names(self._label_names),
                                    self._index_names(self._part_names), default)
        B, K = packed.anchor_inds.shape
        P = packed.part_inds.shape[1]
        assert len(annotations) == B
        device = packed.anchor_out.device
        M, N = len(self._label_index), len(self._part_index)
        (gt_a, n_a, wa), (gt_p, n_p, wp), scale, owner = self._pack_ground_truth(annotations, device)
        a_stats = torch.empty(B, M, 3, dtype=torch.int32, device=device)
        p_stats = torch.empty(B, N, 3, dtype=torch.int32, device=device)
        a_acc = torch.empty(B, K, dtype=torch.float64, device=device)
        p_acc = torch.empty(B, P, dtype=torch.float64, device=device)
        # per-class thresholds: M + N doubles (labels, then parts); `conf` covers classes the table has no entry for
        conf_class = torch.tensor(conf, dtype=torch.float64, device=device) if isinstance(conf, list) else None
        conf = float(default) if conf_class is not None else conf
        out_w, out_h = out_size
        in_w, in_h = int(self.args.down_ratio * out_w), int(self.args.down_ratio * out_h)  # decoders.py:37-38
        prm = _native.SdnetMatchParams()
        prm.struct_size = ctypes.sizeof(_native.SdnetMatchParams)
        prm.B, prm.M, prm.N, prm.K, prm.P = B, M, N, K, P
        prm.max_gt_anchors, prm.max_gt_parts = wa, wp
        prm.conf, prm.sx, prm.sy = float(conf), in_w / out_w, in_h / out_h
        prm.anchor_out, prm.part_out = packed.anchor_out.data_ptr(), packed.part_out.data_ptr()
        prm.image_scale = scale.data_ptr()
        prm.gt_anchors, prm.n_gt_anchors = gt_a.data_ptr(), n_a.data_ptr()
        prm.gt_parts, prm.n_gt_parts = gt_p.data_ptr(), n_p.data_ptr()
        prm.anchor_stats, prm.part_stats = a_stats.data_ptr(), p_stats.data_ptr()
        prm.anchor_acc, prm.part_acc = a_acc.data_ptr(), p_acc.data_ptr()
        prm.conf_class = conf_class.data_ptr() if conf_class is not None else None
        stream = torch.cuda.current_stream(device).cuda_stream
        _native.check(self.lib.sdnet_match_launch(ctypes.byref(prm), ctypes.c_void_p(stream)), "sdnet_match_launch")
        a_cls = packed.anchor_out[:, :, 3].to(torch.int32)
        p_cls = packed.part_out[:, :, 3].to(torch.int32)
        host = [t.cpu().numpy() for t in (a_stats, p_stats, a_acc, p_acc, a_cls, p_cls)]
        self._absorb(self.anchor_eval, self._label_names, host[0], host[2], host[4])
        self._absorb(self.part_eval, self._part_names, host[1], host[3], host[5])
        if not (eval_csi or eval_classif):
            return
        # ---- object-level metrics: eval_csi / compute_csi and eval_classif (evaluator.py:380-474, 539-581)
        groups = self._classification_groups(device)
        c_stats = torch.empty(B, M, 3, dtype=torch.int32, device=device)
        k_stats = torch.empty(B, 20, 3, dtype=torch.int32, device=device)
        c_acc = torch.empty(B, K, dtype=torch.float64, device=device)
        k_acc = torch.empty(B, K, dtype=torch.float64, device=device)
        n_parts = torch.empty(B, K, dtype=torch.int32, device=device)
        op = _native.SdnetObjectMatchParams()
        op.struct_size = ctypes.sizeof(_native.SdnetObjectMatchParams)
        op.B, op.M, op.N, op.K, op.P = B, M, N, K, P
        op.max_gt_objects, op.max_gt_parts = wa, wp
        op.conf, op.sx, op.sy = float(conf), in_w / out_w, in_h / out_h
        op.csi_threshold = float(getattr(self.args, "csi_threshold", 0.75))
        op.anchor_out, op.part_out, op.assign = packed.anchor_out.data_ptr(), packed.part_out.data_ptr(), packed.assign.data_ptr()
        op.image_scale = scale.data_ptr()
        op.gt_objects, op.n_gt_objects = gt_a.data_ptr(), n_a.data_ptr()
        op.gt_parts, op.gt_part_owner, op.n_gt_parts = gt_p.data_ptr(), owner.data_ptr(), n_p.data_ptr()
        op.cls_group = groups.data_ptr()
        op.csi_stats, op.csi_acc = c_stats.data_ptr(), c_acc.data_ptr()
        op.classif_stats, op.classif_acc, op.pred_parts = k_stats.data_ptr(), k_acc.data_ptr(), n_parts.data_ptr()
        op.conf_class = prm.conf_class
        _native.check(self.lib.sdnet_match_objects_launch(ctypes.byref(op), ctypes.c_void_p(stream)), "sdnet_match_objects_launch")
        c_stats, k_stats, c_acc, k_acc, n_parts = (t.cpu().numpy() for t in (c_stats, k_stats, c_acc, k_acc, n_parts))
        if eval_csi:
            self._absorb(self.csi_eval, self._label_names, c_stats, c_acc, host[4])
        if eval_classif:
            group_np = groups.cpu().numpy()
            key = np.where((n_parts >= 0) & (n_parts <= 9), group_np[np.clip(host[4], 0, M - 1)] * 10 + n_parts, -1)
            key = np.where(group_np[np.clip(host[4], 0, M - 1)] >= 0, key, -1)
            self._absorb(self.classification_eval, dict(enumerate(Evaluator.get_classification_labels())), k_stats, k_acc, key)

    @staticmethod
    def _index_names(names):
        """Name of every index 0 .. max, None where an index has no name."""
        return [names.get(i) for i in range(max(names, default=-1) + 1)]

    def _classification_groups(self, device):
        """cls_group of the object matchers: 0 / 1 for the classes named "bean" / "maize", -1 for the others."""
        return torch.tensor([{"bean": 0, "maize": 1}.get(self._label_names.get(i), -1) for i in range(len(self._label_index))],
                            dtype=torch.int32, device=device)

    @staticmethod
    def _absorb(target: Evaluations, names, stats, acc, cls):
        totals = stats.sum(axis=0)  # (classes, 3): ndet, npos, tp
        for index, name in names.items():
            res = target[name]
            res.ndet += int(totals[index, 0])
            res.npos += int(totals[index, 1])
            res.tp += int(totals[index, 2])
            hit = (cls == index) & ~np.isnan(acc)
            res.acc += acc[hit].tolist()  # image-major, slot (= score) order: the order the reference appends in

    def _results(self):
        return {"Anchor Location": self.anchor_eval, "Part Location": self.part_eval, "All Kps Location": self.kps_eval,
                "CSI": self.csi_eval, "Classification": self.classification_eval}

    def pretty_print(self):
        for title, evals in self._results().items():
            _print_table(title, evals)

    def save_kps_csv(self, path):
        """label, recall, precision, f1, average localisation error per keypoint label (evaluator.py:606-626)."""
        evals = self.kps_eval
        lines = [",".join((label, str(evals[label].recall), str(evals[label].precision), str(evals[label].f1_score),
                           str(evals[label].avg_acc))) for label in sorted(evals.labels)]
        Path(path).write_text("\n".join(lines))

    def __repr__(self):
        text = ""
        for title, evals in self._results().items():
            text += f"{title}\n"
            if len(evals) > 1:
                text += f"  total: {evals.reduce()}\n"
            for label, evaluation in sorted(evals.items(), key=lambda item: item[0]):
                text += f"  {label}: {evaluation}\n"
        return text


# Device bytes one sweep launch may write; accumulate_packed splits a larger batch into consecutive image slices.
SWEEP_OUTPUT_BUDGET = 1 << 30


class ThresholdSweep:
    """The evaluator at a grid of confidence thresholds, and optionally of grouping distances, from one decode.

    ``at(t)`` is a plain ``Evaluator`` holding exactly what ``Evaluator.accumulate_packed(decode at t, ...,
    conf_thresh=t)`` would hold, for every decode and evaluation this sweep has accumulated: the detections a decoder
    keeps do not depend on its threshold, only its grouping does, and ``sdnet_sweep_launch`` redoes the grouping at
    every grid point (the full nearest-anchor search of the decoder, in the same fp32 arithmetic) before matching.
    ``curve`` and ``best_threshold`` read the precision / recall / F1 curve off the grid.

    ``thresholds``: finite, strictly increasing, at most 256.  ``dtype``: the dtype of the heat maps the detections
    were decoded from -- the grouping compares ``score > t`` in that dtype, as the decoder does.  ``dist_thresh``: the
    decoder's grouping distance (default ``args.decoder_dist_thresh``); ``args`` as for ``Evaluator``.

    ``gates``: a grid of grouping distances instead of the one ``dist_thresh`` -- ``decoder_dist_thresh`` values
    (fractions of min(W, H)), finite, >= 0, strictly increasing, at most 64.  ``at(t, gate)`` is then what a decode at
    (t, gate) evaluated at t would hold; ``surface`` and ``best`` read the (threshold x gate) grid.  The nearest-anchor
    search and the location tables do not depend on the gate: they are computed once per threshold.
    """

    TABLES = {"anchor": "anchor_eval", "part": "part_eval", "kps": "kps_eval", "csi": "csi_eval",
              "classification": "classification_eval"}
    _LOCATION = ("anchor_eval", "part_eval")

    def __init__(self, args, thresholds, *, dtype: torch.dtype = torch.float32, dist_thresh=None, gates=None):
        values = [float(t) for t in thresholds]
        if not values or len(values) > _native.MAX_THRESHOLDS:
            raise ValueError(f"{len(values)} thresholds; a sweep takes 1 to {_native.MAX_THRESHOLDS}")
        if not all(math.isfinite(v) for v in values):
            raise ValueError("thresholds must be finite")
        if any(b <= a for a, b in zip(values, values[1:])):
            raise ValueError("thresholds must be strictly increasing")
        if dtype not in ops._DTYPES:
            raise ValueError(f"dtype {dtype} is not a heat-map dtype of the decoder (float32, float16, bfloat16)")
        if gates is not None:
            if dist_thresh is not None:
                raise ValueError("pass either dist_thresh or gates, not both")
            gate_values = [float(g) for g in gates]
            if not gate_values or len(gate_values) > _native.MAX_GATES:
                raise ValueError(f"{len(gate_values)} gates; a sweep takes 1 to {_native.MAX_GATES}")
            if not all(math.isfinite(g) and g >= 0 for g in gate_values):
                raise ValueError("gates must be finite and >= 0")
            if any(b <= a for a, b in zip(gate_values, gate_values[1:])):
                raise ValueError("gates must be strictly increasing")
        self.args = args
        self.thresholds = np.array(values, dtype=np.float64)
        self.dtype = dtype
        if gates is None:
            self.dist_thresh = float(args.decoder_dist_thresh if dist_thresh is None else dist_thresh)
            self.gates = np.array([self.dist_thresh], dtype=np.float64)
        else:
            self.dist_thresh = None
            self.gates = np.array(gate_values, dtype=np.float64)
        self._gated = gates is not None  # launch with the gate grid (G >= 1) rather than the one dist_abs_f32 (G = 0)
        self._grid = [[Evaluator(args) for _ in self.gates] for _ in values]  # [threshold][gate]
        self.lib = _native.load()
        self.last_copy_bytes = 0  # device -> host bytes of the last accumulate_packed

    def reset(self):
        for row in self._grid:
            for ev in row:
                ev.reset()

    def _gate_index(self, gate) -> int:
        if gate is None:
            if len(self.gates) != 1:
                raise KeyError(f"this sweep has {len(self.gates)} gates: name one")
            return 0
        hit = np.flatnonzero(self.gates == float(gate))
        if hit.size == 0:
            raise KeyError(gate)
        return int(hit[0])

    def at(self, t, gate=None) -> Evaluator:
        """The ``Evaluator`` of grid point (``t``, ``gate``); ``gate`` may be left out when the sweep has one gate
        (``KeyError`` otherwise, and for a point not on the grid)."""
        hit = np.flatnonzero(self.thresholds == float(t))
        if hit.size == 0:
            raise KeyError(t)
        return self._grid[int(hit[0])][self._gate_index(gate)]

    def accumulate_packed(self, packed: ops.PackedDetections, annotations, out_size, eval_csi=False, eval_classif=False):
        """Add one decoded batch at every point of the grid.  Arguments as for ``Evaluator.accumulate_packed``, but
        ``packed`` must come from a decode WITH grouping (``Decoder``, ``CoreMLDecoder``, ``ops.decode_packed(...,
        group=True)``), because the part origins are regrouped; the threshold and gate it was decoded at do not matter:
        its ``assign`` and ``counts`` are not read."""
        ev0 = self._grid[0][0]
        B, K = packed.anchor_inds.shape
        P = packed.part_inds.shape[1]
        T, G = len(self.thresholds), len(self.gates)
        if len(annotations) != B:
            raise ValueError(f"{len(annotations)} annotations for a batch of {B} images")
        device = packed.anchor_out.device
        M, N = len(ev0._label_index), len(ev0._part_index)
        gt = ev0._pack_ground_truth(annotations, device)
        if device.type != "cuda":
            raise RuntimeError(f"the packed detections live on {device}: the sweep runs on a CUDA device only")
        objects = eval_csi or eval_classif
        # device bytes one image's outputs take; the batch goes through in slices that stay under the budget
        per_image = T * (12 * (M + N) + 8 * (K + P))
        if objects:
            per_image += T * G * (12 * M + 240 + 20 * K)
        step = max(1, SWEEP_OUTPUT_BUDGET // per_image)
        self.last_copy_bytes = 0
        for b0 in range(0, B, step):
            self._accumulate_slice(packed, gt, b0, min(B, b0 + step), out_size, eval_csi, eval_classif)

    def _accumulate_slice(self, packed, gt, b0, b1, out_size, eval_csi, eval_classif):
        """One launch over images b0 .. b1-1 of the batch (``gt`` = the whole batch's packed ground truth), absorbed
        into every grid point after the images before b0."""
        ev0 = self._grid[0][0]
        B, K, P = b1 - b0, packed.anchor_inds.shape[1], packed.part_inds.shape[1]
        T, G = len(self.thresholds), len(self.gates)
        device = packed.anchor_out.device
        M, N = len(ev0._label_index), len(ev0._part_index)
        (gt_a, n_a, wa), (gt_p, n_p, wp), scale, owner = gt
        gt_a, n_a, gt_p, n_p, scale, owner = (x[b0:b1] for x in (gt_a, n_a, gt_p, n_p, scale, owner))
        anchor_out, part_out = packed.anchor_out[b0:b1], packed.part_out[b0:b1]
        objects = eval_csi or eval_classif
        out_w, out_h = out_size
        in_w, in_h = int(self.args.down_ratio * out_w), int(self.args.down_ratio * out_h)  # decoders.py:37-38
        i32, f64 = {"dtype": torch.int32, "device": device}, {"dtype": torch.float64, "device": device}
        conf = torch.tensor(self.thresholds, **f64)
        conf_group = torch.tensor([ops._f32(t, self.dtype) for t in self.thresholds], dtype=torch.float32, device=device)
        a_stats, p_stats = torch.empty(B, T, M, 3, **i32), torch.empty(B, T, N, 3, **i32)
        a_acc, p_acc = torch.empty(B, T, K, **f64), torch.empty(B, T, P, **f64)
        prm = _native.SdnetSweepParams()
        prm.struct_size = ctypes.sizeof(_native.SdnetSweepParams)
        prm.B, prm.M, prm.N, prm.K, prm.P, prm.T = B, M, N, K, P, T
        prm.max_gt_objects, prm.max_gt_parts = wa, wp
        if self._gated:  # as ops.decode_packed rounds its gate
            grid = torch.tensor([ops._f32(g * min(out_w, out_h)) for g in self.gates], dtype=torch.float32, device=device)
            prm.G, prm.dist_abs_grid = G, grid.data_ptr()
        else:
            prm.dist_abs_f32 = ops._f32(self.dist_thresh * min(out_w, out_h))  # as ops.decode_packed
        prm.sx, prm.sy = in_w / out_w, in_h / out_h
        prm.csi_threshold = float(getattr(self.args, "csi_threshold", 0.75))
        prm.conf, prm.conf_group = conf.data_ptr(), conf_group.data_ptr()
        prm.anchor_out, prm.part_out = anchor_out.data_ptr(), part_out.data_ptr()
        prm.image_scale = scale.data_ptr()
        prm.gt_objects, prm.n_gt_objects = gt_a.data_ptr(), n_a.data_ptr()
        prm.gt_parts, prm.gt_part_owner, prm.n_gt_parts = gt_p.data_ptr(), owner.data_ptr(), n_p.data_ptr()
        prm.anchor_stats, prm.part_stats = a_stats.data_ptr(), p_stats.data_ptr()
        prm.anchor_acc, prm.part_acc = a_acc.data_ptr(), p_acc.data_ptr()
        a_cls = anchor_out[:, :, 3].to(torch.int32)
        p_cls = part_out[:, :, 3].to(torch.int32)
        # (evaluations of each grid point, names, stats (B, R, C, 3), acc (B, R, slots), label of each acc (B, R, slots)):
        # R = T rows for the location tables, T * G rows (threshold-major) for the object tables
        tables = [("anchor_eval", ev0._label_names, a_stats, a_acc, a_cls[:, None].expand(B, T, K)),
                  ("part_eval", ev0._part_names, p_stats, p_acc, p_cls[:, None].expand(B, T, P))]
        if objects:
            groups = ev0._classification_groups(device)
            c_stats, k_stats = torch.empty(B, T * G, M, 3, **i32), torch.empty(B, T * G, 20, 3, **i32)
            c_acc, k_acc = torch.empty(B, T * G, K, **f64), torch.empty(B, T * G, K, **f64)
            n_parts = torch.empty(B, T * G, K, **i32)
            prm.flags = _native.SWEEP_OBJECTS
            prm.cls_group = groups.data_ptr()
            prm.csi_stats, prm.csi_acc = c_stats.data_ptr(), c_acc.data_ptr()
            prm.classif_stats, prm.classif_acc, prm.pred_parts = k_stats.data_ptr(), k_acc.data_ptr(), n_parts.data_ptr()
        stream = torch.cuda.current_stream(device).cuda_stream
        _native.check(self.lib.sdnet_sweep_launch(ctypes.byref(prm), ctypes.c_void_p(stream)), "sdnet_sweep_launch")
        if eval_csi:
            tables.append(("csi_eval", ev0._label_names, c_stats, c_acc, a_cls[:, None].expand(B, T * G, K)))
        if eval_classif:
            g = groups[a_cls.clamp(0, M - 1).long()][:, None]  # as Evaluator.accumulate_packed's classification key
            key = torch.where((n_parts >= 0) & (n_parts <= 9), g * 10 + n_parts, -1)
            tables.append(("classification_eval", dict(enumerate(Evaluator.get_classification_labels())), k_stats, k_acc,
                           torch.where(g >= 0, key, -1)))
        # Only the true positives' values cross to the host: per table, the non-NaN accumulators in (row, image, slot)
        # order with their labels, and the per-row totals.
        stats, hits, vals, labs = [], [], [], []
        for _, _, st, acc, cls in tables:
            acc, cls = acc.transpose(0, 1), cls.transpose(0, 1)  # (R, B, slots)
            hit = ~torch.isnan(acc)
            stats.append(st.sum(dim=0, dtype=torch.int64).flatten())
            hits.append(hit.sum(dim=(1, 2)))
            vals.append(acc[hit])
            labs.append(cls[hit].to(torch.int32))
        host = [torch.cat(x).cpu().numpy() for x in (stats, hits, vals, labs)]
        self.last_copy_bytes += sum(x.nbytes for x in host)
        h_stats, h_hits, h_vals, h_labs = host
        s_off = h_off = v_off = 0
        for attr, names, st, _, _ in tables:
            per_row, rows = st.shape[2] * 3, st.shape[1]
            for r in range(rows):
                n = int(h_hits[h_off + r])
                # a location row is threshold r at every gate; an object row is (threshold r // G, gate r % G)
                targets = self._grid[r] if attr in self._LOCATION else [self._grid[r // G][r % G]]
                for ev in targets:
                    Evaluator._absorb(getattr(ev, attr), names, h_stats[s_off: s_off + per_row].reshape(1, -1, 3),
                                      h_vals[v_off: v_off + n], h_labs[v_off: v_off + n])
                s_off += per_row
                v_off += n
            h_off += rows

    def _rows(self, table, label, cells):
        if table not in self.TABLES:
            raise ValueError(f"unknown table {table!r}; one of {sorted(self.TABLES)}")
        rows = []
        for ev in cells:
            evals = getattr(ev, self.TABLES[table])
            e = evals.reduce() if label is None else evals[label]
            rows.append((e.tp, e.npos, e.ndet, e.precision, e.recall, e.f1_score))
        cols = list(zip(*rows))
        out = {}
        for i, name in enumerate(("tp", "npos", "ndet")):
            out[name] = np.array(cols[i], dtype=np.int64)
        for i, name in enumerate(("precision", "recall", "f1_score"), start=3):
            out[name] = np.array(cols[i], dtype=np.float64)
        return out

    def curve(self, table: str, label=None, gate=None) -> dict:
        """Per grid threshold, at ``gate`` (may be left out when the sweep has one gate): threshold, tp, npos, ndet,
        precision, recall, f1_score of ``table`` (anchor, part, kps, csi, classification) for ``label``, or for all its
        labels together (``Evaluations.reduce``) when ``label`` is None."""
        j = self._gate_index(gate)
        return {"threshold": self.thresholds.copy(), **self._rows(table, label, [row[j] for row in self._grid])}

    def best_threshold(self, table: str, label=None, gate=None) -> float:
        """The grid threshold with the highest F1 score of ``table`` / ``label`` at ``gate`` (the lowest one on a tie)."""
        return float(self.thresholds[int(np.argmax(self.curve(table, label, gate)["f1_score"]))])

    def best_thresholds(self, gate=None) -> dict:
        """``{name: threshold}``: every label's ``best_threshold`` of the ``anchor`` table and every part kind's of the
        ``part`` table, at ``gate``.  Pass it as ``conf_thresh`` to ``Decoder`` and ``Evaluator.accumulate_packed``:
        a decode with these thresholds has, label by label, exactly the location tables of ``at(best)`` for that label,
        because a label's detections are matched against that label's ground truth only."""
        ev = self._grid[0][0]
        best = {name: self.best_threshold("anchor", name, gate) for name in ev.labels}
        best.update({name: self.best_threshold("part", name, gate) for name in ev.kp_labels})
        return best

    def surface(self, table: str, label=None) -> dict:
        """``curve`` over the whole grid: threshold (T,), gate (G,), and tp, npos, ndet, precision, recall, f1_score
        as (T, G) arrays."""
        T, G = len(self.thresholds), len(self.gates)
        out = self._rows(table, label, [ev for row in self._grid for ev in row])
        return {"threshold": self.thresholds.copy(), "gate": self.gates.copy(),
                **{name: v.reshape(T, G) for name, v in out.items()}}

    def best(self, table: str, label=None) -> tuple:
        """The (threshold, gate) with the highest F1 score of ``table`` / ``label``; on a tie the lowest threshold, then
        the lowest gate."""
        t, g = np.unravel_index(int(np.argmax(self.surface(table, label)["f1_score"])), (len(self.thresholds), len(self.gates)))
        return float(self.thresholds[t]), float(self.gates[g])
