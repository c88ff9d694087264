"""Per-class confidence thresholds on the host: the C ABI's table fields and their argument errors, name mappings,
the C object assembly (csrc/fastobj.c) with a threshold per class against the oracle's object loop, and
``ThresholdSweep.best_thresholds`` on hand-filled evaluations."""
import ctypes
import json
import math
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import sdnet_oracle as O
from tests import per_class_oracle as PC
from structuredetector_b200 import Decoder, _native, ops
from structuredetector_b200.evaluator import Evaluation, Evaluator, ThresholdSweep


def _decode_params():
    """Every pointer the decode's validation asks for set (never dereferenced: validation fails first)."""
    p = _native.SdnetDecodeParams()
    p.struct_size = ctypes.sizeof(_native.SdnetDecodeParams)
    p.dtype, p.radius = 0, 2
    p.B, p.M, p.N, p.H, p.W, p.K, p.P = 1, 2, 1, 8, 8, 10, 10
    for t in ("anchor_hm", "part_hm", "offsets", "embeddings"):
        setattr(p, t, _native.SdnetTensor4(4096, 0, 0, 8, 1))
    for name in ("anchor_out", "part_out", "anchor_inds", "part_inds", "assign", "counts"):
        setattr(p, name, 4096)
    return p


def test_table_fields_follow_the_abi_conventions():
    lib = _native.load()
    assert _native.ABI_VERSION == 11
    p = _decode_params()
    p.conf_class_f32 = 4098  # not 4-byte aligned
    assert lib.sdnet_decode_launch(ctypes.byref(p), None) == -8
    assert lib.sdnet_decode_peaks_path(ctypes.byref(p)) == -8
    p.conf_class_f32 = 4096  # aligned: validation goes on to the (missing) workspace
    assert lib.sdnet_decode_launch(ctypes.byref(p), None) == -5
    assert "per-class threshold" in _native.error_string(-8)
    with pytest.raises(ValueError):
        _native.check(-8, "x")
    for struct, launch in ((_native.SdnetMatchParams, lib.sdnet_match_launch),
                           (_native.SdnetObjectMatchParams, lib.sdnet_match_objects_launch)):
        m = struct()
        m.struct_size = ctypes.sizeof(struct)
        m.B, m.M, m.N, m.K, m.P = 1, 2, 1, 10, 10
        for name, kind in struct._fields_:
            if kind is ctypes.c_void_p and name != "conf_class":
                setattr(m, name, 4096)
        m.conf_class = 4100  # 4-byte, not 8-byte aligned
        assert launch(ctypes.byref(m), None) == -8, struct.__name__


def test_zeroed_table_fields_mean_no_table():
    """A zero-initialised struct is the scalar decode / match of ABI version 10."""
    assert _native.SdnetDecodeParams().conf_class_f32 is None
    assert _native.SdnetMatchParams().conf_class is None and _native.SdnetObjectMatchParams().conf_class is None


def test_name_mappings():
    classes, kinds = ["bean", "maize", None], ["leaf"]
    assert ops.class_thresholds(0.3, classes, kinds, 0.5) == 0.3
    assert ops.class_thresholds({"maize": 0.55, "leaf": 0.25}, classes, kinds, 0.4) == [0.4, 0.55, 0.4, 0.25]
    assert ops.class_thresholds({}, classes, kinds, 0.4) == [0.4] * 4
    assert ops.class_thresholds({"stem": 0.1}, ["stem"], ["stem"], 0.4) == [0.1, 0.1]  # a class and a kind of one name
    for bad in ({"weed": 0.3}, {None: 0.3}, {"bean": float("nan")}, {"leaf": float("inf")}, {"bean": -math.inf}):
        with pytest.raises(ValueError):
            ops.class_thresholds(bad, classes, kinds, 0.4)


def test_decoder_and_evaluator_refuse_bad_mappings_before_any_launch():
    outputs = {"anchor_hm": torch.zeros(1, 2, 8, 8), "part_hm": torch.zeros(1, 1, 8, 8)}
    dec = Decoder(SimpleNamespace(_r_labels={0: "bean", 1: "maize"}, _r_parts={0: "leaf"}, anchor_name="stem",
                                  down_ratio=4.0, max_objects=5, max_parts=5, conf_threshold=0.4, decoder_dist_thresh=0.1))
    assert dec._conf(outputs, {"leaf": 0.2}) == [0.4, 0.4, 0.2]
    assert dec._conf(outputs, None) == 0.4 and dec._conf(outputs, 0.25) == 0.25
    for bad in ({"weed": 0.3}, {"bean": float("nan")}):
        with pytest.raises(ValueError):
            dec(outputs, conf_thresh=bad)
        with pytest.raises(ValueError):
            dec.detections_json(outputs, conf_thresh=bad)
    ev = Evaluator(SimpleNamespace(labels={"bean": 0, "maize": 1}, parts={"leaf": 0}, width=32, height=32,
                                   dist_threshold=0.1, conf_threshold=0.4, down_ratio=4.0))
    with pytest.raises(ValueError, match="neither"):
        ev.accumulate_packed(None, [], (8, 8), conf_thresh={"weed": 0.3})


def test_per_class_tables_of_a_decode():
    """ops._conf_arg: M + N entries, each rounded to the heat maps' dtype as the scalar is."""
    conf, table = ops._conf_arg([0.1, 0.35, 1 / 3], 2, 1, torch.float16, "cpu")
    assert conf == 0.0 and table.dtype == torch.float32
    assert table.tolist() == [ops._f32(v, torch.float16) for v in (0.1, 0.35, 1 / 3)]
    assert ops._conf_arg(0.35, 2, 1, torch.bfloat16, "cpu") == (ops._f32(0.35, torch.bfloat16), None)
    assert ops._conf_arg(np.float32(0.5), 2, 1, torch.float32, "cpu") == (0.5, None)
    with pytest.raises(ValueError, match="M \\+ N = 3"):
        ops._conf_arg([0.1, 0.2], 2, 1, torch.float32, "cpu")
    with pytest.raises(ValueError, match="finite"):
        ops._conf_arg([0.1, 0.2, float("nan")], 2, 1, torch.float32, "cpu")


# ----------------------------------------------------------------------------------------------- object assembly
def _random_packed(rng, B, K, P, M, N):
    blob = torch.zeros(ops.packed_nbytes(B, K, P, M + N), dtype=torch.uint8)
    host = ops._carve(blob, B, K, P, M + N)
    a, p = host.anchor_out.numpy(), host.part_out.numpy()
    a[..., 0], a[..., 1] = rng.uniform(0, 600, (B, K)), rng.uniform(0, 500, (B, K))
    a[..., 2] = -np.sort(-rng.uniform(0.05, 1.0, (B, K)).astype(np.float32), axis=1)
    a[..., 3] = rng.integers(0, M, (B, K))
    p[..., 0], p[..., 1] = rng.uniform(0, 600, (B, P)), rng.uniform(0, 500, (B, P))
    p[..., 2] = -np.sort(-rng.uniform(0.05, 1.0, (B, P)).astype(np.float32), axis=1)
    p[..., 3] = rng.integers(0, N, (B, P))
    host.assign.numpy()[:] = rng.integers(-1, K, (B, P))
    return host


def _tables(host, M, N, mode):
    """Per-class thresholds that sit exactly at a score of their class, at the next double above or below it, or far
    apart (a strict class above every score next to a lenient one)."""
    a, p = host.anchor_out.numpy(), host.part_out.numpy()
    score_of = lambda rows, c: float(rows[0][rows[0][:, 3] == c][len(rows[0][rows[0][:, 3] == c]) // 2, 2])
    at = [score_of(a, c) for c in range(M)] + [score_of(p, c) for c in range(N)]
    if mode == "at_score":
        return at
    if mode == "next_up":
        return [float(np.nextafter(v, 2.0)) for v in at]
    if mode == "next_down":
        return [float(np.nextafter(v, -1.0)) for v in at]
    return [0.99 if c % 2 == 0 else 0.05 for c in range(M)] + [0.05 if c % 2 == 0 else 0.99 for c in range(N)]


@pytest.mark.parametrize("mode", ["at_score", "next_up", "next_down", "strict_and_lenient"])
def test_c_object_assembly_per_class_matches_the_oracle(mode):
    """fastobj assemble / keypoints / json_text with one threshold per class against the oracle's object loop: objects
    need score > conf[class], raw parts not score < conf[kind], parts grouped onto a slot that is not emitted drop."""
    rng = np.random.default_rng(11)
    B, K, P, M, N = 4, 29, 37, 3, 2
    host = _random_packed(rng, B, K, P, M, N)
    table = _tables(host, M, N, mode)
    labels, kinds = {i: f"label{i}" for i in range(M)}, {i: f"part{i}" for i in range(N)}
    dec = Decoder(SimpleNamespace(_r_labels=labels, _r_parts=kinds, anchor_name="stem", down_ratio=4.0, max_objects=K,
                                  max_parts=P, conf_threshold=0.4, decoder_dist_thresh=0.1))
    out_size, in_size = (612, 512), (2448, 2051)
    packed = {"anchor_out": host.anchor_out.numpy(), "part_out": host.part_out.numpy(), "assign": host.assign.numpy()}
    conf = dec._host_conf(table, M)
    anns = dec._assemble(host, conf, out_size, in_size)
    want = PC.assemble(packed, labels, kinds, "stem", table[:M], out_size, in_size)
    got = [[(o.name, (o.anchor.kind, o.anchor.x, o.anchor.y, o.anchor.score), [(k.kind, k.x, k.y, k.score) for k in o.parts])
            for o in ann.objects] for ann in anns]
    assert got == want
    emitted = sum(len(img) for img in want)
    assert 0 < emitted < B * K, "the thresholds should keep some objects and drop others"
    raw = dec._raw_parts(host, conf, out_size, in_size)
    want_raw = PC.raw_parts(packed, kinds, table[M:], out_size, in_size)
    assert [[(k.kind, k.x, k.y, k.score) for k in img] for img in raw] == want_raw
    texts = dec._json_from_host(host, conf, out_size, in_size)
    assert texts == [json.dumps(ann.json_repr(), indent=2) for ann in anns]
    # every entry equal to t: the scalar's results
    t = table[0]
    flat = lambda anns: [[(o.name, o.anchor.x, o.anchor.score, [(k.kind, k.x) for k in o.parts]) for o in a.objects] for a in anns]
    assert flat(dec._assemble(host, dec._host_conf([t] * (M + N), M), out_size, in_size)) == \
        flat(dec._assemble(host, t, out_size, in_size))
    assert O.assemble(packed, labels, kinds, "stem", t, out_size, in_size) == \
        PC.assemble(packed, labels, kinds, "stem", [t] * M, out_size, in_size)


def test_c_object_assembly_tables_compare_in_double():
    """A threshold exactly at a float32 score does not emit the object but keeps the raw part; the next double below
    emits both."""
    from structuredetector_b200 import _fastobj
    from structuredetector_b200.annotations import ImageAnnotation, Keypoint, Object

    s = float(np.float32(0.3))
    a = np.array([[[1.0, 2.0, s, 1.0], [3.0, 4.0, s, 0.0]]], dtype=np.float32)
    p = np.array([[[1.0, 2.0, s, 0.0, 0.0, 0.0]]], dtype=np.float32)
    assign = np.array([[0]], dtype=np.int32)
    for table, n_objects, n_parts in (([0.9, s], 0, 0), ([0.9, float(np.nextafter(s, 0.0))], 1, 1)):
        anns = _fastobj.assemble(a, p, assign, 1, 2, 1, table, 1.0, 1.0, ["b", "m"], ["leaf"], "stem", Keypoint, Object,
                                 ImageAnnotation)
        assert len(anns[0].objects) == n_objects
        assert sum(len(o.parts) for o in anns[0].objects) == n_parts
    assert len(_fastobj.keypoints(p, 1, 1, 6, [s], 1.0, 1.0, ["leaf"], Keypoint)[0]) == 1
    assert len(_fastobj.keypoints(p, 1, 1, 6, [float(np.nextafter(s, 1.0))], 1.0, 1.0, ["leaf"], Keypoint)[0]) == 0
    with pytest.raises(IndexError):  # a class the table (and the label map) does not cover is reported, not skipped
        _fastobj.keypoints(p, 1, 1, 6, [], 1.0, 1.0, [], Keypoint)
    with pytest.raises(TypeError):
        _fastobj.keypoints(p, 1, 1, 6, ["x"], 1.0, 1.0, ["leaf"], Keypoint)


# ----------------------------------------------------------------------------------------------- best_thresholds
def test_best_thresholds_on_hand_filled_evaluations():
    """Anchor classes take their best threshold from the anchor table, part kinds from the part table; the highest F1
    wins and the lowest threshold on a tie."""
    args = SimpleNamespace(labels={"bean": 0, "maize": 1}, parts={"leaf": 0, "flower": 1}, width=512, height=512,
                           dist_threshold=0.1, conf_threshold=0.4, down_ratio=4.0, decoder_dist_thresh=0.1)
    grid = [0.2, 0.35, 0.5, 0.65]
    sweep = ThresholdSweep(args, grid)
    f1 = {  # (tp, npos, ndet) per threshold
        ("anchor_eval", "bean"): [(5, 10, 20), (8, 10, 10), (6, 10, 7), (2, 10, 2)],    # best at 0.35
        ("anchor_eval", "maize"): [(4, 10, 10), (4, 10, 10), (6, 10, 10), (6, 10, 10)],  # tie at 0.5 and 0.65
        ("part_eval", "leaf"): [(9, 10, 9), (1, 10, 1), (0, 10, 0), (0, 10, 0)],         # best at 0.2
        ("part_eval", "flower"): [(0, 0, 0)] * 4,                                         # F1 = 1 everywhere: lowest
    }
    for (table, label), rows in f1.items():
        for t, (tp, npos, ndet) in zip(grid, rows):
            getattr(sweep.at(t), table)[label] = Evaluation(tp, npos, ndet)
    # the part table's "bean" would pull the other way if the tables were mixed up
    best = sweep.best_thresholds()
    assert best == {"bean": 0.35, "maize": 0.5, "leaf": 0.2, "flower": 0.2}
    assert all(best[name] == sweep.best_threshold("anchor", name) for name in ("bean", "maize"))
    assert all(best[name] == sweep.best_threshold("part", name) for name in ("leaf", "flower"))
    gated = ThresholdSweep(args, grid, gates=[0.05, 0.1])
    with pytest.raises(KeyError):
        gated.best_thresholds()
    assert set(gated.best_thresholds(gate=0.1)) == {"bean", "maize", "leaf", "flower"}


# ----------------------------------------------------------------------------------------------- the per-class oracle
@pytest.mark.parametrize("mode", ["blobs", "noise", "ties"])
def test_per_class_oracle_with_an_equal_table_is_the_oracle(mode):
    """tests/per_class_oracle.py restates the oracle's grouping with per-class compares: with every entry equal to t it
    gives the oracle's own decode at t, field by field."""
    from structuredetector_b200.synth import DecodeConfig, make_raw
    from tests import per_class_oracle as PC

    cfg = DecodeConfig("pc-oracle", 2, 3, 2, 48, 56, 40, 40, cfg_id=70)
    f = make_raw(cfg, mode).numpy()
    planes = f[:, :3], f[:, 3:5], f[:, 5:7], f[:, 7:]
    for t in (0.05, 0.4, float(np.float32(0.7))):
        want = O.decode_packed(*planes, 40, 40, t, 0.1)
        got = PC.decode_packed(*planes, 40, 40, [t] * 5, 0.1)
        for key in ("anchor_out", "part_out", "anchor_inds", "part_inds", "part_emb", "assign", "counts",
                    "anchor_scores_masked", "part_scores_masked"):
            np.testing.assert_array_equal(got[key], want[key], err_msg=f"{mode} t={t}: {key}")
