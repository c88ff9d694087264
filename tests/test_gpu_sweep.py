"""-m gpu: ThresholdSweep / sdnet_sweep_launch against the per-threshold pipeline it replaces.

The contract, bit for bit: for every grid threshold t, ``sweep.at(t)`` holds what a fresh ``Evaluator`` holds after
``accumulate_packed(ops.decode_packed(outputs, K, P, t, dist), ..., conf_thresh=t, eval_csi=True, eval_classif=True)``
-- tp, npos and ndet equal and the accumulated values equal under ``==`` in all five tables -- and the regrouped
assignment at t equals that decode's ``assign``.
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import sweep_oracle as SO
from oracle import sdnet_oracle as O
from oracle import torch_port as TP
from structuredetector_b200 import _native, ops
from structuredetector_b200.evaluator import Evaluator, ThresholdSweep
from structuredetector_b200.synth import DecodeConfig, make_raw, split_outputs
from tests.helpers import np_inputs, packed_np, torch_sigmoid_fn
from tests.test_gpu_evaluator_limits import KINDS, LABELS, _annotations, _args, _ground_truth
from tests.test_gpu_limits import FAR_CASES, _far_raw
from tests.test_sweep import EVAL_OBJECTS, GOLDEN, _golden_case, golden_expectation

pytestmark = pytest.mark.gpu

TABLES = ("anchor_eval", "part_eval", "kps_eval", "csi_eval", "classification_eval")
GRID = [round(0.05 * i, 2) for i in range(1, 20)]  # 0.05 ... 0.95


def _assert_same(got: Evaluator, want: Evaluator, what):
    for table in TABLES:
        g, w = getattr(got, table), getattr(want, table)
        assert set(g.labels) == set(w.labels), (what, table)
        for label, e in w.items():
            assert (g[label].tp, g[label].npos, g[label].ndet) == (e.tp, e.npos, e.ndet), (what, table, label)
            assert g[label].acc == e.acc, (what, table, label)


def _regroup(packed, grid, dtype, dist_abs):
    """sdnet_sweep_launch's regrouped assignment (B, T, P), location half only and no ground truth."""
    B, K = packed.anchor_inds.shape
    P = packed.part_inds.shape[1]
    T, dev = len(grid), packed.anchor_out.device
    C = max(int(packed.anchor_out[..., 3].max()), int(packed.part_out[..., 3].max())) + 1  # classes and kinds
    conf = torch.tensor(grid, dtype=torch.float64, device=dev)
    conf_group = torch.tensor([ops._f32(t, dtype) for t in grid], dtype=torch.float32, device=dev)
    zeros = torch.zeros(B, 4, dtype=torch.float64, device=dev)
    n_gt = torch.zeros(B, dtype=torch.int32, device=dev)
    out = {"a_stats": torch.empty(B, T, C, 3, dtype=torch.int32, device=dev),
           "p_stats": torch.empty(B, T, C, 3, dtype=torch.int32, device=dev),
           "a_acc": torch.empty(B, T, K, dtype=torch.float64, device=dev),
           "p_acc": torch.empty(B, T, P, dtype=torch.float64, device=dev),
           "assign": torch.full((B, T, P), -7, dtype=torch.int32, device=dev)}
    p = _native.SdnetSweepParams()
    p.struct_size = ctypes.sizeof(p)
    p.B, p.M, p.N, p.K, p.P, p.T = B, C, C, K, P, T
    p.dist_abs_f32, p.sx, p.sy = dist_abs, 4.0, 4.0
    p.conf, p.conf_group = conf.data_ptr(), conf_group.data_ptr()
    p.anchor_out, p.part_out, p.image_scale = packed.anchor_out.data_ptr(), packed.part_out.data_ptr(), zeros.data_ptr()
    p.n_gt_objects = p.n_gt_parts = n_gt.data_ptr()
    p.anchor_stats, p.part_stats = out["a_stats"].data_ptr(), out["p_stats"].data_ptr()
    p.anchor_acc, p.part_acc, p.assign_out = out["a_acc"].data_ptr(), out["p_acc"].data_ptr(), out["assign"].data_ptr()
    _native.check(_native.load().sdnet_sweep_launch(ctypes.byref(p), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)),
                  "sdnet_sweep_launch")
    return out["assign"].cpu().numpy()


def _contract(outs, grid, K, P, dist, anns, out_size, args, *, dtype=torch.float32, what="", **kw):
    """Sweep one decode and compare with the per-threshold pipeline; returns the sweep."""
    packed = ops.decode_packed(outs, K, P, 0.5, dist, **kw)
    sweep = ThresholdSweep(args, grid, dtype=dtype, dist_thresh=dist)
    sweep.accumulate_packed(packed, anns, out_size, eval_csi=True, eval_classif=True)
    assign = _regroup(packed, grid, dtype, ops._f32(dist * min(out_size)))
    for i, t in enumerate(grid):
        pk = ops.decode_packed(outs, K, P, t, dist, **kw)
        want = Evaluator(args)
        want.accumulate_packed(pk, anns, out_size, conf_thresh=t, eval_csi=True, eval_classif=True)
        _assert_same(sweep.at(t), want, f"{what} t={t!r}")
        np.testing.assert_array_equal(assign[:, i], pk.assign.cpu().numpy(), err_msg=f"{what} t={t!r}: assign")
    return sweep


def _batch(cfg, mode, device, *, seed=None, dtype=torch.float32):
    """(outputs, annotations, args, out_size, packed fields of a decode at 0.2) for a cfg-shaped batch with ground truth
    derived from its detections."""
    raw = make_raw(cfg, mode, seed=seed).to(dtype)
    outs = split_outputs(raw.to(device), cfg.labels, cfg.parts)
    labels = {name: i for name, i in list(LABELS.items())[: cfg.labels]}
    kinds = {name: i for name, i in list(KINDS.items())[: cfg.parts]}
    out_size = (cfg.width, cfg.height)
    args = _args(out_size, 0.02, labels=labels)
    args.parts = kinds
    pk = packed_np(ops.decode_packed(outs, cfg.max_objects, cfg.max_parts, 0.2, cfg.dist_thresh))
    objs = O.assemble(pk, {i: n for n, i in labels.items()}, {i: k for k, i in kinds.items()}, "stem", 0.2, out_size,
                      (4 * cfg.width, 4 * cfg.height))
    rng = np.random.default_rng(cfg.cfg_id + len(mode))
    gts = [_ground_truth(o, rng) for o in objs]
    gts = [[g for g in gt if g[0] in labels] for gt in gts]
    sizes = [(2448, 2048) if b % 2 else (1296, 1536) for b in range(len(gts))]
    return outs, _annotations(gts, sizes), args, out_size, pk


def _boundary_grid(pk, base):
    """`base` plus the exact doubles of some detections' scores, their neighbouring doubles, 0.4 and float32(0.4)."""
    scores = [float(pk["anchor_out"][0, i, 2]) for i in (2, 7)] + [float(pk["part_out"][0, i, 2]) for i in (3, 11)]
    extra = {0.4, float(np.float32(0.4))}
    for s in scores:
        extra |= {s, float(np.nextafter(s, 0.0)), float(np.nextafter(s, 1.0))}
    return sorted(set(base) | extra)


CFG3 = DecodeConfig("cfg3-small", 4, 2, 1, 128, 152, 100, 100, cfg_id=3)


@pytest.mark.parametrize("mode", ["blobs", "noise"])
def test_sweep_matches_per_threshold_pipeline(cuda_device, mode):
    """cfg3-shaped maps, fp32, T = 19 plus boundary thresholds: anchors' `score > t`, raw parts' `not score < t` and
    the grouping's fp32 compare on either side of a detection's exact score."""
    outs, anns, args, out_size, pk = _batch(CFG3, mode, cuda_device)
    grid = _boundary_grid(pk, GRID)
    sweep = _contract(outs, grid, CFG3.max_objects, CFG3.max_parts, CFG3.dist_thresh, anns, out_size, args, what=mode)
    f1 = sweep.curve("anchor")["f1_score"]
    assert f1.max() > 0.2 and len(set(f1.tolist())) > 3, f1
    assert sweep.at(0.4).anchor_eval.reduce().tp > 0 and sweep.at(0.4).csi_eval.reduce().tp > 0
    assert sweep.last_copy_bytes > 0


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
def test_sweep_on_reduced_precision_maps(cuda_device, dtype):
    """The grouping compares `score > t` in the maps' dtype: the sweep rounds its grid the same way."""
    outs, anns, args, out_size, pk = _batch(CFG3, "blobs", cuda_device, dtype=dtype)
    _contract(outs, _boundary_grid(pk, GRID), CFG3.max_objects, CFG3.max_parts, CFG3.dist_thresh, anns, out_size, args,
              dtype=dtype, what=str(dtype))


def test_sweep_on_pre_activated_maps(cuda_device):
    cfg = CFG3
    raw = make_raw(cfg, "blobs")
    raw[:, :3] = TP.suppress(TP.activate(raw[:, :3].to(cuda_device)), 2).cpu()
    outs = split_outputs(raw.to(cuda_device), cfg.labels, cfg.parts)
    _, anns, args, out_size, _ = _batch(cfg, "blobs", cuda_device)
    _contract(outs, GRID, cfg.max_objects, cfg.max_parts, cfg.dist_thresh, anns, out_size, args, pre_activated=True,
              what="pre-activated")


def test_decode_threshold_does_not_matter(cuda_device):
    """A decode at 0.05 and one at 0.9 (different `assign` and `counts`) sweep to identical results."""
    outs, anns, args, out_size, _ = _batch(CFG3, "noise", cuda_device)
    sweeps = []
    for conf in (0.05, 0.9):
        packed = ops.decode_packed(outs, CFG3.max_objects, CFG3.max_parts, conf, CFG3.dist_thresh)
        sweep = ThresholdSweep(args, GRID, dist_thresh=CFG3.dist_thresh)
        sweep.accumulate_packed(packed, anns, out_size, eval_csi=True, eval_classif=True)
        sweeps.append(sweep)
    for t in GRID:
        _assert_same(sweeps[0].at(t), sweeps[1].at(t), f"t={t}")


def test_two_batches_accumulate(cuda_device):
    """Two batches into one sweep against two batches into one Evaluator per threshold; reset() empties it."""
    batches = [_batch(CFG3, mode, cuda_device, seed=seed) for mode, seed in (("blobs", 11), ("noise", 12))]
    args, out_size = batches[0][2], batches[0][3]
    sweep = ThresholdSweep(args, GRID, dist_thresh=CFG3.dist_thresh)
    for outs, anns, _, _, _ in batches:
        sweep.accumulate_packed(ops.decode_packed(outs, 100, 100, 0.5, CFG3.dist_thresh), anns, out_size, True, True)
    for t in GRID:
        want = Evaluator(args)
        for outs, anns, _, _, _ in batches:
            want.accumulate_packed(ops.decode_packed(outs, 100, 100, t, CFG3.dist_thresh), anns, out_size, conf_thresh=t,
                                   eval_csi=True, eval_classif=True)
        _assert_same(sweep.at(t), want, f"t={t}")
    sweep.reset()
    assert all(sweep.curve(table)["ndet"].sum() == 0 for table in ("anchor", "part", "kps", "csi", "classification"))


# ----------------------------------------------------------------------------------------------- at the limits
def test_sweep_at_k_p_1024(cuda_device):
    """K = P = 1024 with one image holding 1,024 ground-truth objects and 1,024 ground-truth parts (the object scratch
    and match_pass's arrays share the dynamic shared memory)."""
    cfg = DecodeConfig("dense", 3, 3, 2, 128, 128, 1024, 1024, cfg_id=44)
    raw = make_raw(cfg, "noise")
    outs = split_outputs(raw.to(cuda_device), 3, 2)
    out_size = (128, 128)
    pk = packed_np(ops.decode_packed(outs, 1024, 1024, 0.4, 0.1))
    objs = O.assemble(pk, {i: n for n, i in LABELS.items()}, {i: k for k, i in KINDS.items()}, "stem", 0.4, out_size, (512, 512))
    rng = np.random.default_rng(44)
    gts = [_ground_truth(objs[0], rng), _ground_truth(objs[1], rng, n_objects=1024), []]
    anns = _annotations(gts, [(1931, 1297), (1297, 1931), (512, 512)])
    _contract(outs, [0.05, 0.3, 0.4, 0.6, 0.9], 1024, 1024, 0.1, anns, out_size, _args(out_size, 0.02), what="K=P=1024")


def test_sweep_with_256_thresholds(cuda_device):
    cfg = DecodeConfig("t256", 2, 2, 1, 48, 64, 40, 40, cfg_id=46)
    outs, anns, args, out_size, _ = _batch(cfg, "blobs", cuda_device)
    grid = sorted(set(np.linspace(0.001, 0.999, 256).tolist()))
    assert len(grid) == _native.MAX_THRESHOLDS
    _contract(outs, grid, cfg.max_objects, cfg.max_parts, cfg.dist_thresh, anns, out_size, args, what="T=256")


@pytest.mark.parametrize("case", FAR_CASES)
def test_sweep_full_grouping_search(cuda_device, case):
    """Valid coordinates beyond +-1e5, gates of 1e5 and more, and the 2.56e6 gate that groups the masked slots: the
    sweep's plain P x K search against the tail kernel's restricted one."""
    raw, dist = _far_raw(case)
    outs = split_outputs(raw.to(cuda_device), 2, 1)
    out_size = (128, 128)
    labels = {"bean": 0, "maize": 1}
    args = _args(out_size, 0.05, labels=labels)
    args.parts = {"leaf": 0}
    pk = packed_np(ops.decode_packed(outs, 100, 100, 0.4, dist))
    objs = O.assemble(pk, {0: "bean", 1: "maize"}, {0: "leaf"}, "stem", 0.4, out_size, (512, 512))
    gts = [[g for g in _ground_truth(objs[0], np.random.default_rng(42)) if g[0] in labels]]
    _contract(outs, [0.1, 0.3, 0.4, float(np.float32(0.4)), 0.7], 100, 100, dist, _annotations(gts, [(512, 512)]), out_size,
              args, what=case)


# ----------------------------------------------------------------------------------------------- references
@pytest.mark.parametrize("name", sorted(EVAL_OBJECTS))
def test_sweep_reproduces_reference_at_golden_conf(cuda_device, name):
    """A grid holding each stored case's conf reproduces what the reference's evaluator stored at that conf: counts
    exact, accumulated values to 1e-9 relative."""
    meta, inputs, args, gts, sizes = _golden_case(name)
    _, m, n, h, w = meta["shape"]
    raw = torch.from_numpy(np.load(GOLDEN / f"{name}.npz")["raw"]).to(cuda_device)
    packed = ops.decode_packed(split_outputs(raw, m, n), meta["K"], meta["P"], 0.9, meta["dist"])
    sweep = ThresholdSweep(args, sorted({0.1, meta["conf"], 0.8}), dist_thresh=meta["dist"])
    sweep.accumulate_packed(packed, _annotations(gts, sizes), (w, h), eval_csi=True, eval_classif=True)
    ev = sweep.at(meta["conf"])
    got = {"anchor": ev.anchor_eval, "part": ev.part_eval, "csi": ev.csi_eval, "classification": ev.classification_eval}
    for key, want in golden_expectation(name).items():
        assert set(got[key].labels) == set(want), (name, key)
        for label, (tp, npos, ndet, acc) in want.items():
            g = got[key][label]
            assert (g.tp, g.npos, g.ndet) == (tp, npos, ndet), (name, key, label)
            np.testing.assert_allclose(g.acc, acc, rtol=1e-9, atol=0)


def test_sweep_against_oracle_sweep(cuda_device):
    """A small batch against the oracle's per-threshold restatement: counts exact, accumulated values to 1e-9."""
    cfg = DecodeConfig("small", 2, 2, 1, 40, 52, 30, 40, cfg_id=47)
    outs, anns, args, out_size, pk = _batch(cfg, "blobs", cuda_device)
    gts = [[(o.name, o.anchor.x, o.anchor.y, [(k.kind, k.x, k.y) for k in o.parts]) for o in a.objects] for a in anns]
    sizes = [a.img_size for a in anns]
    grid = _boundary_grid(pk, [0.1, 0.3, 0.5, 0.7, 0.9])
    sweep = ThresholdSweep(args, grid, dist_thresh=cfg.dist_thresh)
    sweep.accumulate_packed(ops.decode_packed(outs, cfg.max_objects, cfg.max_parts, 0.5, cfg.dist_thresh), anns, out_size,
                            eval_csi=True, eval_classif=True)
    tables = SO.sweep(np_inputs(outs), grid, cfg.max_objects, cfg.max_parts, cfg.dist_thresh,
                      gts, sizes, args, sigmoid_fn=torch_sigmoid_fn(cuda_device))
    names = {"anchor": "anchor_eval", "part": "part_eval", "csi": "csi_eval", "classification": "classification_eval"}
    for t, want in zip(grid, tables):
        ev = sweep.at(t)
        for key, tab in want.items():
            for label, (tp, npos, ndet, acc) in tab.items():
                g = getattr(ev, names[key])[label]
                assert (g.tp, g.npos, g.ndet) == (tp, npos, ndet), (t, key, label)
                np.testing.assert_allclose(g.acc, acc, rtol=1e-9, atol=0, err_msg=f"{t} {key} {label}")


def test_sweep_with_more_decoded_classes_than_labels(cuda_device):
    """Maps with 3 classes and 2 part kinds, evaluated with 2 labels and 1 kind: the other classes' detections are
    counted nowhere, as Evaluator counts them, with and without the object tables (the location matcher's label counters
    take every class a decode can emit)."""
    cfg = DecodeConfig("extra", 2, 3, 2, 64, 80, 60, 60, cfg_id=48)
    outs = split_outputs(make_raw(cfg, "noise").to(cuda_device), 3, 2)
    out_size = (80, 64)
    args = _args(out_size, 0.05, labels={"bean": 0, "maize": 1})
    args.parts = {"leaf": 0}
    pk = packed_np(ops.decode_packed(outs, 60, 60, 0.3, 0.1))
    assert (pk["anchor_out"][..., 3] == 2).any() and (pk["part_out"][..., 3] == 1).any()
    objs = O.assemble(pk, {0: "bean", 1: "maize", 2: "weed"}, {0: "leaf", 1: "flower"}, "stem", 0.3, out_size, (320, 256))
    rng = np.random.default_rng(48)
    gts = [[(n, x, y, [k for k in kps if k[0] == "leaf"]) for n, x, y, kps in _ground_truth(o, rng) if n != "weed"] for o in objs]
    anns = _annotations(gts, [(640, 512), (512, 640)])
    _contract(outs, GRID, 60, 60, 0.1, anns, out_size, args, what="extra classes")
    sweep = ThresholdSweep(args, GRID, dist_thresh=0.1)
    sweep.accumulate_packed(ops.decode_packed(outs, 60, 60, 0.5, 0.1), anns, out_size)
    for t in GRID:
        want = Evaluator(args)
        want.accumulate_packed(ops.decode_packed(outs, 60, 60, t, 0.1), anns, out_size, conf_thresh=t)
        _assert_same(sweep.at(t), want, f"location only t={t}")
