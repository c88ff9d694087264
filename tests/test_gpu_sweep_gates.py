"""-m gpu: ThresholdSweep(..., gates=...) / sdnet_sweep_launch with G >= 1 against the per-point pipeline it replaces.

The contract, bit for bit: for every grid threshold t and gate g, ``sweep.at(t, g)`` holds what a fresh ``Evaluator``
holds after ``accumulate_packed(ops.decode_packed(outputs, K, P, t, g), ..., conf_thresh=t, eval_csi=True,
eval_classif=True)`` -- tp, npos and ndet equal and the accumulated values equal under ``==`` in all five tables -- and
the regrouped assignment at (t, g) equals that decode's ``assign``.
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import sdnet_oracle as O
from oracle import torch_port as TP
from structuredetector_b200 import _native, evaluator, ops
from structuredetector_b200.evaluator import Evaluator, ThresholdSweep
from structuredetector_b200.synth import DecodeConfig, make_raw, split_outputs
from tests.helpers import packed_np
from tests.test_gpu_evaluator_limits import KINDS, LABELS, _annotations, _args, _ground_truth
from tests.test_gpu_limits import FAR_CASES, _far_raw
from tests.test_gpu_sweep import CFG3, GRID, _assert_same, _batch, _boundary_grid

pytestmark = pytest.mark.gpu

GATES = [0.05, 0.1, 0.2]


def _raw_sweep(packed, grid, dtype, args, anns, out_size, *, G=0, dist_abs=0.0, gates_abs=(), objects=True):
    """Every output of one sdnet_sweep_launch over `packed` with `args`' labels and `anns`' ground truth (host tensors)."""
    B, K = packed.anchor_inds.shape
    P = packed.part_inds.shape[1]
    T, R, dev = len(grid), len(grid) * max(G, 1), packed.anchor_out.device
    ev = Evaluator(args)
    M, N = len(args.labels), len(args.parts)
    (gt_a, n_a, wa), (gt_p, n_p, wp), scale, owner = ev._pack_ground_truth(anns, dev)
    i32, f64 = {"dtype": torch.int32, "device": dev}, {"dtype": torch.float64, "device": dev}
    conf = torch.tensor(grid, **f64)
    conf_group = torch.tensor([ops._f32(t, dtype) for t in grid], dtype=torch.float32, device=dev)
    gates = torch.tensor(list(gates_abs) or [0.0], dtype=torch.float32, device=dev)
    out = {"anchor_stats": torch.full((B, T, M, 3), -7, **i32), "part_stats": torch.full((B, T, N, 3), -7, **i32),
           "anchor_acc": torch.full((B, T, K), -7.0, **f64), "part_acc": torch.full((B, T, P), -7.0, **f64),
           "csi_stats": torch.full((B, R, M, 3), -7, **i32), "csi_acc": torch.full((B, R, K), -7.0, **f64),
           "classif_stats": torch.full((B, R, 20, 3), -7, **i32), "classif_acc": torch.full((B, R, K), -7.0, **f64),
           "pred_parts": torch.full((B, R, K), -7, **i32), "assign_out": torch.full((B, R, P), -7, **i32)}
    p = _native.SdnetSweepParams()
    p.struct_size = ctypes.sizeof(p)
    p.B, p.M, p.N, p.K, p.P, p.T, p.G = B, M, N, K, P, T, G
    p.max_gt_objects, p.max_gt_parts = wa, wp
    p.flags = _native.SWEEP_OBJECTS if objects else 0
    out_w, out_h = out_size
    p.dist_abs_f32, p.dist_abs_grid = dist_abs, gates.data_ptr()
    p.sx, p.sy = int(args.down_ratio * out_w) / out_w, int(args.down_ratio * out_h) / out_h
    p.csi_threshold = args.csi_threshold
    p.conf, p.conf_group = conf.data_ptr(), conf_group.data_ptr()
    p.anchor_out, p.part_out, p.image_scale = packed.anchor_out.data_ptr(), packed.part_out.data_ptr(), scale.data_ptr()
    p.gt_objects, p.n_gt_objects, p.gt_parts, p.n_gt_parts = gt_a.data_ptr(), n_a.data_ptr(), gt_p.data_ptr(), n_p.data_ptr()
    p.gt_part_owner, p.cls_group = owner.data_ptr(), ev._classification_groups(dev).data_ptr()
    for name, t in out.items():
        setattr(p, name, t.data_ptr())
    _native.check(_native.load().sdnet_sweep_launch(ctypes.byref(p), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)),
                  "sdnet_sweep_launch")
    return {name: t.cpu() for name, t in out.items()}


def _abs(gates, out_size):
    return [ops._f32(g * min(out_size)) for g in gates]  # as ops.decode_packed rounds its gate


def _contract(outs, grid, gates, K, P, anns, out_size, args, *, dtype=torch.float32, what="", points=None, **kw):
    """Sweep one decode over (grid x gates) and compare with a decode and an Evaluator per point (every point, or those
    of `points`); the regrouped assignment is compared at every point.  Returns the sweep and the assignment."""
    packed = ops.decode_packed(outs, K, P, 0.5, 0.1, **kw)
    sweep = ThresholdSweep(args, grid, dtype=dtype, gates=gates)
    sweep.accumulate_packed(packed, anns, out_size, eval_csi=True, eval_classif=True)
    G = len(gates)
    assign = _raw_sweep(packed, grid, dtype, args, anns, out_size, G=G, gates_abs=_abs(gates, out_size),
                        objects=False)["assign_out"].numpy()
    B = assign.shape[0]
    assign = assign.reshape(B, len(grid), G, -1)
    for i, t in enumerate(grid):
        for j, g in enumerate(gates):
            pk = ops.decode_packed(outs, K, P, t, g, **kw)
            np.testing.assert_array_equal(assign[:, i, j], pk.assign.cpu().numpy(), err_msg=f"{what} t={t!r} g={g!r}: assign")
            if points is None or (i, j) in points:
                want = Evaluator(args)
                want.accumulate_packed(pk, anns, out_size, conf_thresh=t, eval_csi=True, eval_classif=True)
                _assert_same(sweep.at(t, g), want, f"{what} t={t!r} g={g!r}")
    return sweep, assign


def _nearest(pk, b, t, dtype=torch.float32):
    """Per part slot of image b: (first nearest anchor slot, its fp32 distance) of the grouping at threshold t, in the
    decoder's op order (each step rounded to fp32)."""
    cg = np.float32(ops._f32(t, dtype))
    a, q = pk["anchor_out"][b].astype(np.float32), pk["part_out"][b].astype(np.float32)
    far = np.float32(1e6)
    ax = np.where(a[:, 2] > cg, a[:, 0], far)
    ay = np.where(a[:, 2] > cg, a[:, 1], far)
    ox = np.where(q[:, 2] > cg, q[:, 4], -far)
    oy = np.where(q[:, 2] > cg, q[:, 5], -far)
    dx, dy = ox[:, None] - ax[None, :], oy[:, None] - ay[None, :]
    d = np.sqrt(dx * dx + dy * dy)
    assert d.dtype == np.float32
    arg = np.argmin(d, axis=1)
    return arg, d[np.arange(len(arg)), arg], q[:, 2] > cg


def _boundary_gates(pk, out_size, t):
    """Two gates that pin `distance < gate`: one whose fp32 absolute gate is exactly a valid part's nearest-anchor
    distance (the part stays ungrouped there), and the next fp32 gate above it (the part is grouped)."""
    arg, dist, valid = _nearest(pk, 0, t)
    cand = np.flatnonzero(valid & (dist > 0))
    q = int(cand[np.argsort(dist[cand])[len(cand) // 2]])
    d = np.float32(dist[q])
    at = float(d) / min(out_size)
    above = float(np.nextafter(d, np.float32(np.inf))) / min(out_size)
    assert _abs([at, above], out_size) == [float(d), float(np.nextafter(d, np.float32(np.inf)))]
    return at, above, q, int(arg[q])


# ----------------------------------------------------------------------------------------------- the contract
@pytest.mark.parametrize("mode", ["blobs", "noise"])
def test_gate_sweep_matches_per_point_pipeline(cuda_device, mode):
    """cfg3-shaped maps, fp32, T = 19 plus boundary thresholds, gates 0, tiny, 0.05, 0.1, 0.2 and two at a part's exact
    nearest-anchor distance."""
    outs, anns, args, out_size, pk = _batch(CFG3, mode, cuda_device)
    grid = _boundary_grid(pk, GRID)
    t0 = 0.4
    at, above, q, a = _boundary_gates(pk, out_size, t0)
    gates = sorted({0.0, 1e-6, 0.05, 0.1, 0.2, at, above})
    sweep, assign = _contract(outs, grid, gates, CFG3.max_objects, CFG3.max_parts, anns, out_size, args, what=mode)
    i = grid.index(t0)
    assert assign[0, i, gates.index(at), q] == -1 and assign[0, i, gates.index(above), q] == a
    assert (assign[:, :, gates.index(0.0)] == -1).all()
    f1 = sweep.surface("csi")["f1_score"]
    assert len(set(f1.ravel().tolist())) > 10, f1
    assert not np.array_equal(f1[:, gates.index(0.05)], f1[:, gates.index(0.2)])
    assert sweep.best("csi") in {(t, g) for t in grid for g in gates}
    assert sweep.last_copy_bytes > 0


@pytest.mark.parametrize("case", FAR_CASES)
def test_gate_sweep_full_grouping_search(cuda_device, case):
    """Coordinates beyond +-1e5 and gates of 1e5 and more, each case with gates bracketing its own: masked slots group
    at some gates and not at others (gate_2.56e6 puts masked parts onto valid anchors)."""
    raw, dist = _far_raw(case)
    outs = split_outputs(raw.to(cuda_device), 2, 1)
    out_size = (128, 128)
    labels = {"bean": 0, "maize": 1}
    args = _args(out_size, 0.05, labels=labels)
    args.parts = {"leaf": 0}
    pk = packed_np(ops.decode_packed(outs, 100, 100, 0.4, dist))
    objs = O.assemble(pk, {0: "bean", 1: "maize"}, {0: "leaf"}, "stem", 0.4, out_size, (512, 512))
    gts = [[g for g in _ground_truth(objs[0], np.random.default_rng(42)) if g[0] in labels]]
    f32_below = float(np.nextafter(np.float32(dist * 128), np.float32(0))) / 128
    gates = sorted({0.1, dist / 2, f32_below, dist, 2 * dist})
    grid = [0.1, 0.3, 0.4, float(np.float32(0.4)), 0.7]
    _, assign = _contract(outs, grid, gates, 100, 100, _annotations(gts, [(512, 512)]), out_size, args, what=case)
    if case == "gate_2.56e6":  # masked parts (at -1e6, -1e6) onto a valid anchor at 2.56e6, not at 1.28e6
        _, _, valid = _nearest(pk, 0, 0.4)
        masked = np.flatnonzero(~valid)
        at_gate, at_half = assign[0, 2, gates.index(dist), masked], assign[0, 2, gates.index(dist / 2), masked]
        assert (at_gate >= 0).all() and (at_half == -1).all()


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
def test_gate_sweep_on_reduced_precision_maps(cuda_device, dtype):
    outs, anns, args, out_size, pk = _batch(CFG3, "blobs", cuda_device, dtype=dtype)
    _contract(outs, _boundary_grid(pk, GRID), GATES, CFG3.max_objects, CFG3.max_parts, anns, out_size, args, dtype=dtype,
              what=str(dtype))


def test_gate_sweep_on_pre_activated_maps(cuda_device):
    raw = make_raw(CFG3, "blobs")
    raw[:, :3] = TP.suppress(TP.activate(raw[:, :3].to(cuda_device)), 2).cpu()
    outs = split_outputs(raw.to(cuda_device), CFG3.labels, CFG3.parts)
    _, anns, args, out_size, _ = _batch(CFG3, "blobs", cuda_device)
    _contract(outs, GRID, GATES, CFG3.max_objects, CFG3.max_parts, anns, out_size, args, pre_activated=True,
              what="pre-activated")


def test_gate_sweep_with_more_decoded_classes_than_labels(cuda_device):
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
    _contract(outs, GRID, GATES, 60, 60, _annotations(gts, [(640, 512), (512, 640)]), out_size, args, what="extra classes")


def test_two_batches_accumulate_over_gates(cuda_device):
    batches = [_batch(CFG3, mode, cuda_device, seed=seed) for mode, seed in (("blobs", 11), ("noise", 12))]
    args, out_size = batches[0][2], batches[0][3]
    sweep = ThresholdSweep(args, GRID, gates=GATES)
    for outs, anns, _, _, _ in batches:
        sweep.accumulate_packed(ops.decode_packed(outs, 100, 100, 0.5, 0.1), anns, out_size, True, True)
    for t in GRID:
        for g in GATES:
            want = Evaluator(args)
            for outs, anns, _, _, _ in batches:
                want.accumulate_packed(ops.decode_packed(outs, 100, 100, t, g), anns, out_size, conf_thresh=t,
                                       eval_csi=True, eval_classif=True)
            _assert_same(sweep.at(t, g), want, f"t={t} g={g}")


def test_gate_sweep_at_k_p_1024_and_256_by_64_points(cuda_device):
    """K = P = 1024, one image with 1,024 ground-truth objects and parts, T x G = 256 x 64.  The assignment is checked at
    all 16,384 points; the tables at every 15th threshold and every 9th gate, the last of each included."""
    cfg = DecodeConfig("dense", 2, 3, 2, 128, 128, 1024, 1024, cfg_id=44)
    outs = split_outputs(make_raw(cfg, "noise").to(cuda_device), 3, 2)
    out_size = (128, 128)
    pk = packed_np(ops.decode_packed(outs, 1024, 1024, 0.4, 0.1))
    objs = O.assemble(pk, {i: n for n, i in LABELS.items()}, {i: k for k, i in KINDS.items()}, "stem", 0.4, out_size, (512, 512))
    gts = [_ground_truth(objs[0], np.random.default_rng(44), n_objects=1024), []]
    assert sum(len(kps) for _, _, _, kps in gts[0]) >= 1024
    anns = _annotations(gts, [(1297, 1931), (512, 512)])
    grid = sorted(set(np.linspace(0.001, 0.999, 256).tolist()))
    gates = [0.005 * j for j in range(64)]
    assert len(grid) == _native.MAX_THRESHOLDS and len(gates) == _native.MAX_GATES
    points = {(i, j) for i in list(range(0, 256, 15)) + [255] for j in list(range(0, 64, 9)) + [63]}
    _contract(outs, grid, gates, 1024, 1024, anns, out_size, _args(out_size, 0.02), what="K=P=1024", points=points)


# ----------------------------------------------------------------------------------------------- layouts and paths
def test_image_slices_equal_one_pass(cuda_device, monkeypatch):
    """With the output budget patched down to one image, a batch goes through one launch per image: the same tables."""
    outs, anns, args, out_size, _ = _batch(CFG3, "noise", cuda_device)
    packed = ops.decode_packed(outs, 100, 100, 0.5, 0.1)
    whole = ThresholdSweep(args, GRID, gates=GATES)
    whole.accumulate_packed(packed, anns, out_size, True, True)
    monkeypatch.setattr(evaluator, "SWEEP_OUTPUT_BUDGET", 1)
    sliced = ThresholdSweep(args, GRID, gates=GATES)
    launches = []
    lib = sliced.lib

    class Counting:
        def sdnet_sweep_launch(self, prm, stream):
            launches.append(prm._obj.B)
            return lib.sdnet_sweep_launch(prm, stream)

    sliced.lib = Counting()
    sliced.accumulate_packed(packed, anns, out_size, True, True)
    assert launches == [1] * len(anns)
    assert sliced.last_copy_bytes > whole.last_copy_bytes > 0
    for t in GRID:
        for g in GATES:
            _assert_same(sliced.at(t, g), whole.at(t, g), f"t={t} g={g}")


def test_zero_gates_is_one_gate_at_dist_abs_f32(cuda_device):
    """The raw ABI: G = 0 with dist_abs_f32 and G = 1 with dist_abs_grid = {dist_abs_f32} (and dist_abs_f32 = 0, which
    it must not read) write bit-identical outputs."""
    outs, anns, args, out_size, pk = _batch(CFG3, "blobs", cuda_device)
    packed = ops.decode_packed(outs, 100, 100, 0.5, 0.1)
    grid = _boundary_grid(pk, GRID)
    gate = _abs([CFG3.dist_thresh], out_size)[0]
    zero = _raw_sweep(packed, grid, torch.float32, args, anns, out_size, G=0, dist_abs=gate)
    one = _raw_sweep(packed, grid, torch.float32, args, anns, out_size, G=1, dist_abs=0.0, gates_abs=[gate])
    for name, t in zero.items():
        bits = (lambda x: x.view(torch.int64)) if t.dtype == torch.float64 else (lambda x: x)
        assert torch.equal(bits(t), bits(one[name])), name
    assert (zero["assign_out"] >= 0).any() and (zero["pred_parts"] > 0).any()


def test_one_gate_equals_dist_thresh(cuda_device):
    """gates=[d] holds what dist_thresh=d holds, and copies the same bytes."""
    outs, anns, args, out_size, _ = _batch(CFG3, "blobs", cuda_device)
    packed = ops.decode_packed(outs, 100, 100, 0.5, 0.1)
    d = 0.07
    plain, gated = ThresholdSweep(args, GRID, dist_thresh=d), ThresholdSweep(args, GRID, gates=[d])
    for sweep in (plain, gated):
        sweep.accumulate_packed(packed, anns, out_size, eval_csi=True, eval_classif=True)
    assert gated.last_copy_bytes == plain.last_copy_bytes
    for t in GRID:
        _assert_same(gated.at(t), plain.at(t, d), f"t={t}")
    assert gated.best("csi") == plain.best("csi") == (plain.best_threshold("csi"), d)
