"""The decoder at the edges of its documented limits (include/sdnet_decode.h, DESIGN section 2): K and P up to 1024,
M + N up to 255, H * W up to 2^24 - 1.  These are the shapes that take branches no realistic map reaches: a tail sort of
more than 1024 composites, grouping in more than one pass, the full P x K grouping search over the masked slots, the
8-bit class and 24-bit index fields of the composite.

-m gpu cases are bit-exact (tests/helpers.py::assert_packed_equal) against the numpy oracle fed the device's own
activation; the unmarked ones check on the host that every limit is refused before any launch.
"""
import ctypes
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import sdnet_oracle as O
from oracle import torch_port as TP
from structuredetector_b200 import _native, ops
from structuredetector_b200.synth import DecodeConfig, make_raw, split_outputs
from tests.helpers import assert_packed_equal, packed_np, torch_sigmoid_fn

gpu = pytest.mark.gpu


def _device_activation(dtype, device):
    """float32 ndarray -> the reference's clamped sigmoid evaluated in `dtype` on the device."""
    def fn(m):
        t = torch.from_numpy(np.ascontiguousarray(m)).to(device).to(dtype)
        return torch.clamp(torch.sigmoid(t), min=1e-6, max=1 - 1e-6).float().cpu().numpy()
    return fn


def _oracle(raw, m, n, k, p, conf, dist, device, *, dtype=torch.float32, radius=2, pre_activated=False):
    """O.decode_packed on the float32 image of `raw` (B, M+N+4, H, W), fed the activation `dtype` gets on the device."""
    f = raw.float().cpu().numpy()
    planes = f[:, :m], f[:, m:m + n], f[:, m + n:m + n + 2], f[:, m + n + 2:]
    if pre_activated:
        kw = {"pre_activated": True}
    elif dtype == torch.float32:
        kw = {"sigmoid_fn": torch_sigmoid_fn(device)}
    else:
        kw = {"activation_fn": _device_activation(dtype, device), "conf_cmp": float(torch.tensor(conf, dtype=dtype))}
    return O.decode_packed(*planes, k, p, conf, dist, radius=radius, **kw)


def _check(raw, m, n, k, p, device, *, conf=0.4, dist=0.1, what="", **kw):
    """Decode `raw` on the device and compare every packed field with the oracle; returns the device's fields."""
    dtype = raw.dtype
    outs = split_outputs(raw.to(device), m, n)
    got = packed_np(ops.decode_packed(outs, k, p, conf, dist, **kw))
    want = _oracle(raw, m, n, k, p, conf, dist, device, dtype=dtype, radius=kw.get("radius", 2),
                   pre_activated=kw.get("pre_activated", False))
    assert_packed_equal(got, want, what=what)
    return got


# ----------------------------------------------------------------------------------------------- large K / P
# 613 is the first K whose histogram cut-off (up to K + 412 composites) can collect more than the 1024 the counting-rank
# sort takes; 1000 and 1024 get there on the radix route too (up to K + 64)
LARGE = [(128, 128, 613), (128, 128, 1000), (128, 128, 1024), (64, 64, 1024), (64, 130, 1024), (32, 32, 1024)]
VARIANTS = [("default", torch.float32, {}), ("warp", torch.float32, {"warp_kernel": True}),
            ("exact", torch.float32, {"exact_select": True}), ("radius1", torch.float32, {"radius": 1}),
            ("fp16", torch.float16, {}), ("bf16", torch.bfloat16, {}), ("pre", torch.float32, {"pre_activated": True})]


@gpu
@pytest.mark.parametrize("mode", ["noise", "ties", "blobs"])
@pytest.mark.parametrize("h,w,k", LARGE)
def test_large_k_and_p(cuda_device, h, w, k, mode):
    """K = P up to 1024 (32 x 32: K = P = H * W, the lists are mostly zero-fill) on both peaks kernels, the exact select,
    radius 1, fp16 / bf16 and pre-activated maps."""
    cfg = DecodeConfig("limits", 2, 3, 2, h, w, k, k, cfg_id=40)
    raw32 = make_raw(cfg, mode, seed=4000 + h + w + k)
    for name, dtype, kw in VARIANTS:
        raw = raw32.to(dtype)
        if kw.get("pre_activated"):  # 64 x 64: fewer non-zero pixels than K, the zeros come from the tail's zero-fill
            raw = raw32.clone()
            raw[:, :5] = TP.suppress(TP.activate(raw32[:, :5].to(cuda_device)), kw.get("radius", 2)).cpu()
        if name in ("default", "warp"):
            outs = split_outputs(raw.to(cuda_device), 3, 2)
            want_path = "warp" if kw.get("warp_kernel") or w % 4 else "tile"
            assert ops.peaks_path(outs, k, k, warp_kernel=bool(kw.get("warp_kernel"))) == want_path
        _check(raw, 3, 2, k, k, cuda_device, what=f"{h}x{w} K=P={k} {mode} {name}", **kw)


def _lattice(n_tied, split, seed, m=2, n=2, h=128, w=128):
    """(1, M+N+4, H, W) maps whose peaks sit on a 3-pixel lattice, so every site survives the 5 x 5 NMS.  In the anchor
    group and in the part group, `n_tied` sites share the logit 4.0 -- all in the group's first plane, or half in each of
    its first two planes (`split`) -- and every other pixel is at least 8 logits lower, with distinct values."""
    g = torch.Generator().manual_seed(seed)
    raw = torch.empty(1, m + n + 4, h, w)
    ys, xs = torch.meshgrid(torch.arange(0, h, 3), torch.arange(0, w, 3), indexing="ij")
    sites = (ys * w + xs).flatten()
    assert sites.numel() >= n_tied
    for c in range(m + n):
        plane = (-30.0 + 16.0 * torch.randperm(h * w, generator=g).double() / (h * w)).float()  # [-30, -14), distinct
        order = sites[torch.randperm(sites.numel(), generator=g)]
        plane[order] = (-12.0 + 8.0 * torch.arange(order.numel()).double() / order.numel()).float()  # [-12, -4)
        first = c in (0, m)
        tied = (n_tied // 2 if first else n_tied - n_tied // 2) if split else (n_tied if first else 0)
        if c in (0, 1, m, m + 1):
            plane[order[:tied]] = 4.0
        raw[0, c] = plane.view(h, w)
    raw[:, m + n:m + n + 2] = torch.rand(1, 2, h, w, generator=g)
    raw[:, m + n + 2:] = 3.0 * torch.randn(1, 2, h, w, generator=g)
    return raw


@gpu
@pytest.mark.parametrize("warp_kernel", [False, True], ids=["tile", "warp"])
@pytest.mark.parametrize("n_tied,split", [(1200, False), (1200, True), (1600, False)], ids=["hist", "hist-split", "radix"])
def test_sort_of_more_than_1024_composites(cuda_device, n_tied, split, warp_kernel):
    """1200 tied composites all fall in the cut-off bin and 1200 <= K + 412: the histogram route collects and sorts all of
    them, more than the counting-rank sort takes.  1600 is more than K + 412 and takes the radix route.  Split across
    two planes, the tie is ordered by the class field."""
    raw = _lattice(n_tied, split, seed=5000 + n_tied + split)
    got = _check(raw, 2, 2, 1024, 1024, cuda_device, what=f"lattice {n_tied} split={split}", warp_kernel=warp_kernel)
    if n_tied <= 1024 + 412:
        assert int(got["diag"][:, 1].max()) == 0, "a plane went through the exact select: not the histogram route"
    tie = O.clamped_sigmoid(np.array([4.0], dtype=np.float32), torch_sigmoid_fn(cuda_device))[0]
    assert (got["anchor_out"][0, :, 2] == tie).all() and (got["part_out"][0, :, 2] == tie).all()
    if split:  # all of the first plane's 600 ties, then the second plane's in index order
        assert (got["anchor_out"][0, :600, 3] == 0).all() and (got["anchor_out"][0, 600:, 3] == 1).all()


@gpu
@pytest.mark.parametrize("warp_kernel", [False, True], ids=["tile", "warp"])
def test_grouping_in_more_than_one_pass(cuda_device, warp_kernel):
    """More than 512 valid parts: a grouping pass covers 512 of them, the rest need a second pass."""
    cfg = DecodeConfig("passes", 2, 2, 2, 128, 128, 1024, 1024, cfg_id=41)
    raw = make_raw(cfg, "noise")
    got = _check(raw, 2, 2, 1024, 1024, cuda_device, conf=0.05, what="two grouping passes", warp_kernel=warp_kernel)
    assert (got["counts"][:, 1] > 512).all(), got["counts"]
    assert (got["assign"][:, 512:] >= 0).any(axis=1).all(), "no part of the second pass was grouped"


# ----------------------------------------------------------------------------------------------- full grouping search
_NEAR = 1e5  # kNearField in csrc/tail.cuh
_F32_BELOW_NEAR = float(np.nextafter(np.float32(_NEAR), np.float32(0)))
_AY, _AX = 10, 10  # an anchor peak of the first class
_PY, _PX = 20, 30  # a part peak


def _far_raw(case):
    """128 x 128 blobs maps (few valid slots, many masked ones) with one anchor and one part peak whose offsets and
    embeddings are set per case.  Returns (raw, dist_thresh)."""
    cfg = DecodeConfig("far", 1, 2, 1, 128, 128, 100, 100, cfg_id=42)
    raw = make_raw(cfg, "blobs")
    ox, oy, ex, ey = 3, 4, 5, 6  # channels of offsets / embeddings
    raw[0, 0, _AY, _AX] = 12.0
    raw[0, 2, _PY, _PX] = 12.0
    raw[0, ox:ey + 1, _AY, _AX] = 0.0
    raw[0, ox:ey + 1, _PY, _PX] = 0.0
    dist = 0.1
    if case == "part_origin_far":
        raw[0, ex, _PY, _PX] = 2e5
    elif case == "part_origin_on_masked_anchors":  # origin exactly (1e6, 1e6): zero distance to every masked anchor
        raw[0, ex, _PY, _PX], raw[0, ey, _PY, _PX] = 1e6 - _PX, 1e6 - _PY
    elif case == "anchor_far":
        raw[0, ox, _AY, _AX] = 2e5
    elif case == "anchor_on_masked_parts":  # anchor exactly at (-1e6, -1e6): zero distance to every masked part
        raw[0, ox, _AY, _AX], raw[0, oy, _AY, _AX] = -1e6 - _AX, -1e6 - _AY
    elif case == "origin_at_1e5":
        raw[0, ex, _PY, _PX] = _NEAR - _PX
    elif case == "origin_below_1e5":
        raw[0, ex, _PY, _PX] = _F32_BELOW_NEAR - _PX
    elif case == "gate_at_1e5":
        dist = _NEAR / 128  # 781.25: the gate is exactly 1e5
    elif case == "gate_below_1e5":
        dist = _F32_BELOW_NEAR / 128
    elif case == "gate_2.56e6":
        dist = 2.56e6 / 128
        raw[0, ex, _PY, _PX], raw[0, ey, _PY, _PX] = 1e6 - _PX, 1e6 - _PY
    else:
        raise ValueError(case)
    return raw, dist


FAR_CASES = ["part_origin_far", "part_origin_on_masked_anchors", "anchor_far", "anchor_on_masked_parts", "origin_at_1e5",
             "origin_below_1e5", "gate_at_1e5", "gate_below_1e5", "gate_2.56e6"]


@gpu
@pytest.mark.parametrize("case", FAR_CASES)
def test_full_grouping_search(cuda_device, case):
    """A valid coordinate at or beyond +-1e5, or a gate of at least 1e5, makes the masked slots (anchors at +1e6, parts
    at -1e6) take part in the grouping: against the oracle and against the reference's op sequence on the device."""
    raw, dist = _far_raw(case)
    got = _check(raw, 2, 1, 100, 100, cuda_device, dist=dist, what=case)
    outs = split_outputs(raw.to(cuda_device), 2, 1)
    port = {key: v.cpu().numpy() for key, v in TP.decode_tensors(outs, 100, 100, 0.4, dist).items()}
    assert_packed_equal(got, port, what=f"torch port {case}")
    n_anchors, n_parts = (int(v) for v in got["counts"][0])
    assert 0 < n_anchors < 100 and 0 < n_parts < 100, "the case needs valid and masked slots of both kinds"
    top_part = int(np.flatnonzero(got["part_inds"][0] == _PY * 128 + _PX)[0])
    if case in ("part_origin_on_masked_anchors", "gate_2.56e6"):
        assert got["assign"][0, top_part] == n_anchors, "the far part belongs to the first masked anchor slot"
    if case == "anchor_on_masked_parts":
        top_anchor = int(np.flatnonzero(got["anchor_inds"][0] == _AY * 128 + _AX)[0])
        assert (got["assign"][0, n_parts:] == top_anchor).all()
    if case == "gate_2.56e6":
        masked = got["assign"][0, n_parts:]
        assert ((masked >= 0) & (masked < n_anchors)).all(), "masked parts group onto valid anchors"


# ----------------------------------------------------------------------------------------------- channel limit
@gpu
@pytest.mark.parametrize("mode", ["noise", "ties"])
@pytest.mark.parametrize("k", [64, 1024])
@pytest.mark.parametrize("m,n", [(200, 55), (254, 1), (1, 254)])
def test_channel_limit(cuda_device, m, n, k, mode):
    """M + N = 255: class indices up to 253 in the composite's 8-bit class field (255 - c)."""
    cfg = DecodeConfig("channels", 1, m, n, 32, 40, k, k, cfg_id=43)
    raw = make_raw(cfg, mode, seed=6000 + m + k)
    _check(raw, m, n, k, k, cuda_device, what=f"M={m} N={n} K=P={k} {mode}")


# ----------------------------------------------------------------------------------------------- index limit
def _last_row_raw(h, w, seed):
    """(1, 6, H, W), M = N = 1: background logits 2 N(0,1) - 6 and, in the last row, peaks every third column whose logits
    (8 to 12) grow with the column -- every selected slot has a flat index within W of H * W."""
    g = torch.Generator().manual_seed(seed)
    raw = torch.empty(1, 6, h, w)
    raw[:, :2] = 2.0 * torch.randn(1, 2, h, w, generator=g) - 6.0
    raw[:, 2:4] = torch.rand(1, 2, h, w, generator=g)
    raw[:, 4:] = 5.0 * torch.randn(1, 2, h, w, generator=g)
    xs = torch.arange(0, w, 3)
    raw[0, :2, h - 1, xs] = 8.0 + 4.0 * xs.float() / w
    return raw


@gpu
@pytest.mark.parametrize("h,w,dtype,path", [(4095, 4096, torch.float32, "tile"), (4095, 4096, torch.float16, "tile"),
                                            (4095, 4097, torch.float32, "warp")], ids=["tile-f32", "tile-f16", "warp-f32"])
def test_index_limit(cuda_device, h, w, dtype, path):
    """Maps of 2^24 - 4096 and 2^24 - 1 pixels, the most H * W may be: flat indices near 2^24 in the composite's 24-bit
    index field (0xFFFFFF - index), the exact select's survivor bitmap and the list capacity at that size."""
    assert (1 << 24) - w - 1 <= h * w < (1 << 24)
    raw = _last_row_raw(h, w, seed=7000 + w).to(dtype)
    outs = split_outputs(raw.to(cuda_device), 1, 1)
    assert ops.peaks_path(outs, 1024, 1024) == path
    # the activation and the NMS once, the oracle's selection per K
    f = raw.float().numpy()
    sig = torch_sigmoid_fn(cuda_device)
    act = (lambda x: O.clamped_sigmoid(x, sig)) if dtype == torch.float32 else _device_activation(dtype, cuda_device)
    nms = [O.nms(np.asarray(act(f[:, c:c + 1]), dtype=np.float32)) for c in (0, 1)]
    conf_cmp = float(torch.tensor(0.4, dtype=dtype))
    runs = [(100, {}), (1024, {})] + ([(1024, {"exact_select": True})] if dtype == torch.float32 and path == "tile" else [])
    want = {}
    for k, kw in runs:
        got = packed_np(ops.decode_packed(outs, k, k, 0.4, 0.1, **kw))
        if k not in want:
            want[k] = O.decode_packed(nms[0], nms[1], f[:, 2:4], f[:, 4:], k, k, 0.4, 0.1, pre_activated=True,
                                      conf_cmp=conf_cmp)
        assert_packed_equal(got, want[k], what=f"{h}x{w} {dtype} K=P={k} {kw}")
        for key in ("anchor_inds", "part_inds"):
            assert int(got[key].min()) >= h * w - w, f"{key}: a selected index outside the last row"
        if kw.get("exact_select"):
            assert int(got["diag"][:, 1].min()) == 1


# ----------------------------------------------------------------------------------------------- host-only limits
def _decode_params(**shape):
    p = _native.SdnetDecodeParams()
    p.struct_size = ctypes.sizeof(_native.SdnetDecodeParams)
    p.dtype, p.radius = _native.DTYPE_F32, 2
    p.B, p.M, p.N, p.H, p.W, p.K, p.P = 1, 2, 1, 64, 64, 1024, 1024
    for key, value in shape.items():
        setattr(p, key, value)
    return p


def test_decode_limits_are_refused_before_any_launch():
    """K or P above 1024, M + N above 255: SDNET_E_SHAPE from the host-side check (the tensors are NULL, so a library
    that skipped the check would answer SDNET_E_NULL instead; nothing is ever launched)."""
    lib = _native.load()
    assert lib.sdnet_decode_launch(ctypes.byref(_decode_params()), None) == -1  # within the limits: the NULL tensors
    for shape in ({"K": 1025}, {"P": 1025}, {"M": 200, "N": 56}, {"M": 255, "N": 1}, {"M": 1, "N": 255}):
        assert lib.sdnet_decode_launch(ctypes.byref(_decode_params(**shape)), None) == -2, shape
    assert lib.sdnet_decode_launch(ctypes.byref(_decode_params(M=200, N=55)), None) == -1


def _match_buffers(B, K, P, M, G):
    """Buffers for one match call with G ground-truth rows, all counts zero.  On a machine with a CUDA device they live
    there, so a launch -- which a correct library never makes for G > 1024 -- would only read zero ground truth."""
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    t = SimpleNamespace(
        anchor_out=torch.zeros(B, K, 4, device=dev), part_out=torch.zeros(B, P, 6, device=dev),
        assign=torch.full((B, P), -1, dtype=torch.int32, device=dev), scale=torch.ones(B, 4, dtype=torch.float64, device=dev),
        gt=torch.zeros(B, G, 3, dtype=torch.float64, device=dev), owner=torch.zeros(B, G, dtype=torch.int32, device=dev),
        n=torch.zeros(B, dtype=torch.int32, device=dev), groups=torch.zeros(M, dtype=torch.int32, device=dev),
        stats=torch.zeros(B, max(M, 20), 3, dtype=torch.int32, device=dev),
        acc=torch.zeros(B, max(K, P), dtype=torch.float64, device=dev), parts=torch.zeros(B, K, dtype=torch.int32, device=dev))
    return t


@pytest.mark.parametrize("which", ["anchors", "parts"])
def test_match_limits_are_refused_before_any_launch(which):
    """Both match launches refuse more than SDNET_MAX_GT ground-truth rows per image with SDNET_E_SHAPE."""
    lib = _native.load()
    B, K, P, M, N, G = 1, 8, 8, 2, 1, _native.MAX_GT + 1
    t = _match_buffers(B, K, P, M, G)
    mp = _native.SdnetMatchParams()
    mp.struct_size = ctypes.sizeof(_native.SdnetMatchParams)
    mp.B, mp.M, mp.N, mp.K, mp.P = B, M, N, K, P
    mp.max_gt_anchors, mp.max_gt_parts = (G, 1) if which == "anchors" else (1, G)
    mp.anchor_out, mp.part_out, mp.image_scale = t.anchor_out.data_ptr(), t.part_out.data_ptr(), t.scale.data_ptr()
    mp.gt_anchors, mp.gt_parts, mp.n_gt_anchors, mp.n_gt_parts = t.gt.data_ptr(), t.gt.data_ptr(), t.n.data_ptr(), t.n.data_ptr()
    mp.anchor_stats, mp.part_stats, mp.anchor_acc, mp.part_acc = (t.stats.data_ptr(), t.stats.data_ptr(), t.acc.data_ptr(),
                                                                  t.acc.data_ptr())
    assert lib.sdnet_match_launch(ctypes.byref(mp), None) == -2
    op = _native.SdnetObjectMatchParams()
    op.struct_size = ctypes.sizeof(_native.SdnetObjectMatchParams)
    op.B, op.M, op.N, op.K, op.P = B, M, N, K, P
    op.max_gt_objects, op.max_gt_parts = (G, 1) if which == "anchors" else (1, G)
    op.anchor_out, op.part_out, op.assign, op.image_scale = (t.anchor_out.data_ptr(), t.part_out.data_ptr(),
                                                             t.assign.data_ptr(), t.scale.data_ptr())
    op.gt_objects, op.n_gt_objects, op.gt_parts, op.gt_part_owner, op.n_gt_parts = (
        t.gt.data_ptr(), t.n.data_ptr(), t.gt.data_ptr(), t.owner.data_ptr(), t.n.data_ptr())
    op.cls_group, op.csi_stats, op.csi_acc = t.groups.data_ptr(), t.stats.data_ptr(), t.acc.data_ptr()
    op.classif_stats, op.classif_acc, op.pred_parts = t.stats.data_ptr(), t.acc.data_ptr(), t.parts.data_ptr()
    assert lib.sdnet_match_objects_launch(ctypes.byref(op), None) == -2


def test_ground_truth_limits_of_the_evaluator():
    """Evaluator._pack_ground_truth refuses an object with 65 parts and an image with 1025 ground-truth parts (the
    1025-anchor image: tests/test_evaluator.py); 64 parts in one object and 1024 in one image pass."""
    from structuredetector_b200 import ImageAnnotation, Keypoint, Object
    from structuredetector_b200.evaluator import Evaluator
    args = SimpleNamespace(labels={"bean": 0}, parts={"leaf": 0}, width=512, height=512, dist_threshold=0.05,
                           conf_threshold=0.4, down_ratio=4.0)
    ev = Evaluator(args)

    def image(parts_per_object):
        objs = [Object("bean", Keypoint("stem", 1.0, 2.0), [Keypoint("leaf", float(i), 3.0) for i in range(n)])
                for n in parts_per_object]
        return ImageAnnotation("x", objs, img_size=(512, 512))

    ev._pack_ground_truth([image([64])], torch.device("cpu"))
    ev._pack_ground_truth([image([64] * 16)], torch.device("cpu"))  # 1024 parts
    with pytest.raises(ValueError, match="64 parts"):
        ev._pack_ground_truth([image([65])], torch.device("cpu"))
    with pytest.raises(ValueError, match="1025 ground-truth points"):
        ev._pack_ground_truth([image([64] * 16 + [1])], torch.device("cpu"))
