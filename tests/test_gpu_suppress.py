"""-m gpu: the suppress kernels (csrc/suppress.cuh, DESIGN section 4.5) at the geometry that is timed, at every row
remainder, and on strided inputs and outputs, bit for bit against the reference's own op sequence on the device,
``TP.suppress(TP.activate(hm), radius)``.

Two kernels compute ``nms(clamped_sigmoid(x))``:

- ``sdnet_suppress_tile_kernel<R>`` takes fp32 maps whose base and pitches are 16-byte aligned (and a 16-byte-aligned
  output). It reads TMA tiles of 4 rows x 128 columns, cuts the line of (plane, panel) columns into the peaks kernel's
  units (whole columns, then chunks of ``chunk_groups`` groups that may run over a column's end), deals them round
  robin, and zero-fills each output word before it overwrites the survivors.
- ``sdnet_suppress_kernel<R, DT>`` takes fp16, bf16 and every layout the tile kernel cannot: 64-row strips, 128-column
  panels, halo lanes, vector or scalar loads and stores depending on alignment.

Every launch here runs under the CUDA profiler and asserts which of the two it reached.  Outputs written through
``suppress_into`` are pre-filled with a sentinel bit pattern; where the output is a view, it sits inside a larger
buffer whose elements outside the view must still hold the sentinel afterwards.  Large references are computed
in slices of 16 images, and every image is compared."""
import functools

import pytest
import torch
from torch.profiler import ProfilerActivity

from oracle import torch_port as TP
from structuredetector_b200 import ops
from structuredetector_b200.synth import CONFIGS, DecodeConfig, make_raw

pytestmark = pytest.mark.gpu

TILE, REG = "sdnet_suppress_tile_kernel", "sdnet_suppress_kernel<"
SENTINEL = 0x7FA5A5A5  # a NaN bit pattern: no kernel writes it
SLICE = 16  # images per reference slice
UNIQUE = 32  # distinct images of a benchmark-sized batch, as in bench.py
TILE_WARPS_PER_SM = 24  # at most 6 resident CTAs of 4 warps (the tile kernel's launch bounds)
CFG5 = CONFIGS["cfg5"]  # 512 x 612 maps: 5 panels of 128 columns, 128 groups of 4 rows per column


def launched(kernel, *calls):
    """Run the calls under the CUDA profiler and return their results; each call must launch exactly one suppress
    kernel, and it must be ``kernel``."""
    with torch.profiler.profile(activities=[ProfilerActivity.CUDA]) as prof:
        results = [call() for call in calls]
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if "sdnet_suppress" in e.name]
    assert len(names) == len(calls) and all(kernel in n for n in names), (kernel, names)
    return results


def bits(t):
    return t.view(torch.int32 if t.dtype == torch.float32 else torch.int16)


def assert_reference(got, hm, radius, what):
    """``got`` equals the reference on ``hm`` bit for bit, image slice by image slice.  ``suppress_into`` writes
    float32 whatever the input's dtype; fp16 / bf16 scores widen to it exactly."""
    for lo in range(0, hm.shape[0], SLICE):
        want = TP.suppress(TP.activate(hm[lo:lo + SLICE]), radius)
        g = got[lo:lo + SLICE]
        want = want.to(g.dtype).contiguous()
        if not torch.equal(bits(g), bits(want)):
            first = tuple((bits(g) != bits(want)).nonzero()[0].tolist())
            n = int((bits(g) != bits(want)).sum())
            raise AssertionError(f"{what}, radius {radius}: {n} pixels differ in images {lo}..{lo + g.shape[0] - 1}, "
                                 f"the first at {(lo + first[0],) + first[1:]}: got {float(g[first])!r} "
                                 f"want {float(want[first])!r}")


def sentinel(shape, device):
    return torch.full(shape, SENTINEL, dtype=torch.int32, device=device).view(torch.float32)


def assert_frame_intact(buf, view_slices, what):
    """Every element of ``buf`` outside ``buf[view_slices]`` still holds the sentinel."""
    outside = torch.ones(buf.shape, dtype=torch.bool, device=buf.device)
    outside[view_slices] = False
    n = int((buf.view(torch.int32)[outside] != SENTINEL).sum())
    assert n == 0, f"{what}: {n} elements written outside the output view"


@functools.lru_cache(maxsize=None)
def _unique_cfg5(mode):
    return make_raw(CFG5, mode, batch=UNIQUE)  # CPU: the device copy is made per case and freed with it


def shard(device, mode, images, channels, dtype):
    """``images`` cfg5 raw outputs (first ``channels`` channels, contiguous) built like bench.py's: 32 distinct
    images tiled with a rotation coprime to 32, so every image appears and no two planes are queued alike."""
    uniq = _unique_cfg5(mode)[:, :channels].to(device)
    idx = (torch.arange(images, device=device) * 7 + 3) % UNIQUE
    return uniq[idx].to(dtype).contiguous()


def assert_tile_regime(device, columns, regime):
    """The tile kernel's schedule the case is meant to reach, from the column count and the SM count: with at most
    24 resident warps per SM, ``columns >= k * SMs * 24`` gives every warp at least k whole columns."""
    full = torch.cuda.get_device_properties(device).multi_processor_count * TILE_WARPS_PER_SM
    if regime == "chunks":  # one wave of chunk units, no whole-column unit
        assert columns < full, (columns, full)
    elif regime == "tier1":  # one whole column per warp, then chunks
        assert full <= columns < 2 * full, (columns, full)
    else:  # "multi": at least two whole columns per warp, so each warp carries its ring across units
        assert columns >= 2 * full, (columns, full)


# --- 1. benchmark geometry, tile kernel -------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["noise", "blobs"])
@pytest.mark.parametrize("images,channels,regime", [(32, 3, "chunks"), (32, 7, "chunks"), (128, 3, "chunks"),
                                                    (128, 7, "tier1"), (256, 3, "tier1"), (256, 7, "multi")])
def test_tile_kernel_bench_geometry(cuda_device, mode, images, channels, regime):
    """cfg5 maps, fp32: C = 3 is what tools/time_suppress.py times, C = 7 every channel of the raw head output.
    Radius 2 through ``suppress_maps``; radius 1 through ``suppress_into`` on a sentinel-filled output, so a group
    row left unwritten shows."""
    assert_tile_regime(cuda_device, images * channels * -(-CFG5.width // 128), regime)
    hm = shard(cuda_device, mode, images, channels, torch.float32)
    what = f"{mode} {images}x{channels}"
    (got,) = launched(TILE, lambda: ops.suppress_maps(hm, 2))
    assert_reference(got, hm, 2, what)
    del got
    out = sentinel(hm.shape, cuda_device)
    launched(TILE, lambda: ops.suppress_into(hm, out, 1))
    assert_reference(out, hm, 1, what)


# --- 2. benchmark geometry, register-window kernel --------------------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("mode", ["noise", "blobs", "ties"])
@pytest.mark.parametrize("images", [128, 256])
def test_register_kernel_bench_geometry(cuda_device, dtype, mode, images):
    """cfg5 maps in fp16 / bf16, all 7 channels: 8 strips of 64 rows, 5 panels of which the last has 100 of 128
    columns.  ``suppress_maps`` returns the input's dtype, compared through an int16 view."""
    hm = shard(cuda_device, mode, images, 7, dtype)
    for radius in (2, 1):
        (got,) = launched(REG, lambda: ops.suppress_maps(hm, radius))
        assert got.dtype == dtype
        assert_reference(got, hm, radius, f"{dtype} {mode} {images}")
        del got


@pytest.mark.parametrize("mode", ["noise", "ladder"])
def test_register_kernel_fp32_misaligned_bench_geometry(cuda_device, mode):
    """fp32 cfg5 maps the tile kernel cannot take: rows start 4 bytes past a 16-byte boundary (a view of a
    wider tensor), so the register-window kernel runs with scalar loads."""
    hm = shard(cuda_device, mode, 64, 7, torch.float32)
    wide = torch.empty(hm.shape[:3] + (hm.shape[3] + 1,), device=cuda_device)
    wide[..., 1:] = hm
    view = wide[..., 1:]
    del hm
    for radius in (2, 1):
        (got,) = launched(REG, lambda: ops.suppress_maps(view, radius))
        assert_reference(got, view, radius, f"misaligned {mode}")
        del got


# --- 3. row and column remainders -------------------------------------------------------------------------------
# H % 4 takes every residue.  With few columns the chunk is at its minimum of 8 groups, so at H = 65, 66, 67
# (17 groups per column) and H = 130 (33 groups) chunks run over column ends; H = 63 (16 groups) makes two chunks per
# column, and H <= 7 (1 or 2 groups) one chunk per column.  The register kernel sees one to three 64-row strips.
HEIGHTS = [2, 3, 5, 6, 7, 63, 65, 66, 67, 130]
MODES = ["noise", "blobs", "ladder", "ties"]


@functools.lru_cache(maxsize=None)
def _maps(h, w, batch, planes, mode):
    """The first ``planes`` channels of a synthetic raw output (CPU)."""
    cfg = DecodeConfig("sup", batch, planes - 1, 1, h, w, 1, 1, cfg_id=41)
    return make_raw(cfg, mode)[:, :planes]


@pytest.mark.parametrize("radius", [2, 1])
@pytest.mark.parametrize("h", HEIGHTS)
def test_tile_kernel_remainders(cuda_device, h, radius):
    """fp32, W a multiple of 4, 2 images x 3 planes; the output is a 16-byte-aligned view inside a sentinel frame
    (one channel, one row and four columns of margin on each side)."""
    widths = [4, 128, 132, 252, 256, 260, 612]
    cases = []
    for i, w in enumerate(widths):
        hm = _maps(h, w, 2, 3, MODES[(i + h) % len(MODES)]).to(cuda_device)
        buf = sentinel((2, 5, h + 2, w + 8), cuda_device)
        sl = (slice(None), slice(1, 4), slice(1, h + 1), slice(4, w + 4))
        cases.append((hm, buf, sl))
    launched(TILE, *[lambda hm=hm, buf=buf, sl=sl: ops.suppress_into(hm, buf[sl], radius) for hm, buf, sl in cases])
    for w, (hm, buf, sl) in zip(widths, cases):
        assert_reference(buf[sl], hm, radius, f"{h}x{w}")
        assert_frame_intact(buf, sl, f"{h}x{w}")


@pytest.mark.parametrize("radius", [2, 1])
@pytest.mark.parametrize("h", HEIGHTS)
def test_register_kernel_remainders(cuda_device, h, radius):
    """fp16, W not a multiple of 4: partial last panels and per-element tails; the output view has an odd pitch and a
    4-byte-misaligned base, so every store is scalar."""
    widths = [1, 3, 5, 127, 129, 257]
    cases = []
    for i, w in enumerate(widths):
        hm = _maps(h, w, 2, 3, MODES[(i + h) % len(MODES)]).to(cuda_device).half()
        buf = sentinel((2, 5, h + 2, w + 3), cuda_device)
        sl = (slice(None), slice(1, 4), slice(1, h + 1), slice(1, w + 1))
        cases.append((hm, buf, sl))
    launched(REG, *[lambda hm=hm, buf=buf, sl=sl: ops.suppress_into(hm, buf[sl], radius) for hm, buf, sl in cases])
    for w, (hm, buf, sl) in zip(widths, cases):
        assert_reference(buf[sl], hm, radius, f"{h}x{w}")
        assert_frame_intact(buf, sl, f"{h}x{w}")


@pytest.mark.parametrize("dtype,kernel", [(torch.float32, TILE), (torch.float16, REG), (torch.bfloat16, REG)])
def test_large_plane(cuda_device, dtype, kernel):
    """One 4095 x 4096 plane (1024 groups per column, 64 strips, 32 panels) into a 16-byte-aligned framed view:
    the tile kernel's chunks straddle column ends, the register kernel stores float4 words."""
    h, w = 4095, 4096
    hm = _maps(h, w, 1, 1, "ties").to(cuda_device).to(dtype)
    buf = sentinel((1, 3, h + 2, w + 8), cuda_device)
    sl = (slice(None), slice(1, 2), slice(1, h + 1), slice(4, w + 4))
    for radius in (2, 1):
        buf.view(torch.int32)[sl] = SENTINEL
        launched(kernel, lambda: ops.suppress_into(hm, buf[sl], radius))
        assert_reference(buf[sl], hm, radius, f"{dtype} {h}x{w}")
        assert_frame_intact(buf, sl, f"{dtype} {h}x{w}")


# --- 4. layouts and stores --------------------------------------------------------------------------------------
B, C, H, W = 3, 5, 70, 260  # 2 strips, 3 panels (the last with 4 columns), H % 4 = 2


def _padded(t, pitch):
    """A copy of ``t`` whose rows are ``pitch`` elements apart (a view of a wider tensor)."""
    big = torch.zeros(t.shape[:3] + (pitch,), dtype=t.dtype, device=t.device)
    big[..., :t.shape[3]] = t
    return big[..., :t.shape[3]]


def _misaligned(t):
    big = torch.zeros(t.shape[:3] + (t.shape[3] + 1,), dtype=t.dtype, device=t.device)
    big[..., 1:] = t
    return big[..., 1:]


# input layout -> the (B, C, H, W) view given to the kernel
INPUTS = {
    "channel_slice": lambda raw: raw[:, :C],  # strided over the batch: 9 channels of which the first 5
    "pitch_mult4": lambda raw: _padded(raw[:, :C], W + 4),
    "pitch_odd": lambda raw: _padded(raw[:, :C], W + 3),
    "misaligned": lambda raw: _misaligned(raw[:, :C]),
}
# output layout -> (buffer shape, the view's slices)
OUTPUTS = {
    "wide_channels": ((B, 9, H, W), (slice(None), slice(0, C))),
    "pitch_aligned": ((B, C + 2, H + 2, W + 8), (slice(None), slice(1, C + 1), slice(1, H + 1), slice(4, W + 4))),
    "pitch_odd": ((B, C + 2, H + 2, W + 1), (slice(None), slice(1, C + 1), slice(1, H + 1), slice(0, W))),
}
LAYOUTS = [  # dtype, input, output, kernel
    (torch.float32, "channel_slice", "wide_channels", TILE),
    (torch.float32, "pitch_mult4", "pitch_aligned", TILE),
    (torch.float32, "channel_slice", "pitch_odd", REG),  # 16-byte loads, scalar stores
    (torch.float32, "pitch_odd", "pitch_aligned", REG),  # scalar loads, 16-byte stores
    (torch.float32, "misaligned", "wide_channels", REG),
    (torch.float16, "channel_slice", "wide_channels", REG),
    (torch.float16, "pitch_odd", "pitch_odd", REG),
    (torch.bfloat16, "pitch_mult4", "pitch_aligned", REG),
    (torch.bfloat16, "misaligned", "pitch_odd", REG),
]


@pytest.mark.parametrize("mode", ["ladder", "ties"])
@pytest.mark.parametrize("dtype,inp,outp,kernel", LAYOUTS,
                         ids=[f"{str(d).split('.')[-1]}-{i}-{o}" for d, i, o, _ in LAYOUTS])
def test_layouts_and_stores(cuda_device, dtype, inp, outp, kernel, mode):
    raw = make_raw(DecodeConfig("sup", B, 3, 2, H, W, 1, 1, cfg_id=43), mode).to(cuda_device).to(dtype)
    hm = INPUTS[inp](raw)
    shape, sl = OUTPUTS[outp]
    buf = sentinel(shape, cuda_device)
    for radius in (2, 1):
        buf.view(torch.int32)[sl] = SENTINEL
        launched(kernel, lambda: ops.suppress_into(hm, buf[sl], radius))
        assert_reference(buf[sl], hm, radius, f"{inp} -> {outp}")
        assert_frame_intact(buf, sl, f"{inp} -> {outp}")
