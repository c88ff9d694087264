"""-m gpu: the peaks kernel's per-channel floor hint.

In a launch with more columns than resident warps, a plane may start at the lowest floor that finished planes of its
channel reached, less a margin, instead of at no floor at all.  That hint is a guess for the plane; the exact-select
kernel checks it against the plane's histogram and redoes the plane when the hint pruned too much.  So results never
depend on the hint: every packed field equals what SDNET_FLAG_NO_FLOOR_HINT gives and what the reference's op sequence
gives (oracle/torch_port.py on the device), except the candidate counts in ``diag``."""
import re
from pathlib import Path

import pytest
import torch

from oracle import torch_port as TP
from structuredetector_b200 import _native, ops
from structuredetector_b200.synth import CONFIGS, DecodeConfig, make_raw, split_outputs

pytestmark = pytest.mark.gpu
FIELDS = ("anchor_inds", "part_inds", "assign", "counts", "anchor_out", "part_out", "part_emb")
# many small planes: 4096 images x 3 channels of 128 x 128 are 12288 one-panel columns, ~3.5 waves of the resident warps
SMALL = DecodeConfig("hint", 4096, 2, 1, 128, 128, 100, 100, cfg_id=12)


def _port(outs, cfg, pre_activated=False, chunk=256):
    parts = []
    for lo in range(0, outs["anchor_hm"].shape[0], chunk):
        sub = {k: v[lo:lo + chunk] for k, v in outs.items()}
        ref = TP.decode_tensors(sub, cfg.max_objects, cfg.max_parts, cfg.conf_threshold, cfg.dist_thresh,
                                pre_activated=pre_activated)
        parts.append({k: ref[k] for k in FIELDS})
    return {k: torch.cat([p[k] for p in parts]) for k in FIELDS}


def _run(plan, outs, cfg, dtype, flags=0):
    conf = float(torch.tensor(cfg.conf_threshold, dtype=dtype))
    got = plan.run(outs["anchor_hm"], outs["part_hm"], outs["offsets"], outs["embeddings"], conf,
                   ops._f32(cfg.dist_thresh * min(cfg.width, cfg.height)), flags=flags)
    torch.cuda.synchronize()
    return {k: v.clone() for k, v in got.as_dict().items()}


def _plan(device, cfg, images, dtype):
    return ops.DecodePlan(device, images, cfg.labels, cfg.parts, cfg.height, cfg.width, cfg.max_objects, cfg.max_parts, dtype)


def _check(device, cfg, outs, dtype, *, flags=0, pre_activated=False, what=""):
    """Decode with and without hints; both must equal the reference.  Returns (hinted, unhinted) fields."""
    images = outs["anchor_hm"].shape[0]
    on = _run(_plan(device, cfg, images, dtype), outs, cfg, dtype, flags)
    off = _run(_plan(device, cfg, images, dtype), outs, cfg, dtype, flags | _native.FLAG_NO_FLOOR_HINT)
    want = _port(outs, cfg, pre_activated)
    for key in FIELDS:
        assert torch.equal(on[key], off[key]), f"{what}: {key} differs with hints on and off"
        assert torch.equal(on[key], want[key].to(on[key].dtype)), f"{what}: {key} differs from the reference"
    return on, off


def _tiled(cfg, mode, images, unique, seed, dtype=torch.float32):
    uniq = make_raw(cfg, mode, batch=unique, seed=seed)
    idx = (torch.arange(images) * 7 + 3) % unique
    return uniq[idx].contiguous().to(dtype)


def test_flag_matches_the_header():
    header = (Path(__file__).resolve().parent.parent / "include" / "sdnet_decode.h").read_text()
    assert int(re.search(r"#define SDNET_FLAG_NO_FLOOR_HINT (\d+)u", header).group(1)) == _native.FLAG_NO_FLOOR_HINT


@pytest.mark.parametrize("mode", ["noise", "blobs"])
def test_bench_batch_fp32(cuda_device, mode):
    cfg = CONFIGS["cfg5"]
    raw = torch.cat([make_raw(cfg, mode, batch=32, seed=500 + s) for s in range(32)])  # 1024 distinct images
    outs = split_outputs(raw.to(cuda_device), cfg.labels, cfg.parts)
    on, off = _check(cuda_device, cfg, outs, torch.float32, what=mode)
    assert on["diag"][:, 0].float().mean() < 0.8 * off["diag"][:, 0].float().mean(), "the hints pruned nothing"


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("mode", ["noise", "blobs"])
def test_bench_batch_half(cuda_device, dtype, mode):
    cfg = CONFIGS["cfg5"]
    raw = _tiled(cfg, mode, 512, 32, seed=600, dtype=dtype)  # 512 images: 1.3 waves of fp16 / bf16 columns
    outs = split_outputs(raw.to(cuda_device), cfg.labels, cfg.parts)
    on, off = _check(cuda_device, cfg, outs, dtype, what=f"{mode} {dtype}")
    cand_on, cand_off = on["diag"][:, 0].float().mean(), off["diag"][:, 0].float().mean()
    assert cand_on < 0.9 * cand_off, f"the hints pruned little: {cand_on:.0f} against {cand_off:.0f} candidates per plane"


def _adversarial(device, high_images):
    """The first `high_images` images lie 4 logits higher than the rest: the planes that finish first set hints far
    above the floors of the planes that start later.  (Blob maps: their planes' floors lie within 3 fine bins of each
    other, so without the shift no hint is too high.)"""
    raw = _tiled(SMALL, "blobs", SMALL.batch, 64, seed=81)
    raw[:high_images, :SMALL.labels + SMALL.parts] += 4.0
    return split_outputs(raw.to(device), SMALL.labels, SMALL.parts)


def test_wrong_hints_are_caught_by_the_exact_select(cuda_device):
    outs = _adversarial(cuda_device, 1600)
    on, off = _check(cuda_device, SMALL, outs, torch.float32, what="adversarial")
    redone = on["diag"][:, 1].view(SMALL.batch, -1)
    assert int(off["diag"][:, 1].sum()) == 0
    assert int(redone[1600:].sum()) > 0, "no hint was too high: the batch does not test the fallback"
    assert int(redone[:1600].sum()) == 0, "a plane of the high images was redone"


def test_pre_activated_maps(cuda_device):
    # noise maps: their planes' K-th scores lie near 0.87.  Blob maps of this size put them near 0.008, and a fine bin of a
    # pre-activated map is 1/128 in score, so the hint's 2-bin margin takes it to 0 there: nothing to see pruned.
    raw = _tiled(SMALL, "noise", SMALL.batch, 64, seed=82)
    outs = split_outputs(raw.to(cuda_device), SMALL.labels, SMALL.parts)
    outs["anchor_hm"] = TP.suppress(TP.activate(outs["anchor_hm"]))
    outs["part_hm"] = TP.suppress(TP.activate(outs["part_hm"]))
    on, off = _check(cuda_device, SMALL, outs, torch.float32, flags=_native.FLAG_PRE_ACTIVATED, pre_activated=True,
                     what="pre-activated")
    assert on["diag"][:, 0].float().mean() < 0.8 * off["diag"][:, 0].float().mean(), "the hints pruned nothing"


def test_channel_whose_planes_all_saturate(cuda_device):
    raw = _tiled(SMALL, "noise", SMALL.batch, 64, seed=83)
    raw[:, 0] = 14.0 + raw[:, 0].abs()  # every score of channel 0 is the clamp's: one plateau per plane
    outs = split_outputs(raw.to(cuda_device), SMALL.labels, SMALL.parts)
    on, _ = _check(cuda_device, SMALL, outs, torch.float32, what="saturated")
    assert int(on["diag"].view(SMALL.batch, -1, 2)[:, 1:, 1].sum()) == 0, "a plane of the other channels was redone"


def test_workspace_reused_with_hints(cuda_device):
    """One plan whose workspace starts as garbage decodes batch after batch with hints.  Hint words left behind by one
    decode would start the next batch's planes at the old batch's floors: a batch of low floors after one of high floors
    would then need the exact select, which a one-off decode of it does not."""
    high = _adversarial(cuda_device, SMALL.batch)
    low = _adversarial(cuda_device, 0)
    mixed = _adversarial(cuda_device, 1600)
    plan = _plan(cuda_device, SMALL, SMALL.batch, torch.float32)
    plan.workspace.fill_(0xA5)
    for it, outs in enumerate((high, low, mixed, low, high, low)):
        got = _run(plan, outs, SMALL, torch.float32)
        want = _run(_plan(cuda_device, SMALL, SMALL.batch, torch.float32), outs, SMALL, torch.float32)
        for key in FIELDS:
            assert torch.equal(got[key], want[key]), f"run {it}: {key}"
        if outs is not mixed:
            assert int(got["diag"][:, 1].sum()) == 0, f"run {it}: planes redone, so hints were left behind"
