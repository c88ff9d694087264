"""-m gpu: dense sigmoid + NMS maps (the reference's RawDecoder, src/sdnet/cli/convert_coreml.py:12-19)
against the reference's own op sequence on the device, and the RawDecoder -> CoreMLDecoder route against
the plain Decoder."""
import pytest
import torch

from oracle import torch_port as TP
from structuredetector_b200 import CoreMLDecoder, CoreMLModel, Decoder, RawDecoder, ops
from structuredetector_b200.synth import CONFIGS, DecodeConfig, make_raw, split_outputs
from tests.helpers import make_args, plain

pytestmark = pytest.mark.gpu


def _reference_maps(hm, radius=2):
    return TP.suppress(TP.activate(hm), radius)  # max_pool2d equality on clamp(sigmoid(x)), in hm's dtype


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("h,w,mode", [(128, 128, "noise"), (128, 128, "ties"), (37, 53, "ties"), (1, 300, "noise"),
                                      (300, 1, "noise"), (33, 257, "blobs"), (64, 612, "noise")])
def test_suppress_maps_bit_exact(cuda_device, dtype, h, w, mode):
    cfg = DecodeConfig("sup", 2, 3, 2, h, w, 1, 1, cfg_id=31)
    raw = make_raw(cfg, mode).to(dtype).to(cuda_device)
    hm = raw[:, :5]  # channel-slice view, not contiguous in the batch dimension
    for radius in (2, 1):
        got = ops.suppress_maps(hm, radius)
        want = _reference_maps(hm, radius)
        assert got.dtype == dtype and got.shape == want.shape
        assert torch.equal(got.view(torch.int32 if dtype == torch.float32 else torch.int16),
                           want.contiguous().view(torch.int32 if dtype == torch.float32 else torch.int16)), (h, w, mode, radius)


def test_saturated_plateaus_survive(cuda_device):
    hm = torch.full((1, 1, 20, 24), 20.0, device=cuda_device)  # every score is the clamp: one big plateau
    hm[0, 0, 5, 5] = 15.0                                       # a lower logit with the SAME clamped score
    got = ops.suppress_maps(hm)
    assert torch.equal(got, _reference_maps(hm)) and int((got > 0).sum()) == 20 * 24


@pytest.mark.parametrize("name,mode,batch,dtype", [
    pytest.param("cfg1", "blobs", 2, torch.float32, id="cfg1-blobs"),
    pytest.param("cfg1", "ladder", 2, torch.float32, id="cfg1-ladder"),
    pytest.param("cfg3", "blobs", 2, torch.float32, id="cfg3-blobs"),
    # the benchmarked geometry: 960 tile-kernel columns (fp32), 8 strips x 5 panels per plane (fp16)
    pytest.param("cfg5", "blobs", 64, torch.float32, id="cfg5-blobs-64-float32"),
    pytest.param("cfg5", "blobs", 64, torch.float16, id="cfg5-blobs-64-float16"),
])
def test_raw_decoder_feeds_coreml_decoder(cuda_device, name, mode, batch, dtype):
    cfg = CONFIGS[name]
    raw = make_raw(cfg, mode, batch=batch).to(dtype).to(cuda_device)
    args = make_args(cfg)
    baked = RawDecoder(cfg.labels + cfg.parts)(raw)
    assert baked.shape == raw.shape and torch.equal(baked[:, cfg.labels + cfg.parts:], raw[:, cfg.labels + cfg.parts:])
    via_coreml = CoreMLDecoder(args)(split_outputs(baked, cfg.labels, cfg.parts))
    direct = Decoder(args)(split_outputs(raw, cfg.labels, cfg.parts))
    assert plain(via_coreml) == plain(direct)


def test_coreml_model_wrapper_bakes_the_heat_maps(cuda_device):
    """CoreMLModel(model, args) = the network followed by RawDecoder (convert_coreml.py:21-29): a stand-in head producing the raw
    (B, M+N+4, H, W) tensor, checked against the reference's op sequence and decoded through CoreMLDecoder."""
    from types import SimpleNamespace

    cfg = CONFIGS["cfg3"]
    raw = make_raw(cfg, "blobs", batch=2).to(cuda_device)

    class Head(torch.nn.Module):  # plays the network: returns the stored raw output whatever the image
        def forward(self, image):
            return raw

    args = make_args(cfg)
    args.labels, args.parts = {"bean": 0, "maize": 1}, {"leaf": 0}
    module = CoreMLModel(Head(), args)
    baked = module(torch.zeros(2, 3, 8, 8, device=cuda_device))
    nb = cfg.labels + cfg.parts
    assert torch.equal(baked[:, :nb], _reference_maps(raw[:, :nb])) and torch.equal(baked[:, nb:], raw[:, nb:])
    assert plain(CoreMLDecoder(args)(split_outputs(baked, cfg.labels, cfg.parts))) == plain(Decoder(args)(split_outputs(raw, cfg.labels, cfg.parts)))


@pytest.mark.parametrize("path", ["tile", "w"])
def test_suppress_into_strided_output(cuda_device, path, monkeypatch):
    """sdnet_suppress_into_launch: the result lands in the first channels of a wider tensor (strided output), on both kernels
    (the per-lane one is forced through a 4-byte-misaligned input view)."""
    cfg = DecodeConfig("supinto", 3, 3, 2, 70, 132, 1, 1, cfg_id=33)
    raw = make_raw(cfg, "noise").to(cuda_device)
    if path == "w":
        wide = torch.zeros(3, 9, 70, 133, device=cuda_device)
        wide[..., 1:] = raw
        raw_in = wide[..., 1:]  # rows start 4 bytes off a 16-byte boundary: TMA cannot describe them
    else:
        raw_in = raw
    out = torch.full((3, 9, 70, 132), -7.0, device=cuda_device)
    ops.suppress_into(raw_in[:, :5], out[:, :5])
    assert torch.equal(out[:, :5], _reference_maps(raw[:, :5])) and bool((out[:, 5:] == -7.0).all())
