"""CPU: the oracle against the golden vectors produced by running the reference itself
(tests/golden/make_golden.py), and against the port of the reference's op sequence on shapes the vectors
do not have.  This is what pins the oracle (SURVEY.md 8c: the reference has no tests of its own)."""
import numpy as np
import pytest
import torch

from oracle import sdnet_oracle as O
from oracle import torch_port as TP
from structuredetector_b200.synth import CONFIGS, DecodeConfig, make_raw, split_outputs
from tests.helpers import (assert_objects_close, assert_topk_equal_up_to_ties, golden_args, golden_names, listify, load_golden,
                           np_inputs, torch_sigmoid_fn)

TIE_FREE = [n for n in golden_names() if not n.startswith(("ties", "half"))]


def _oracle_on_golden(name, sigmoid_fn):
    meta, arr = load_golden(name)
    b, m, n, h, w = meta["shape"]
    raw = arr["raw"]
    pk = O.decode_packed(raw[:, :m], raw[:, m:m + n], raw[:, m + n:m + n + 2], raw[:, m + n + 2:], meta["K"], meta["P"],
                         meta["conf"], meta["dist"], sigmoid_fn=sigmoid_fn)
    return meta, arr, pk


@pytest.mark.parametrize("name", TIE_FREE)
def test_oracle_matches_reference_golden_bit_exact(name):
    """Fed torch-CPU's sigmoid (what the reference used), the oracle must reproduce every number."""
    meta, arr, pk = _oracle_on_golden(name, torch_sigmoid_fn("cpu"))
    np.testing.assert_array_equal(pk["anchor_inds"], arr["a_inds"])
    np.testing.assert_array_equal(pk["part_inds"], arr["p_inds"])
    np.testing.assert_array_equal(pk["anchor_scores_masked"], arr["a_scores_masked"])
    np.testing.assert_array_equal(pk["part_scores_masked"], arr["p_scores_masked"])
    np.testing.assert_array_equal(pk["anchor_out"][..., 3], arr["a_labels"])
    np.testing.assert_array_equal(pk["part_out"][..., 3], arr["p_labels"])
    np.testing.assert_array_equal(pk["anchor_out"][..., 0], arr["a_xs"])  # the reference adds offsets in place
    np.testing.assert_array_equal(pk["anchor_out"][..., 1], arr["a_ys"])
    np.testing.assert_array_equal(pk["part_out"][..., 0], arr["p_xs"])
    np.testing.assert_array_equal(pk["part_out"][..., 1], arr["p_ys"])
    np.testing.assert_array_equal(pk["part_emb"], arr["embeddings"])
    args = golden_args(meta)
    b, m, n, h, w = meta["shape"]
    objs = O.assemble(pk, args._r_labels, args._r_parts, args.anchor_name, meta["conf"], (w, h), (4 * w, 4 * h))
    assert listify(objs) == meta["annotation"]
    rp = O.raw_parts(pk, args._r_parts, meta["conf"], (w, h), (4 * w, 4 * h))
    assert listify(rp) == meta["raw_parts"]
    if "anchor_sig" in arr:
        np.testing.assert_array_equal(pk["anchor_sig"], arr["anchor_sig"])
        np.testing.assert_array_equal(pk["part_sig"], arr["part_sig"])


@pytest.mark.parametrize("name", TIE_FREE)
def test_oracle_default_sigmoid_agrees_within_tolerance(name):
    """With its own (correctly rounded) sigmoid the oracle keeps every index and assignment and
    moves scores by at most a couple of ulps."""
    meta, arr, pk = _oracle_on_golden(name, None)
    np.testing.assert_array_equal(pk["anchor_inds"], arr["a_inds"])
    np.testing.assert_array_equal(pk["part_inds"], arr["p_inds"])
    np.testing.assert_allclose(pk["anchor_scores_masked"], arr["a_scores_masked"], rtol=0, atol=1e-6)
    args = golden_args(meta)
    b, m, n, h, w = meta["shape"]
    objs = O.assemble(pk, args._r_labels, args._r_parts, args.anchor_name, meta["conf"], (w, h), (4 * w, 4 * h))
    assert_objects_close(listify(objs), meta["annotation"], score_atol=1e-6, coord_rtol=1e-5, what=name)


def test_oracle_on_ties_matches_reference_up_to_tie_order():
    meta, arr, pk = _oracle_on_golden("ties_small", torch_sigmoid_fn("cpu"))
    assert_topk_equal_up_to_ties(pk["anchor_scores_masked"], pk["anchor_out"][..., 3], pk["anchor_inds"],
                                 arr["a_scores_masked"], arr["a_labels"], arr["a_inds"], what="anchors")
    assert_topk_equal_up_to_ties(pk["part_scores_masked"], pk["part_out"][..., 3], pk["part_inds"],
                                 arr["p_scores_masked"], arr["p_labels"], arr["p_inds"], what="parts")


@pytest.mark.parametrize("name", TIE_FREE)
def test_oracle_variants_match_reference_golden(name):
    meta, arr = load_golden(name)
    b, m, n, h, w = meta["shape"]
    raw = arr["raw"]
    args = golden_args(meta)
    sig = torch_sigmoid_fn("cpu")
    # KeypointDecoder (reference decoders.py:345-423)
    kps = O.keypoint_decode(raw[:, :m], raw[:, m:m + n], raw[:, m + n:m + n + 2], meta["K"], meta["P"], meta["conf"],
                            meta["down_ratio"], args._r_labels, args._r_parts, sigmoid_fn=sig)
    assert listify(kps) == meta["keypoints"]
    # CoreMLDecoder (reference decoders.py:182-342): maps arrive already activated and suppressed
    a_pre = O.nms(O.clamped_sigmoid(raw[:, :m], sig))
    p_pre = O.nms(O.clamped_sigmoid(raw[:, m:m + n], sig))
    pk = O.decode_packed(a_pre, p_pre, raw[:, m + n:m + n + 2], raw[:, m + n + 2:], meta["K"], meta["P"], meta["conf"],
                         meta["dist"], pre_activated=True)
    np.testing.assert_array_equal(pk["anchor_inds"], arr["coreml_a_inds"])
    np.testing.assert_array_equal(pk["part_inds"], arr["coreml_p_inds"])
    objs = O.assemble(pk, args._r_labels, args._r_parts, args.anchor_name, meta["conf"], (w, h), (4 * w, 4 * h))
    assert listify(objs) == meta["coreml_annotation"]


@pytest.mark.parametrize("name", TIE_FREE)
def test_torch_port_matches_reference_golden(name):
    """The travelling torch port (CPU baseline / on-device checker) reproduces the reference too."""
    meta, arr = load_golden(name)
    b, m, n, h, w = meta["shape"]
    args = golden_args(meta)
    outs = split_outputs(torch.from_numpy(arr["raw"]), m, n)
    pk = TP.decode_tensors(outs, meta["K"], meta["P"], meta["conf"], meta["dist"])
    np.testing.assert_array_equal(pk["anchor_inds"].numpy(), arr["a_inds"])
    np.testing.assert_array_equal(pk["part_inds"].numpy(), arr["p_inds"])
    np.testing.assert_array_equal(pk["anchor_scores_masked"].numpy(), arr["a_scores_masked"])
    objs = TP.decode(outs, args._r_labels, args._r_parts, args.anchor_name, args.down_ratio, meta["K"], meta["P"],
                     meta["conf"], meta["dist"])
    assert listify(objs) == meta["annotation"]


def test_oracle_helpers_semantics():
    """Window is 5x5 with -inf padding, plateaus survive whole, k > H*W raises like torch.topk."""
    hm = np.zeros((1, 1, 8, 8), dtype=np.float32)
    hm[0, 0, 0, 2] = 0.6  # border peak survives (padding is -inf, SURVEY A.1)
    hm[0, 0, 1, 3] = 0.5  # within 2 px of it: suppressed
    out = O.nms(hm)
    assert out[0, 0, 0, 2] == np.float32(0.6) and out[0, 0, 1, 3] == 0
    flat = np.full((1, 1, 16, 16), 20.0, dtype=np.float32)  # saturated plateau: every member survives (A.2)
    assert (O.nms(O.clamped_sigmoid(flat)) == O.CLAMP_HI).all()
    with pytest.raises(RuntimeError):
        O.topk(hm, 65)
    # canonical tie rule: equal values come out in ascending index order, lower class first
    t = np.zeros((1, 2, 2, 4), dtype=np.float32)
    t[0, 1, 0, 1] = t[0, 0, 1, 2] = t[0, 0, 0, 3] = 0.7
    s, ind, cls, ys, xs = O.topk(t, 3)
    assert ind.tolist() == [[3, 6, 1]] and cls.tolist() == [[0.0, 0.0, 1.0]]
    # fp32 compare of `score > conf` (A.5): a score equal to float32(0.4) is NOT above 0.4
    assert not (np.float32(0.4) > np.float32(0.4))


@pytest.mark.parametrize("mode", ["noise", "blobs", "ladder"])
def test_oracle_matches_torch_port_off_the_golden_shapes(mode):
    """3 labels x 2 parts on 56x72 maps with K = 50, P = 60, a shape none of the stored vectors has: the oracle and the
    port of the reference's op sequence (both pinned to the reference's stored outputs above) return the same objects."""
    cfg = DecodeConfig("live", 2, 3, 2, 56, 72, 50, 60, cfg_id=77)
    raw = make_raw(cfg, mode)
    outs = split_outputs(raw, cfg.labels, cfg.parts)
    from tests.helpers import make_args

    args = make_args(cfg)
    port = TP.decode({k: v.clone() for k, v in outs.items()}, args._r_labels, args._r_parts, args.anchor_name,
                     args.down_ratio, cfg.max_objects, cfg.max_parts, cfg.conf_threshold, cfg.dist_thresh)
    pk = O.decode_packed(*np_inputs(outs), cfg.max_objects, cfg.max_parts, cfg.conf_threshold, cfg.dist_thresh,
                         sigmoid_fn=torch_sigmoid_fn("cpu"))
    objs = O.assemble(pk, args._r_labels, args._r_parts, args.anchor_name, cfg.conf_threshold,
                      (cfg.width, cfg.height), (4 * cfg.width, 4 * cfg.height))
    assert sum(len(o) for o in objs) > 0
    assert listify(port) == listify(objs)


@pytest.mark.parametrize("name", ["half_f16", "half_bf16"])
def test_oracle_reduced_precision_matches_reference_golden(name):
    """fp16 / bf16 inputs (the reference under --amp): scores sit on a coarse grid, so torch-CPU's
    unspecified tie order shuffles slots; what does not depend on it must match exactly -- the
    activated maps, the sorted score lists, and how many objects / parts each image yields."""
    meta, arr = load_golden(name)
    dtype = {"float16": torch.float16, "bfloat16": torch.bfloat16}[meta["dtype"]]
    b, m, n, h, w = meta["shape"]
    raw = arr["raw"]

    def act(x):  # the reference's clamped sigmoid in `dtype`, evaluated by torch on the CPU
        t = torch.from_numpy(np.ascontiguousarray(x)).to(dtype)
        return torch.clamp(torch.sigmoid(t), min=1e-6, max=1 - 1e-6).float().numpy()

    pk = O.decode_packed(raw[:, :m], raw[:, m:m + n], raw[:, m + n:m + n + 2], raw[:, m + n + 2:], meta["K"], meta["P"],
                         meta["conf"], meta["dist"], activation_fn=act,
                         conf_cmp=float(torch.tensor(meta["conf"], dtype=dtype)))
    np.testing.assert_array_equal(pk["anchor_sig"], arr["anchor_sig"])
    np.testing.assert_array_equal(pk["anchor_scores_masked"], arr["a_scores_masked"])
    np.testing.assert_array_equal(pk["part_scores_masked"], arr["p_scores_masked"])
    args = golden_args(meta)
    objs = O.assemble(pk, args._r_labels, args._r_parts, args.anchor_name, meta["conf"], (w, h), (4 * w, 4 * h))
    assert [len(o) for o in objs] == meta["objects_per_image"]
