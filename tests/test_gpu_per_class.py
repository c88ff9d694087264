"""-m gpu: per-class confidence thresholds through the decoder and the evaluator.

A table with every entry equal to t decodes bit for bit like the scalar t.  Tables whose valid slots are not a prefix
of the score order (a strict class next to a lenient one, thresholds at a detection's exact score) decode bit for bit
like the numpy oracle's decode with the same table (tests/per_class_oracle.py).  Objects, raw parts, metadata masks and
JSON follow its object loop; the evaluator follows ``oracle/evaluator_oracle.py``, and, label by label, the sweep's table at that label's
threshold.
"""
import json

import numpy as np
import pytest
import torch

from oracle import evaluator_oracle as EO
from oracle import sdnet_oracle as O
from oracle import torch_port as TP
from tests import per_class_oracle as PC
from structuredetector_b200 import CoreMLDecoder, Decoder, ops
from structuredetector_b200.evaluator import Evaluator, ThresholdSweep
from structuredetector_b200.synth import CONFIGS, DecodeConfig, make_raw, split_outputs
from tests.helpers import assert_packed_equal, make_args, packed_np, torch_sigmoid_fn
from tests.test_gpu_evaluator_limits import KINDS, LABELS, _annotations, _args, _ground_truth
from tests.test_gpu_limits import FAR_CASES, _device_activation, _far_raw

pytestmark = pytest.mark.gpu

# every packed field but `diag`, whose candidate counts depend on how the peaks kernel's units were scheduled
FIELDS = ("anchor_out", "part_out", "anchor_inds", "part_inds", "part_emb", "assign", "counts")


def _pre_activate(raw, m, n, device):
    raw = raw.clone()
    raw[:, :m + n] = TP.suppress(TP.activate(raw[:, :m + n].to(device)), 2).cpu()
    return raw


def _bits_equal(got, want, what):
    for key in FIELDS:
        g, w = got[key], want[key]
        if g.dtype == np.float32:
            g, w = g.view(np.uint32), w.view(np.uint32)
        np.testing.assert_array_equal(g, w, err_msg=f"{what}: {key}")


# ----------------------------------------------------------------------------------------------- equal table == scalar
@pytest.mark.parametrize("variant", ["fp32", "fp16", "bf16", "pre"])
@pytest.mark.parametrize("mode", ["blobs", "noise"])
@pytest.mark.parametrize("cfg", [CONFIGS["cfg3"], DecodeConfig("cfg5-128", 128, 2, 1, 512, 612, 100, 100, cfg_id=5)],
                         ids=["cfg3", "cfg5-128"])
def test_equal_table_is_the_scalar(cuda_device, cfg, mode, variant):
    m, n = cfg.labels, cfg.parts
    raw = make_raw(cfg, mode)
    if variant == "pre":
        raw = _pre_activate(raw, m, n, cuda_device)
    raw = raw.to({"fp16": torch.float16, "bf16": torch.bfloat16}.get(variant, torch.float32))
    outs = split_outputs(raw.to(cuda_device), m, n)
    for t in (0.4, 0.1, 0.7):
        kw = {"pre_activated": variant == "pre"}
        want = packed_np(ops.decode_packed(outs, cfg.max_objects, cfg.max_parts, t, cfg.dist_thresh, **kw))
        got = packed_np(ops.decode_packed(outs, cfg.max_objects, cfg.max_parts, [t] * (m + n), cfg.dist_thresh, **kw))
        _bits_equal(got, want, f"{cfg.name} {mode} {variant} t={t}")
        assert want["counts"].sum() > 0


# ----------------------------------------------------------------------------------------------- against the oracle
def _oracle(raw, m, n, k, p, table, dist, device, *, dtype=torch.float32, pre_activated=False):
    f = raw.float().cpu().numpy()
    planes = f[:, :m], f[:, m:m + n], f[:, m + n:m + n + 2], f[:, m + n + 2:]
    if pre_activated:
        kw = {"pre_activated": True}
    elif dtype == torch.float32:
        kw = {"sigmoid_fn": torch_sigmoid_fn(device)}
    else:
        kw = {"activation_fn": _device_activation(dtype, device)}
    conf_class = [ops._f32(v, dtype) for v in table]
    return PC.decode_packed(*planes, k, p, conf_class, dist, **kw)


def _check(raw, m, n, k, p, table, device, *, dist=0.1, what="", non_prefix=True, **kw):
    outs = split_outputs(raw.to(device), m, n)
    got = packed_np(ops.decode_packed(outs, k, p, table, dist, **kw))
    want = _oracle(raw, m, n, k, p, table, dist, device, dtype=raw.dtype, pre_activated=kw.get("pre_activated", False))
    assert_packed_equal(got, want, what=what)
    if non_prefix:  # some image has a masked slot ahead of a valid one
        a_mask = want["anchor_scores_masked"] >= 0
        p_mask = want["part_scores_masked"] >= 0
        gaps = lambda mask: [(~mask[b, : np.flatnonzero(mask[b])[-1]]).any() if mask[b].any() else False
                             for b in range(mask.shape[0])]
        assert any(gaps(a_mask)) or any(gaps(p_mask)), f"{what}: the valid slots are a prefix"
    return got, want


@pytest.mark.parametrize("variant", ["fp32", "fp16", "bf16", "pre"])
@pytest.mark.parametrize("mode", ["blobs", "noise"])
def test_strict_and_lenient_classes(cuda_device, mode, variant):
    cfg = DecodeConfig("pc", 4, 3, 2, 128, 152, 100, 100, cfg_id=60)
    raw = make_raw(cfg, mode, seed=600 + len(mode))
    if variant == "pre":
        raw = _pre_activate(raw, 3, 2, cuda_device)
    raw = raw.to({"fp16": torch.float16, "bf16": torch.bfloat16}.get(variant, torch.float32))
    for table in ([0.99, 0.05, 0.4, 0.05, 0.99], [0.05, 0.99, 0.3, 0.6, 0.1]):
        _check(raw, 3, 2, 100, 100, table, cuda_device, what=f"{mode} {variant} {table}", pre_activated=variant == "pre")


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16], ids=["fp32", "fp16"])
def test_thresholds_at_a_score_and_the_next_value(cuda_device, dtype):
    """Each class's threshold exactly at one of its detections' scores, then at the next value of the maps' dtype."""
    cfg = DecodeConfig("pc-at", 2, 2, 1, 128, 152, 100, 100, cfg_id=61)
    raw = make_raw(cfg, "blobs", seed=610).to(dtype)
    pk = packed_np(ops.decode_packed(split_outputs(raw.to(cuda_device), 2, 1), 100, 100, 0.05, 0.1))
    at = []
    for rows, c in ((pk["anchor_out"][0], 0), (pk["anchor_out"][0], 1), (pk["part_out"][0], 0)):
        scores = rows[(rows[:, 3] == c) & (rows[:, 2] > 0.1), 2]
        at.append(float(scores[len(scores) // 2]))
    step = lambda v: float(torch.tensor(v, dtype=dtype).view(torch.int16 if dtype == torch.float16 else torch.int32).add(1)
                           .view(dtype))
    for name, table in (("at", at), ("next", [step(v) for v in at]), ("mixed", [at[0], step(at[1]), 0.99])):
        _check(raw, 2, 1, 100, 100, table, cuda_device, what=f"{dtype} {name}", non_prefix=False)


def test_every_anchor_class_above_one(cuda_device):
    cfg = DecodeConfig("pc-none", 2, 2, 1, 128, 152, 100, 100, cfg_id=62)
    raw = make_raw(cfg, "noise", seed=620)
    got, _ = _check(raw, 2, 1, 100, 100, [1.5, 2.0, 0.2], cuda_device, what="no anchor", non_prefix=False)
    assert (got["counts"][:, 0] == 0).all() and (got["counts"][:, 1] > 0).all() and (got["assign"] == -1).all()


def test_k_and_p_1024(cuda_device):
    cfg = DecodeConfig("pc-1024", 2, 3, 2, 128, 128, 1024, 1024, cfg_id=63)
    raw = make_raw(cfg, "noise", seed=630)
    for table in ([0.9, 0.05, 0.5, 0.2, 0.95], [0.3, 0.7, 0.99, 0.9, 0.05]):
        _check(raw, 3, 2, 1024, 1024, table, cuda_device, what=f"K=P=1024 {table}")


@pytest.mark.parametrize("case", FAR_CASES)
def test_full_grouping_search(cuda_device, case):
    """The far-coordinate and huge-gate cases: with per-class thresholds the masked slots are no longer the tail of the
    slot order, and the full search covers them wherever they are."""
    raw, dist = _far_raw(case)
    table = [0.05, 0.99, 0.3]  # the far anchor peak is of class 0
    _check(raw, 2, 1, 100, 100, table, cuda_device, dist=dist, what=case)


@pytest.mark.parametrize("m,n", [(200, 55), (254, 1), (1, 254)])
def test_channel_limit(cuda_device, m, n):
    cfg = DecodeConfig("pc-channels", 1, m, n, 32, 40, 64, 64, cfg_id=64)
    raw = make_raw(cfg, "noise", seed=640 + m)
    table = np.random.default_rng(m).uniform(0.05, 0.95, m + n).tolist()
    # the classes of the top anchor and the top part admit nothing: the valid slots cannot be a prefix
    pk = packed_np(ops.decode_packed(split_outputs(raw.to(cuda_device), m, n), 64, 64, 0.05, 0.1))
    table[int(pk["anchor_out"][0, 0, 3])] = 1.5
    table[m + int(pk["part_out"][0, 0, 3])] = 1.5
    _check(raw, m, n, 64, 64, table, cuda_device, what=f"M={m} N={n}")


def test_pinned_host_inputs(cuda_device):
    cfg = DecodeConfig("pc-host", 2, 2, 1, 128, 152, 100, 100, cfg_id=65)
    raw = make_raw(cfg, "blobs", seed=650)
    table = [0.99, 0.05, 0.3]
    dev = packed_np(ops.decode_packed(split_outputs(raw.to(cuda_device), 2, 1), 100, 100, table, 0.1))
    host = packed_np(ops.decode_packed(split_outputs(raw.pin_memory(), 2, 1), 100, 100, table, 0.1))
    _bits_equal(host, dev, "pinned host")


def test_plan_and_pipeline_take_the_table(cuda_device):
    cfg = DecodeConfig("pc-plan", 2, 2, 1, 128, 152, 100, 100, cfg_id=66)
    raw = make_raw(cfg, "noise", seed=660).to(cuda_device)
    outs = split_outputs(raw, 2, 1)
    table = [0.99, 0.05, 0.3]
    want = packed_np(ops.decode_packed(outs, 100, 100, table, 0.1))
    conf_class = torch.tensor(table, dtype=torch.float32, device=cuda_device)
    dist = ops._f32(0.1 * 128)
    args = (outs["anchor_hm"], outs["part_hm"], outs["offsets"], outs["embeddings"], 0.0, dist)
    plan = ops.DecodePlan(cuda_device, 2, 2, 1, 128, 152, 100, 100)
    _bits_equal(packed_np(plan.run(*args, conf_class=conf_class)), want, "DecodePlan.run")
    assert len(plan.run_timed(*args, conf_class=conf_class)) == 3
    _bits_equal(packed_np(plan.out), want, "DecodePlan.run_timed")
    pipe = ops.DecodePipeline.for_shape(cuda_device, 2, 2, 2, 1, 128, 152, 100, 100)
    out, event = pipe.submit(*args, conf_class=conf_class)
    event.synchronize()
    _bits_equal(packed_np(out), want, "DecodePipeline.submit")
    with pytest.raises(ValueError):
        plan.run(*args, conf_class=conf_class[:2])
    with pytest.raises(ValueError):
        plan.run(*args, conf_class=conf_class.double())


# ----------------------------------------------------------------------------------------------- objects
@pytest.mark.parametrize("pre", [False, True], ids=["Decoder", "CoreMLDecoder"])
def test_decoder_objects_with_a_name_mapping(cuda_device, tmp_path, pre):
    cfg = CONFIGS["cfg3"]
    raw = make_raw(cfg, "blobs")[:4]
    if pre:
        raw = _pre_activate(raw, 2, 1, cuda_device)
    args = make_args(cfg)  # bean, maize / leaf
    mapping = {"bean": 0.9, "leaf": 0.2}  # maize takes args.conf_threshold
    table = [0.9, args.conf_threshold, 0.2]
    dec = (CoreMLDecoder if pre else Decoder)(args)
    outs = split_outputs(raw.to(cuda_device), 2, 1)
    meta = dec(outs, conf_thresh=mapping, return_metadata=True)
    pk = _oracle(raw, 2, 1, 100, 100, table, cfg.dist_thresh, cuda_device, pre_activated=pre)
    out_size, in_size = (cfg.width, cfg.height), (4 * cfg.width, 4 * cfg.height)
    labels, kinds = {0: "bean", 1: "maize"}, {0: "leaf"}
    want = PC.assemble(pk, labels, kinds, "stem", table[:2], out_size, in_size)
    got = [[(o.name, (o.anchor.kind, o.anchor.x, o.anchor.y, o.anchor.score), [(k.kind, k.x, k.y, k.score) for k in o.parts])
            for o in ann.objects] for ann in meta["annotation"]]
    assert got == want
    assert any(want)
    raw_parts = PC.raw_parts(pk, kinds, table[2:], out_size, in_size)
    assert [[(k.kind, k.x, k.y, k.score) for k in img] for img in meta["raw_parts"]] == raw_parts
    a_scores = meta["topk_anchor"][0].cpu().numpy()
    p_scores = meta["topk_kp"][0].cpu().numpy()
    a_conf = np.float32(table)[pk["anchor_out"][..., 3].astype(int)]
    p_conf = np.float32(table)[2 + pk["part_out"][..., 3].astype(int)]
    np.testing.assert_array_equal(a_scores, np.where(pk["anchor_out"][..., 2] > a_conf, pk["anchor_out"][..., 2], -1.0))
    np.testing.assert_array_equal(p_scores, np.where(pk["part_out"][..., 2] > p_conf, pk["part_out"][..., 2], -1.0))
    texts = dec.detections_json(outs, conf_thresh=mapping)
    assert texts == [json.dumps(ann.json_repr(), indent=2) for ann in meta["annotation"]]
    saved = dec.save_detections_json(outs, tmp_path, conf_thresh=mapping)
    assert saved == texts and (tmp_path / "batch_0.json").read_text() == texts[0]
    # the same decode under the equal table and the scalar
    scalar = dec(outs, conf_thresh=0.4)
    equal = dec(outs, conf_thresh={"bean": 0.4, "maize": 0.4, "leaf": 0.4})
    assert [[(o.name, o.anchor.x, o.anchor.score, len(o.parts)) for o in a.objects] for a in scalar] == \
        [[(o.name, o.anchor.x, o.anchor.score, len(o.parts)) for o in a.objects] for a in equal]


# ----------------------------------------------------------------------------------------------- evaluator
def _oracle_tables(pk, gts, img_sizes, args, out_size, table):
    """The evaluator oracle on the oracle's objects and raw parts under per-class thresholds (labels, then kinds)."""
    label_map = {i: name for name, i in args.labels.items()}
    part_map = {i: name for name, i in args.parts.items()}
    M = len(label_map)
    in_size = (int(args.down_ratio * out_size[0]), int(args.down_ratio * out_size[1]))
    objs = PC.assemble(pk, label_map, part_map, "stem", table[:M], out_size, in_size)
    raw_parts = PC.raw_parts(pk, part_map, table[M:], out_size, in_size)
    labels, kinds = list(args.labels), list(args.parts)
    net = (args.width, args.height)
    tables = {"anchor": {l: [0, 0, 0, []] for l in labels}, "part": {k: [0, 0, 0, []] for k in kinds},
              "csi": {l: [0, 0, 0, []] for l in labels}, "classification": {l: [0, 0, 0, []] for l in EO.CLASSIFICATION_LABELS}}
    for b, (gt, size) in enumerate(zip(gts, img_sizes)):
        loc = EO.evaluate_image([(name, a[1], a[2], a[3]) for name, a, _ in objs[b]], raw_parts[b], gt, size, net,
                                args.dist_threshold, labels, kinds)
        rx, ry = size[0] / net[0], size[1] / net[1]
        thresh, norm = min(size) * args.dist_threshold, min(size)
        preds = [(name, a[1] * rx, a[2] * ry, a[3], [(k[0], k[1] * rx, k[2] * ry, k[3]) for k in kps]) for name, a, kps in objs[b]]
        g = [(name, x * rx, y * ry, [(k, px * rx, py * ry) for k, px, py in kps]) for name, x, y, kps in gt]
        for key, res in (("anchor", loc["anchor"]), ("part", loc["part"]),
                         ("csi", EO.eval_csi_image(preds, g, labels, thresh, args.csi_threshold)),
                         ("classification", EO.eval_classif_image(preds, g, thresh, norm))):
            for label, (tp, npos, ndet, acc) in res.items():
                t = tables[key][label]
                t[0], t[1], t[2] = t[0] + tp, t[1] + npos, t[2] + ndet
                t[3] += acc
    return tables


def _batch(cfg, device, seed):
    """Maps, ground truth derived from their detections, args (LABELS / KINDS), out_size."""
    raw = make_raw(cfg, "noise" if cfg.max_objects > 200 else "blobs", seed=seed)
    outs = split_outputs(raw.to(device), cfg.labels, cfg.parts)
    out_size = (cfg.width, cfg.height)
    labels = dict(list(LABELS.items())[: cfg.labels])
    args = _args(out_size, 0.02, labels=labels)
    pk = packed_np(ops.decode_packed(outs, cfg.max_objects, cfg.max_parts, 0.2, cfg.dist_thresh))
    objs = O.assemble(pk, {i: n for n, i in labels.items()}, {i: k for k, i in KINDS.items()}, "stem", 0.2, out_size,
                      (4 * cfg.width, 4 * cfg.height))
    rng = np.random.default_rng(seed)
    gts = [[g for g in _ground_truth(o, rng) if g[0] in labels] for o in objs]
    sizes = [(2448, 2048) if b % 2 else (1296, 1536) for b in range(len(gts))]
    return outs, gts, sizes, args, out_size


def test_evaluator_with_a_name_mapping_against_the_oracle(cuda_device):
    cfg = DecodeConfig("pc-eval", 4, 3, 2, 128, 152, 100, 100, cfg_id=67)
    outs, gts, sizes, args, out_size = _batch(cfg, cuda_device, 670)
    mapping = {"bean": 0.6, "weed": 0.15, "leaf": 0.5, "flower": 0.1}  # maize takes args.conf_threshold
    table = [0.6, args.conf_threshold, 0.15, 0.5, 0.1]
    packed = ops.decode_packed(outs, 100, 100, table, cfg.dist_thresh)
    ev = Evaluator(args)
    ev.accumulate_packed(packed, _annotations(gts, sizes), out_size, conf_thresh=mapping, eval_csi=True, eval_classif=True)
    want = _oracle_tables(packed_np(packed), gts, sizes, args, out_size, table)
    got = {"anchor": ev.anchor_eval, "part": ev.part_eval, "csi": ev.csi_eval, "classification": ev.classification_eval}
    for key, tab in want.items():
        for label, (tp, npos, ndet, acc) in tab.items():
            g = got[key][label]
            assert (g.tp, g.npos, g.ndet) == (tp, npos, ndet), (key, label)
            np.testing.assert_allclose(g.acc, acc, rtol=1e-9, atol=0, err_msg=f"{key} {label}")
    assert ev.anchor_eval.reduce().tp > 0 and ev.csi_eval.reduce().tp > 0
    # the equal mapping is the scalar
    scalar, equal = Evaluator(args), Evaluator(args)
    pk = ops.decode_packed(outs, 100, 100, 0.35, cfg.dist_thresh)
    scalar.accumulate_packed(pk, _annotations(gts, sizes), out_size, conf_thresh=0.35, eval_csi=True, eval_classif=True)
    equal.accumulate_packed(pk, _annotations(gts, sizes), out_size, conf_thresh={n: 0.35 for n in (*LABELS, *KINDS)},
                            eval_csi=True, eval_classif=True)
    for table_name in ("anchor_eval", "part_eval", "csi_eval", "classification_eval"):
        for label, e in getattr(scalar, table_name).items():
            o = getattr(equal, table_name)[label]
            assert (o.tp, o.npos, o.ndet, o.acc) == (e.tp, e.npos, e.ndet, e.acc), (table_name, label)


@pytest.mark.parametrize("cfg", [DecodeConfig("pc-link", 4, 3, 2, 128, 152, 100, 100, cfg_id=68),
                                 DecodeConfig("pc-link-dense", 2, 3, 2, 128, 128, 500, 500, cfg_id=69)],
                         ids=["blobs", "noise-500"])
def test_sweep_best_thresholds_decode_to_the_sweep_tables(cuda_device, cfg):
    """Decode at best_thresholds() of a sweep: label by label, the per-class Evaluator's location tables are the sweep's
    at that label's threshold."""
    outs, gts, sizes, args, out_size = _batch(cfg, cuda_device, 680 + cfg.cfg_id)
    anns = _annotations(gts, sizes)
    grid = [round(0.05 * i, 2) for i in range(1, 20)]
    sweep = ThresholdSweep(args, grid, dist_thresh=cfg.dist_thresh)
    sweep.accumulate_packed(ops.decode_packed(outs, cfg.max_objects, cfg.max_parts, 0.5, cfg.dist_thresh), anns, out_size)
    best = sweep.best_thresholds()
    assert set(best) == set(args.labels) | set(args.parts)
    table = ops.class_thresholds(best, list(args.labels), list(args.parts), args.conf_threshold)
    packed = ops.decode_packed(outs, cfg.max_objects, cfg.max_parts, table, cfg.dist_thresh)
    ev = Evaluator(args)
    ev.accumulate_packed(packed, anns, out_size, conf_thresh=best)
    for attr, names in (("anchor_eval", args.labels), ("part_eval", args.parts)):
        for name in names:
            got, want = getattr(ev, attr)[name], getattr(sweep.at(best[name]), attr)[name]
            assert (got.tp, got.npos, got.ndet) == (want.tp, want.npos, want.ndet), (attr, name, best[name])
            assert got.acc == want.acc, (attr, name)


def test_more_decoded_classes_than_labels(cuda_device):
    """Maps with 3 classes and 2 kinds evaluated with 2 labels and 1 kind under a mapping: the matchers read no table
    entry for the other classes (they compare against args.conf_threshold) and the labels' tables are the scalar
    evaluator's at each label's threshold."""
    cfg = DecodeConfig("pc-extra", 2, 3, 2, 64, 80, 60, 60, cfg_id=48)
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
    mapping = {"bean": 0.6, "maize": 0.2, "leaf": 0.45}
    packed = ops.decode_packed(outs, 60, 60, [0.6, 0.2, 0.9, 0.45, 0.05], 0.1)
    ev = Evaluator(args)
    ev.accumulate_packed(packed, anns, out_size, conf_thresh=mapping, eval_csi=True, eval_classif=True)
    for attr, name in (("anchor_eval", "bean"), ("anchor_eval", "maize"), ("part_eval", "leaf")):
        want = Evaluator(args)
        t = mapping[name]
        want.accumulate_packed(ops.decode_packed(outs, 60, 60, t, 0.1), anns, out_size, conf_thresh=t)
        g, w = getattr(ev, attr)[name], getattr(want, attr)[name]
        assert (g.tp, g.npos, g.ndet, g.acc) == (w.tp, w.npos, w.ndet, w.acc), (attr, name)
