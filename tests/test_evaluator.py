"""Evaluator matching (SURVEY 8f-4): the CPU restatement against the reference's golden output (CPU),
the CUDA kernel against both (GPU)."""
import json
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import evaluator_oracle as EO

GOLDEN = Path(__file__).parent / "golden"
INDEX = json.loads((GOLDEN / "index.json").read_text())
EVAL = json.loads((GOLDEN / "eval.json").read_text())
EVAL_OBJECTS = json.loads((GOLDEN / "eval_objects.json").read_text())  # eval_csi + eval_classif of the same cases


def _names(name):
    _, m, n, _, _ = INDEX[name]["shape"]
    return [f"label{i}" for i in range(m)], [f"part{i}" for i in range(n)]


@pytest.mark.parametrize("name", sorted(EVAL))
def test_oracle_reproduces_reference_evaluator(name):
    labels, kinds = _names(name)
    got = EO.evaluate_batch(INDEX[name]["annotation"], INDEX[name]["raw_parts"], EVAL[name], labels, kinds)
    for key in ("anchor", "part"):
        for label, want in EVAL[name]["result"][key].items():
            tp, npos, ndet, acc = got[key][label]
            assert (tp, npos, ndet) == (want["tp"], want["npos"], want["ndet"]), (name, key, label)
            assert acc == want["acc"], (name, key, label)  # same Python-float arithmetic: bit-exact


def _object_case(name):
    """eval.json's ground truth + eval_objects.json's thresholds and expected CSI / classification tables."""
    return {**EVAL[name], "csi_threshold": EVAL_OBJECTS[name]["csi_threshold"]}, EVAL_OBJECTS[name]


@pytest.mark.parametrize("name", sorted(EVAL_OBJECTS))
def test_oracle_reproduces_reference_object_metrics(name):
    """eval_csi / compute_csi / eval_classif (evaluator.py:380-474, 539-581) restated, against what the reference's own
    Evaluator.accumulate(..., True, True) produced: counts and every accumulated value bit for bit."""
    case, want = _object_case(name)
    labels, _ = _names(name)
    got = EO.evaluate_objects_batch(INDEX[name]["annotation"], case, labels, rename=want["rename"])
    for key in ("csi", "classification"):
        for label, w in want["result"][key].items():
            tp, npos, ndet, acc = got[key][label]
            assert (tp, npos, ndet) == (w["tp"], w["npos"], w["ndet"]), (name, key, label)
            assert acc == w["acc"], (name, key, label)


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(EVAL_OBJECTS))
def test_cuda_object_matching_reproduces_reference_evaluator(cuda_device, name):
    """sdnet_match_objects_launch on the packed detections against the reference's Decoder + Evaluator on CPU:
    counts exact, CSI values exact ratios of small integers, localisation errors to 1e-9 relative."""
    from structuredetector_b200 import ImageAnnotation, Keypoint, Object, ops
    from structuredetector_b200.evaluator import Evaluator
    from structuredetector_b200.synth import split_outputs
    meta = INDEX[name]
    case, want = _object_case(name)
    rename = want["rename"]
    _, m, n, h, w = meta["shape"]
    labels, kinds = _names(name)
    labels = [rename.get(l, l) for l in labels]
    raw = torch.from_numpy(np.load(GOLDEN / f"{name}.npz")["raw"]).to(cuda_device)
    packed = ops.decode_packed(split_outputs(raw, m, n), meta["K"], meta["P"], meta["conf"], meta["dist"])
    args = SimpleNamespace(labels={l: i for i, l in enumerate(labels)}, parts={k: i for i, k in enumerate(kinds)},
                           width=case["width"], height=case["height"], dist_threshold=case["dist_threshold"],
                           conf_threshold=meta["conf"], down_ratio=meta["down_ratio"], csi_threshold=case["csi_threshold"])
    anns = []
    for image in case["images"]:
        objs = [Object(rename.get(nm, nm), Keypoint("stem", x, y), [Keypoint(k, px, py) for k, px, py in kps]) for nm, x, y, kps in image["gt"]]
        anns.append(ImageAnnotation("gt", objs, img_size=tuple(image["img_size"])))
    ev = Evaluator(args)
    ev.accumulate_packed(packed, anns, (w, h), eval_csi=True, eval_classif=True)
    for key, evals in (("csi", ev.csi_eval), ("classification", ev.classification_eval)):
        assert set(evals.labels) == set(want["result"][key])
        for label, wnt in want["result"][key].items():
            got = evals[label]
            assert (got.tp, got.npos, got.ndet) == (wnt["tp"], wnt["npos"], wnt["ndet"]), (name, key, label)
            np.testing.assert_allclose(got.acc, wnt["acc"], rtol=1e-9, atol=0)
    # the location tables are unaffected by the extra flags
    for key, evals in (("anchor", ev.anchor_eval), ("part", ev.part_eval)):
        for label, wnt in EVAL[name]["result"][key].items():
            label = rename.get(label, label)
            assert (evals[label].tp, evals[label].npos, evals[label].ndet) == (wnt["tp"], wnt["npos"], wnt["ndet"])
    assert "CSI" in repr(ev) and "Classification" in repr(ev)


def _annotations(case):
    from structuredetector_b200 import ImageAnnotation, Keypoint, Object
    anns = []
    for image in case["images"]:
        objs = [Object(name, Keypoint("stem", x, y), [Keypoint(k, px, py) for k, px, py in kps]) for name, x, y, kps in image["gt"]]
        anns.append(ImageAnnotation("gt", objs, img_size=tuple(image["img_size"])))
    return anns


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(EVAL))
def test_cuda_matching_reproduces_reference_evaluator(cuda_device, name):
    """Decode the stored raw input on the GPU, match on the GPU, compare with what the reference's
    Decoder + Evaluator produced on CPU: counts exact; localisation errors to 1e-9 relative (positions are
    bit-identical fp32, the distance is a double hypot on both sides)."""
    from structuredetector_b200 import ops
    from structuredetector_b200.evaluator import Evaluator
    from structuredetector_b200.synth import split_outputs
    meta, case = INDEX[name], EVAL[name]
    _, m, n, h, w = meta["shape"]
    labels, kinds = _names(name)
    raw = torch.from_numpy(np.load(GOLDEN / f"{name}.npz")["raw"]).to(cuda_device)
    packed = ops.decode_packed(split_outputs(raw, m, n), meta["K"], meta["P"], meta["conf"], meta["dist"])
    args = SimpleNamespace(labels={l: i for i, l in enumerate(labels)}, parts={k: i for i, k in enumerate(kinds)},
                           width=case["width"], height=case["height"], dist_threshold=case["dist_threshold"],
                           conf_threshold=meta["conf"], down_ratio=meta["down_ratio"])
    ev = Evaluator(args)
    ev.accumulate_packed(packed, _annotations(case), (w, h))
    for key, evals in (("anchor", ev.anchor_eval), ("part", ev.part_eval)):
        for label, want in case["result"][key].items():
            got = evals[label]
            assert (got.tp, got.npos, got.ndet) == (want["tp"], want["npos"], want["ndet"]), (name, key, label)
            np.testing.assert_allclose(got.acc, want["acc"], rtol=1e-9, atol=0)
    # formulas of Evaluation (evaluator.py:40-75)
    total = ev.kps_eval.reduce()
    assert total.tp == sum(r["tp"] for k in ("anchor", "part") for r in case["result"][k].values())
    assert 0.0 <= total.f1_score <= 1.0 and 0.0 <= total.recall <= 1.0


@pytest.mark.gpu
def test_cuda_matching_against_oracle_on_dense_batch(cuda_device):
    """cfg2-sized noise batch with seeded ground truth: the kernel against the CPU restatement."""
    from structuredetector_b200 import Decoder, ImageAnnotation, Keypoint, Object, ops
    from structuredetector_b200.evaluator import Evaluator
    from structuredetector_b200.synth import CONFIGS, make_raw, split_outputs
    from tests.helpers import make_args
    cfg = CONFIGS["cfg2"]
    raw = make_raw(cfg, "noise", batch=6).to(cuda_device)
    outs = split_outputs(raw, cfg.labels, cfg.parts)
    dargs = make_args(cfg)
    meta = Decoder(dargs)(outs, return_metadata=True)
    packed = ops.decode_packed(outs, cfg.max_objects, cfg.max_parts, cfg.conf_threshold, cfg.dist_thresh)
    labels, kinds = list(dargs._r_labels.values()), list(dargs._r_parts.values())
    rng = np.random.default_rng(11)
    anns, plain_gt = [], []
    for ann in meta["annotation"]:
        objs = []
        for o in ann.objects:
            if rng.random() < 0.7:
                kps = [Keypoint(p.kind, p.x + rng.normal(0, 3), p.y + rng.normal(0, 3)) for p in o.parts if rng.random() < 0.7]
                objs.append(Object(o.name, Keypoint("a", o.anchor.x + rng.normal(0, 4), o.anchor.y + rng.normal(0, 4)), kps))
        anns.append(ImageAnnotation("gt", objs, img_size=(1931, 1297)))
        plain_gt.append([(o.name, o.anchor.x, o.anchor.y, [(p.kind, p.x, p.y) for p in o.parts]) for o in objs])
    args = SimpleNamespace(labels={l: i for i, l in enumerate(labels)}, parts={k: i for i, k in enumerate(kinds)},
                           width=4 * cfg.width, height=4 * cfg.height, dist_threshold=0.02,
                           conf_threshold=cfg.conf_threshold, down_ratio=4.0)
    ev = Evaluator(args)
    ev.accumulate_packed(packed, anns, (cfg.width, cfg.height))
    want = {"anchor": {l: [0, 0, 0, []] for l in labels}, "part": {k: [0, 0, 0, []] for k in kinds}}
    for ann, raw_parts, gts in zip(meta["annotation"], meta["raw_parts"], plain_gt):
        res = EO.evaluate_image([(o.name, o.anchor.x, o.anchor.y, o.anchor.score) for o in ann.objects],
                                [(p.kind, p.x, p.y, p.score) for p in raw_parts], gts, (1931, 1297),
                                (args.width, args.height), args.dist_threshold, labels, kinds)
        for key in want:
            for label, (tp, npos, ndet, acc) in res[key].items():
                t = want[key][label]
                t[0] += tp; t[1] += npos; t[2] += ndet; t[3] += acc
    for key, evals in (("anchor", ev.anchor_eval), ("part", ev.part_eval)):
        for label, (tp, npos, ndet, acc) in want[key].items():
            got = evals[label]
            assert (got.tp, got.npos, got.ndet) == (tp, npos, ndet), (key, label)
            np.testing.assert_allclose(got.acc, acc, rtol=1e-9, atol=0)
    assert ev.anchor_eval.reduce().tp > 50 and ev.part_eval.reduce().tp > 50


def test_evaluation_classes_mirror_the_reference_formulas():
    """Evaluation / Evaluations (evaluator.py:13-206): counters, derived metrics, +, |, reduce -- against
    fixed expectations and, where the reference is importable, against its own classes."""
    from structuredetector_b200.evaluator import Evaluation, Evaluations
    a = Evaluation(tp=3, npos=5, ndet=4, acc=[0.01, 0.02, 0.03])
    assert (a.fp, a.fn) == (1, 2) and a.precision == 0.75 and a.recall == 0.6
    assert a.f1_score == pytest.approx(2 * 3 / 9) and a.csi == pytest.approx(3 / 6)
    assert a.avg_acc == pytest.approx(0.02) and a.acc_err == pytest.approx(np.std([0.01, 0.02, 0.03]) / np.sqrt(3))
    empty = Evaluation()
    assert (empty.precision, empty.recall, empty.f1_score, empty.csi) == (1, 1, 1, 1) and np.isnan(empty.avg_acc)
    assert Evaluation(tp=0, npos=0, ndet=2).precision == 0 and Evaluation(tp=0, npos=2, ndet=0).recall == 0
    with pytest.raises(AssertionError):
        Evaluation(tp=2, npos=1, ndet=2)
    total = a + Evaluation(tp=1, npos=1, ndet=2, acc=[0.5])
    assert (total.tp, total.npos, total.ndet, total.acc) == (4, 6, 6, [0.01, 0.02, 0.03, 0.5]) and a.tp == 3
    x, y = Evaluations(["l0", "l1"]), Evaluations(["l0", "l1"])
    x["l0"] += a
    y["l1"] += Evaluation(tp=1, npos=2, ndet=1, acc=[0.1])
    both = x + y
    assert (both["l0"].tp, both["l1"].tp, both.reduce().npos) == (3, 1, 7) and len(both) == 2
    parts = Evaluations(["p0"])
    parts["p0"] += Evaluation(tp=2, npos=2, ndet=3, acc=[0.2, 0.3])
    merged = both | parts
    assert set(merged.labels) == {"l0", "l1", "p0"} and merged.reduce().tp == 6
    acc = Evaluations(["l0"])
    acc["l0"] += Evaluation(tp=1, npos=1, ndet=1, acc=[0.4])
    acc |= both          # in-place union: shared labels summed, new ones adopted (evaluator.py:180-185)
    assert set(acc.labels) == {"l0", "l1"} and acc["l0"].tp == 4 and acc["l1"].tp == 1
    assert [c if isinstance(c, str) else c.header for c in Evaluation.columns()] == list(Evaluation.COLUMNS)
    ref_src = Path("/root/reference/src")
    if ref_src.exists():
        import sys
        sys.dont_write_bytecode = True
        sys.path.insert(0, str(ref_src))
        try:
            from sdnet.model.evaluator import Evaluation as RefEvaluation
        finally:
            sys.path.remove(str(ref_src))
        rng = np.random.default_rng(3)
        for _ in range(50):
            npos, ndet = int(rng.integers(0, 20)), int(rng.integers(0, 20))
            tp = int(rng.integers(0, min(npos, ndet) + 1))
            acc = rng.random(tp).tolist()
            ours, ref = Evaluation(tp, npos, ndet, list(acc)), RefEvaluation(tp, npos, ndet, list(acc))
            for name in ("fp", "fn", "csi", "precision", "recall", "f1_score"):
                assert getattr(ours, name) == getattr(ref, name), name
            if tp:
                assert ours.avg_acc == ref.avg_acc and ours.acc_err == ref.acc_err
            assert ours.stats() == ref.stats() and repr(ours) == repr(ref)


def test_ground_truth_packing_host_logic():
    """Evaluator._pack_ground_truth: row layout, unknown labels (-1, never matched or counted), per-image
    scale rows (evaluator.py:245-250), and the SDNET_MAX_GT limit.  Host only: loads the library, no launch."""
    from structuredetector_b200 import ImageAnnotation, Keypoint, Object, _native
    from structuredetector_b200.evaluator import Evaluator
    args = SimpleNamespace(labels={"maize": 0, "bean": 1}, parts={"leaf": 0}, width=512, height=256, dist_threshold=0.05,
                           conf_threshold=0.4, down_ratio=4.0)
    ev = Evaluator(args)
    anns = [
        ImageAnnotation("a", [Object("bean", Keypoint("stem", 10.0, 20.0), [Keypoint("leaf", 1.0, 2.0), Keypoint("leaf", 3.0, 4.0)]),
                              Object("weed", Keypoint("stem", 5.0, 6.0), [Keypoint("flower", 7.0, 8.0)])], img_size=(2048, 1024)),
        ImageAnnotation("b", [], img_size=(1000, 3000)),
    ]
    (gt_a, n_a, wa), (gt_p, n_p, wp), scale, owner = ev._pack_ground_truth(anns, torch.device("cpu"))
    assert owner.tolist() == [[0, 0, 1], [0, 0, 0]]  # object index of every ground-truth part (object order)
    assert (wa, wp) == (2, 3) and n_a.tolist() == [2, 0] and n_p.tolist() == [3, 0]
    assert gt_a[0].tolist() == [[10.0, 20.0, 1.0], [5.0, 6.0, -1.0]]
    assert gt_p[0].tolist() == [[1.0, 2.0, 0.0], [3.0, 4.0, 0.0], [7.0, 8.0, -1.0]]
    assert scale[0].tolist() == [2048 / 512, 1024 / 256, 1024 * 0.05, 1024.0]
    assert scale[1].tolist() == [1000 / 512, 3000 / 256, 1000 * 0.05, 1000.0]
    crowd = ImageAnnotation("c", [Object("bean", Keypoint("stem", 0.0, 0.0)) for _ in range(_native.MAX_GT + 1)], img_size=(10, 10))
    with pytest.raises(ValueError):
        ev._pack_ground_truth([crowd], torch.device("cpu"))
