"""-m gpu: the evaluator's matchers (sdnet_match_kernel, sdnet_match_objects_kernel) at their limits -- K = P = 1024,
1024 ground-truth points in one image, a 64-part ground-truth object -- and at their comparison boundaries: location
matching keeps a distance `< thresh`, classification `<= thresh`, CSI `>= csi_threshold`; the first nearest (or best)
ground truth in annotation order wins; objects need score `> conf`, raw parts score `>= conf`.

Every case goes through ``Evaluator.accumulate_packed(..., eval_csi=True, eval_classif=True)`` and is compared with
``oracle/evaluator_oracle.py`` on the objects ``oracle.sdnet_oracle.assemble`` builds from the same packed detections:
counts exactly, accumulated values to 1e-9 relative -- exactly where every offset is axis-aligned, so that ``hypot``
is exact.
"""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import evaluator_oracle as EO
from oracle import sdnet_oracle as O
from structuredetector_b200 import ImageAnnotation, Keypoint, Object, ops
from structuredetector_b200.evaluator import Evaluator
from structuredetector_b200.synth import DecodeConfig, make_raw, split_outputs
from tests.helpers import assert_packed_equal, np_inputs, packed_np, torch_sigmoid_fn

pytestmark = pytest.mark.gpu

LABELS = {"bean": 0, "maize": 1, "weed": 2}  # "weed" is in no classification group (cls_group -1)
KINDS = {"leaf": 0, "flower": 1}
TABLES = ("anchor", "part", "csi", "classification")


def _args(out_size, dist_threshold, conf=0.4, csi_threshold=0.5, labels=LABELS):
    return SimpleNamespace(labels=dict(labels), parts=dict(KINDS), width=4 * out_size[0], height=4 * out_size[1],
                           dist_threshold=dist_threshold, conf_threshold=conf, down_ratio=4.0, csi_threshold=csi_threshold)


def _annotations(gts, img_sizes):
    """Plain ground truth [(name, x, y, [(kind, x, y), ...]), ...] per image -> ImageAnnotation list."""
    return [ImageAnnotation("gt", [Object(name, Keypoint("stem", x, y), [Keypoint(k, px, py) for k, px, py in kps])
                                   for name, x, y, kps in gt], img_size=size) for gt, size in zip(gts, img_sizes)]


def _oracle_tables(pk, gts, img_sizes, args, out_size):
    """eval_anchor / eval_part / eval_csi / eval_classif of the reference, restated, over the batch:
    {table: {label: [tp, npos, ndet, acc]}}."""
    label_map = {i: name for name, i in args.labels.items()}
    part_map = {i: name for name, i in args.parts.items()}
    in_size = (int(args.down_ratio * out_size[0]), int(args.down_ratio * out_size[1]))
    objs = O.assemble(pk, label_map, part_map, "stem", args.conf_threshold, out_size, in_size)
    raw_parts = O.raw_parts(pk, part_map, args.conf_threshold, out_size, in_size)
    labels, kinds = list(args.labels), list(args.parts)
    net = (args.width, args.height)
    tables = {"anchor": {l: [0, 0, 0, []] for l in labels}, "part": {k: [0, 0, 0, []] for k in kinds},
              "csi": {l: [0, 0, 0, []] for l in labels}, "classification": {l: [0, 0, 0, []] for l in EO.CLASSIFICATION_LABELS}}
    for b, (gt, size) in enumerate(zip(gts, img_sizes)):
        loc = EO.evaluate_image([(name, a[1], a[2], a[3]) for name, a, _ in objs[b]], raw_parts[b], gt, size, net,
                                args.dist_threshold, labels, kinds)
        rx, ry = size[0] / net[0], size[1] / net[1]  # evaluate_objects_batch
        thresh, norm = min(size) * args.dist_threshold, min(size)
        preds = [(name, a[1] * rx, a[2] * ry, a[3], [(k[0], k[1] * rx, k[2] * ry, k[3]) for k in kps]) for name, a, kps in objs[b]]
        g = [(name, x * rx, y * ry, [(k, px * rx, py * ry) for k, px, py in kps]) for name, x, y, kps in gt]
        results = (("anchor", loc["anchor"]), ("part", loc["part"]),
                   ("csi", EO.eval_csi_image(preds, g, labels, thresh, args.csi_threshold)),
                   ("classification", EO.eval_classif_image(preds, g, thresh, norm)))
        for key, res in results:
            for label, (tp, npos, ndet, acc) in res.items():
                t = tables[key][label]
                t[0] += tp
                t[1] += npos
                t[2] += ndet
                t[3] += acc
    return tables


def _evaluate(packed, gts, img_sizes, args, out_size, *, exact=False, what=""):
    """The device's tables against the oracle's; returns the Evaluator."""
    ev = Evaluator(args)
    ev.accumulate_packed(packed, _annotations(gts, img_sizes), out_size, eval_csi=True, eval_classif=True)
    want = _oracle_tables(packed_np(packed), gts, img_sizes, args, out_size)
    got = {"anchor": ev.anchor_eval, "part": ev.part_eval, "csi": ev.csi_eval, "classification": ev.classification_eval}
    for key in TABLES:
        assert set(got[key].labels) == set(want[key]), (what, key)
        for label, (tp, npos, ndet, acc) in want[key].items():
            g = got[key][label]
            assert (g.tp, g.npos, g.ndet) == (tp, npos, ndet), (what, key, label)
            if exact:
                assert g.acc == acc, (what, key, label)
            else:
                np.testing.assert_allclose(g.acc, acc, rtol=1e-9, atol=0, err_msg=f"{what} {key} {label}")
    return ev


# ----------------------------------------------------------------------------------------------- dense, at the limits
def _ground_truth(objs, rng, n_objects=None):
    """Ground truth derived from assembled detections: jittered, some dropped, some duplicated, spurious ones added.
    With `n_objects`, padded or cut to exactly that many objects, holding exactly that many parts in all."""
    gt = []
    for name, a, kps in objs:
        if rng.random() < 0.15:
            continue
        parts = [(k[0], k[1] + rng.normal(0, 2), k[2] + rng.normal(0, 2)) for k in kps if rng.random() < 0.8]
        gt.append((name, a[1] + rng.normal(0, 2), a[2] + rng.normal(0, 2), parts))
        if rng.random() < 0.05:
            gt.append(gt[-1])
    for _ in range(20):
        gt.append((str(rng.choice(list(LABELS))), float(rng.uniform(0, 512)), float(rng.uniform(0, 512)), []))
    if n_objects is None:
        return gt
    gt = gt[:n_objects]
    while len(gt) < n_objects:
        gt.append((str(rng.choice(list(LABELS))), float(rng.uniform(0, 512)), float(rng.uniform(0, 512)), []))
    parts = sum(len(o[3]) for o in gt)
    for i in range(len(gt) - 1, -1, -1):  # cut parts from the back, or give the spurious objects some
        name, x, y, kps = gt[i]
        if parts > n_objects:
            keep = max(0, len(kps) - (parts - n_objects))
            parts -= len(kps) - keep
            kps = kps[:keep]
        elif parts < n_objects and not kps:
            add = min(3, n_objects - parts)
            kps = [(str(rng.choice(list(KINDS))), x + rng.normal(0, 5), y + rng.normal(0, 5)) for _ in range(add)]
            parts += add
        gt[i] = (name, x, y, kps)
    assert len(gt) == n_objects and sum(len(o[3]) for o in gt) == n_objects
    return gt


def test_dense_batch_at_k_p_1024(cuda_device):
    """Noise maps decoded at K = P = 1024 (about a thousand objects per image): one image with ground truth derived from
    its detections, one with exactly 1024 ground-truth objects and 1024 ground-truth parts, one without ground truth,
    one without a detection above conf."""
    cfg = DecodeConfig("dense", 4, 3, 2, 128, 128, 1024, 1024, cfg_id=44)
    raw = make_raw(cfg, "noise")
    raw[3, :5] -= 12.0  # logits below -7: no score reaches conf
    out_size = (128, 128)
    packed = ops.decode_packed(split_outputs(raw.to(cuda_device), 3, 2), 1024, 1024, 0.4, 0.1)
    pk = packed_np(packed)
    assert (pk["counts"][:3] > 900).all() and (pk["counts"][3] == 0).all(), pk["counts"]
    args = _args(out_size, 0.02)
    objs = O.assemble(pk, {i: n for n, i in LABELS.items()}, {i: k for k, i in KINDS.items()}, "stem", 0.4, out_size, (512, 512))
    rng = np.random.default_rng(44)
    gts = [_ground_truth(objs[0], rng), _ground_truth(objs[1], rng, n_objects=1024), [], _ground_truth(objs[0], rng)]
    sizes = [(1931, 1297), (1297, 1931), (512, 512), (2048, 1024)]
    ev = _evaluate(packed, gts, sizes, args, out_size, what="dense")
    assert ev.anchor_eval.reduce().tp > 500 and ev.part_eval.reduce().tp > 500
    assert ev.csi_eval.reduce().tp > 100 and ev.classification_eval.reduce().tp > 100


# ----------------------------------------------------------------------------------------------- exact boundaries
# Network input 512 x 512 = image size (no resize), heat maps 128 x 128 (x 4), dist_threshold 1/16: thresh = 32 exactly.
OUT = (128, 128)
SIZE = (512, 512)
THRESH = 32.0


def _packed(device, anchors, parts, assign, K=16, P=32, M=3, N=2):
    """Packed detections as the tail kernel leaves them, one image: `anchors` = [(x, y, score, class)] and `parts` =
    [(x, y, score, kind)] in slot (score) order, heat-map frame; every other slot scores 0."""
    blob = torch.zeros(ops.packed_nbytes(1, K, P, M + N), dtype=torch.uint8)
    host = ops._carve(blob, 1, K, P, M + N)
    host.assign.fill_(-1)
    for i, row in enumerate(anchors):
        host.anchor_out[0, i] = torch.tensor(row, dtype=torch.float32)
    for i, row in enumerate(parts):
        host.part_out[0, i, :4] = torch.tensor(row, dtype=torch.float32)
    for i, slot in enumerate(assign):
        host.assign[0, i] = slot
    return ops._carve(blob.to(device), 1, K, P, M + N)


def test_location_and_classification_boundaries(cuda_device):
    """Axis-aligned distances of exactly 32 (location: false positive, classification: true positive) and of the largest
    double below 32 (true positive for both); two ground truths mirrored at +-10 (the first in annotation order wins);
    a duplicated ground truth (the second copy stays unmatched).  The same for raw parts."""
    below = float(np.nextafter(133.0, 0.0))  # detection at x = 101: distance the largest double below 32
    bean, maize, weed = 0, 1, 2
    anchors = [(25.25, 30.5, 0.9, bean),     # x = 101: ground truth at 133 (distance 32)
               (33.5, 30.5, 0.85, bean),     # x = 134: the same ground truth at distance 1
               (50.25, 30.5, 0.8, maize),    # x = 201: ground truth at 233 - ulp
               (75.25, 75.0, 0.7, bean),     # x = 301: ground truths at 291 and 311
               (72.75, 75.0, 0.6, bean),     # x = 291
               (100.25, 100.0, 0.5, maize),  # x = 401: two copies of a ground truth at (401, 410)
               (100.5, 100.0, 0.45, maize),  # x = 402
               (10.0, 120.0, 0.42, weed)]
    parts = [(25.25, 50.0, 0.9, 0), (33.5, 50.0, 0.85, 0), (50.25, 50.0, 0.8, 0), (75.25, 50.0, 0.7, 1),
             (72.75, 50.0, 0.6, 1), (100.25, 50.0, 0.5, 0), (100.5, 50.0, 0.45, 0)]
    gt = [("bean", 133.0, 122.0, []), ("maize", below + 100.0, 122.0, []), ("bean", 291.0, 300.0, []),
          ("bean", 311.0, 300.0, []), ("maize", 401.0, 410.0, []), ("maize", 401.0, 410.0, []),
          ("weed", 40.0, 480.0, [("leaf", 133.0, 200.0), ("leaf", below + 100.0, 200.0), ("flower", 291.0, 200.0),
                                 ("flower", 311.0, 200.0), ("leaf", 401.0, 210.0), ("leaf", 401.0, 210.0)])]
    assert below + 100.0 == float(np.nextafter(233.0, 0.0))
    packed = _packed(cuda_device, anchors, parts, [])
    ev = _evaluate(packed, [gt], [SIZE], _args(OUT, THRESH / SIZE[0]), OUT, exact=True, what="boundaries")
    # location: 101 misses at 32, 134 takes it; 301 takes 291 (first of two at 10), 291 then finds it taken
    assert (ev.anchor_eval["bean"].tp, ev.anchor_eval["bean"].acc) == (2, [1 / 512, 10 / 512])
    assert ev.anchor_eval["maize"].tp == 2 and ev.part_eval["leaf"].tp == 3 and ev.part_eval["flower"].tp == 1
    # classification: 101 takes the ground truth at exactly 32, so 134 finds it taken
    assert (ev.classification_eval["bean_0"].tp, ev.classification_eval["bean_0"].acc) == (2, [32 / 512, 10 / 512])


CSI_HALF = float(np.nextafter(0.5, 1.0))


@pytest.mark.parametrize("csi_threshold", [0.5, CSI_HALF, 0.01], ids=["half", "above-half", "low"])
def test_csi_boundaries(cuda_device, csi_threshold):
    """A CSI of exactly 2/4 against csi_threshold 0.5 and the next double above it; two identical ground-truth objects
    (the first maximum wins); a 64-part ground-truth object of which only the 64th part is matched, by two predicted
    parts (the second finds it taken); an object with 10 grouped parts, which classification counts nowhere."""
    bean, maize, weed = 0, 1, 2
    anchors = [(25.25, 30.5, 0.9, bean),    # (101, 122): CSI (1 + 1) / (3 + 3 - 2) = 1/2
               (75.25, 30.5, 0.8, maize),   # (301, 122) and (302, 122): two identical ground truths
               (75.5, 30.5, 0.79, maize),
               (25.25, 100.0, 0.7, weed),   # (101, 400): the 64-part ground truth
               (75.25, 100.0, 0.6, bean)]   # (301, 400): 10 parts
    parts, assign = [], []

    def part(x, y, kind, owner):
        parts.append((x, y, 0.95 - 0.01 * len(parts), kind))
        assign.append(owner)

    part(25.25, 35.0, 0, 0)     # (101, 140): matches
    part(25.25, 40.0, 1, 0)     # (101, 160): its ground truth is 40 away
    part(75.25, 35.0, 0, 1)
    part(75.5, 35.0, 0, 2)
    part(25.25, 107.5, 0, 3)    # (101, 430) and (102, 430): nearest to the 64th part
    part(25.5, 107.5, 0, 3)
    for i in range(10):
        part(75.25 + i, 110.0, 0, 4)
    gt = [("bean", 101.0, 122.0, [("leaf", 101.0, 140.0), ("flower", 101.0, 200.0)]),
          ("maize", 301.0, 122.0, [("leaf", 301.0, 140.0)]), ("maize", 301.0, 122.0, [("leaf", 301.0, 140.0)]),
          ("weed", 101.0, 400.0, [("leaf", 480.0, 5.0 + 7.0 * i) for i in range(63)] + [("leaf", 101.0, 430.0)]),
          ("bean", 301.0, 400.0, [("leaf", 301.0 + 4 * i, 440.0) for i in range(10)])]
    packed = _packed(cuda_device, anchors, parts, assign)
    ev = _evaluate(packed, [gt], [SIZE], _args(OUT, THRESH / SIZE[0], csi_threshold=csi_threshold), OUT, exact=True,
                   what=f"csi {csi_threshold}")
    half_tp = 1 if csi_threshold <= 0.5 else 0
    assert ev.csi_eval["bean"].tp == half_tp + 1 and ev.csi_eval["maize"].tp == 1
    assert ev.csi_eval["weed"].acc == ([2 / 66] if csi_threshold < 2 / 66 else [])
    assert ev.classification_eval.reduce().ndet == 3  # bean_2, maize_1 twice; the 10-part bean is in no class


def test_score_equal_to_conf(cuda_device):
    """conf = 0.5 and logits of exactly 0 (score 0.5): such an anchor is no object and such a part is a raw part that is
    never grouped -- in the decoder's counts and in the evaluator's detection counts."""
    cfg = DecodeConfig("atconf", 1, 2, 1, 64, 64, 10, 10, cfg_id=45)
    raw = make_raw(cfg, "ladder")
    raw[:, :3] = -8.0 - torch.rand(1, 3, 64, 64, generator=torch.Generator().manual_seed(45))
    raw[:, 3:] = 0.0
    raw[0, 0, 10, 10] = 2.0   # bean, valid
    raw[0, 0, 10, 30] = 0.0   # bean at exactly conf
    raw[0, 1, 40, 40] = 0.0   # maize at exactly conf
    raw[0, 2, 30, 50] = 0.0   # leaf at exactly conf
    raw[0, 2, 12, 12] = 1.0   # leaf, valid, 2.8 pixels from the valid bean
    outs = split_outputs(raw.to(cuda_device), 2, 1)
    packed = ops.decode_packed(outs, 10, 10, 0.5, 0.1)
    pk = packed_np(packed)
    want = O.decode_packed(*np_inputs(split_outputs(raw, 2, 1)), 10, 10, 0.5, 0.1, sigmoid_fn=torch_sigmoid_fn(cuda_device))
    assert_packed_equal(pk, want, what="score = conf")
    assert pk["counts"].tolist() == [[1, 1]]
    at_conf = np.flatnonzero(pk["part_out"][0, :, 2] == 0.5)
    assert at_conf.size == 1 and pk["assign"][0, at_conf[0]] == -1
    labels = {"bean": 0, "maize": 1}
    gt = [("bean", 40.0, 40.0, [("leaf", 44.0, 44.0), ("leaf", 48.0, 48.0)]), ("maize", 160.0, 160.0, [])]
    ev = _evaluate(packed, [gt], [(256, 256)], _args((64, 64), 0.1, conf=0.5, labels=labels), (64, 64), what="score = conf")
    assert ev.anchor_eval.reduce().ndet == 1 and ev.part_eval["leaf"].ndet == 2
