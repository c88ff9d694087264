"""CPU restatement of the evaluator's threshold sweep -- TEST INFRASTRUCTURE ONLY (imported by tests/ and nothing
else; the product path is ThresholdSweep in structuredetector_b200/evaluator.py on the GPU).

The long way round: one whole decode (oracle/sdnet_oracle.py) and one whole evaluation (oracle/evaluator_oracle.py)
per threshold, which is what a user without the sweep runs.  It is a module of its own so that evaluator_oracle.py, the
restatement the reference's stored evaluator output pins, stays exactly as those tests checked it.
"""
from __future__ import annotations

import numpy as np

from oracle import sdnet_oracle as O
from oracle.evaluator_oracle import CLASSIFICATION_LABELS, eval_classif_image, eval_csi_image, evaluate_image


# ---------------------------------------------------------------------------------------------------------------
# all four tables of one decoded batch, and the same at a grid of confidence thresholds
def evaluate_tables(objs, raw_parts, gts, img_sizes, args):
    """eval_anchor / eval_part / eval_csi / eval_classif over a batch.  `objs` / `raw_parts` as sdnet_oracle.assemble /
    raw_parts return them (network-input frame), `gts` per image [(name, x, y, [(kind, x, y), ...])] in the same frame;
    `args` as the evaluator's (labels, parts, width, height, dist_threshold, csi_threshold).
    Returns {"anchor" | "part" | "csi" | "classification": {label: [tp, npos, ndet, acc]}}."""
    labels, kinds = list(args.labels), list(args.parts)
    net = (args.width, args.height)
    tables = {"anchor": {l: [0, 0, 0, []] for l in labels}, "part": {k: [0, 0, 0, []] for k in kinds},
              "csi": {l: [0, 0, 0, []] for l in labels}, "classification": {l: [0, 0, 0, []] for l in CLASSIFICATION_LABELS}}
    for b, (gt, size) in enumerate(zip(gts, img_sizes)):
        loc = evaluate_image([(name, a[1], a[2], a[3]) for name, a, _ in objs[b]], raw_parts[b], gt, size, net,
                             args.dist_threshold, labels, kinds)
        rx, ry = size[0] / net[0], size[1] / net[1]
        thresh, norm = min(size) * args.dist_threshold, min(size)
        preds = [(name, a[1] * rx, a[2] * ry, a[3], [(k[0], k[1] * rx, k[2] * ry, k[3]) for k in kps]) for name, a, kps in objs[b]]
        g = [(name, x * rx, y * ry, [(k, px * rx, py * ry) for k, px, py in kps]) for name, x, y, kps in gt]
        results = (("anchor", loc["anchor"]), ("part", loc["part"]),
                   ("csi", eval_csi_image(preds, g, labels, thresh, args.csi_threshold)),
                   ("classification", eval_classif_image(preds, g, thresh, norm)))
        for key, res in results:
            for label, (tp, npos, ndet, acc) in res.items():
                t = tables[key][label]
                t[0] += tp
                t[1] += npos
                t[2] += ndet
                t[3] += acc
    return tables


def sweep(inputs, thresholds, max_objects, max_parts, dist_thresh, gts, img_sizes, args, *, conf_cmp=None, **decode_kw):
    """The evaluator at every threshold of a grid, the long way round: per threshold t, one sdnet_oracle.decode_packed
    grouping at `conf_cmp(t)` (t rounded to the heat maps' dtype; float32 when None), then assemble / raw_parts at t and
    evaluate_tables.  `inputs` = (anchor_hm, part_hm, offsets, embeddings) arrays, `decode_kw` goes to decode_packed.
    Returns one evaluate_tables result per threshold."""
    h, w = np.asarray(inputs[0]).shape[2:]
    out_size, in_size = (w, h), (int(args.down_ratio * w), int(args.down_ratio * h))
    label_map = {i: name for name, i in args.labels.items()}
    part_map = {i: name for name, i in args.parts.items()}
    out = []
    for t in thresholds:
        pk = O.decode_packed(*inputs, max_objects, max_parts, t, dist_thresh,
                             conf_cmp=None if conf_cmp is None else conf_cmp(t), **decode_kw)
        objs = O.assemble(pk, label_map, part_map, "stem", t, out_size, in_size)
        out.append(evaluate_tables(objs, O.raw_parts(pk, part_map, t, out_size, in_size), gts, img_sizes, args))
    return out
