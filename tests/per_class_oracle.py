"""Per-class confidence thresholds in the numpy oracle's terms -- test infrastructure.

``oracle.sdnet_oracle`` restates the reference decoder with one threshold.  This module restates the same decode with
one threshold per anchor class and part kind, on top of it and without changing it: the selection, gathers and
coordinates come from ``sdnet_oracle.decode_packed(..., group=False)``, and the grouping of the reference
(decoders.py:78-100) is redone here with every slot's ``score > conf`` taken against its own class's entry.  The
object loops (decoders.py:103-159) are restated the same way.
"""
from __future__ import annotations

import numpy as np

from oracle import sdnet_oracle as O

F32 = np.float32


def decode_packed(anchor_hm, part_hm, offsets, embeddings, max_objects, max_parts, conf_class, dist_thresh, **kw):
    """``sdnet_oracle.decode_packed`` with ``conf_class``: M + N thresholds (anchor classes, then part kinds), each
    already rounded to the heat maps' dtype, instead of the one threshold.  ``kw``: the oracle's activation options."""
    out = O.decode_packed(anchor_hm, part_hm, offsets, embeddings, max_objects, max_parts, 0.0, dist_thresh, group=False,
                          **kw)
    m = np.asarray(anchor_hm).shape[1]
    h, w = np.asarray(anchor_hm).shape[2:]
    table = np.asarray(conf_class, dtype=F32)
    a, p = out["anchor_out"], out["part_out"]
    a_score, p_score = a[..., 2], p[..., 2]
    a_conf, p_conf = table[a[..., 3].astype(np.int64)], table[m + p[..., 3].astype(np.int64)]
    one = F32(1.0)
    p_mask = (p_score > p_conf).astype(F32)
    a_mask = (a_score > a_conf).astype(F32)
    out["part_scores_masked"] = (-(one - p_mask) + p_mask * p_score).astype(F32)
    out["anchor_scores_masked"] = (-(one - a_mask) + a_mask * a_score).astype(F32)
    ori_x = (-O.MASKED_FAR * (one - p_mask) + p_mask * p[..., 4]).astype(F32)
    ori_y = (-O.MASKED_FAR * (one - p_mask) + p_mask * p[..., 5]).astype(F32)
    pos_x = (O.MASKED_FAR * (one - a_mask) + a_mask * a[..., 0]).astype(F32)
    pos_y = (O.MASKED_FAR * (one - a_mask) + a_mask * a[..., 1]).astype(F32)
    dx = (ori_x[:, None, :] - pos_x[:, :, None]).astype(F32)
    dy = (ori_y[:, None, :] - pos_y[:, :, None]).astype(F32)
    dist = O.hypot(np.stack((dx, dy), axis=-1))  # (B, K, P)
    min_inds = np.argmin(dist, axis=1)  # first minimum wins
    min_vals = np.take_along_axis(dist, min_inds[:, None, :], axis=1)[:, 0, :]
    gate = F32(float(dist_thresh) * min(w, h))
    out["assign"] = np.where(min_vals < gate, min_inds, -1).astype(np.int32)
    out["counts"] = np.stack((a_mask.sum(axis=1), p_mask.sum(axis=1)), axis=1).astype(np.int32)
    return out


def assemble(packed, label_map, part_map, anchor_name, anchor_conf, out_size, in_size):
    """``sdnet_oracle.assemble`` with ``anchor_conf``: one threshold per anchor class (objects: score > conf[class],
    in double; parts grouped onto an anchor that is not emitted are dropped)."""
    (ow, oh), (iw, ih) = out_size, in_size
    rx, ry = iw / ow, ih / oh
    anchors = packed["anchor_out"].astype(np.float64)
    parts = packed["part_out"].astype(np.float64)
    images = []
    for b in range(anchors.shape[0]):
        buckets = {}
        for i, slot in enumerate(packed["assign"][b].tolist()):
            if slot >= 0:
                buckets.setdefault(slot, []).append(i)
        objects = []
        for a_i in range(anchors.shape[1]):
            ax, ay, score, cls = anchors[b, a_i].tolist()
            if score <= anchor_conf[int(cls)]:
                continue
            kps = [(part_map[int(parts[b, i, 3])], parts[b, i, 0] * rx, parts[b, i, 1] * ry, parts[b, i, 2])
                   for i in buckets.get(a_i, ())]
            objects.append((label_map[int(cls)], (anchor_name, ax * rx, ay * ry, score), kps))
        images.append(objects)
    return images


def raw_parts(packed, part_map, part_conf, out_size, in_size):
    """``sdnet_oracle.raw_parts`` with ``part_conf``: one threshold per part kind (skip score < conf[kind], in double)."""
    (ow, oh), (iw, ih) = out_size, in_size
    rx, ry = iw / ow, ih / oh
    parts = packed["part_out"].astype(np.float64)
    return [[(part_map[int(pc)], px * rx, py * ry, ps) for px, py, ps, pc in parts[b, :, :4].tolist()
             if not ps < part_conf[int(pc)]] for b in range(parts.shape[0])]
