"""Port of the reference decoder onto stock torch ops -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The reference (laclouis5/StructureDetector) is pure-Python PyTorch and does not exist on
the GPU box, so this module is the thing that *can travel*: the same stock ATen calls the
reference issues (sigmoid, clamp, max_pool2d, topk, gather, min; reference:
src/sdnet/data/decoders.py:44-100 and src/sdnet/utils/utils.py:342-361,422-467),
composed by our own code, runnable on ``cpu`` (the CPU baseline / ``--impl reference``
arm of bench.py) or on ``cuda`` (the on-device checker used by ``-m gpu`` tests).

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline legs may
import it.  ``tests/test_oracle.py`` validates it against the reference's stored outputs in
``tests/golden/`` and against the oracle on other shapes.

Differences from the reference that are deliberate:
  * returns packed tensors (same layout as the C-ABI outputs) and builds Python objects
    from one ``.tolist()`` per tensor instead of one ``.item()`` per scalar -- this makes
    the CPU baseline *faster* than the true reference, never slower;
  * no in-place mutation of inputs.
"""
from __future__ import annotations

import torch
import torch.nn.functional as tnf


def _select(scores: torch.Tensor, k: int):
    """Two-stage top-k of reference utils.py:447-467 on an already NMS'd (B, C, H, W) map."""
    b, c, _, w = scores.shape
    s1, i1 = torch.topk(scores.reshape(b, c, -1), k)
    i1f = i1.float()
    ys1 = torch.div(i1f, w, rounding_mode="floor")
    xs1 = torch.remainder(i1f, w)
    s2, pos = torch.topk(s1.reshape(b, -1), k)
    cls = torch.div(pos.float(), k, rounding_mode="floor")
    take = lambda t: t.reshape(b, -1).gather(1, pos)
    return s2, take(i1), cls, take(ys1), take(xs1)


def _pick(feat: torch.Tensor, ind: torch.Tensor) -> torch.Tensor:
    """(B, Cf, H, W) sampled at flat indices (B, n) -> (B, n, Cf)  (reference utils.py:347-351)."""
    b, cf = feat.shape[:2]
    return feat.reshape(b, cf, -1).gather(2, ind.unsqueeze(1).expand(-1, cf, -1)).permute(0, 2, 1)


def activate(hm: torch.Tensor) -> torch.Tensor:
    return torch.clamp(torch.sigmoid(hm), min=1e-6, max=1 - 1e-6)


def suppress(sig: torch.Tensor, radius: int = 2) -> torch.Tensor:
    mx = tnf.max_pool2d(sig, kernel_size=2 * radius + 1, stride=1, padding=radius)
    return (sig == mx) * sig


@torch.no_grad()
def decode_tensors(outputs: dict, max_objects: int, max_parts: int, conf_thresh: float, dist_thresh: float,
                   *, pre_activated: bool = False, radius: int = 2, group: bool = True) -> dict:
    a_hm, p_hm = outputs["anchor_hm"], outputs["part_hm"]
    h, w = a_hm.shape[2:]
    if pre_activated:
        a_sig, p_sig, a_nms, p_nms = a_hm, p_hm, a_hm, p_hm
    else:
        a_sig, p_sig = activate(a_hm), activate(p_hm)
        a_nms, p_nms = suppress(a_sig, radius), suppress(p_sig, radius)

    a_score, a_ind, a_cls, a_ys, a_xs = _select(a_nms, max_objects)
    a_off = _pick(outputs["offsets"], a_ind)
    a_x, a_y = a_xs + a_off[..., 0], a_ys + a_off[..., 1]

    p_score, p_ind, p_cls, p_ys, p_xs = _select(p_nms, max_parts)
    p_off = _pick(outputs["offsets"], p_ind)
    p_emb = _pick(outputs["embeddings"], p_ind)
    p_x, p_y = p_xs + p_off[..., 0], p_ys + p_off[..., 1]
    o_x, o_y = p_x + p_emb[..., 0], p_y + p_emb[..., 1]

    out = {
        "anchor_out": torch.stack((a_x, a_y, a_score, a_cls.float()), dim=2),
        "part_out": torch.stack((p_x, p_y, p_score, p_cls.float(), o_x, o_y), dim=2),
        "anchor_inds": a_ind,
        "part_inds": p_ind,
        "part_emb": p_emb.contiguous(),
        "anchor_sig": a_sig,
        "part_sig": p_sig,
    }
    if not group:
        return out

    p_keep = (p_score > conf_thresh).float()
    a_keep = (a_score > conf_thresh).float()
    out["part_scores_masked"] = -(1 - p_keep) + p_keep * p_score
    out["anchor_scores_masked"] = -(1 - a_keep) + a_keep * a_score
    far = 1e6
    ori = torch.stack((-far * (1 - p_keep) + p_keep * o_x, -far * (1 - p_keep) + p_keep * o_y), dim=-1)  # (B,P,2)
    pos = torch.stack((far * (1 - a_keep) + a_keep * a_x, far * (1 - a_keep) + a_keep * a_y), dim=-1)  # (B,K,2)
    diff = ori.unsqueeze(1) - pos.unsqueeze(2)  # (B,K,P,2)
    dist = torch.empty(diff.shape[:-1], device=diff.device)
    torch.sum(torch.square(diff), dim=-1, out=dist)
    torch.sqrt(dist, out=dist)
    min_vals, min_inds = dist.min(dim=1)
    ok = min_vals < (dist_thresh * min(w, h))
    out["min_inds"] = min_inds
    out["min_vals"] = min_vals
    out["assign"] = torch.where(ok, min_inds, torch.full_like(min_inds, -1)).to(torch.int32)
    out["counts"] = torch.stack((a_keep.sum(1), p_keep.sum(1)), dim=1).to(torch.int32)
    return out


def assemble(packed: dict, label_map, part_map, anchor_name, conf_thresh, out_size, in_size):
    """Plain-tuple objects, same structure as ``oracle.sdnet_oracle.assemble``."""
    (ow, oh), (iw, ih) = out_size, in_size
    rx, ry = iw / ow, ih / oh
    anchors = packed["anchor_out"].cpu().tolist()
    parts = packed["part_out"].cpu().tolist()
    assign = packed["assign"].cpu().tolist()
    images = []
    for b, slots in enumerate(assign):
        buckets = {}
        for i, slot in enumerate(slots):
            if slot >= 0:
                buckets.setdefault(slot, []).append(i)
        objects = []
        for a_i, (ax, ay, score, cls) in enumerate(anchors[b]):
            if score <= conf_thresh:
                continue
            kps = [(part_map[int(parts[b][i][3])], parts[b][i][0] * rx, parts[b][i][1] * ry, parts[b][i][2])
                   for i in buckets.get(a_i, ())]
            objects.append((label_map[int(cls)], (anchor_name, ax * rx, ay * ry, score), kps))
        images.append(objects)
    return images


def decode(outputs: dict, label_map, part_map, anchor_name, down_ratio, max_objects, max_parts,
           conf_thresh, dist_thresh):
    """Whole reference call (tensors + objects); what ``bench.py --impl reference`` times."""
    h, w = outputs["anchor_hm"].shape[2:]
    packed = decode_tensors(outputs, max_objects, max_parts, conf_thresh, dist_thresh)
    return assemble(packed, label_map, part_map, anchor_name, conf_thresh, (w, h),
                    (int(down_ratio * w), int(down_ratio * h)))
