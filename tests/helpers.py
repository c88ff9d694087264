"""Shared test plumbing: plain-tuple views of decoder outputs, sigmoid adapters, arg namespaces."""
from __future__ import annotations

from pathlib import Path
from types import SimpleNamespace

import numpy as np
import torch

GOLDEN_DIR = Path(__file__).resolve().parent / "golden"


def make_args(cfg, conf=None, dist=None, anchor_name="stem", down_ratio=4.0, max_objects=None, max_parts=None):
    labels = {i: f"label{i}" for i in range(cfg.labels)}
    parts = {i: f"part{i}" for i in range(cfg.parts)}
    if cfg.labels == 2 and cfg.parts == 1:  # reference labels.json
        labels, parts = {0: "bean", 1: "maize"}, {0: "leaf"}
    return SimpleNamespace(
        _r_labels=labels, _r_parts=parts, anchor_name=anchor_name, down_ratio=down_ratio,
        max_objects=cfg.max_objects if max_objects is None else max_objects,
        max_parts=cfg.max_parts if max_parts is None else max_parts,
        conf_threshold=cfg.conf_threshold if conf is None else conf,
        decoder_dist_thresh=cfg.dist_thresh if dist is None else dist,
    )


def plain(annotations):
    """ImageAnnotation list (ours or the reference's) -> nested tuples for equality checks."""
    return [[(o.name, (o.anchor.kind, o.anchor.x, o.anchor.y, o.anchor.score),
              [(p.kind, p.x, p.y, p.score) for p in o.parts]) for o in ann.objects] for ann in annotations]


def plain_keypoints(images):
    return [[(k.kind, k.x, k.y, k.score) for k in kps] for kps in images]


def torch_sigmoid_fn(device="cpu"):
    """numpy->numpy sigmoid evaluated by torch on ``device`` (bit-identical to what the
    reference computes there)."""
    def fn(x):
        t = torch.from_numpy(np.ascontiguousarray(x)).to(device)
        return torch.sigmoid(t).cpu().numpy()
    return fn


def np_inputs(outputs):
    return [outputs[k].detach().cpu().numpy() for k in ("anchor_hm", "part_hm", "offsets", "embeddings")]


def packed_np(packed):
    return {k: v.detach().cpu().numpy() for k, v in packed.as_dict().items()}


def assert_packed_equal(got: dict, want: dict, *, what=""):
    """Bit-exact comparison of every packed field the oracle also produces."""
    for key in ("anchor_inds", "part_inds", "assign", "counts"):
        if key in want and key in got:
            np.testing.assert_array_equal(got[key], want[key], err_msg=f"{what}: {key}")
    for key in ("anchor_out", "part_out", "part_emb"):
        if key in want and key in got:
            g, w = np.ascontiguousarray(got[key]).view(np.uint32), np.ascontiguousarray(want[key]).view(np.uint32)
            bad = np.argwhere(g != w)
            assert bad.size == 0, f"{what}: {key} differs at {bad[:5].tolist()} got {got[key][tuple(bad[0])]} want {want[key][tuple(bad[0])]}"


# ----------------------------------------------------------------------------- golden fixtures
def load_golden(name):
    """(meta dict, arrays dict) of one fixture written by tests/golden/make_golden.py."""
    import json

    index = json.loads((GOLDEN_DIR / "index.json").read_text())
    return index[name], dict(np.load(GOLDEN_DIR / f"{name}.npz"))


def golden_names():
    import json

    return sorted(json.loads((GOLDEN_DIR / "index.json").read_text()))


def golden_args(meta):
    _, m, n, _, _ = meta["shape"]
    return SimpleNamespace(
        _r_labels={i: f"label{i}" for i in range(m)}, _r_parts={i: f"part{i}" for i in range(n)},
        anchor_name=meta["anchor_name"], down_ratio=meta["down_ratio"], max_objects=meta["K"], max_parts=meta["P"],
        conf_threshold=meta["conf"], decoder_dist_thresh=meta["dist"])


def listify(objs):
    """tuples -> lists, so oracle/our output compares equal to what came back from JSON."""
    if isinstance(objs, (list, tuple)):
        return [listify(o) for o in objs]
    return objs


def assert_objects_close(got, want, *, score_atol=0.0, coord_rtol=0.0, what=""):
    """Same structure, names and ordering; scores / coordinates within the given tolerances."""
    assert len(got) == len(want), f"{what}: {len(got)} images vs {len(want)}"
    for b, (gi, wi) in enumerate(zip(got, want)):
        assert len(gi) == len(wi), f"{what}: image {b}: {len(gi)} objects vs {len(wi)}"
        for o, (go, wo) in enumerate(zip(gi, wi)):
            assert go[0] == wo[0], f"{what}: image {b} object {o}: label {go[0]} vs {wo[0]}"
            kps_g, kps_w = [go[1]] + list(go[2]), [wo[1]] + list(wo[2])
            assert len(kps_g) == len(kps_w), f"{what}: image {b} object {o}: {len(kps_g) - 1} parts vs {len(kps_w) - 1}"
            for kg, kw in zip(kps_g, kps_w):
                assert kg[0] == kw[0], f"{what}: image {b} object {o}: kind {kg[0]} vs {kw[0]}"
                for a, c in ((kg[1], kw[1]), (kg[2], kw[2])):
                    assert abs(a - c) <= coord_rtol * max(abs(c), 1.0), f"{what}: image {b} object {o}: coord {a} vs {c}"
                assert abs(kg[3] - kw[3]) <= score_atol, f"{what}: image {b} object {o}: score {kg[3]} vs {kw[3]}"


def assert_topk_equal_up_to_ties(got_scores, got_cls, got_inds, ref_scores, ref_cls, ref_inds, *, what=""):
    """Scores identical slot by slot; (class, index) identical as SETS inside each run of equal
    scores -- except the last run of a row, whose membership depends on torch.topk's tie rule."""
    np.testing.assert_array_equal(got_scores, ref_scores, err_msg=f"{what}: scores")
    for r in range(got_scores.shape[0]):
        row = got_scores[r]
        k = len(row)
        start = 0
        while start < k:
            end = start
            while end + 1 < k and row[end + 1] == row[start]:
                end += 1
            if end < k - 1:  # run closed inside the list: membership is unambiguous
                g = sorted(zip(got_cls[r, start:end + 1].tolist(), got_inds[r, start:end + 1].tolist()))
                w = sorted(zip(ref_cls[r, start:end + 1].tolist(), ref_inds[r, start:end + 1].tolist()))
                assert g == w, f"{what}: row {r} slots {start}..{end}"
            start = end + 1
