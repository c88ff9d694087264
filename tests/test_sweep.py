"""CPU: the host side of the threshold sweep -- the SdnetSweepParams layout, the argument errors sdnet_sweep_launch
returns before any launch, ThresholdSweep's own checks, curve / best_threshold on hand-filled evaluations -- and the
oracle's restatement of the sweep against the reference's stored evaluator output."""
import ctypes
import json
import math
import shutil
import subprocess
from pathlib import Path
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from oracle import sweep_oracle as SO
from structuredetector_b200 import ImageAnnotation, Keypoint, Object, _native, ops
from structuredetector_b200.evaluator import Evaluation, ThresholdSweep
from tests.helpers import load_golden, torch_sigmoid_fn

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = ROOT / "tests" / "golden"
EVAL = json.loads((GOLDEN / "eval.json").read_text())
EVAL_OBJECTS = json.loads((GOLDEN / "eval_objects.json").read_text())


def _args(**kw):
    base = dict(labels={"bean": 0, "maize": 1}, parts={"leaf": 0}, width=512, height=512, dist_threshold=0.05,
                conf_threshold=0.4, down_ratio=4.0, csi_threshold=0.5, decoder_dist_thresh=0.1)
    base.update(kw)
    return SimpleNamespace(**base)


def test_sweep_params_layout_matches_the_header_under_gcc(tmp_path):
    """sizeof and every offsetof of SdnetSweepParams as the C compiler sees the public header."""
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    fields = _native.SdnetSweepParams._fields_
    src = ["#include <stdio.h>", "#include <stddef.h>", '#include "sdnet_decode.h"', "int main(void) {",
           'printf("size %zu\\n", sizeof(SdnetSweepParams));']
    src += [f'printf("{name} %zu\\n", offsetof(SdnetSweepParams, {name}));' for name, _ in fields]
    src += [f'printf("MAX_THRESHOLDS %d\\n", SDNET_MAX_THRESHOLDS);', f'printf("SWEEP_OBJECTS %u\\n", SDNET_SWEEP_OBJECTS);',
            "return 0; }"]
    (tmp_path / "layout.c").write_text("\n".join(src))
    subprocess.run([cc, "-std=c99", "-Wall", "-Werror", f"-I{ROOT / 'include'}", str(tmp_path / "layout.c"), "-o",
                    str(tmp_path / "layout")], check=True)
    out = dict(line.split() for line in subprocess.run([str(tmp_path / "layout")], check=True, capture_output=True,
                                                        text=True).stdout.split("\n") if line)
    assert int(out.pop("size")) == ctypes.sizeof(_native.SdnetSweepParams)
    assert int(out.pop("MAX_THRESHOLDS")) == _native.MAX_THRESHOLDS
    assert int(out.pop("SWEEP_OBJECTS")) == _native.SWEEP_OBJECTS
    assert {name: int(v) for name, v in out.items()} == {name: getattr(_native.SdnetSweepParams, name).offset
                                                         for name, _ in fields}


def _sweep_buffers():
    """Zeroed buffers large enough for every shape the tests below pass (T up to 257, K = P up to 1025, 256 classes,
    1025 ground-truth rows), on the CUDA device when there is one.  A library that let one of these calls through its
    checks would launch on zeros within bounds, never on bad memory."""
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    T, S, C, G = _native.MAX_THRESHOLDS + 1, 1025, 256, _native.MAX_GT + 1
    f64, i32 = {"dtype": torch.float64, "device": dev}, {"dtype": torch.int32, "device": dev}
    return {"conf": torch.zeros(T, **f64), "conf_group": torch.zeros(T, device=dev),
            "anchor_out": torch.zeros(1, S, 4, device=dev), "part_out": torch.zeros(1, S, 6, device=dev),
            "image_scale": torch.ones(1, 4, **f64), "gt_objects": torch.zeros(1, G, 3, **f64),
            "n_gt_objects": torch.zeros(1, **i32), "gt_parts": torch.zeros(1, G, 3, **f64),
            "gt_part_owner": torch.zeros(1, G, **i32), "n_gt_parts": torch.zeros(1, **i32), "cls_group": torch.zeros(C, **i32),
            "anchor_stats": torch.zeros(T, C, 3, **i32), "part_stats": torch.zeros(T, C, 3, **i32),
            "anchor_acc": torch.zeros(T, S, **f64), "part_acc": torch.zeros(T, S, **f64),
            "csi_stats": torch.zeros(T, C, 3, **i32), "csi_acc": torch.zeros(T, S, **f64),
            "classif_stats": torch.zeros(T, 20, 3, **i32), "classif_acc": torch.zeros(T, S, **f64),
            "pred_parts": torch.zeros(T, S, **i32)}


def _params(bufs, objects=True, **shape):
    """A well-formed single-image sweep over `bufs`, with `shape` overriding its sizes."""
    p = _native.SdnetSweepParams()
    p.struct_size = ctypes.sizeof(_native.SdnetSweepParams)
    p.B, p.M, p.N, p.K, p.P, p.T = 1, 2, 1, 100, 100, 19
    p.max_gt_objects, p.max_gt_parts = 10, 20
    p.flags = _native.SWEEP_OBJECTS if objects else 0
    for name, t in bufs.items():
        setattr(p, name, t.data_ptr())
    for key, value in shape.items():
        setattr(p, key, value)
    return p


@pytest.mark.parametrize("field", ["conf", "conf_group", "anchor_out", "part_out", "image_scale", "gt_objects", "n_gt_objects",
                                   "gt_parts", "n_gt_parts", "anchor_stats", "part_stats", "anchor_acc", "part_acc",
                                   "gt_part_owner", "cls_group", "csi_stats", "csi_acc", "classif_stats", "classif_acc",
                                   "pred_parts"])
def test_sweep_refuses_a_null_pointer(field):
    """SDNET_E_NULL for each required pointer.  T = 0 as well, so a library that skipped the pointer check would answer
    SDNET_E_SHAPE instead; nothing is ever launched."""
    lib = _native.load()
    assert lib.sdnet_sweep_launch(None, None) == -1
    p = _params(_sweep_buffers(), T=0)
    setattr(p, field, None)
    assert lib.sdnet_sweep_launch(ctypes.byref(p), None) == -1


def test_sweep_argument_errors_are_reported_before_any_launch():
    lib = _native.load()
    bufs = _sweep_buffers()
    p = _params(bufs)
    p.struct_size -= 8
    assert lib.sdnet_sweep_launch(ctypes.byref(p), None) == -7
    # the object-level inputs and outputs are only required with SDNET_SWEEP_OBJECTS: without it, refuse on the shape
    p = _params(bufs, objects=False, T=0)
    for name in ("gt_part_owner", "cls_group", "csi_stats", "csi_acc", "classif_stats", "classif_acc", "pred_parts"):
        setattr(p, name, None)
    assert lib.sdnet_sweep_launch(ctypes.byref(p), None) == -2
    # no ground truth at all: the ground-truth arrays may be NULL
    p = _params(bufs, max_gt_objects=0, max_gt_parts=0, T=_native.MAX_THRESHOLDS + 1)
    p.gt_objects = p.gt_parts = p.gt_part_owner = None
    assert lib.sdnet_sweep_launch(ctypes.byref(p), None) == -2
    for shape in ({"T": 0}, {"T": _native.MAX_THRESHOLDS + 1}, {"K": 1025}, {"P": 1025}, {"K": 0}, {"B": 0}, {"M": 0},
                  {"N": 0}, {"M": 200, "N": 56}, {"max_gt_objects": _native.MAX_GT + 1},
                  {"max_gt_parts": _native.MAX_GT + 1}, {"max_gt_objects": -1}):
        assert lib.sdnet_sweep_launch(ctypes.byref(_params(bufs, **shape)), None) == -2, shape


@pytest.mark.parametrize("grid", [[0.5, 0.4], [0.4, 0.4], [0.1, math.nan], [0.1, math.inf], [-math.inf, 0.1], [],
                                  list(np.linspace(0.0, 1.0, 257))],
                         ids=["decreasing", "repeated", "nan", "inf", "minus-inf", "empty", "257"])
def test_threshold_grid_is_checked(grid):
    with pytest.raises(ValueError):
        ThresholdSweep(_args(), grid)


def test_sixty_five_part_object_is_refused():
    """The object matcher tracks a ground-truth object's parts in a 64-bit mask; the sweep refuses more before any
    device work."""
    K, P, C = 8, 8, 3
    packed = ops._carve(torch.zeros(ops.packed_nbytes(1, K, P, C), dtype=torch.uint8), 1, K, P, C)
    obj = Object("bean", Keypoint("stem", 10.0, 10.0), [Keypoint("leaf", 10.0 + i, 12.0) for i in range(65)])
    sweep = ThresholdSweep(_args(), [0.3, 0.5])
    with pytest.raises(ValueError, match="64"):
        sweep.accumulate_packed(packed, [ImageAnnotation("gt", [obj], img_size=(512, 512))], (128, 128), eval_csi=True)


def test_at_takes_grid_points_only():
    sweep = ThresholdSweep(_args(), [0.1, 0.4, float(np.float32(0.4))])
    assert sweep.at(0.4) is not sweep.at(np.float32(0.4))
    with pytest.raises(KeyError):
        sweep.at(0.2)


def test_curve_and_best_threshold_on_hand_filled_evaluations():
    sweep = ThresholdSweep(_args(), [0.1, 0.3, 0.5, 0.7, 0.9])
    # (tp, npos, ndet) of "bean" and "maize" per threshold; 0.3 and 0.5 tie for the best F1 of "bean" and of the total
    bean = [(3, 6, 10), (3, 6, 6), (2, 6, 2), (1, 6, 1), (0, 6, 0)]
    maize = [(1, 2, 6), (1, 2, 2), (2, 2, 6), (0, 2, 0), (0, 0, 0)]
    for t, b, m in zip(sweep.thresholds, bean, maize):
        sweep.at(t).anchor_eval["bean"] = Evaluation(*b)
        sweep.at(t).anchor_eval["maize"] = Evaluation(*m)
    c = sweep.curve("anchor", "bean")
    np.testing.assert_array_equal(c["threshold"], sweep.thresholds)
    np.testing.assert_array_equal(c["tp"], [3, 3, 2, 1, 0])
    np.testing.assert_array_equal(c["ndet"], [10, 6, 2, 1, 0])
    np.testing.assert_array_equal(c["precision"], [0.3, 0.5, 1.0, 1.0, 0.0])  # 0 / 0 with ground truth: 0
    np.testing.assert_array_equal(c["recall"], [0.5, 0.5, 2 / 6, 1 / 6, 0.0])
    np.testing.assert_array_equal(c["f1_score"], [6 / 16, 6 / 12, 4 / 8, 2 / 7, 0.0])
    assert sweep.best_threshold("anchor", "bean") == 0.3  # tie of 0.5 at 0.3 and 0.5: the lower threshold
    m = sweep.curve("anchor", "maize")
    assert m["precision"][-1] == 1.0 and m["recall"][-1] == 1.0 and m["f1_score"][-1] == 1.0  # nothing to find, nothing found
    assert sweep.best_threshold("anchor", "maize") == 0.9
    total = sweep.curve("anchor")
    np.testing.assert_array_equal(total["tp"], [4, 4, 4, 1, 0])
    np.testing.assert_array_equal(total["npos"], [8, 8, 8, 8, 6])
    np.testing.assert_array_equal(total["f1_score"], [8 / 24, 8 / 16, 8 / 16, 2 / 9, 0.0])
    assert sweep.best_threshold("anchor") == 0.3
    kps = sweep.curve("kps")  # anchors | parts; the part table is empty
    np.testing.assert_array_equal(kps["tp"], total["tp"])
    with pytest.raises(ValueError):
        sweep.curve("objects")
    sweep.reset()
    assert sweep.curve("anchor")["ndet"].tolist() == [0] * 5


# ----------------------------------------------------------------------------------------------- the oracle's sweep
def _golden_case(name):
    """(raw inputs, args, ground truth, image sizes) of one stored evaluator case, labels renamed as eval_objects.json
    evaluated them."""
    meta, arr = load_golden(name)
    _, m, n, _, _ = meta["shape"]
    case, objects = EVAL[name], EVAL_OBJECTS[name]
    rename = objects["rename"]
    raw = arr["raw"]
    inputs = (raw[:, :m], raw[:, m:m + n], raw[:, m + n:m + n + 2], raw[:, m + n + 2:])
    args = SimpleNamespace(labels={rename.get(f"label{i}", f"label{i}"): i for i in range(m)},
                           parts={f"part{i}": i for i in range(n)}, width=case["width"], height=case["height"],
                           dist_threshold=case["dist_threshold"], csi_threshold=objects["csi_threshold"],
                           down_ratio=meta["down_ratio"], conf_threshold=meta["conf"], decoder_dist_thresh=meta["dist"])
    gts = [[(rename.get(nm, nm), x, y, [tuple(k) for k in kps]) for nm, x, y, kps in image["gt"]] for image in case["images"]]
    return meta, inputs, args, gts, [tuple(image["img_size"]) for image in case["images"]]


def golden_expectation(name):
    """{table: {label: (tp, npos, ndet, acc)}} the reference stored for a golden case at its conf."""
    rename = EVAL_OBJECTS[name]["rename"]
    want = {key: {rename.get(l, l): r for l, r in EVAL[name]["result"][key].items()} for key in ("anchor", "part")}
    want.update({key: EVAL_OBJECTS[name]["result"][key] for key in ("csi", "classification")})
    return {key: {l: (r["tp"], r["npos"], r["ndet"], r["acc"]) for l, r in tab.items()} for key, tab in want.items()}


@pytest.mark.parametrize("name", sorted(EVAL_OBJECTS))
def test_oracle_sweep_reproduces_reference_at_each_golden_conf(name):
    """The oracle's sweep over a grid holding the case's conf: at that conf, every table the reference stored, bit for
    bit (same Python-float arithmetic)."""
    meta, inputs, args, gts, sizes = _golden_case(name)
    grid = sorted({0.2, meta["conf"], 0.7})
    tables = SO.sweep(inputs, grid, meta["K"], meta["P"], meta["dist"], gts, sizes, args, sigmoid_fn=torch_sigmoid_fn("cpu"))
    at_conf = tables[grid.index(meta["conf"])]
    for key, want in golden_expectation(name).items():
        assert set(at_conf[key]) == set(want), (name, key)
        for label, (tp, npos, ndet, acc) in want.items():
            assert tuple(at_conf[key][label][:3]) == (tp, npos, ndet), (name, key, label)
            assert at_conf[key][label][3] == acc, (name, key, label)
