"""CPU: the host side of the (threshold x gate) sweep -- SDNET_MAX_GATES, the gate arguments sdnet_sweep_launch refuses
before any launch, ThresholdSweep's gate checks, at / curve / surface / best / best_threshold on hand-filled evaluations
-- and the gate sweep restated the long way round, with the oracle, against the reference's stored evaluator output."""
import ctypes
import math
import shutil
import subprocess
from pathlib import Path

import pytest
import torch

from oracle import sweep_oracle as SO
from structuredetector_b200 import _native
from structuredetector_b200.evaluator import Evaluation, ThresholdSweep
from tests.helpers import torch_sigmoid_fn
from tests.test_sweep import EVAL_OBJECTS, _args, _golden_case, _params, _sweep_buffers, golden_expectation

ROOT = Path(__file__).resolve().parent.parent


def sweep_gates(inputs, thresholds, gates, max_objects, max_parts, gts, img_sizes, args, **kw):
    """The evaluator at every (threshold, gate) of a grid, the long way round: per point (t, g), one
    sdnet_oracle.decode_packed at t with grouping distance g, then evaluate_tables at t (the oracle's threshold sweep
    once per gate).  Returns [threshold][gate] evaluate_tables results."""
    per_gate = [SO.sweep(inputs, thresholds, max_objects, max_parts, g, gts, img_sizes, args, **kw) for g in gates]
    return [[per_gate[j][i] for j in range(len(gates))] for i in range(len(thresholds))]


def test_max_gates_matches_the_header_under_gcc(tmp_path):
    cc = shutil.which("gcc") or shutil.which("cc")
    if cc is None:
        pytest.skip("no C compiler")
    src = ["#include <stdio.h>", '#include "sdnet_decode.h"',
           'int main(void) { printf("%d\\n", SDNET_MAX_GATES); return 0; }']
    (tmp_path / "gates.c").write_text("\n".join(src))
    subprocess.run([cc, "-std=c99", "-Wall", "-Werror", f"-I{ROOT / 'include'}", str(tmp_path / "gates.c"), "-o",
                    str(tmp_path / "gates")], check=True)
    out = subprocess.run([str(tmp_path / "gates")], check=True, capture_output=True, text=True).stdout
    assert int(out) == _native.MAX_GATES == 64


def test_gate_argument_errors_are_reported_before_any_launch():
    """G outside 0..64 is SDNET_E_SHAPE, a NULL gate grid with G >= 1 is SDNET_E_NULL.  The
    zeroed buffers are large enough for every call, so a library that let one through would launch within bounds."""
    lib = _native.load()
    bufs = _sweep_buffers()
    grid = torch.zeros(_native.MAX_GATES + 1, device=bufs["conf"].device)
    for G in (-1, _native.MAX_GATES + 1):
        p = _params(bufs, G=G, dist_abs_grid=grid.data_ptr())
        assert lib.sdnet_sweep_launch(ctypes.byref(p), None) == -2, G
    p = _params(bufs, G=1, dist_abs_grid=None)
    assert lib.sdnet_sweep_launch(ctypes.byref(p), None) == -1
    # the grid is not read with G = 0: a NULL grid is fine there (refused here on T = 0 only)
    p = _params(bufs, G=0, dist_abs_grid=None, T=0)
    assert lib.sdnet_sweep_launch(ctypes.byref(p), None) == -2


@pytest.mark.skipif(torch.cuda.is_available(), reason="no buffer can hold 2^31 output rows: checked only where a call "
                    "that passed the library's checks fails before it launches, for want of a device")
def test_gate_rows_above_int_max_are_refused():
    """B * T fits an int, B * T * G does not: SDNET_E_SHAPE."""
    lib = _native.load()
    bufs = _sweep_buffers()
    grid = torch.zeros(_native.MAX_GATES)
    p = _params(bufs, B=(1 << 31) // (256 * 64) + 1, T=256, G=64, dist_abs_grid=grid.data_ptr())
    assert p.B * p.T <= 0x7fffffff < p.B * p.T * p.G
    assert lib.sdnet_sweep_launch(ctypes.byref(p), None) == -2


@pytest.mark.parametrize("gates", [[], [0.01 * i for i in range(65)], [0.1, math.nan], [0.1, math.inf], [-0.01, 0.1],
                                   [0.1, 0.1], [0.2, 0.1]],
                         ids=["empty", "65", "nan", "inf", "negative", "repeated", "decreasing"])
def test_gate_grid_is_checked(gates):
    with pytest.raises(ValueError):
        ThresholdSweep(_args(), [0.3, 0.5], gates=gates)


def test_gates_and_dist_thresh_together_are_refused():
    with pytest.raises(ValueError, match="both"):
        ThresholdSweep(_args(), [0.3, 0.5], dist_thresh=0.1, gates=[0.05, 0.1])


def test_one_gate_attributes():
    plain = ThresholdSweep(_args(), [0.3, 0.5])
    assert plain.dist_thresh == 0.1 and plain.gates.tolist() == [0.1]
    assert plain.at(0.3) is plain.at(0.3, 0.1)
    gated = ThresholdSweep(_args(), [0.3, 0.5], gates=[0.0, 0.05])
    assert gated.gates.tolist() == [0.0, 0.05]
    assert gated.at(0.3, 0.0) is not gated.at(0.3, 0.05) is not gated.at(0.5, 0.05)
    for bad in ((0.3,), (0.3, 0.1), (0.4, 0.05)):
        with pytest.raises(KeyError):
            gated.at(*bad)
    with pytest.raises(KeyError):
        gated.curve("anchor")
    with pytest.raises(KeyError):
        gated.best_threshold("anchor")


def test_surface_and_best_on_hand_filled_evaluations():
    thresholds, gates = [0.1, 0.3, 0.5], [0.02, 0.05, 0.1, 0.2]
    sweep = ThresholdSweep(_args(), thresholds, gates=gates)
    # "bean" CSI (tp, npos, ndet): the best F1 (0.5) ties across gates at 0.3 (0.05 and 0.1) and across thresholds at
    # 0.05 (0.3 and 0.5): best is (0.3, 0.05), the row-major first
    bean = {0.1: [(1, 6, 10), (2, 6, 10), (2, 6, 10), (1, 6, 10)],
            0.3: [(2, 6, 6), (3, 6, 6), (3, 6, 6), (2, 6, 6)],
            0.5: [(1, 6, 2), (2, 6, 2), (1, 6, 2), (0, 6, 2)]}
    maize = {0.1: [(0, 2, 0)] * 4, 0.3: [(0, 2, 0)] * 4, 0.5: [(0, 2, 0), (0, 2, 0), (0, 2, 0), (2, 2, 2)]}
    for t in thresholds:
        for g, b, m in zip(gates, bean[t], maize[t]):
            sweep.at(t, g).csi_eval["bean"] = Evaluation(*b)
            sweep.at(t, g).csi_eval["maize"] = Evaluation(*m)
    s = sweep.surface("csi", "bean")
    assert s["threshold"].tolist() == thresholds and s["gate"].tolist() == gates
    assert s["tp"].tolist() == [[1, 2, 2, 1], [2, 3, 3, 2], [1, 2, 1, 0]]
    assert s["ndet"].shape == (3, 4) and (s["npos"] == 6).all()
    assert s["f1_score"][1].tolist() == [4 / 12, 6 / 12, 6 / 12, 4 / 12]
    assert s["f1_score"][2, 1] == 4 / 8 == s["f1_score"][1, 1]
    assert s["precision"][2].tolist() == [0.5, 1.0, 0.5, 0.0] and s["recall"][0, 0] == 1 / 6
    assert sweep.best("csi", "bean") == (0.3, 0.05)
    # maize alone: one point finds both objects
    assert sweep.best("csi", "maize") == (0.5, 0.2)
    # the total: bean + maize; (0.5, 0.2) gives (2, 8, 4) -> 1/3, below (0.3, 0.05)'s (3, 8, 6) -> 3/7
    assert sweep.best("csi") == (0.3, 0.05)
    total = sweep.surface("csi")
    assert total["tp"][2, 3] == 2 and total["npos"][2, 3] == 8
    # curve / best_threshold along one gate
    c = sweep.curve("csi", "bean", gate=0.2)
    assert c["threshold"].tolist() == thresholds and c["tp"].tolist() == [1, 2, 0]
    assert sweep.best_threshold("csi", "bean", gate=0.05) == 0.3  # 0.3 and 0.5 tie at 0.5: the lower threshold
    assert sweep.best_threshold("csi", "maize", gate=0.2) == 0.5
    with pytest.raises(ValueError):
        sweep.surface("objects")
    sweep.reset()
    assert (sweep.surface("csi")["ndet"] == 0).all()


def test_best_on_a_one_gate_sweep_is_best_threshold():
    sweep = ThresholdSweep(_args(), [0.1, 0.3, 0.5])
    for t, b in zip(sweep.thresholds, [(3, 6, 10), (3, 6, 6), (2, 6, 2)]):
        sweep.at(t).anchor_eval["bean"] = Evaluation(*b)
    assert sweep.best("anchor", "bean") == (0.3, 0.1) and sweep.best_threshold("anchor", "bean") == 0.3
    assert sweep.surface("anchor", "bean")["f1_score"][:, 0].tolist() == sweep.curve("anchor", "bean")["f1_score"].tolist()


# ----------------------------------------------------------------------------------------------- the oracle's sweep
@pytest.mark.parametrize("name", sorted(EVAL_OBJECTS))
def test_oracle_gate_sweep_reproduces_reference_at_each_golden_point(name):
    """The gate sweep the long way round over a grid holding the case's (conf, decoder_dist_thresh): at that point, every table
    the reference stored, bit for bit; with one gate it is the oracle's threshold sweep."""
    meta, inputs, args, gts, sizes = _golden_case(name)
    grid = sorted({0.2, meta["conf"], 0.7})
    gates = sorted({0.02, meta["dist"], 0.3})
    sig = torch_sigmoid_fn("cpu")
    tables = sweep_gates(inputs, grid, gates, meta["K"], meta["P"], gts, sizes, args, sigmoid_fn=sig)
    assert len(tables) == len(grid) and all(len(row) == len(gates) for row in tables)
    at = tables[grid.index(meta["conf"])][gates.index(meta["dist"])]
    for key, want in golden_expectation(name).items():
        assert set(at[key]) == set(want), (name, key)
        for label, (tp, npos, ndet, acc) in want.items():
            assert tuple(at[key][label][:3]) == (tp, npos, ndet), (name, key, label)
            assert at[key][label][3] == acc, (name, key, label)
    one = sweep_gates(inputs, grid, [meta["dist"]], meta["K"], meta["P"], gts, sizes, args, sigmoid_fn=sig)
    assert [row[0] for row in one] == SO.sweep(inputs, grid, meta["K"], meta["P"], meta["dist"], gts, sizes, args,
                                               sigmoid_fn=sig)
