"""Time the (threshold x gate) sweep against one threshold sweep per gate, on 1024 cfg5 images.

    python tools/time_sweep_gates.py [--images 1024] [--baseline-lib PATH] [--out FILE]

Workload: tools/time_sweep.py's (cfg5 `blobs` maps, 32 generated images repeated to the batch, decoded once; its ground
truth), T = 19 thresholds 0.05 ... 0.95 and G = 8 gates 0.02 ... 0.16.  Reports
  - sdnet_sweep_launch's device time (CUDA events over many launches after a warm-up) at G = 1 and G = 8;
  - the wall time of ThresholdSweep(..., gates=8 gates).accumulate_packed(..., True, True), ending in a synchronise,
    against eight one-gate ThresholdSweeps on the same decode, with the bytes each copies to the host and whether both
    give identical tables at all 152 points;
  - with --baseline-lib (a build of the parent commit's library, whose SdnetSweepParams ends before `G`): G = 0 of this
    build against that build, alternating the two in rounds.
"""
import argparse
import ctypes
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path
from types import SimpleNamespace

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
from structuredetector_b200 import _native, ops  # noqa: E402
from structuredetector_b200.evaluator import ThresholdSweep  # noqa: E402
from structuredetector_b200.synth import CONFIGS, make_raw, split_outputs  # noqa: E402
from time_sweep import GRID, event_ms, ground_truth, same_tables  # noqa: E402

GATES = [round(0.02 * i, 2) for i in range(1, 9)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=1024)
    ap.add_argument("--baseline-lib", default=None)
    ap.add_argument("--out", default=None)
    opt = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("no CUDA device: nothing to time")
    cfg, B, dev = CONFIGS["cfg5"], opt.images, torch.device("cuda:0")
    K, P, dist = cfg.max_objects, cfg.max_parts, cfg.dist_thresh
    raw = make_raw(cfg, "blobs", batch=32).to(dev).repeat((B + 31) // 32, 1, 1, 1)[:B].contiguous()
    outs = split_outputs(raw, cfg.labels, cfg.parts)
    out_size = (cfg.width, cfg.height)
    packed = ops.decode_packed(outs, K, P, 0.05, dist)
    anns = ground_truth(packed, B, seed=5)
    args = SimpleNamespace(labels={"bean": 0, "maize": 1}, parts={"leaf": 0}, width=4 * cfg.width, height=4 * cfg.height,
                           dist_threshold=0.05, conf_threshold=0.4, down_ratio=4.0, csi_threshold=0.5,
                           decoder_dist_thresh=dist)
    res = {"gpu": torch.cuda.get_device_name(dev), "images": B, "thresholds": len(GRID), "gates": GATES, "K": K, "P": P}
    try:
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                            capture_output=True, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError):
        res["power_limit"] = "unknown"

    # ---- the 2-D sweep call, end to end, against one 1-D sweep per gate on the same decode
    sweep = ThresholdSweep(args, GRID, gates=GATES)
    walls = []
    for _ in range(4):
        sweep.reset()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sweep.accumulate_packed(packed, anns, out_size, eval_csi=True, eval_classif=True)
        torch.cuda.synchronize()
        walls.append(time.perf_counter() - t0)
    res["grid_call_ms"] = [round(1e3 * w, 2) for w in walls[1:]]
    res["grid_copy_bytes"] = sweep.last_copy_bytes
    loops, per_gate = [], None
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        per_gate = []
        for g in GATES:
            one = ThresholdSweep(args, GRID, dist_thresh=g)
            one.accumulate_packed(packed, anns, out_size, eval_csi=True, eval_classif=True)
            per_gate.append(one)
        torch.cuda.synchronize()
        loops.append(time.perf_counter() - t0)
    res["per_gate_loop_ms"] = [round(1e3 * w, 2) for w in loops[1:]]
    res["per_gate_copy_bytes"] = sum(one.last_copy_bytes for one in per_gate)
    res["identical_points"] = sum(same_tables(sweep.at(t, g), one.at(t)) and same_tables(one.at(t), sweep.at(t, g))
                                  for g, one in zip(GATES, per_gate) for t in GRID)
    res["points"] = len(GRID) * len(GATES)
    res["loop_over_grid"] = round(statistics.median(loops[1:]) / statistics.median(walls[1:]), 2)

    # ---- the kernel alone: the launch the call makes, at G = 1 and G = 8, and at G = 0
    ev0 = sweep.at(GRID[0], GATES[0])
    (gt_a, n_a, wa), (gt_p, n_p, wp), scale, owner = ev0._pack_ground_truth(anns, dev)
    T, M, N = len(GRID), 2, 1
    i32, f64 = {"dtype": torch.int32, "device": dev}, {"dtype": torch.float64, "device": dev}
    conf = torch.tensor(GRID, **f64)
    conf_group = torch.tensor([ops._f32(t) for t in GRID], dtype=torch.float32, device=dev)
    gate_abs = torch.tensor([ops._f32(g * min(out_size)) for g in GATES], dtype=torch.float32, device=dev)
    groups = ev0._classification_groups(dev)
    R = T * len(GATES)
    bufs = [torch.empty(B, T, M, 3, **i32), torch.empty(B, T, N, 3, **i32), torch.empty(B, T, K, **f64),
            torch.empty(B, T, P, **f64), torch.empty(B, R, M, 3, **i32), torch.empty(B, R, K, **f64),
            torch.empty(B, R, 20, 3, **i32), torch.empty(B, R, K, **f64), torch.empty(B, R, K, **i32)]

    def params(cls, G):
        p = cls()
        p.struct_size = ctypes.sizeof(p)
        p.B, p.M, p.N, p.K, p.P, p.T, p.max_gt_objects, p.max_gt_parts = B, M, N, K, P, T, wa, wp
        p.flags, p.sx, p.sy, p.csi_threshold = _native.SWEEP_OBJECTS, 4.0, 4.0, 0.5
        p.dist_abs_f32 = ops._f32(dist * min(out_size))
        if G:
            p.G, p.dist_abs_grid = G, gate_abs.data_ptr()
        p.conf, p.conf_group = conf.data_ptr(), conf_group.data_ptr()
        p.anchor_out, p.part_out, p.image_scale = packed.anchor_out.data_ptr(), packed.part_out.data_ptr(), scale.data_ptr()
        p.gt_objects, p.n_gt_objects, p.gt_parts, p.n_gt_parts = gt_a.data_ptr(), n_a.data_ptr(), gt_p.data_ptr(), n_p.data_ptr()
        p.gt_part_owner, p.cls_group = owner.data_ptr(), groups.data_ptr()
        (p.anchor_stats, p.part_stats, p.anchor_acc, p.part_acc, p.csi_stats, p.csi_acc, p.classif_stats, p.classif_acc,
         p.pred_parts) = (x.data_ptr() for x in bufs)
        return p

    lib, stream = _native.load(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def runner(which, p):
        return lambda: _native.check(which.sdnet_sweep_launch(ctypes.byref(p), stream), "sdnet_sweep_launch")

    for G, key in ((1, "kernel_g1_ms"), (len(GATES), "kernel_g8_ms")):
        run = runner(lib, params(_native.SdnetSweepParams, G))
        event_ms(run, 5)
        res[key] = [round(event_ms(run, 50), 4) for _ in range(3)]

    if opt.baseline_lib:
        base = ctypes.CDLL(str(Path(opt.baseline_lib).resolve()))
        v9 = type("SdnetSweepParamsV9", (ctypes.Structure,), {"_fields_": _native.SdnetSweepParams._fields_[:-2]})
        base.sdnet_sweep_launch.restype = ctypes.c_int
        base.sdnet_sweep_launch.argtypes = [ctypes.POINTER(v9), ctypes.c_void_p]
        new_fn, base_fn = runner(lib, params(_native.SdnetSweepParams, 0)), runner(base, params(v9, 0))
        event_ms(new_fn, 5)
        event_ms(base_fn, 5)
        rounds = {"this": [], "baseline": []}
        for _ in range(8):
            rounds["this"].append(round(event_ms(new_fn, 50), 4))
            rounds["baseline"].append(round(event_ms(base_fn, 50), 4))
        res["kernel_g0_ms_rounds"] = rounds
        res["kernel_g0_ms_median"] = {k: round(statistics.median(v), 4) for k, v in rounds.items()}
        res["kernel_g0_ms_spread"] = {k: round(max(v) - min(v), 4) for k, v in rounds.items()}
    text = json.dumps(res, indent=1)
    print(text)
    if opt.out:
        Path(opt.out).parent.mkdir(parents=True, exist_ok=True)
        Path(opt.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
