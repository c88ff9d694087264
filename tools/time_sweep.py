"""Time the evaluator's threshold sweep against the per-threshold loop it replaces, on 1024 cfg5 images.

    python tools/time_sweep.py [--images 1024] [--baseline-lib PATH] [--out FILE]

Workload: cfg5 `blobs` maps (32 generated images repeated to the batch), decoded once; ground truth derived from every
image's detections with its own seed: jittered, 15 % dropped, 2 spurious objects per image, 1 to 6 parts per object.
Grid: T = 19 thresholds, 0.05 ... 0.95.  Reports
  - sdnet_sweep_launch's device time (CUDA events over many launches after a warm-up);
  - the wall time of ThresholdSweep.accumulate_packed(..., True, True), ending in a synchronise;
  - the wall time of the loop it replaces: per threshold ops.decode_packed + Evaluator.accumulate_packed(..., True, True);
  - whether both produce the same tables, and the bytes the sweep copies to the host.
With --baseline-lib (a build of the parent commit's library), also sdnet_match_objects_kernel of that build and of
this one, alternating the two in rounds, to show the move of its body into a shared device function costs nothing.
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

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from structuredetector_b200 import ImageAnnotation, Keypoint, Object, _native, ops  # noqa: E402
from structuredetector_b200.evaluator import Evaluator, ThresholdSweep  # noqa: E402
from structuredetector_b200.synth import CONFIGS, make_raw, split_outputs  # noqa: E402

GRID = [round(0.05 * i, 2) for i in range(1, 20)]


def ground_truth(packed, B, seed):
    a = packed.anchor_out.cpu().numpy()
    rng = np.random.default_rng(seed)
    names = ("bean", "maize")
    anns = []
    for b in range(B):
        objs = []
        for x, y, s, c in a[b]:
            if s <= 0.2 or rng.random() < 0.15:
                continue
            ax, ay = 4 * x + rng.normal(0, 6), 4 * y + rng.normal(0, 6)
            parts = [Keypoint("leaf", ax + rng.normal(0, 25), ay + rng.normal(0, 25)) for _ in range(rng.integers(1, 7))]
            objs.append(Object(names[int(c)], Keypoint("stem", ax, ay), parts))
        for _ in range(2):
            ax, ay = rng.uniform(0, 2448), rng.uniform(0, 2048)
            objs.append(Object(str(rng.choice(names)), Keypoint("stem", ax, ay),
                               [Keypoint("leaf", ax + rng.normal(0, 25), ay) for _ in range(rng.integers(1, 7))]))
        anns.append(ImageAnnotation("gt", objs, img_size=(2448, 2048)))
    return anns


def event_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def same_tables(a, b):
    for table in ("anchor_eval", "part_eval", "csi_eval", "classification_eval"):
        for label, e in getattr(b, table).items():
            g = getattr(a, table)[label]
            if (g.tp, g.npos, g.ndet, g.acc) != (e.tp, e.npos, e.ndet, e.acc):
                return False
    return True


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
    res = {"gpu": torch.cuda.get_device_name(dev), "images": B, "thresholds": len(GRID), "K": K, "P": P,
           "gt_objects_per_image": float(np.mean([len(x.objects) for x in anns]))}
    try:
        res["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                                            capture_output=True, text=True, check=True).stdout.strip()
    except (OSError, subprocess.CalledProcessError):
        res["power_limit"] = "unknown"

    # ---- the sweep call, end to end
    sweep = ThresholdSweep(args, GRID, dist_thresh=dist)
    walls = []
    for _ in range(4):
        sweep.reset()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sweep.accumulate_packed(packed, anns, out_size, eval_csi=True, eval_classif=True)
        torch.cuda.synchronize()
        walls.append(time.perf_counter() - t0)
    res["sweep_call_ms"] = [round(1e3 * w, 2) for w in walls[1:]]
    res["sweep_copy_bytes"] = sweep.last_copy_bytes

    # ---- the loop it replaces
    loops, evs = [], None
    for _ in range(2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        evs = []
        for t in GRID:
            ev = Evaluator(args)
            ev.accumulate_packed(ops.decode_packed(outs, K, P, t, dist), anns, out_size, conf_thresh=t, eval_csi=True,
                                 eval_classif=True)
            evs.append(ev)
        torch.cuda.synchronize()
        loops.append(time.perf_counter() - t0)
    res["loop_ms"] = [round(1e3 * w, 2) for w in loops]
    res["identical"] = all(same_tables(sweep.at(t), ev) for t, ev in zip(GRID, evs))
    res["loop_over_sweep"] = round(min(loops) / statistics.median(walls[1:]), 2)

    # ---- the kernel alone: the same launch the call makes
    ev0 = sweep.at(GRID[0])
    (gt_a, n_a, wa), (gt_p, n_p, wp), scale, owner = ev0._pack_ground_truth(anns, dev)
    T, M, N = len(GRID), 2, 1
    i32, f64 = {"dtype": torch.int32, "device": dev}, {"dtype": torch.float64, "device": dev}
    conf = torch.tensor(GRID, **f64)
    conf_group = torch.tensor([ops._f32(t) for t in GRID], dtype=torch.float32, device=dev)
    groups = ev0._classification_groups(dev)
    bufs = [torch.empty(B, T, M, 3, **i32), torch.empty(B, T, N, 3, **i32), torch.empty(B, T, K, **f64),
            torch.empty(B, T, P, **f64), torch.empty(B, T, M, 3, **i32), torch.empty(B, T, K, **f64),
            torch.empty(B, T, 20, 3, **i32), torch.empty(B, T, K, **f64), torch.empty(B, T, K, **i32)]
    p = _native.SdnetSweepParams()
    p.struct_size = ctypes.sizeof(p)
    p.B, p.M, p.N, p.K, p.P, p.T, p.max_gt_objects, p.max_gt_parts = B, M, N, K, P, T, wa, wp
    p.flags, p.dist_abs_f32, p.sx, p.sy, p.csi_threshold = _native.SWEEP_OBJECTS, ops._f32(dist * min(out_size)), 4.0, 4.0, 0.5
    p.conf, p.conf_group = conf.data_ptr(), conf_group.data_ptr()
    p.anchor_out, p.part_out, p.image_scale = packed.anchor_out.data_ptr(), packed.part_out.data_ptr(), scale.data_ptr()
    p.gt_objects, p.n_gt_objects, p.gt_parts, p.n_gt_parts = gt_a.data_ptr(), n_a.data_ptr(), gt_p.data_ptr(), n_p.data_ptr()
    p.gt_part_owner, p.cls_group = owner.data_ptr(), groups.data_ptr()
    (p.anchor_stats, p.part_stats, p.anchor_acc, p.part_acc, p.csi_stats, p.csi_acc, p.classif_stats, p.classif_acc,
     p.pred_parts) = (x.data_ptr() for x in bufs)
    lib, stream = _native.load(), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    launch = lambda: _native.check(lib.sdnet_sweep_launch(ctypes.byref(p), stream), "sdnet_sweep_launch")  # noqa: E731
    event_ms(launch, 5)
    res["sweep_kernel_ms"] = [round(event_ms(launch, 50), 4) for _ in range(3)]
    res["pair_distances"] = B * T * K * P

    # ---- sdnet_match_objects_kernel: this build against the baseline build, alternating
    if opt.baseline_lib:
        base = ctypes.CDLL(str(Path(opt.baseline_lib).resolve()))
        base.sdnet_match_objects_launch.restype = ctypes.c_int
        base.sdnet_match_objects_launch.argtypes = lib.sdnet_match_objects_launch.argtypes
        packed40 = ops.decode_packed(outs, K, P, 0.4, dist)
        o = _native.SdnetObjectMatchParams()
        o.struct_size = ctypes.sizeof(o)
        o.B, o.M, o.N, o.K, o.P, o.max_gt_objects, o.max_gt_parts = B, M, N, K, P, wa, wp
        o.conf, o.sx, o.sy, o.csi_threshold = 0.4, 4.0, 4.0, 0.5
        o.anchor_out, o.part_out, o.assign = packed40.anchor_out.data_ptr(), packed40.part_out.data_ptr(), packed40.assign.data_ptr()
        o.image_scale, o.gt_objects, o.n_gt_objects = scale.data_ptr(), gt_a.data_ptr(), n_a.data_ptr()
        o.gt_parts, o.gt_part_owner, o.n_gt_parts, o.cls_group = gt_p.data_ptr(), owner.data_ptr(), n_p.data_ptr(), groups.data_ptr()
        outs_new = [torch.empty(B, M, 3, **i32), torch.empty(B, K, **f64), torch.empty(B, 20, 3, **i32),
                    torch.empty(B, K, **f64), torch.empty(B, K, **i32)]
        outs_base = [torch.empty_like(x) for x in outs_new]

        def runner(which, bufs_):
            def run():
                o.csi_stats, o.csi_acc, o.classif_stats, o.classif_acc, o.pred_parts = (x.data_ptr() for x in bufs_)
                _native.check(which.sdnet_match_objects_launch(ctypes.byref(o), stream), "sdnet_match_objects_launch")
            return run

        new_fn, base_fn = runner(lib, outs_new), runner(base, outs_base)
        event_ms(new_fn, 5)
        event_ms(base_fn, 5)
        rounds = {"this": [], "baseline": []}
        for _ in range(8):
            rounds["this"].append(round(1e3 * event_ms(new_fn, 100), 2))
            rounds["baseline"].append(round(1e3 * event_ms(base_fn, 100), 2))
        res["match_objects_us"] = rounds
        res["match_objects_same_output"] = all(torch.equal(a, b) if a.dtype != torch.float64 else
                                               torch.equal(torch.nan_to_num(a, nan=-1.0), torch.nan_to_num(b, nan=-1.0))
                                               for a, b in zip(outs_new, outs_base))
    text = json.dumps(res, indent=1)
    print(text)
    if opt.out:
        Path(opt.out).parent.mkdir(parents=True, exist_ok=True)
        Path(opt.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
