"""Time the peaks kernel's floor hint on 1024 distinct cfg5 images (not the benchmark's 32 images tiled 32 times).

    python tools/time_floor_hint.py [--reps 30] [--dtype f32] [--out results.json]

The images are ``make_raw(cfg5, mode, batch=32, seed=s)`` for 32 seeds, copied to the device.  For noise and blobs, one
plan decodes with hints (the default) and one with SDNET_FLAG_NO_FLOOR_HINT, alternating rep by rep in this process.
Per build: the median per-kernel device times of ``sdnet_decode_launch_timed``, the step time of back-to-back decodes,
candidates per plane, and the planes the exact select redid (a hint that pruned too much).  Every rep's packed outputs
must be equal bit for bit between the two, ``diag`` (candidate counts) excepted."""
import argparse
import json
import statistics
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import torch  # noqa: E402

from structuredetector_b200 import _native, ops  # noqa: E402
from structuredetector_b200.synth import CONFIGS, make_raw, split_outputs  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--dtype", default="f32", choices=("f32", "f16", "bf16"))
    ap.add_argument("--out", default=None, help="also write the results as JSON to this file")
    args = ap.parse_args()
    cfg = CONFIGS["cfg5"]
    dev = torch.device("cuda:0")
    tdtype = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}[args.dtype]
    M, N, H, W, K, P = cfg.labels, cfg.parts, cfg.height, cfg.width, cfg.max_objects, cfg.max_parts
    conf = float(torch.tensor(cfg.conf_threshold, dtype=tdtype))
    dist = ops._f32(cfg.dist_thresh * min(W, H))
    builds = {"hint": 0, "no_hint": _native.FLAG_NO_FLOOR_HINT}
    result = {"device": torch.cuda.get_device_name(dev), "dtype": args.dtype, "images": 1024, "reps": args.reps, "modes": {}}
    for mode in ("noise", "blobs"):
        raw = torch.cat([make_raw(cfg, mode, batch=32, seed=1000 + s) for s in range(32)]).to(tdtype).to(dev)
        o = split_outputs(raw, M, N)
        call = (o["anchor_hm"], o["part_hm"], o["offsets"], o["embeddings"], conf, dist)
        plans = {name: ops.DecodePlan(dev, raw.shape[0], M, N, H, W, K, P, tdtype) for name in builds}
        for name, plan in plans.items():
            for _ in range(3):
                plan.run(*call, flags=builds[name])
        torch.cuda.synchronize()
        kms = {name: [] for name in builds}
        redone = {name: [] for name in builds}
        cand = {name: [] for name in builds}
        for _ in range(args.reps):
            blobs = {}
            for name, plan in plans.items():
                kms[name].append(plan.run_timed(*call, flags=builds[name]))
                out = plan.out
                redone[name].append(int(out.diag[:, 1].sum()))
                cand[name].append(float(out.diag[:, 0].float().mean()))
                blobs[name] = out.blob[:out.blob.numel() - out.diag.numel() * 4].clone()
            if not torch.equal(blobs["hint"], blobs["no_hint"]):
                raise SystemExit(f"{mode}: packed outputs differ with hints on and off")
        steps = {}
        for _ in range(2):  # alternating back-to-back windows, the second one kept
            for name, plan in plans.items():
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
                for _ in range(args.reps):
                    plan.run(*call, flags=builds[name])
                ev1.record()
                torch.cuda.synchronize()
                steps[name] = ev0.elapsed_time(ev1) / args.reps
        rows = {}
        for name in builds:
            rows[name] = {
                "peaks_ms": statistics.median(k[0] for k in kms[name]),
                "exact_ms": statistics.median(k[1] for k in kms[name]),
                "tail_ms": statistics.median(k[2] for k in kms[name]),
                "serial_step_ms": steps[name],
                "candidates_per_plane_mean": statistics.mean(cand[name]),
                "planes_via_exact_select_max": max(redone[name]),
                "planes_via_exact_select_mean": statistics.mean(redone[name]),
            }
            r = rows[name]
            print(f"{mode:6s} {name:8s} peaks {r['peaks_ms']:.4f} ms  exact {r['exact_ms']:.4f}  tail {r['tail_ms']:.4f}  "
                  f"step {r['serial_step_ms']:.4f}  cand/plane {r['candidates_per_plane_mean']:.0f}  "
                  f"exact-select planes max {r['planes_via_exact_select_max']}", flush=True)
        rows["peaks_gain"] = 1.0 - rows["hint"]["peaks_ms"] / rows["no_hint"]["peaks_ms"]
        rows["step_gain"] = 1.0 - rows["hint"]["serial_step_ms"] / rows["no_hint"]["serial_step_ms"]
        rows["bit_exact"] = True
        print(f"{mode:6s} peaks kernel {100 * rows['peaks_gain']:.1f} % faster, step {100 * rows['step_gain']:.1f} % faster, "
              f"outputs bit-exact", flush=True)
        result["modes"][mode] = rows
        del plans
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
