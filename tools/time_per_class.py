"""Time the tail kernel with one confidence threshold and with per-class thresholds.

    python tools/time_per_class.py [--reps 200] [--label NAME] [--out FILE]

Workloads: cfg5 (1024 images, 512 x 612, K = P = 100) with `blobs` and `noise` maps, and cfg4 (16 images, 256 x 256,
20 classes, 10 kinds, K = P = 500) with `noise` maps.  For each: the tail kernel's device time from
DecodePlan.run_timed (CUDA events between the three kernels; median of --reps decodes after a warm-up), with the scalar
threshold 0.4 and -- where the library takes a table -- with a table of every class at 0.4 and with a table whose
classes alternate between 0.9 and 0.1 (the valid slots are then not a prefix of the score order).  The script runs on
any build that has DecodePlan.run_timed; a build without per-class thresholds reports the scalar only, so the same file
times a parent build next to this one.  Prints one JSON line (card name and power limit included).
"""
import argparse
import inspect
import json
import statistics
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from structuredetector_b200 import ops  # noqa: E402
from structuredetector_b200.synth import CONFIGS, make_raw, split_outputs  # noqa: E402

WORKLOADS = [("cfg5", "blobs"), ("cfg5", "noise"), ("cfg4", "noise")]


def tail_ms(plan, outs, dist_abs, reps, **kw):
    args = (outs["anchor_hm"], outs["part_hm"], outs["offsets"], outs["embeddings"], ops._f32(0.4), dist_abs)
    for _ in range(10):
        plan.run_timed(*args, **kw)
    return statistics.median(plan.run_timed(*args, **kw)[2] for _ in range(reps))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--label", default="")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: the tail kernel's time is measured on the GPU only")
    dev = torch.device("cuda", 0)
    per_class = "conf_class" in inspect.signature(ops.DecodePlan.run_timed).parameters
    res = {"label": a.label, "per_class_supported": per_class, "reps": a.reps, "tail_ms": {}}
    query = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True)
    res["gpu"] = query.stdout.strip()
    for name, mode in WORKLOADS:
        cfg = CONFIGS[name]
        m, n = cfg.labels, cfg.parts
        raw = make_raw(cfg, mode).to(dev)
        outs = split_outputs(raw, m, n)
        plan = ops.DecodePlan(dev, cfg.batch, m, n, cfg.height, cfg.width, cfg.max_objects, cfg.max_parts)
        dist_abs = ops._f32(cfg.dist_thresh * min(cfg.width, cfg.height))
        row = {"scalar": tail_ms(plan, outs, dist_abs, a.reps)}
        if per_class:
            equal = torch.full((m + n,), ops._f32(0.4), dtype=torch.float32, device=dev)
            mixed = torch.tensor([0.9 if c % 2 else 0.1 for c in range(m + n)], dtype=torch.float32, device=dev)
            row["table_equal"] = tail_ms(plan, outs, dist_abs, a.reps, conf_class=equal)
            row["table_mixed"] = tail_ms(plan, outs, dist_abs, a.reps, conf_class=mixed)
            row["scalar_again"] = tail_ms(plan, outs, dist_abs, a.reps)
        res["tail_ms"][f"{name}-{mode}"] = row
        del raw, outs, plan
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
