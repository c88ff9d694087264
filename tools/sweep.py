"""Time several builds of the decode library side by side in ONE process (kernel experiments).

    python tools/sweep.py [--images 1024,128] [--modes noise,blobs] [--dtype f32] [--reps 20] name ...

``name`` = ``base`` (the product library) or a build made by ``tools/xbuild.sh <name>``
(``structuredetector_b200/csrc/exp/lib_<name>.so``).  For every (build, images, mode): the per-kernel
device times of ``sdnet_decode_launch_timed`` (mean of --reps), the peaks kernel's fraction of the
measured copy peak, candidates per plane, and whether the packed result equals the base build's
bit for bit.  Output: one line per case + gpurun_out/sweep.json."""
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
    ap.add_argument("names", nargs="+")
    ap.add_argument("--images", default="1024,128")
    ap.add_argument("--modes", default="noise,blobs")
    ap.add_argument("--dtype", default="f32")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default="gpurun_out/sweep.json")
    args = ap.parse_args()
    cfg = CONFIGS["cfg5"]
    dev = torch.device("cuda:0")
    tdtype = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}[args.dtype]
    esize = 4 if args.dtype == "f32" else 2
    peak = 6549.1
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        peak = float(json.loads(pk.read_text())["hbm_gbs"])
    M, N, H, W, K, P = cfg.labels, cfg.parts, cfg.height, cfg.width, cfg.max_objects, cfg.max_parts
    conf = float(torch.tensor(cfg.conf_threshold, dtype=tdtype))
    dist = float(torch.tensor(cfg.dist_thresh * min(W, H), dtype=torch.float32))

    libs = {}
    for name in args.names:
        path = _native.LIB_PATH if name == "base" else ROOT / "structuredetector_b200" / "csrc" / "exp" / f"lib_{name}.so"
        libs[name] = _native.load_from(path)
    results = []
    for mode in args.modes.split(","):
        uniq = make_raw(cfg, mode, batch=32).to(dev)
        for images in map(int, args.images.split(",")):
            idx = torch.arange(images, device=dev) % 32
            raw = uniq[idx].contiguous().to(tdtype)
            o = split_outputs(raw, M, N)
            ref_blob = None
            for name, lib in libs.items():
                plan = ops.DecodePlan(dev, images, M, N, H, W, K, P, tdtype, lib=lib)
                call = (o["anchor_hm"], o["part_hm"], o["offsets"], o["embeddings"], conf, dist)
                for _ in range(3):
                    plan.run(*call)
                torch.cuda.synchronize()
                kms = [plan.run_timed(*call) for _ in range(args.reps)]
                # throughput of back-to-back decodes on one stream (no pipelining): the step time a single caller sees
                ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                ev0.record()
                for _ in range(args.reps):
                    plan.run(*call)
                ev1.record()
                torch.cuda.synchronize()
                serial_ms = ev0.elapsed_time(ev1) / args.reps
                out = plan.out
                n_det = out.blob.numel() - out.diag.numel() * 4
                blob = out.blob[:n_det].clone()
                same = None
                if ref_blob is None:
                    ref_blob = blob
                else:
                    same = bool(torch.equal(blob, ref_blob))
                pm = statistics.mean(k[0] for k in kms)
                pmin = min(k[0] for k in kms)
                r = {"name": name, "mode": mode, "images": images, "peaks_ms": pm, "peaks_min_ms": pmin,
                     "exact_ms": statistics.mean(k[1] for k in kms), "tail_ms": statistics.mean(k[2] for k in kms),
                     "serial_step_ms": serial_ms, "frac": images * (M + N) * H * W * esize / (pm * 1e-3) / 1e9 / peak,
                     "cand_per_plane": float(out.diag[:, 0].float().mean()), "exact_planes": int(out.diag[:, 1].sum()),
                     "same_as_first": same}
                try:
                    r["sched"] = plan.schedule(*call[:4])
                except Exception as exc:  # noqa: BLE001
                    r["sched"] = repr(exc)
                results.append(r)
                print(f"{name:32s} {mode:6s} {images:5d}  peaks {pm:.4f} (min {pmin:.4f}) frac {r['frac']:.3f}  tail {r['tail_ms']:.4f}  "
                      f"serial {serial_ms:.4f}  cand {r['cand_per_plane']:.0f}  same {same}", flush=True)
                del plan
    Path(args.out).parent.mkdir(exist_ok=True)
    Path(args.out).write_text(json.dumps(results, indent=1))


if __name__ == "__main__":
    main()
