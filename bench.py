#!/usr/bin/env python
"""bench.py -- decoded images/s of the SDNet decoding path on 1..8 B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--mode both|noise|blobs]
                    [--workload cfg5|cfg2|cfg3|cfg4] [--dtype f32|f16|bf16] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

Default workload: BASELINE.json configs[4] ("cfg5"): a global batch of 1024 network outputs of the
2448x2048-input configuration, i.e. raw (1024, 2+1+4, 512, 612) fp32, K = P = 100, conf 0.4, dist 0.1,
split evenly over the ranks (strong scaling).  One *step* = one decode of the whole global batch: every
rank decodes its shard (3 kernels through the C ABI) and -- for N > 1 -- the packed detections end up on
every rank (fused into the tail kernel's stores, or ncclAllGather).  Inputs are resident in HBM and
larger than L2 (8.98 GB / N per rank); the small workloads (cfg2-cfg4) rotate over enough distinct input
buffers to exceed L2 twice.

Both synthetic modes of SURVEY 8(d) are timed (``modes``); the headline ``value`` is the SLOWER one.
Outside the timed region the very plan that was timed is checked, bit for bit, against the reference's
own op sequence on the device (``parity_checked``) and, for N > 1, every rank checks the gathered result
against a single-GPU decode of the whole batch (``gather_bit_exact``).

``--dump-outputs DIR`` writes what the last timed step of each mode returned (the packed detections of the whole
global batch, as rank 0 holds them after the gather) as ``DIR/<mode>_<field>.npy``, so that two builds can be
compared output for output on identical inputs.  Past 64 MB a fixed sample of images is written instead, and
``DIR/<mode>_images.npy`` lists which.

Prints ONE JSON line.  ``--impl reference`` times the reference decoder on the host CPU instead: the
UNMODIFIED reference ``Decoder`` from ``oracle/_ref`` when that archive exists (``kind: "reference"``),
else the port ``oracle/torch_port.py`` (``kind: "port"``), all host threads, on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

UNIQUE_IMAGES = 32  # distinct synthetic images generated on the CPU; tiled to fill a cfg5 shard
CPU_BATCH = 16  # images per CPU-baseline step (the reference's cfg3 batch)
L2_BYTES = 126 * 1024 * 1024
DUMP_BYTES = 63 << 20  # --dump-outputs array data over all modes; the rest of 64 MB is left for the .npy headers


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=("ours", "reference"), default="ours")
    ap.add_argument("--mode", choices=("both", "noise", "blobs"), default="both",
                    help="synthetic input mode(s); 'both' times noise and blobs and headlines the slower")
    ap.add_argument("--workload", choices=("cfg5", "cfg2", "cfg3", "cfg4"), default="cfg5",
                    help="BASELINE.json config: cfg5 = the metric's (1024 x 2448x2048 inputs); cfg2-cfg4 = the other configs")
    ap.add_argument("--dtype", choices=("f32", "f16", "bf16"), default="f32",
                    help="element type of the network outputs (f32 = the headline; f16/bf16 = the --amp validation path)")
    ap.add_argument("--global-batch", type=int, default=None, help="override the workload's batch (debug only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-objects", action="store_true", help="skip the Decoder -> Python objects legs")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity checks outside the timed region")
    ap.add_argument("--e2e-steps", type=int, default=4)
    ap.add_argument("--pipeline", type=int, default=0,
                    help="decodes in flight: consecutive steps alternate between this many plans/streams; 0 = auto "
                         "(3 for shards of >= 512 images, 4 down to 161, 12 for smaller ones)")
    ap.add_argument("--gather-wait", choices=("lazy", "step"), default="lazy",
                    help="fused gather: wait for every rank's rows after each step, or only before a result buffer is "
                         "written again (two runs later) and at the end of the timed region")
    ap.add_argument("--gather", choices=("fused", "nccl"), default="fused",
                    help="N > 1: tail kernel stores into every peer (symmetric memory) + barrier, or ncclAllGather")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the packed detections of the last timed step of each mode as "
                         "DIR/<mode>_<field>.npy (float32, or float64 for integer fields; a fixed sample of images "
                         "when they exceed 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's results: not available with --impl reference")
    return args


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    REASONS = {  # nvmlClocksEventReasons bits
        0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
        0x80: "hw_power_brake_slowdown",
    }

    def __init__(self, index: int, period_s: float = 0.005):
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception as exc:  # noqa: BLE001
            self.nv, self.error = None, repr(exc)

    def _loop(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                bits = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                for bit, name in self.REASONS.items():
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if self.nv is None or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0,
                    "note": "NVML unavailable" if self.nv is None else "timed region shorter than one sample"}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except (ValueError, IndexError):
            pass
    return local_rank


def workload_name(cfg, dtype="f32") -> str:
    what = {"cfg5": "2448x2048 inputs", "cfg3": "2448x2048 inputs", "cfg2": "512x512 inputs",
            "cfg4": "1024x1024 inputs, 20 labels + 10 parts"}.get(cfg.name, "inputs")
    return (f"{cfg.name}: global batch {cfg.batch} of {what} -> raw ({cfg.batch}, {cfg.channels}, {cfg.height}, "
            f"{cfg.width}) {'fp32' if dtype == 'f32' else dtype}, K=P={cfg.max_objects}, conf {cfg.conf_threshold}, "
            f"dist {cfg.dist_thresh}")


# ----------------------------------------------------------------------------- CPU reference arm
def cpu_reference_rate(cfg, mode: str, seconds: float, steps: int | None = None, warmup: int = 1, threads: int | None = None,
                       force_port: bool = False):
    """images/s of the reference decoder on the host CPU: the unmodified reference ``Decoder`` when
    ``oracle/_ref`` holds it (``kind: "reference"``), else the oracle port of its op sequence."""
    import torch

    from oracle import torch_port
    from oracle.build_ref import load_reference_decoders
    from structuredetector_b200.synth import make_raw, split_outputs

    # all the host threads the process may use (torchrun exports OMP_NUM_THREADS=1, which would make
    # the CPU arm ten times slower than the same code started with plain `python`)
    try:
        usable = len(os.sched_getaffinity(0))
    except AttributeError:
        usable = os.cpu_count() or 1
    torch.set_num_threads(max(1, usable if threads is None else threads))
    batch = min(CPU_BATCH, cfg.batch)
    raw = make_raw(cfg, mode, batch=batch)
    outs = split_outputs(raw, cfg.labels, cfg.parts)
    labels = {i: f"label{i}" for i in range(cfg.labels)}
    parts = {i: f"part{i}" for i in range(cfg.parts)}
    ref = None if force_port else load_reference_decoders()
    if ref is not None:
        from types import SimpleNamespace

        dec = ref.Decoder(SimpleNamespace(_r_labels=labels, _r_parts=parts, anchor_name="anchor", down_ratio=4.0,
                                          max_objects=cfg.max_objects, max_parts=cfg.max_parts,
                                          conf_threshold=cfg.conf_threshold, decoder_dist_thresh=cfg.dist_thresh))
        run = lambda: dec(outs)  # the reference never writes into its inputs (decoders.py:44-100)
        kind, what = "reference", "unmodified reference Decoder.__call__ (sdnet.data.decoders, oracle/_ref archive)"
    else:
        run = lambda: torch_port.decode(outs, labels, parts, "anchor", 4.0, cfg.max_objects, cfg.max_parts,
                                        cfg.conf_threshold, cfg.dist_thresh)
        kind, what = "port", "oracle/torch_port.py (the reference's op sequence, one .tolist() per tensor)"
    for _ in range(max(1, warmup)):
        run()
    times = []
    t_end = time.perf_counter() + seconds
    while (steps is not None and len(times) < steps) or (steps is None and (time.perf_counter() < t_end or len(times) < 2)):
        t0 = time.perf_counter()
        run()
        times.append(time.perf_counter() - t0)
    total = sum(times)
    return {
        "value": batch * len(times) / total,
        "unit": "images/s",
        "cores": torch.get_num_threads(),
        "host_cpus": os.cpu_count(),
        "kind": kind,
        "sample": f"{len(times)} steps x {batch} images of {cfg.name} maps ({cfg.height}x{cfg.width}, mode {mode}): {what}, "
                  f"tensor ops + Python object assembly, torch {torch.__version__} CPU",
        "ms_per_step": 1e3 * total / len(times),
        "steps": len(times),
    }


def run_reference_arm(args, cfg, modes):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # the CPU arm runs once, on rank 0
    per_mode = {m: cpu_reference_rate(cfg, m, seconds=0.0, steps=max(1, args.steps), warmup=max(1, args.warmup)) for m in modes}
    head = min(per_mode, key=lambda m: per_mode[m]["value"])
    res = per_mode[head]
    batch = min(CPU_BATCH, cfg.batch)
    line = {
        "impl": "reference",
        "metric": "decoded images/s",
        "value": res["value"],
        "unit": "images/s",
        "n_gpus": args.gpus,
        "steps": res["steps"],
        "warmup": max(1, args.warmup),
        "ms_per_step": res["ms_per_step"],
        "higher_is_better": True,
        "scaling": "strong",
        "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_name(cfg), "mode": head, "images_per_step": batch,
                   "note": f"CPU arm: each step decodes a bounded sample of the workload ({batch} images), all host threads"},
        "modes": {m: {"value": r["value"], "ms_per_step": r["ms_per_step"]} for m, r in per_mode.items()},
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": res["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------- our arm
def emit(line: dict):
    """The ONE JSON line goes to the real stdout; everything else any library prints to fd 1 while
    the bench runs (e.g. NCCL's version banner) was diverted to stderr by main()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1
FIELDS = ("anchor_inds", "part_inds", "assign", "counts", "anchor_out", "part_out", "part_emb")


def port_reference(outs, cfg, chunk=32):
    """The reference's own op sequence on the device tensors (oracle/torch_port.py), in chunks."""
    import torch

    from oracle import torch_port as TP

    acc = {k: [] for k in FIELDS}
    n = outs["anchor_hm"].shape[0]
    for lo in range(0, n, chunk):
        sub = {k: v[lo:lo + chunk] for k, v in outs.items()}
        ref = TP.decode_tensors(sub, cfg.max_objects, cfg.max_parts, cfg.conf_threshold, cfg.dist_thresh)
        for k in FIELDS:
            acc[k].append(ref[k])
    return {k: torch.cat(v) for k, v in acc.items()}


def fields_equal(got, want, got_rows=None):
    """Names of the packed fields that differ (bit-exact compare; ``got_rows`` = the images of ``got`` that ``want`` covers)."""
    import torch

    bad = []
    for k in FIELDS:
        g, w = getattr(got, k) if not isinstance(got, dict) else got[k], want[k] if isinstance(want, dict) else getattr(want, k)
        if got_rows is not None:
            g = g[got_rows]
        if g.shape != w.shape or not torch.equal(g, w.to(g.dtype)):
            bad.append(k)
    return bad


def dump_outputs(directory, per_mode: dict):
    """Write ``{mode: {field: host tensor}}`` as ``directory/<mode>_<field>.npy``: float fields as float32, integer
    fields as float64 (exact for every index and count here).  Every field is indexed by image first; when a mode's
    arrays exceed its share of ``DUMP_BYTES`` they are cut to a fixed, seeded sample of images, whose indices are
    written as ``<mode>_images.npy``."""
    import numpy as np

    out = Path(directory)
    out.mkdir(parents=True, exist_ok=True)
    budget = DUMP_BYTES // len(per_mode)
    for mode, fields in per_mode.items():
        arrays = {k: v.numpy().astype(np.float32 if v.dtype.is_floating_point else np.float64) for k, v in fields.items()}
        images = next(iter(arrays.values())).shape[0]
        per_image = sum(a.nbytes for a in arrays.values()) // images
        if per_image * images > budget:
            rows = np.random.default_rng(0).choice(images, budget // (per_image + 8), replace=False)
            rows.sort()
            arrays = {k: a[rows] for k, a in arrays.items()}
            arrays["images"] = rows.astype(np.float64)
        for k, a in arrays.items():
            np.save(out / f"{mode}_{k}.npy", a)


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    from structuredetector_b200.synth import CONFIGS, DecodeConfig, make_raw, split_outputs

    cfg = CONFIGS[args.workload]
    if args.global_batch:
        cfg = DecodeConfig(cfg.name, args.global_batch, cfg.labels, cfg.parts, cfg.height, cfg.width,
                           cfg.max_objects, cfg.max_parts, cfg.conf_threshold, cfg.dist_thresh, cfg.cfg_id)
    modes = ("noise", "blobs") if args.mode == "both" else (args.mode,)
    if args.workload == "cfg4" and args.mode == "both":
        modes = ("noise",)  # BASELINE config 4 is "dense peaks" by definition
    if args.impl == "reference":
        run_reference_arm(args, cfg, modes)
        return

    import torch
    import torch.distributed as dist

    from structuredetector_b200 import ops

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run for N > 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the decode path has no CPU fallback")
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    if cfg.batch % world:
        raise SystemExit(f"global batch {cfg.batch} does not divide over {world} ranks")
    shard = cfg.batch // world
    M, N, H, W, K, P = cfg.labels, cfg.parts, cfg.height, cfg.width, cfg.max_objects, cfg.max_parts
    tdtype = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}[args.dtype]
    esize = 4 if args.dtype == "f32" else 2
    conf32 = float(torch.tensor(cfg.conf_threshold, dtype=tdtype))
    dist32 = float(torch.tensor(cfg.dist_thresh * min(W, H), dtype=torch.float32))

    # ---- synthetic inputs: identical bits on every run; each rank takes its slice of the global batch.
    # `buffers[mode]` = list of distinct resident input tensors the steps rotate over (one when it exceeds L2).
    def global_index(n_unique):
        return torch.arange(cfg.batch, device=device) % n_unique

    buffers, uniq_dev = {}, {}
    shard_bytes = shard * (M + N + 4) * H * W * esize
    n_rot = 1 if shard_bytes > 2 * L2_BYTES else -(-2 * L2_BYTES // shard_bytes) + 1
    for mode in modes:
        uniq = make_raw(cfg, mode, batch=min(UNIQUE_IMAGES, cfg.batch)).to(device)
        uniq_dev[mode] = uniq
        idx = global_index(uniq.shape[0])[rank * shard:(rank + 1) * shard]
        buffers[mode] = [uniq[(idx + r) % uniq.shape[0]].contiguous().to(tdtype) for r in range(n_rot)]
    outs_of = {mode: [split_outputs(raw, M, N) for raw in buffers[mode]] for mode in modes}

    plan = ops.DecodePlan(device, shard, M, N, H, W, K, P, tdtype)
    blob_bytes = plan.out.blob.numel()
    gathered = None
    fused = None
    gather_kind = "none"
    if world > 1 and args.gather == "fused":
        try:
            from structuredetector_b200.parallel import FusedGatherPlan

            fused = FusedGatherPlan(device, cfg.batch, M, N, H, W, K, P, dtype=tdtype)
            fused.lazy = args.gather_wait == "lazy"
            how = ("one multimem.st per value to the blob's NVSwitch multicast mapping" if fused.stores == "multicast"
                   else "one st.global per peer over NVLink")
            sync = ("the tail kernel's last CTA releases the rank's completion flag into every copy, a one-CTA wait kernel spins on the local flags"
                    if fused.sync == "flags" else "one symmetric-memory barrier")
            when = ("arrival is waited for before a result buffer is written again (two runs later) and at the end of the timed region"
                    if fused.lazy and fused.sync == "flags" else "arrival is waited for after every step")
            gather_kind = (f"fused: tail kernel stores each rank's packed detections into every rank's copy (symmetric memory, {how}); "
                           f"{sync}; {when}; results double-buffered")
        except Exception as exc:  # noqa: BLE001
            print(f"[bench] symmetric memory unavailable ({exc!r}); falling back to ncclAllGather", file=sys.stderr)
            fused = None
    if world > 1 and fused is None:
        gathered = torch.empty(world * blob_bytes, dtype=torch.uint8, device=device)
        gather_kind = "ncclAllGather of packed detections (every rank holds all results)"

    # Software pipeline over batches: consecutive steps alternate between `depth` plans (own workspace,
    # own outputs, own gather buffer) on `depth` streams, so one batch's tail kernel and gather overlap
    # the next batch's peaks kernel.  --pipeline 1 = strictly one decode at a time.
    # measured on one B200 (profiles/r02_pipeline_depth.log): 1024 images 0.806 / 0.784 / 0.774 ms per step at depth 1 / 2 / 3;
    # 128 images 0.139 / 0.122 / 0.117 ms at 2 / 4 / 6 -- consecutive kernels overlap at their ends, and a small shard's
    # kernel is all warm-up at its start and all streaming at its end, so more of them in flight mix those phases
    # (8 GPUs x 128 images, profiles/r02_gather_n8.log: 0.131 ms per step at depth 6, 0.128 at 8; with lazy arrival waits
    # 0.1199 at 8, 0.1188 at 12)
    depth = args.pipeline if args.pipeline > 0 else (3 if shard >= 512 else (4 if shard > 160 else 12))
    pipe = None
    if depth > 1:
        if fused is not None:
            extra = [FusedGatherPlan(device, cfg.batch, M, N, H, W, K, P, dtype=tdtype) for _ in range(depth - 1)]
            for e in extra:
                e.lazy = fused.lazy
            pipe = ops.DecodePipeline(device, depth, lambda i: fused if i == 0 else extra[i - 1])
        elif world == 1:
            pipe = ops.DecodePipeline(device, depth, lambda i: plan if i == 0 else ops.DecodePlan(device, shard, M, N, H, W, K, P, tdtype))
        else:
            depth = 1  # the ncclAllGather baseline stays serial

    def step(o):
        """Enqueue one decode of the batch; returns the PackedDetections it writes."""
        if pipe is not None:
            return pipe.submit(o["anchor_hm"], o["part_hm"], o["offsets"], o["embeddings"], conf32, dist32)[0]
        if fused is not None:
            return fused.run(o["anchor_hm"], o["part_hm"], o["offsets"], o["embeddings"], conf32, dist32)
        res = plan.run(o["anchor_hm"], o["part_hm"], o["offsets"], o["embeddings"], conf32, dist32)
        if world > 1:
            dist.all_gather_into_tensor(gathered, plan.out.blob)
        return res

    def fence():
        torch.cuda.synchronize(device)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    peaks_file = ROOT / "MEASURED_PEAKS.json"
    if peaks_file.exists():
        peak_gbs, peak_src = float(json.loads(peaks_file.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak_gbs, peak_src = 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"
    peaks_bytes = shard * (M + N) * H * W * esize  # algorithmic bytes of the dominant kernel: heat maps read once

    per_mode, dumped = {}, {}
    align = torch.zeros(1, device=device)
    for mode in modes:
        rot = outs_of[mode]
        for i in range(max(3, args.warmup)):
            step(rot[i % len(rot)])
        fence()
        # ---- timed region: exactly K steps, CUDA events on the launching stream, max over ranks
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ClockSampler(physical_gpu_index(local_rank)) as clocks:
            fence()
            if world > 1:
                # start the clock at the same moment on every GPU: a stream-ordered collective right before the first
                # event, so a rank whose host reaches this line late delays everybody's start instead of being waited
                # for inside the others' timed regions (a 3 ms host skew is 12 % of a 200-step region at 8 GPUs)
                dist.all_reduce(align)
            ev0.record()
            for i in range(args.steps):
                last = step(rot[i % len(rot)])
            if pipe is not None:
                pipe.drain()  # fused gather in lazy mode: includes the wait for every rank's rows of each plan's last run
            elif fused is not None:
                fused.wait_arrival()
            ev1.record()
            fence()
        if args.dump_outputs and rank == 0:  # copied now: the untimed runs below reuse the timed plans' outputs
            if gathered is not None:  # ncclAllGather: the caller's result is every rank's blob, merged
                from structuredetector_b200.parallel import merge_packed

                last = merge_packed([gathered[r * blob_bytes:(r + 1) * blob_bytes] for r in range(world)], [shard] * world,
                                    K, P, M + N)
            dumped[mode] = {k: getattr(last, k).cpu() for k in FIELDS}
        ms_total = ev0.elapsed_time(ev1)
        by_rank = None
        if world > 1:
            t = torch.tensor([ms_total], dtype=torch.float64, device=device)
            every = torch.empty(world, dtype=torch.float64, device=device)
            dist.all_gather_into_tensor(every, t)
            by_rank = [round(v / args.steps, 5) for v in every.tolist()]
            ms_total = max(every.tolist())  # the job's time is the slowest rank's
        ms_per_step = ms_total / args.steps

        # ---- one more (untimed) step through the timed objects, then look at what they produced
        o = rot[0]
        if fused is not None:
            res = fused.run(o["anchor_hm"], o["part_hm"], o["offsets"], o["embeddings"], conf32, dist32)
            fused.wait_arrival()
        else:
            res = plan.run(o["anchor_hm"], o["part_hm"], o["offsets"], o["embeddings"], conf32, dist32)
        fence()
        local_rows = slice(rank * shard, (rank + 1) * shard) if fused is not None else None
        counts = res.counts.sum(dim=0).tolist()  # fused: the whole batch, gathered; else this rank's shard
        if fused is None and world > 1:
            counts = [c * world for c in counts]
        diag_overflow = int(res.diag[:, 1].sum())
        cand_mean = float(res.diag[:, 0].float().mean())

        # ---- parity of the timed path, outside the timed region (bit-exact, every packed field)
        parity = None
        if not args.no_parity:
            want = port_reference(o, cfg)
            bad = fields_equal(res, want, got_rows=local_rows)
            parity = {"ok": not bad, "fields_differing": bad, "images": shard,
                      "against": "oracle/torch_port.py (the reference's stock torch ops) on the same device tensors"}
        gather_ok = None
        if world > 1 and not args.no_parity:
            # every rank decodes the WHOLE global batch alone and compares it with what the gather left here
            uniq = uniq_dev[mode]
            full = uniq[global_index(uniq.shape[0])].contiguous().to(tdtype)
            fo = split_outputs(full, M, N)
            solo_plan = ops.DecodePlan(device, cfg.batch, M, N, H, W, K, P, tdtype)
            solo = solo_plan.run(fo["anchor_hm"], fo["part_hm"], fo["offsets"], fo["embeddings"], conf32, dist32)
            torch.cuda.synchronize(device)
            if fused is not None:
                got = res
            else:
                from structuredetector_b200.parallel import merge_packed

                dist.all_gather_into_tensor(gathered, plan.out.blob)
                got = merge_packed([gathered[r * blob_bytes:(r + 1) * blob_bytes] for r in range(world)], [shard] * world, K, P, M + N)
            bad = fields_equal(got, solo)
            flag = torch.tensor([0 if bad else 1], dtype=torch.int32, device=device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            gather_ok = bool(flag.item())
            del full, fo, solo_plan, solo

        # ---- roofline leg: device time of each kernel (events between the launches), averaged
        reps = 20
        kms = [plan.run_timed(o["anchor_hm"], o["part_hm"], o["offsets"], o["embeddings"], conf32, dist32) for _ in range(reps)]
        kernel_ms = {"peaks": statistics.mean(k[0] for k in kms), "exact_select": statistics.mean(k[1] for k in kms),
                     "tail": statistics.mean(k[2] for k in kms)}
        achieved = peaks_bytes / (kernel_ms["peaks"] * 1e-3) / 1e9
        if fused is not None:  # the same three kernels with the tail storing into every peer's copy
            fk = [fused.plan.run_timed(o["anchor_hm"], o["part_hm"], o["offsets"], o["embeddings"], conf32, dist32) for _ in range(reps)]
            kernel_ms["tail_storing_to_peers"] = statistics.mean(k[2] for k in fk)
            fence()
        per_mode[mode] = {
            "value": cfg.batch / (ms_per_step * 1e-3), "ms_per_step": ms_per_step, "ms_per_step_by_rank": by_rank, "kernel_ms": kernel_ms,
            "peaks_achieved_gbs": achieved, "peaks_frac": achieved / peak_gbs,
            "parity": parity, "gather_bit_exact": gather_ok, "clocks": clocks.summary(),
            "detections": {"anchors_above_conf": counts[0], "parts_above_conf": counts[1],
                           "planes_via_exact_select": diag_overflow, "candidates_per_plane_mean": cand_mean},
        }

    if dumped:
        dump_outputs(args.dump_outputs, dumped)
    head = min(per_mode, key=lambda m: per_mode[m]["value"])  # the slower mode is the headline
    hm = per_mode[head]
    ms_per_step, value, kernel_ms = hm["ms_per_step"], hm["value"], hm["kernel_ms"]
    o = outs_of[head][0]
    raw = buffers[head][0]
    sched = plan.schedule(o["anchor_hm"], o["part_hm"], o["offsets"], o["embeddings"])
    # DRAM bytes per launch of the peaks kernel from the ncu capture of the same case (images per rank, input mode,
    # dtype), when profiles/ holds one; null otherwise
    traffic = traffic_source = None
    traffic_path = ROOT / "profiles" / "peaks_kernel_traffic.json"
    if traffic_path.exists() and args.workload == "cfg5":
        try:
            for cap in json.loads(traffic_path.read_text()).get("captures", []):
                if (cap.get("images"), cap.get("mode"), cap.get("dtype")) == (shard, head, args.dtype):
                    traffic, traffic_source = cap["dram_bytes_per_launch"], cap.get("source")
        except Exception:  # noqa: BLE001
            traffic = traffic_source = None
    step_s = ms_per_step * 1e-3
    roofline = {
        "bound": "hbm",
        "kernel": {"tile": "sdnet_peaks_tile_kernel (TMA tiles)", "tile_row_pairs": "sdnet_peaks_tile_kernel (TMA tiles over row pairs)",
                   "warp": "sdnet_peaks_kernel (per-lane feed)"}[sched["path"]],
        "achieved": hm["peaks_achieved_gbs"], "peak": peak_gbs, "unit": "GB/s", "frac": hm["peaks_frac"], "traffic": traffic, "traffic_source": traffic_source,
        "peak_source": peak_src, "mode": head, "kernel_ms": kernel_ms,
        "kernel_share_of_step": kernel_ms["peaks"] / (kernel_ms["peaks"] + kernel_ms["exact_select"] + kernel_ms["tail"]),
        "algorithmic_bytes_per_launch": peaks_bytes,
        "schedule": sched,
        # whole step (all kernels + gather), per rank, under the two denominators of SURVEY 8(d)
        "step_achieved_min_gbs": shard * cfg.min_bytes_per_image * esize / 4 / step_s / 1e9,
        "step_achieved_contract_gbs": shard * cfg.contract_bytes_per_image * esize / 4 / step_s / 1e9,
        "frac_of_8tbs_min": shard * cfg.min_bytes_per_image * esize / 4 / step_s / 8e12,
        "frac_of_8tbs_contract": shard * cfg.contract_bytes_per_image * esize / 4 / step_s / 8e12,
    }

    from types import SimpleNamespace

    from structuredetector_b200 import Decoder

    dec = Decoder(SimpleNamespace(_r_labels={i: f"label{i}" for i in range(M)}, _r_parts={i: f"part{i}" for i in range(N)},
                                  anchor_name="anchor", down_ratio=4.0, max_objects=K, max_parts=P,
                                  conf_threshold=cfg.conf_threshold, decoder_dist_thresh=cfg.dist_thresh))

    # ---- the reference-facing Python call: device tensors -> list[ImageAnnotation] (decode + ONE D2H copy +
    # Python object assembly), reported separately (SURVEY 8d); rank 0, bounded sample
    objects = None
    if rank == 0 and not args.no_objects:
        n_obj = min(shard, 256)
        sample = {k: v[:n_obj] for k, v in o.items()}
        dec(sample)
        torch.cuda.synchronize(device)
        t0 = time.perf_counter()
        reps_obj = 3
        for _ in range(reps_obj):
            anns = dec(sample)
        dt = (time.perf_counter() - t0) / reps_obj
        objects = {"value": n_obj / dt, "unit": "images/s", "ms_per_image": dt / n_obj * 1e3,
                   "objects_per_image": sum(len(a.objects) for a in anns) / n_obj,
                   "parts_per_image": sum(a.nb_parts for a in anns) / n_obj, "mode": head,
                   "sample": f"Decoder(args)(outputs) on {n_obj} images resident on the device -> list[ImageAnnotation], wall clock, 1 Python thread"}

    # ---- end to end with HOST buffers: pinned inputs -> packed results on the host (C ABI), and -> Python objects
    e2e = e2e_objects = None
    if not args.no_e2e:
        host_raw = torch.empty(raw.shape, dtype=raw.dtype, pin_memory=True)
        host_raw.copy_(raw)
        h_outs = split_outputs(host_raw, M, N)
        lanes = 2  # two streams x (plan, staging, host result): batch i+1's upload overlaps batch i's kernels and download
        plans = [plan] + [ops.DecodePlan(device, shard, M, N, H, W, K, P, tdtype) for _ in range(lanes - 1)]
        stagings = [torch.empty(shard * (M + N) * H * W * esize, dtype=torch.uint8, device=device) for _ in range(lanes)]
        host_blobs = [torch.empty(blob_bytes, dtype=torch.uint8, pin_memory=True) for _ in range(lanes)]
        streams = [torch.cuda.Stream(device) for _ in range(lanes)]

        def e2e_step(i):
            k = i % lanes
            with torch.cuda.stream(streams[k]):
                plans[k].run_host(h_outs["anchor_hm"], h_outs["part_hm"], h_outs["offsets"], h_outs["embeddings"],
                                  conf32, dist32, stagings[k], stream=streams[k])
                host_blobs[k].copy_(plans[k].out.blob, non_blocking=True)

        e2e_step(0)
        fence()
        t0 = time.perf_counter()
        for i in range(args.e2e_steps):
            e2e_step(i)
        fence()
        dt = (time.perf_counter() - t0) / args.e2e_steps
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        want = plan.run(o["anchor_hm"], o["part_hm"], o["offsets"], o["embeddings"], conf32, dist32)
        torch.cuda.synchronize(device)
        n_det = blob_bytes - want.diag.numel() * 4  # everything but the trailing diagnostics is deterministic
        same = bool(torch.equal(host_blobs[(args.e2e_steps - 1) % lanes][:n_det], want.blob.cpu()[:n_det]))
        heat = shard * (M + N) * H * W * esize
        gathers = shard * (K + 2 * P) * 2 * 32  # zero-copy reads of offsets/embeddings, one 32 B sector each
        e2e = {"value": cfg.batch / dt, "unit": "images/s", "h2d_bytes_per_step": (heat + gathers) * world,
               "d2h_bytes_per_step": blob_bytes * world, "ms_per_step": dt * 1e3, "steps": args.e2e_steps, "mode": head,
               "path": "sdnet_decode_host_launch: heat planes cudaMemcpy2DAsync from pinned host, offsets/embeddings read "
                       "in place at the selected peaks, packed results copied back to pinned host; two batches in flight",
               "host_results_match_device_path": same}
        del stagings, plans
        # the same through the drop-in Decoder: pinned host tensors in, list[ImageAnnotation] out (what the CPU arm returns)
        if rank == 0 and not args.no_objects:
            n_e = min(shard, 256)
            h_sample = {k: v[:n_e] for k, v in h_outs.items()}
            dec(h_sample)
            t0 = time.perf_counter()
            reps_e = 3
            for _ in range(reps_e):
                anns = dec(h_sample)
            dt = (time.perf_counter() - t0) / reps_e
            e2e_objects = {"value": n_e / dt, "unit": "images/s", "ms_per_step": dt * 1e3, "images_per_step": n_e,
                           "h2d_bytes_per_step": n_e * ((M + N) * H * W * esize + (K + 2 * P) * 64),
                           "d2h_bytes_per_step": ops.packed_nbytes(n_e, K, P, M + N),
                           "objects_per_image": sum(len(a.objects) for a in anns) / n_e,
                           "path": "Decoder(args)(outputs in pinned host memory) -> list[ImageAnnotation]: upload, 3 kernels, "
                                   "ONE download, object assembly; wall clock, 1 Python thread, rank 0"}
        del host_raw

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.dtype == "f32":
        res = cpu_reference_rate(cfg, head, seconds=10.0)
        cpu_baseline = {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")}
        cpu_baseline["host_cpus"] = res["host_cpus"]
        one = cpu_reference_rate(cfg, head, seconds=6.0, threads=1)
        cpu_baseline["one_thread"] = {"value": one["value"], "cores": 1, "steps": one["steps"]}

    if rank == 0:
        parity_all = None if args.no_parity else all(m["parity"]["ok"] for m in per_mode.values())
        gather_all = None
        if world > 1 and not args.no_parity:
            gather_all = all(m["gather_bit_exact"] for m in per_mode.values())
        line = {
            "metric": "decoded images/s",
            "value": value,
            "unit": "images/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": max(3, args.warmup),
            "ms_per_step": ms_per_step,
            "higher_is_better": True,
            "scaling": "strong",
            "vs_baseline": None,
            "dtype": args.dtype,
            "data": "synthetic",
            "config": {
                "workload": workload_name(cfg, args.dtype),
                "mode": f"{head} (headline = the slower of {', '.join(modes)}; both under 'modes')" if len(modes) > 1 else head,
                "images_per_rank": shard, "parallelism": f"batch-shard x{world}",
                "gather": gather_kind,
                "l2": (f"inputs larger than L2 ({raw.numel() * esize / 1e9:.2f} GB per rank, no flush needed)" if n_rot == 1 else
                       f"steps rotate over {n_rot} distinct input buffers of {raw.numel() * esize / 1e6:.1f} MB ({n_rot * raw.numel() * esize / 1e6:.0f} MB > 2 x L2)"),
                "unique_images": int(min(UNIQUE_IMAGES, cfg.batch)),
                "pipeline": (f"{depth} decodes in flight: consecutive steps alternate between {depth} plans (own workspace, outputs"
                             f"{' and gather buffer' if world > 1 else ''}) on {depth} streams; every step is a full decode of the batch")
                            if depth > 1 else "1 (each step waits for the one before)",
            },
            "modes": {m: {k: v for k, v in r.items() if k != "clocks"} for m, r in per_mode.items()},
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
            "e2e": e2e,
            "e2e_objects": e2e_objects,
            "python_objects": objects,
            "parity_checked": parity_all,
            "gather_bit_exact": gather_all,
            "gpu_launches": ops.gpu_launches_per_decode() * args.steps,
            "clocks": hm["clocks"],
            "detections": hm["detections"],
        }
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
