"""bench.py's contract: the reference arm's JSON line (speed-up ratios are computed from it), the refusal to time 'our'
arm without a CUDA device (no CPU fallback), and --dump-outputs (host side on CPU, end to end on the GPU)."""
import importlib.util
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
FIELDS = ("anchor_inds", "part_inds", "assign", "counts", "anchor_out", "part_out", "part_emb")


def _run(*flags, timeout=600, env=None):
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *flags], capture_output=True, text=True, timeout=timeout, cwd=ROOT,
                          env=env)


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench", ROOT / "bench.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    done = _run("--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "1", "--mode", "noise")
    assert done.returncode == 0, done.stderr[-2000:]
    lines = [ln for ln in done.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, "exactly ONE JSON line on stdout"
    line = json.loads(lines[0])
    assert line["impl"] == "reference" and line["metric"] == "decoded images/s" and line["unit"] == "images/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["steps"] == 1 and line["warmup"] == 1
    assert line["value"] > 0 and line["ms_per_step"] > 0 and line["gpu_launches"] == 0 and line["vs_baseline"] is None
    assert line["config"]["workload"].startswith("cfg5") and line["data"] == "synthetic" and line["dtype"] == "f32"
    base = line["cpu_baseline"]
    assert base["kind"] in ("reference", "port") and base["cores"] >= 1 and base["value"] == line["value"]
    assert "Decoder" in base["sample"] or "torch_port" in base["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_our_arm_refuses_to_run_without_a_cuda_device():
    done = _run("--steps", "1", "--warmup", "1", timeout=300, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
    assert done.returncode != 0 and done.stdout.strip() == ""
    assert "no CPU fallback" in done.stderr


def test_bench_refuses_zero_steps():
    done = _run("--steps", "0", timeout=300)
    assert done.returncode != 0 and done.stdout.strip() == "" and "--steps" in done.stderr


def test_dump_outputs_types_names_and_size_cap(tmp_path, monkeypatch):
    """Integer fields become float64 and float fields float32, one file per mode and field; past the size cap every
    field keeps the same fixed sample of images, listed in <mode>_images.npy."""
    bench = _bench_module()
    gen = torch.Generator().manual_seed(0)
    B = 40

    def fields():
        return {"anchor_inds": torch.randint(0, 1 << 20, (B, 5), generator=gen), "assign": torch.randint(-1, 5, (B, 3), dtype=torch.int32, generator=gen),
                "anchor_out": torch.rand(B, 5, 4, generator=gen)}

    small = {"noise": fields(), "blobs": fields()}
    bench.dump_outputs(tmp_path / "all", small)
    for mode, arrays in small.items():
        for k, v in arrays.items():
            got = np.load(tmp_path / "all" / f"{mode}_{k}.npy")
            assert got.dtype == (np.float32 if v.dtype.is_floating_point else np.float64)
            np.testing.assert_array_equal(got, v.numpy())
    assert not list((tmp_path / "all").glob("*_images.npy"))

    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * 10 * (5 * 8 + 3 * 8 + 5 * 4 * 4 + 8))  # room for 10 images per mode
    for name in ("a", "b"):
        bench.dump_outputs(tmp_path / name, small)
    for mode, arrays in small.items():
        rows = np.load(tmp_path / "a" / f"{mode}_images.npy")
        assert len(rows) == 10 and (np.diff(rows) > 0).all()
        np.testing.assert_array_equal(rows, np.load(tmp_path / "b" / f"{mode}_images.npy"))
        for k, v in arrays.items():
            np.testing.assert_array_equal(np.load(tmp_path / "a" / f"{mode}_{k}.npy"), v.numpy()[rows.astype(np.int64)])
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= bench.DUMP_BYTES + (1 << 20)


@pytest.mark.gpu
def test_dump_outputs_is_what_the_last_timed_step_computed(cuda_device, tmp_path):
    """bench.py on the small config: the dumped arrays equal a decode of the input its last timed step read.  With two
    timed steps that is the second of the rotating input buffers, the 32 unique images tiled over the batch shifted by
    one image, not the first buffer that the untimed parity step reads."""
    from structuredetector_b200 import ops
    from structuredetector_b200.synth import CONFIGS, make_raw, split_outputs

    done = _run("--workload", "cfg2", "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--no-e2e", "--no-objects",
                "--dump-outputs", str(tmp_path))
    assert done.returncode == 0, done.stderr[-2000:]
    line = json.loads(done.stdout)
    assert line["steps"] == 2 and line["parity_checked"] is True
    cfg = CONFIGS["cfg2"]
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(f"{m}_{k}.npy" for m in ("noise", "blobs") for k in FIELDS)
    for mode in ("noise", "blobs"):
        raw = make_raw(cfg, mode, batch=32)[(torch.arange(cfg.batch) + 1) % 32].to(cuda_device)
        want = ops.decode_packed(split_outputs(raw, cfg.labels, cfg.parts), cfg.max_objects, cfg.max_parts, cfg.conf_threshold,
                                 cfg.dist_thresh)
        for k in FIELDS:
            got = np.load(tmp_path / f"{mode}_{k}.npy")
            assert got.dtype in (np.float32, np.float64)
            np.testing.assert_array_equal(got, getattr(want, k).cpu().numpy().astype(got.dtype), err_msg=f"{mode} {k}")
