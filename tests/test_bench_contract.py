"""bench.py keeps the driver's JSON contract (one line on stdout, required keys) for both arms."""
import json
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e"}


def run(*args, timeout=900):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True, text=True,
                       timeout=timeout)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def test_reference_arm_line_on_cpu():
    d = run("--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-sample-batch", "1")
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == "mLSTM fwd+bwd tokens/s/GPU" and d["unit"] == "tokens/s" and d["higher_is_better"] is True
    assert d["config"]["workload"].startswith("cfg2_") and d["vs_baseline"] is None and d["value"] > 0
    # "reference": the reference's own chunkwise_simple from oracle/_ref (placed by oracle/make_ref.py); "port" without it
    want_kind = "reference" if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "backends.py")) else "port"
    assert d["cpu_baseline"]["kind"] == want_kind and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert "full batch 32/32" in d["cpu_baseline"]["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_b200_arm_line():
    d = run("--steps", "5", "--warmup", "3", "--cpu-sample-batch", "1")
    assert BASE_KEYS | {"clocks", "gpu_launches", "roofline", "cpu_baseline"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 5 and d["warmup"] >= 3 and d["dtype"] == "bf16" and d["data"] == "synthetic"
    assert d["config"]["workload"] == "cfg2_B32_NH4_S400_DH64" and d["config"]["kernel_family"] == "tcgen05"
    assert d["gpu_launches"] >= 2 * d["steps"]   # forward + the fused backward walk (3+ with the multi-kernel backward)
    rf = d["roofline"]
    assert rf["bound"] == "hbm" and rf["unit"] == "GB/s" and 0 < rf["frac"] < 1 and abs(rf["frac"] - rf["achieved"] / rf["peak"]) < 1e-9
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and 0 < d["e2e"]["value"] < d["value"]
    # the whole result comes back inside the timed region: h, dq, dk, dv (bf16) + di, df (fp32)
    B, NH, S, DH = 32, 4, 400, 64
    assert d["e2e"]["d2h_bytes_per_step"] == 4 * B * NH * S * DH * 2 + 2 * B * NH * S * 4
    assert d["e2e"]["checksum_variant"]["d2h_bytes_per_step"] == 16 and d["e2e"]["checksum_variant"]["value"] > 0
    also = {a["workload"]: a for a in d["also"]}
    assert set(also) == {"cfg3_B32_NH4_S1600_DH128", "cfg3_B32_NH4_S6400_DH128", "ddp_B8_NH4_S1600_DH128", "cfg3alt_B32_NH4_S1600_DH256",
                         "refdefault_B32_NH32_S1600_DH16"}
    assert also["refdefault_B32_NH32_S1600_DH16"]["roofline"]["kernel"].startswith("tcgen05")   # zero-padded inside the library
    assert 0.7 < also["cfg3alt_B32_NH4_S1600_DH256"]["roofline"]["step_tensor_ceiling"] < 0.8
    for a in also.values():
        assert a["steps"] == d["steps"]
        assert a["value"] > 0 and a["gpu_launches"] >= 2 * a["steps"] and 0 < a["roofline"]["step_hbm_frac"] < 1
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["value"] > 0 and "full batch" in cb["sample"]


def test_dump_outputs_samples_the_same_elements_within_the_budget(tmp_path, monkeypatch):
    import numpy as np
    import torch
    import bench
    g = torch.Generator().manual_seed(0)
    outs = {"h": torch.randn(2, 3, 50, 8, generator=g).bfloat16(), "di": torch.randn(2, 3, 50, generator=g)}
    bench.dump_outputs(torch, outs, str(tmp_path / "whole"))
    for name, t in outs.items():
        got = np.load(tmp_path / "whole" / f"{name}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, t.float().numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 2000)
    for tag in ("a", "b"):
        bench.dump_outputs(torch, outs, str(tmp_path / tag))
    files = [tmp_path / tag / f"{name}.npy" for tag in ("a", "b") for name in outs]
    assert sum(os.path.getsize(f) for f in files[:2]) <= 2000
    for name, t in outs.items():
        a, b = (np.load(tmp_path / tag / f"{name}.npy") for tag in ("a", "b"))
        assert a.ndim == 1 and 0 < a.size < t.numel() and np.array_equal(a, b)
        assert np.isin(a, t.float().numpy().ravel()).all()


@pytest.mark.gpu
def test_b200_arm_dumps_the_last_steps_outputs(tmp_path):
    import numpy as np
    args = ("--steps", "3", "--warmup", "3", "--no-also", "--no-cpu-baseline")
    for tag in ("a", "b"):
        d = run(*args, "--dump-outputs", str(tmp_path / tag))
    assert d["steps"] == 3
    B, NH, S, DH = 32, 4, 400, 64
    shapes = {"h": (B, NH, S, DH), "dq": (B, NH, S, DH), "dk": (B, NH, S, DH), "dv": (B, NH, S, DH), "di": (B, NH, S),
              "df": (B, NH, S)}
    assert sorted(os.listdir(tmp_path / "a")) == sorted(f"{n}.npy" for n in shapes)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64e6
    for name, shape in shapes.items():
        a, b = (np.load(tmp_path / tag / f"{name}.npy") for tag in ("a", "b"))
        assert a.dtype == np.float32 and a.shape == shape and np.isfinite(a).all() and np.abs(a).max() > 0
        assert np.array_equal(a, b), name          # seeded inputs, deterministic kernels: the same arrays run to run
    # the last timed step ran on input set (K - 1) mod nsets (graph replay) or (W + K - 1) mod nsets (eager launches)
    import torch
    import bench
    from oracle import mlstm_oracle as O
    nsets = int(re.search(r"rotate over (\d+) sets", d["config"]["l2"]).group(1))
    last = (3 - 1 if d["config"]["launch"].startswith("CUDA graph") else d["warmup"] + 3 - 1) % nsets
    ins = bench.make_inputs(torch, B, NH, S, DH, last, "cpu", torch.bfloat16)
    want = O.mlstm_fwbw(*(t[:1].transpose(1, 2).double() for t in ins), chunk_size=64, eps=1e-6)
    for name, w in zip(shapes, want):
        got = torch.from_numpy(np.load(tmp_path / "a" / f"{name}.npy")[:1]).double()
        err = float((got - w).abs().max() / w.abs().max())
        assert err < (1e-2 if name == "h" else 2e-2), (name, err)
