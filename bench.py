#!/usr/bin/env python
"""bench.py — mLSTM cell fwd+bwd throughput (BASELINE.json metric) on B200.

    python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
    python bench.py --impl reference --gpus N ...           # reference CPU path (oracle port)

One "step" = one forward + one backward of the mLSTM cell over one synthetic batch of the
workload (default: BASELINE.json configs[1]: B=32, NH=4, S=400, DH=64, bf16).  Prints ONE JSON
line (see the repo contract).  Timing: CUDA events on the launching stream, >=3 warm-up
steps, inputs rotate over enough independent sets that the working set exceeds L2, max over
ranks for N>1 (one process per GPU, torchrun env).

The same line carries an ``also`` block (N=1): the north-star shapes of BASELINE.json configs[2] (B32 NH4 DH128 at 1600
and 6400 tokens) and the per-GPU shape of batch-64 DDP on 8 GPUs (B8), measured the same way in the same run, so the
driver's clock covers them too.  The headline workload stays configs[1].
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (B, NH, S, DH)  — BASELINE.json configs
    "cfg2_B32_NH4_S400_DH64": (32, 4, 400, 64),
    "cfg2alt_B32_NH4_S400_DH128": (32, 4, 400, 128),
    "cfg3_B32_NH4_S1600_DH128": (32, 4, 1600, 128),
    "cfg3_B32_NH4_S6400_DH128": (32, 4, 6400, 128),
    "ddp_B8_NH4_S1600_DH128": (8, 4, 1600, 128),
    # BASELINE configs[2] read as d = 512 with the layer's expansion 2 (inner 1024 / 4 heads): head dim 256, the shape on which
    # the north star's ">= 50 % of tensor peak" lies below the HBM roofline (csrc/mlstm_tc_256.cu)
    "cfg3alt_B32_NH4_S1600_DH256": (32, 4, 1600, 256),
    # the reference's DEFAULT head dim: qkv_block_size = 16 (vision_lstm2.py:416-417) at inner 512 -> 32 heads of 16; runs the
    # DH = 64 tcgen05 kernels on zero-padded copies made inside the library (csrc/mlstm_api.cu, DESIGN.md §3.2d)
    "refdefault_B32_NH32_S1600_DH16": (32, 32, 1600, 16),
    # developer shapes (dispatch thresholds of the DH = 64 backward variants; not BASELINE configs)
    "dev_B32_NH4_S800_DH64": (32, 4, 800, 64),
    "dev_B32_NH4_S1600_DH64": (32, 4, 1600, 64),
}
DEFAULT_WORKLOAD = "cfg2_B32_NH4_S400_DH64"
ALSO_WORKLOADS = ["cfg3_B32_NH4_S1600_DH128", "cfg3_B32_NH4_S6400_DH128", "ddp_B8_NH4_S1600_DH128", "cfg3alt_B32_NH4_S1600_DH256",
                  "refdefault_B32_NH32_S1600_DH16"]
CHUNK = 64          # the config's chunk size (algorithmic FLOP formula; kernels tile on their own)
L2_BYTES = 126e6


def algorithmic(B, NH, S, DH):
    """SURVEY.md §8(d): per token-head FLOPs and HBM bytes (bf16 I/O, fp32 gates/rows)."""
    th = B * NH * S
    flops_fwd = 4 * DH * DH + 2 * (CHUNK + 1) * DH
    return {
        "token_heads": th,
        "flops_fwdbwd": 3 * flops_fwd * th,
        "bytes_fwd": (8 * DH + 16) * th,
        "bytes_bwd": (14 * DH + 24) * th,
        # per-kernel minimal traffic of the two-kernel backward (DESIGN.md §kernels)
        "bytes_bwd_dq": (10 * DH + 24) * th,     # read q,k,v,dh + i,f,n,m ; write dq + dn,R
        "bytes_bwd_dkv": (12 * DH + 32) * th,    # read q,k,v,dh + i,f,n,m,dn,R ; write dk,dv + di,df
    }


# DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) per launch of the kernels behind each timed
# part, from the `ncu --set full` captures (profiles/r0*_ncu_full_*_summary.csv).  Writes that
# stay in the 126 MB L2 until after the kernel are not counted by ncu.
NCU_TRAFFIC_BYTES = {
    # round 2 captures (profiles/r02_ncu_full_<workload>_summary.csv)
    "cfg2_B32_NH4_S400_DH64": {"fwd": 20.1e6, "bwd_dq": None, "bwd_dkv": 38.0e6 + 0.25e6},   # fused backward: one kernel; its outputs stay in L2
    "cfg3_B32_NH4_S1600_DH128": {"fwd": 159.1e6 + 73.0e6, "bwd_dq": None, "bwd_dkv": 326.5e6 + 129.3e6},   # DH = 128 fused walk
    # DH = 256 family: state walk + F | A | adjoint-state walk + B1 + B2 + scan
    "cfg3alt_B32_NH4_S1600_DH256": {"fwd": (405.5 + 189.8 + 536.1 + 91.5) * 1e6, "bwd_dq": (747.5 + 100.4) * 1e6,
                                    "bwd_dkv": (620.1 + 201.2 + 536.1 + 88.8 + 643.4 + 97.5 + 14.0) * 1e6},
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as fh:
            d = json.load(fh)
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def make_inputs(torch, B, NH, S, DH, seed, device, dtype, on_device=False):
    """SURVEY.md §8(d) synthetic inputs in the reference's memory layout: (B,S,NH,DH) storage
    viewed as (B,NH,S,DH); gates (B,S,NH) viewed (B,NH,S).  q,k in the post-projection regime.
    ``on_device``: draw them with the device's generator (the large `also` shapes; the device-resident arm only)."""
    gdev = device if on_device else "cpu"
    g = torch.Generator(device=gdev).manual_seed(seed)
    std = DH ** -0.5
    rn = lambda *shape: torch.randn(*shape, generator=g, device=gdev)
    q = (rn(B, S, NH, DH) * std).to(dtype)
    k = (rn(B, S, NH, DH) * std).to(dtype)
    v = rn(B, S, NH, DH).to(dtype)
    dh = rn(B, S, NH, DH).to(dtype)
    i = rn(B, S, NH)
    f = torch.linspace(3.0, 6.0, NH, device=gdev).view(1, 1, NH) + rn(B, S, NH)
    return [t.to(device) if (device != "cpu" and not on_device) else t for t in (q, k, v, i, f, dh)]


def as_heads(ts):
    return [t.transpose(1, 2) for t in ts]


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.samples, self.reasons, self.max_mhz = index, False, [], set(), None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.01)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def cpu_fwbw_step(torch, O, cpu_inputs):
    q, k, v, i, f, dh = cpu_inputs
    return O.mlstm_fwbw(q, k, v, i, f, dh, chunk_size=CHUNK, eps=1e-6)


def ref_chunk(S):
    """The reference's chunkwise_simple needs chunk_size | S (backends.py:164): the divisor of S nearest the config's 64."""
    divs = [d for d in range(8, min(S, 256) + 1) if S % d == 0]
    return min(divs, key=lambda d: (abs(d - CHUNK), d)) if divs else S


def reference_step_fn(torch):
    """(step(inputs) -> None, kind, what): the reference's own chunkwise_simple (oracle/_ref/backends.py, placed there by
    oracle/make_ref.py) when present, else the oracle port."""
    from oracle import make_ref
    mod = make_ref.load()
    if mod is not None:
        def step(cin):
            q, k, v, i, f, dh = cin
            leaves = [t.detach().requires_grad_(True) for t in (q, k, v, i, f)]
            h = mod.chunkwise_simple(*leaves, chunk_size=ref_chunk(q.shape[2]), eps=1e-6)
            h.backward(dh)
        return step, "reference", "reference chunkwise_simple (backends.py:149-263) + autograd"
    from oracle import mlstm_oracle as O
    return (lambda cin: cpu_fwbw_step(torch, O, cin)), "port", "oracle port of backends.py:149-263 + autograd"


def cpu_inputs(torch, B, NH, S, DH):
    # contiguous (B,NH,S,DH) fp32: what the reference's .view() calls need
    return [t.float().transpose(1, 2).contiguous() for t in make_inputs(torch, B, NH, S, DH, 0, "cpu", torch.bfloat16)]


def run_reference(args):
    """Reference arm: the reference's CPU implementation of the path on the box's host cores (all threads), the FULL batch of
    the same workload, same metric / unit, the same number of steps (capped so the run ends within minutes)."""
    import torch
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    B, NH, S, DH = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step, kind, what = reference_step_fn(torch)
    inputs = cpu_inputs(torch, B, NH, S, DH)
    t0 = time.perf_counter()
    step(inputs)                                   # warm-up (also sizes the run)
    t_one = time.perf_counter() - t0
    for _ in range(max(0, min(args.warmup, 3) - 1)):
        step(inputs)
    steps = max(1, min(args.steps, int(120.0 / max(t_one, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(steps):
        step(inputs)
    dt = (time.perf_counter() - t0) / steps
    val = B * S / dt
    sample = f"full batch {B}/{B} of {args.workload}, {steps} steps, chunk_size {ref_chunk(S)}, fp32, {what}"
    out = {
        "impl": "reference", "metric": "mLSTM fwd+bwd tokens/s/GPU", "value": val, "unit": "tokens/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": args.workload, "B_per_gpu": B, "NH": NH, "S": S, "DH": DH, "chunk_size": CHUNK},
        "cpu_baseline": {"value": val, "unit": "tokens/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(out)
    return 0


_OUT_FD = None


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _OUT_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_OUT_FD, line)


def launches_of(variant_fwd, variant_bwd, DH):
    """kernels behind each timed part, per variant (csrc/mlstm_tc_*.cu)"""
    if DH not in (64, 128, 256) and variant_fwd != "simt":   # zero-padded to the next kernel width inside the library (csrc/mlstm_api.cu)
        DP = 64 if DH <= 64 else (128 if DH <= 128 else 256)
        inner = launches_of(variant_fwd, variant_bwd, DP)
        if DP <= 128:   # the tensor maps carry the true row length: TMA supplies the zero columns and clips the stores, no copies
            note = "(width-%d kernel on %d-wide rows, zero columns from TMA)" % (DP, DH)
            return {k_: [x + " " + note for x in v_] for k_, v_ in inner.items()}
        return {"fwd": ["pad_rows_kernel (q, k, v -> width %d)" % DP] + inner["fwd"] + ["pad_rows_kernel (crop h)"],
                "bwd_dq": inner["bwd_dq"],
                "bwd_dkv": ["pad_rows_kernel (dh)"] + inner["bwd_dkv"] + ["pad_rows_kernel (crop dq, dk, dv)"]}
    if DH == 256 and variant_fwd == "two_phase":   # the slice-streaming family (csrc/mlstm_tc_256.cu)
        return {"fwd": ["tc_state_fwd_kernel<128> on 2x2 blocks of C", "tc256_par_kernel<F>"],
                "bwd_dq": ["tc256_par_kernel<A>"],
                "bwd_dkv": ["tc_state_bwd_kernel<128> on 2x2 blocks of dC", "tc256_par_kernel<B1> (dv)", "tc256_par_kernel<B2> (dk)",
                            "tc_dfscan_kernel"]}
    return {
        "fwd": {"single_pass": ["tc_fwd_ws_kernel (warp-specialised walk; MLSTM_FWD_WS=0: tc_fwd_kernel)"], "two_phase": ["tc_state_fwd_kernel", "tc_fwd_par_kernel"],
                "simt": ["simt_fwd_kernel"]}[variant_fwd],
        "bwd_dq": {"single_pass": ["tc_bwd_dq_kernel"],
                   "chunk_parallel": ["tc_bwd_par_kernel<A> (whole-backward calls with 2*B*NH <= #SM: tc_dn_kernel + tc_bwd_sa_kernel, "
                                      "the state walk and A in one launch)"],
                   "fused_walk": [], "simt": ["simt_bwd_dq_kernel"]}[variant_bwd],
        "bwd_dkv": {"single_pass": ["tc_bwd_dkv12_kernel (dv and dk walks co-resident)" if DH == 64 else "tc_bwd_dkv_kernel<1>, <2>"],
                    "chunk_parallel": ["tc_state_bwd_kernel", "tc_bwd_b12_kernel (B1 dv | B2 dk side by side)", "tc_dfscan_kernel"],
                    "fused_walk": [("tc_bwd_fused_kernel" if DH == 64 else "tc_bwd_fused128_kernel") + " (dq, dk, dv, di, df in one reverse walk)"],
                    "simt": ["simt_bwd_dkv_kernel"]}[variant_bwd],
    }


def measure_device(torch, dist, ops, _lib, name, K, W, dev, rank, world, reverse=False, on_device=False, keep_outputs=False):
    """Device-resident arm of one workload: K steps between two CUDA events (CUDA-graph replay of one round over the rotating
    input sets), then the same K steps eager with an event pair around every launch for the per-kernel durations.
    ``keep_outputs``: the result also carries "outputs", copies of what the last timed step computed."""
    B, NH, S, DH = WORKLOADS[name]
    alg = algorithmic(B, NH, S, DH)
    pk = peaks()
    set_bytes = alg["bytes_fwd"] + alg["bytes_bwd"]
    nsets = max(2, int(2.2 * L2_BYTES / set_bytes) + 1)
    plans = []
    for s_ in range(nsets):
        q, k, v, i, f, dh = as_heads(make_inputs(torch, B, NH, S, DH, 1000 * rank + s_, dev, torch.bfloat16, on_device=on_device))
        plans.append(ops.MLSTMPlan(q, k, v, i, f, dh, eps=1e-6, chunk_size=CHUNK, reverse=bool(reverse)))
    pl0 = plans[0]

    def step(pl, evs=None):
        # timed step: forward + the whole backward in one call, as mLSTMBackend's autograd node makes it (with few (batch, head)
        # pairs the library then runs the adjoint-state walk and the dq kernel in one launch); the per-kernel pass (evs) calls
        # the backward's two parts separately to put events between them
        if evs is None:
            pl.forward()
            pl.backward()
            return
        evs[0].record()
        pl.forward()
        evs[1].record()
        pl.backward(0)
        evs[2].record()
        pl.backward(1)
        evs[3].record()

    for w in range(W):
        step(plans[w % nsets])
    torch.cuda.synchronize()
    l0 = _lib.launch_count()
    step(plans[W % nsets])
    launches_per_step = _lib.launch_count() - l0
    torch.cuda.synchronize()

    # The timed region replays a CUDA graph of one round over the input sets (nsets steps, so the L2 rotation is kept): the
    # kernels are the same launches with the same arguments, without the Python / ctypes time per step that otherwise competes
    # with a 60 us step (and with the other ranks' host threads at N > 1).  BENCH_NO_GRAPH=1 times eager launches instead.
    graph = None
    if not os.environ.get("BENCH_NO_GRAPH"):
        try:
            cap = torch.cuda.Stream(device=dev)
            cap.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(cap):
                graph = torch.cuda.CUDAGraph()
                # thread_local: other threads of the process (NCCL's watchdog at N > 1) may keep calling the CUDA runtime
                with torch.cuda.graph(graph, stream=cap, capture_error_mode="thread_local"):
                    for s_ in range(nsets):
                        step(plans[s_])
            torch.cuda.current_stream(dev).wait_stream(cap)
            graph.replay()
            torch.cuda.synchronize()
        except Exception as exc:   # capture unsupported: fall back to eager launches, say so
            print(f"bench: CUDA graph capture failed ({exc}); timing eager launches", file=sys.stderr)
            graph = None
            torch.cuda.synchronize()

    def run_steps(n, first):
        """n steps; returns the plan of the last one."""
        if graph is not None:
            for _ in range(n // nsets):
                graph.replay()
            for s_ in range(n - n % nsets, n):
                step(plans[s_ % nsets])
            return plans[(n - 1) % nsets]
        for s_ in range(n):
            step(plans[(first + s_) % nsets])
        return plans[(first + n - 1) % nsets]

    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_start = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    t_start.record()
    last = run_steps(K, W)
    t_end.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    elapsed_ms = t_start.elapsed_time(t_end)
    # copied before the passes below write the plans' output buffers again
    outputs = {n_: t.clone() for n_, t in zip(("h", "dq", "dk", "dv", "di", "df"),
                                              (last.h, last.dq, last.dk, last.dv, last.di, last.df))} if keep_outputs else None
    # The same K steps as eager launches through the plan's C-ABI calls (no graph): what the step costs with the host in the loop
    eager_value = None
    if graph is not None and world == 1:
        t_a, t_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for s_ in range(3):
            step(plans[s_ % nsets])
        torch.cuda.synchronize()
        t_a.record()
        for s_ in range(K):
            step(plans[(W + s_) % nsets])
        t_b.record()
        torch.cuda.synchronize()
        eager_value = B * S / (t_a.elapsed_time(t_b) / K * 1e-3)
    # Second pass, same K steps, eager, with an event pair around every launch: the per-kernel durations the roofline uses.
    # Kept out of the headline region because the events themselves cost ~2.7 us per pair (the fused backward's empty
    # part 0 measures exactly that) and serialise consecutive launches.
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(K)]
    for s_ in range(K):
        step(plans[(W + s_) % nsets], evs[s_])
    torch.cuda.synchronize()
    fwd_ms = sum(e[0].elapsed_time(e[1]) for e in evs) / K
    dq_ms = sum(e[1].elapsed_time(e[2]) for e in evs) / K
    dkv_ms = sum(e[2].elapsed_time(e[3]) for e in evs) / K
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / K
    value = world * B * S / (ms_per_step * 1e-3)

    parts = {"fwd": (fwd_ms, alg["bytes_fwd"]), "bwd_dq": (dq_ms, alg["bytes_bwd_dq"]), "bwd_dkv": (dkv_ms, alg["bytes_bwd_dkv"])}
    if pl0.variant_bwd == "fused_walk":   # one kernel does the whole backward (part 0 launches nothing): SURVEY.md §8(d)'s 14 DH + 24 B
        parts["bwd_dkv"] = (dkv_ms, alg["bytes_bwd"])
    dom = max(parts, key=lambda n: parts[n][0])
    dom_ms, dom_bytes = parts[dom]
    lo = launches_of(pl0.variant_fwd, pl0.variant_bwd, DH)
    achieved = dom_bytes / (dom_ms * 1e-3) / 1e9
    roofline = {
        "bound": "hbm", "kernel": f"{pl0.family}:{'bwd_fused' if (dom == 'bwd_dkv' and pl0.variant_bwd == 'fused_walk') else dom}",
        "launches": lo[dom], "variants": {"fwd": pl0.variant_fwd, "bwd": pl0.variant_bwd}, "achieved": achieved,
        "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": achieved / pk["hbm_gbs"], "traffic": NCU_TRAFFIC_BYTES.get(name, {}).get(dom),
        "traffic_unit": "bytes/launch (ncu dram read+write, profiles/r0*_ncu_full_*)",
        "algorithmic_bytes": dom_bytes, "peak_source": pk["source"],
        "per_kernel_ms": {"fwd": fwd_ms, "bwd_dq": dq_ms, "bwd_dkv": dkv_ms},
        "step_hbm_frac": (alg["bytes_fwd"] + alg["bytes_bwd"]) / (ms_per_step * 1e-3) / 1e9 / pk["hbm_gbs"],
        "step_tensor_frac": alg["flops_fwdbwd"] / (ms_per_step * 1e-3) / 1e12 / pk["bf16_tflops_sustained"],
        # the tensor fraction a step running exactly at the HBM roofline would show (0.41 at DH 128, 0.74 at DH 256)
        "step_tensor_ceiling": min(1.0, alg["flops_fwdbwd"] / (alg["bytes_fwd"] + alg["bytes_bwd"]) * pk["hbm_gbs"] * 1e9 / 1e12
                                   / pk["bf16_tflops_sustained"]),
    }
    return {
        "value": value, "ms_per_step": ms_per_step, "roofline": roofline, "launches_per_step": int(launches_per_step),
        "family": pl0.family, "nsets": nsets, "set_bytes": set_bytes, "graph": graph is not None, "plans": plans, "step": step,
        "eager_value": eager_value, "outputs": outputs,
    }


DUMP_BYTES = 64_000_000


def dump_outputs(torch, outputs, out_dir):
    """Writes each output as ``out_dir/<name>.npy`` in float32 ((B, NH, S, DH) or (B, NH, S), the layout a caller of the cell
    receives).  When they come to more than DUMP_BYTES together, each is replaced by a flat sample of its elements, the same
    share of every output, at positions drawn from a fixed seed: two runs of the same workload sample the same elements."""
    import numpy as np
    total = sum(t.numel() for t in outputs.values()) * 4
    budget = DUMP_BYTES - 256 * len(outputs)       # room for the .npy headers
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        t = t.float()
        if total > budget:
            n = t.numel() * budget // total
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:n].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(out_dir, name + ".npy"), t.contiguous().cpu().numpy())


def measure_e2e(torch, dist, name, K, dev, rank, world, full_result):
    """End-to-end arm: host buffers -> public API (mLSTMBackend + autograd) -> host, every copy inside the timed region.
    Inputs come from pinned host memory on a copy stream (double-buffered, so step s+1's H2D overlaps step s's kernels — what a
    training input pipeline does).  ``full_result``: the whole result (h, dq, dk, dv, di, df) is copied back to pinned host
    memory on a third stream; otherwise a 4-float checksum of it (the round-1 variant, kept as the second number)."""
    from xlstm_yolo_b200.backend import mLSTMBackend, mLSTMBackendConfig
    B, NH, S, DH = WORKLOADS[name]
    be = mLSTMBackend(mLSTMBackendConfig(chunk_size=CHUNK, eps=1e-6, autocast_kernel_dtype="bfloat16"))
    NBUF = 2

    def flat_views(like, device, pinned=False):
        """One flat byte buffer with a view per tensor of `like` (same dtype, shape, strides; 256-byte aligned offsets): the six
        operands of a step travel as ONE copy instead of six (two of them 0.2 MB: per-copy latency, not bandwidth)."""
        offs, total = [], 0
        for t in like:
            offs.append(total)
            total += (t.numel() * t.element_size() + 255) // 256 * 256
        flat = torch.empty(total, dtype=torch.uint8, device=device, pin_memory=pinned)
        views = [flat[o:o + t.numel() * t.element_size()].view(t.dtype).as_strided(t.shape, t.stride()) for o, t in zip(offs, like)]
        return flat, views

    src = make_inputs(torch, B, NH, S, DH, 77 + rank, "cpu", torch.bfloat16)
    host_flat, host = flat_views(src, "cpu", pinned=True)
    for hv, t in zip(host, src):
        hv.copy_(t)
    dev_flat, dev_in = [], []
    for _ in range(NBUF):
        fl, vs = flat_views(src, dev)
        dev_flat.append(fl)
        dev_in.append(vs)
    res_host = [torch.empty(4, dtype=torch.float32).pin_memory() for _ in range(NBUF)]
    # static device-side result slots: a non_blocking D2H copy from a freshly allocated tensor makes the
    # caching allocator cudaMalloc every step (measured: 2.7 mallocs/step, 1.4-35 ms of host time)
    res_dev = [torch.zeros(4, dtype=torch.float32, device=dev) for _ in range(NBUF)]
    res_full = [None] * NBUF          # pinned host tensors with the strides of the results, made on first use
    res_slot = [None] * NBUF          # static device-side copies of the results (same strides)
    res_full_flat, res_slot_flat = [None] * NBUF, [None] * NBUF   # the flat buffers behind them: one copy each way per step
    h2d = sum(t.numel() * t.element_size() for t in host)
    d2h = [res_host[0].numel() * 4]
    main_stream = torch.cuda.current_stream(dev)
    copy_stream = main_stream if os.environ.get("BENCH_E2E_SERIAL") else torch.cuda.Stream(device=dev)
    back_stream = main_stream if os.environ.get("BENCH_E2E_SERIAL") else torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event() for _ in range(NBUF)]
    freed = [torch.cuda.Event() for _ in range(NBUF)]
    done = [torch.cuda.Event() for _ in range(NBUF)]
    copied = [torch.cuda.Event() for _ in range(NBUF)]
    for ev in freed + copied:
        ev.record(main_stream)

    def e2e_copy(sidx):
        b_ = sidx % NBUF
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[b_])
            dev_flat[b_].copy_(host_flat, non_blocking=True)     # q, k, v, i, f, dh in one DMA
            ready[b_].record(copy_stream)

    def e2e_compute(sidx):
        b_ = sidx % NBUF
        main_stream.wait_event(ready[b_])
        q, k, v, i, f, dh = as_heads(dev_in[b_])
        leaves = [t.detach().requires_grad_(True) for t in (q, k, v, i, f)]
        h = be(*leaves)
        h.backward(dh)
        outs = [h.detach()] + [l.grad for l in leaves]
        freed[b_].record(main_stream)
        if full_result:
            if res_full[b_] is None:
                # pinned host tensors with exactly the results' strides ((B,S,NH,DH) storage viewed (B,NH,S,DH)): each copy is
                # then one plain DMA, not a transposing kernel plus a staged copy.  Static device-side slots of the same
                # layout in between: a D2H copy straight from the step's own (freshly allocated) tensors on another stream
                # needs record_stream, which keeps their blocks out of the caching allocator for a step or two and makes
                # it cudaMalloc inside the timed region (measured: 1.2-4.5 ms per step, erratic, against 0.7 ms here).
                res_full_flat[b_], res_full[b_] = flat_views(outs, "cpu", pinned=True)
                res_slot_flat[b_], res_slot[b_] = flat_views(outs, dev)
                d2h[0] = sum(o.numel() * o.element_size() for o in outs)
            main_stream.wait_event(copied[b_])          # the slot's previous content has reached the host
            with torch.no_grad():
                for o, r in zip(outs, res_slot[b_]):
                    r.copy_(o)
            done[b_].record(main_stream)
            with torch.cuda.stream(back_stream):
                back_stream.wait_event(done[b_])
                res_full_flat[b_].copy_(res_slot_flat[b_], non_blocking=True)     # h, dq, dk, dv, di, df in one DMA
                copied[b_].record(back_stream)
        else:
            with torch.no_grad():
                torch.stack([outs[0].abs().mean(dtype=torch.float32), outs[1].abs().mean(dtype=torch.float32),
                             outs[4].abs().mean(), outs[5].abs().mean()], out=res_dev[b_])
            res_host[b_].copy_(res_dev[b_], non_blocking=True)

    def e2e_run(n):
        e2e_copy(0)
        for s_ in range(n):
            if s_ + 1 < n:
                e2e_copy(s_ + 1)
            e2e_compute(s_)

    e2e_run(3)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    e2e_run(K)
    if back_stream is not main_stream:
        main_stream.wait_stream(back_stream)     # the result's way back to the host is inside the timed region
    e1.record()
    torch.cuda.synchronize()
    e2e_ms = e0.elapsed_time(e1) / K
    if world > 1:
        t = torch.tensor([e2e_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t.item())
    return {"value": world * B * S / (e2e_ms * 1e-3), "unit": "tokens/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h[0],
            "ms_per_step": e2e_ms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--reverse", type=int, default=0)
    ap.add_argument("--cpu-sample-batch", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the `also` block (the other BASELINE shapes)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the workload computed (h, dq, dk, dv, di, df) as DIR/<name>.npy, "
                         "float32, at most 64 MB in all (a fixed sample of each output beyond that); the inputs are seeded")
    args = ap.parse_args()
    # stdout carries exactly one JSON line: whatever libraries print there (NCCL's version banner under NCCL_DEBUG=VERSION,
    # for one) is sent to stderr by pointing fd 1 at fd 2; emit() writes to the saved descriptor
    global _OUT_FD
    sys.stdout.flush()
    _OUT_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from xlstm_yolo_b200 import _lib, ops

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.load()

    B, NH, S, DH = WORKLOADS[args.workload]
    W = max(3, args.warmup)
    K = max(1, args.steps)

    # ---- device-resident arm ("value") of the headline workload, clocks sampled during it --------
    sampler = ClockSampler(local_rank)
    sampler.start()
    m = measure_device(torch, dist, ops, _lib, args.workload, K, W, dev, rank, world, reverse=bool(args.reverse),
                       keep_outputs=bool(args.dump_outputs) and rank == 0)
    # keep the sampler alive long enough for at least a few samples of a very short region
    t_hold = time.time()
    while len(sampler.samples) < 3 and time.time() - t_hold < 0.2:
        m["step"](m["plans"][0])
    torch.cuda.synchronize()
    sampler.stop_flag = True
    sampler.join(timeout=1.0)
    del m["plans"]
    if m["outputs"] is not None:
        dump_outputs(torch, m.pop("outputs"), args.dump_outputs)

    # ---- end-to-end arm: the whole result comes back (headline); the checksum variant beside it --------
    e2e = measure_e2e(torch, dist, args.workload, K, dev, rank, world, full_result=True)
    e2e_ck = measure_e2e(torch, dist, args.workload, K, dev, rank, world, full_result=False)
    e2e.update({"api": "xlstm_yolo_b200.mLSTMBackend + autograd",
                "pipeline": "H2D of step s+1 on a copy stream overlaps step s; the full result (h, dq, dk, dv, di, df) goes back "
                            "to pinned host memory on a third stream",
                "checksum_variant": {"value": e2e_ck["value"], "ms_per_step": e2e_ck["ms_per_step"],
                                     "d2h_bytes_per_step": e2e_ck["d2h_bytes_per_step"],
                                     "what": "4-float checksum of the result reduced on the device and copied back (round-1 e2e)"}})

    out = {
        "metric": "mLSTM fwd+bwd tokens/s/GPU", "value": m["value"], "unit": "tokens/s", "n_gpus": world, "steps": K,
        "warmup": W, "ms_per_step": m["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": args.workload, "B_per_gpu": B, "NH": NH, "S": S, "DH": DH, "chunk_size": CHUNK,
                   "reverse": int(args.reverse), "kernel_family": m["family"],
                   "l2": f"inputs rotate over {m['nsets']} sets x {m['set_bytes'] / 1e6:.0f} MB > 126 MB L2", "parallelism": f"dp{world}",
                   "launch": (f"CUDA graph of {m['nsets']} steps (one per input set) replayed" if m["graph"] else "eager ctypes launches"),
                   "per_kernel_ms": "second pass of the same K steps with an event pair around every launch",
                   "eager_tokens_per_s": m["eager_value"]},   # the same steps launched eagerly through the C ABI (no graph)
        "clocks": sampler.result(),
        "e2e": e2e,
        "gpu_launches": int(m["launches_per_step"] * K),
        "roofline": m["roofline"],
    }

    # ---- the other BASELINE shapes, same method, same run (N = 1) --------------------------------------
    if world == 1 and not args.no_also and args.workload == DEFAULT_WORKLOAD:
        also = []
        for name in ALSO_WORKLOADS:
            torch.cuda.empty_cache()
            ma = measure_device(torch, dist, ops, _lib, name, K, 3, dev, rank, world, on_device=True)
            del ma["plans"]
            Ba, NHa, Sa, DHa = WORKLOADS[name]
            also.append({"workload": name, "B_per_gpu": Ba, "NH": NHa, "S": Sa, "DH": DHa, "value": ma["value"], "unit": "tokens/s",
                         "steps": K, "warmup": 3, "ms_per_step": ma["ms_per_step"], "gpu_launches": int(ma["launches_per_step"] * K),
                         "roofline": ma["roofline"], "data": "synthetic, drawn on the device"})
        out["also"] = also

    # ---- CPU baseline (rank 0, N=1): the reference's CPU path on the host cores, bounded sample ------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        torch.set_num_threads(cores)
        step_cpu, kind, what = reference_step_fn(torch)
        cin = cpu_inputs(torch, B, NH, S, DH)
        t0 = time.perf_counter()
        step_cpu(cin)
        t_one = time.perf_counter() - t0
        n = max(1, min(10, int(15.0 / max(t_one, 1e-3))))
        t0 = time.perf_counter()
        for _ in range(n):
            step_cpu(cin)
        dt = (time.perf_counter() - t0) / n
        out["cpu_baseline"] = {"value": B * S / dt, "unit": "tokens/s", "cores": cores, "kind": kind,
                               "sample": f"full batch {B}/{B} of {args.workload}, {n} steps, chunk_size {ref_chunk(S)}, fp32, {what}"}
    if rank == 0:
        emit(out)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
