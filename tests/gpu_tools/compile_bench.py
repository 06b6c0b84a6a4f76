"""Whole ViLBlockPair forward + backward under torch.compile, at the three layer_bench.py shapes (bf16 model and input).

Arms, each timed with CUDA events over --steps steps after --warmup steps (compilation happens in the warm-up):
  eager             the autograd.Functions of ops.py
  eager_ops         eager mode through the registered custom ops instead (what a single-path design would run)
  inductor          torch.compile(pair)
  inductor_unfused  torch.compile(pair) with fused_gates / fused_producer / fused_tail off: cuDNN conv, bmm producer,
                    F.linear gates and the group-norm tail around the bare cell op
Each line also gives the library's kernel launches per step (mlstm_b200_launch_count) of every arm.  The arms run
round-robin --rounds times on the same inputs; every timing of every round is printed."""
import argparse
import copy
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch

from xlstm_yolo_b200 import ViLBlockPair, _lib, ops

SHAPES = [(32, 20, 128, 64), (32, 40, 256, 128), (8, 80, 256, 128)]   # (B, grid, dim, qkv_block_size)


def card():
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return f"{torch.cuda.get_device_name(0)}, power limit {pl}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=2)
    a = ap.parse_args()
    print(f"# {card()}; torch {torch.__version__}", flush=True)
    for B, grid, dim, bs in SHAPES:
        S = grid * grid
        torch.manual_seed(0)
        pair = ViLBlockPair(dim=dim, chunk_size=64, qkv_block_size=bs).cuda().to(torch.bfloat16).train()
        unfused = copy.deepcopy(pair)
        for blk in (unfused.rowwise_from_top_left, unfused.rowwise_from_bot_right):
            blk.layer.fused_producer = False
            blk.layer.fused_tail = False
            blk.layer.mlstm_cell.fused_gates = False
        x = torch.randn(B, S, dim, device="cuda", dtype=torch.bfloat16, requires_grad=True)
        dy = torch.randn(B, S, dim, device="cuda", dtype=torch.bfloat16)
        torch._dynamo.reset()
        arms = {"eager": (pair, False), "eager_ops": (pair, True), "inductor": (torch.compile(pair), False),
                "inductor_unfused": (torch.compile(unfused), False)}
        use_ops = ops._use_custom_ops

        def step(m, force_ops):
            ops._use_custom_ops = (lambda: True) if force_ops else use_ops
            try:
                m(x).backward(dy)
            finally:
                ops._use_custom_ops = use_ops

        times = {k: [] for k in arms}
        launches = {}
        for name, (m, force) in arms.items():
            for _ in range(a.warmup):
                step(m, force)
            torch.cuda.synchronize()
            n0 = _lib.launch_count()
            step(m, force)
            torch.cuda.synchronize()
            launches[name] = _lib.launch_count() - n0
        for _ in range(a.rounds):
            for name, (m, force) in arms.items():
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.steps):
                    step(m, force)
                e1.record()
                torch.cuda.synchronize()
                times[name].append(e0.elapsed_time(e1) / a.steps)
        cols = "  ".join(f"{k} {'/'.join(f'{t:.3f}' for t in v)} ms ({launches[k]} launches)" for k, v in times.items())
        print(f"ViLBlockPair dim={dim} inner={2 * dim} DH={bs} B={B} S={S} fwd+bwd: {cols}", flush=True)


if __name__ == "__main__":
    main()
