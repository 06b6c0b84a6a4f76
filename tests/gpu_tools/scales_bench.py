"""The x-scale ViL layer pieces on the GPU, one JSON line per measurement:

  * the layer tail at inner dim 1536 (x scale) against the PyTorch ops it replaces (group_norm + skip + SiLU(z));
  * the gate projection forward at the detector's (D, NH) pairs, whichever kernel the loaded library picks;
  * ViLBlockPair forward + backward at the x-scale P4 and P5 shapes, every layer kernel on and all switched off.

Every timed call starts L2-cold: a 256 MB buffer is overwritten before it, outside the CUDA events that time the call.
``--root`` imports ``xlstm_yolo_b200`` from another checkout (for an A/B run against an older library)."""
import argparse
import copy
import json
import os
import sys

ap = argparse.ArgumentParser()
ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
ap.add_argument("--tag", default="this tree")
ap.add_argument("--reps", type=int, default=20)
ap.add_argument("--only", default="", help="run one section: tail, gates or pair")
args = ap.parse_args()
sys.path.insert(0, os.path.abspath(args.root))

import torch
import torch.nn.functional as F
from xlstm_yolo_b200 import ViLBlockPair, _lib, ops

DEV = torch.cuda.get_device_name()
FLUSH = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")


def cold_ms(fn, reps=args.reps, warm=3):
    """Median of ``reps`` calls, each after an L2 flush, each between its own pair of events."""
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(reps):
        FLUSH.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    ts.sort()
    return ts[len(ts) // 2]


def emit(**kw):
    print(json.dumps({"device": DEV, "lib": args.tag, **kw}), flush=True)


# ---- layer tail -----------------------------------------------------------------------------------------------------
for (B, S, NH, DH) in [(32, 1600, 12, 128), (32, 400, 12, 128)] if args.only in ("", "tail") else []:
    D, T = NH * DH, B * S
    h = torch.randn(B, S, NH, DH, device="cuda", dtype=torch.bfloat16).transpose(1, 2).requires_grad_(True)
    c = torch.randn(B, S, D, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    up = torch.randn(B, S, 2 * D, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    w = torch.zeros(D, device="cuda", requires_grad=True)
    b = torch.zeros(D, device="cuda", requires_grad=True)
    skip = torch.ones(D, device="cuda", requires_grad=True)
    dy = torch.randn(B, S, D, device="cuda", dtype=torch.bfloat16)

    def plain_y():
        x = h.transpose(1, 2).reshape(T, D)
        n = F.group_norm(x, NH, (1 + w).to(x.dtype), b.to(x.dtype), 1e-3).view(B, S, D)
        return (n + skip.to(x.dtype) * c) * F.silu(up[..., D:])

    arms = {"torch ops": plain_y}
    if ops.glue_supported(h, c, up[..., D:]):
        arms["fused tail"] = lambda: ops.layer_tail(h, c, up[..., D:], w, b, skip, 1e-3)
    for name, fn in arms.items():
        with torch.no_grad():
            t_f = cold_ms(fn)
        t_fb = cold_ms(lambda: fn().backward(dy))
        emit(bench="layer_tail", arm=name, B=B, S=S, D=D, NH=NH, fwd_ms=t_f, fwd_bwd_ms=t_fb,
             fwd_bwd_GBps=T * D * 2 * (4 + 7) / (t_fb * 1e-3) / 1e9 if name == "fused tail" else None)

# ---- gate projection forward ----------------------------------------------------------------------------------------
lib = _lib.load()
for (B, S, D, NH) in [(32, 1600, 256, 4), (32, 400, 512, 4), (32, 1600, 512, 8), (32, 400, 1024, 8),
                      (32, 1600, 1024, 8), (32, 400, 1536, 12), (32, 1600, 1536, 12), (32, 1600, 2048, 16)] if args.only in ("", "gates") else []:
    q, k, v = (torch.randn(B, S, D, device="cuda", dtype=torch.bfloat16) for _ in range(3))
    w_i, w_f = (torch.randn(NH, 3 * D, device="cuda") * 0.05 for _ in range(2))
    b_i, b_f = (torch.randn(NH, device="cuda") for _ in range(2))
    kernel = "not reported by this library"
    if hasattr(lib, "mlstm_b200_gates_fwd_workspace_bytes"):
        p = ops._gate_params(q, k, v, w_i, b_i, w_f, b_f, NH)
        lib.mlstm_b200_gates_fwd_workspace_bytes.restype = _lib.C.c_size_t
        streamed = lib.mlstm_b200_gates_fwd_workspace_bytes(_lib.C.byref(p))   # every shape here is bf16, D % 64 == 0, 2 NH <= 32
        kernel = "tensor cores, streamed weights" if streamed else "tensor cores, resident weights"
    t = cold_ms(lambda: ops.gate_proj_fwd_raw(q, k, v, w_i, b_i, w_f, b_f, NH))
    emit(bench="gate_fwd", kernel=kernel, B=B, S=S, D=D, NH=NH, ms=t, GBps=B * S * 3 * D * 2 / (t * 1e-3) / 1e9)

# ---- x-scale ViLBlockPair -------------------------------------------------------------------------------------------
for (B, grid) in [(32, 40), (32, 20)] if args.only in ("", "pair") else []:
    S, dim = grid * grid, 768
    torch.manual_seed(0)
    pair = ViLBlockPair(dim=dim, chunk_size=64, qkv_block_size=128).cuda().to(torch.bfloat16).train()
    plain = copy.deepcopy(pair)
    for blk in (plain.rowwise_from_top_left, plain.rowwise_from_bot_right):
        blk.layer.fused_producer = False
        blk.layer.fused_tail = False
        blk.layer.mlstm_cell.fused_gates = False
    x = torch.randn(B, S, dim, device="cuda", dtype=torch.bfloat16, requires_grad=True)
    dy = torch.randn(B, S, dim, device="cuda", dtype=torch.bfloat16)
    for name, m in (("layer kernels", pair), ("switches off", plain)):
        t = cold_ms(lambda: m(x).backward(dy), reps=max(5, args.reps // 2))
        emit(bench="vil_pair_fwd_bwd", arm=name, B=B, S=S, dim=dim, ms=t)
