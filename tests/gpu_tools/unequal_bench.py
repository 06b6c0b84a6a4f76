"""Developer tool: forward + backward of the cell at head dims the tcgen05 kernels are not written for — DHqk = DHv / 2
(mLSTMLayerVision's qk_dim_factor = 0.5), DH = 16 (the reference's default qkv_block_size), 32, 192: the zero-padded tensor-core
path of mlstm_api.cu."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
from xlstm_yolo_b200 import ops

for (B, NH, S, DK, DV) in [(32, 4, 1600, 64, 128), (32, 4, 400, 32, 64), (8, 4, 1600, 64, 128), (32, 4, 1600, 128, 256),
                          (32, 32, 1600, 16, 16), (32, 16, 400, 16, 16), (32, 8, 1600, 32, 32), (16, 4, 1600, 192, 192)]:
    g = torch.Generator().manual_seed(0)
    act = lambda d: (torch.randn(B, S, NH, d, generator=g) * 0.3).to(torch.bfloat16).cuda().transpose(1, 2)
    q, k, v, dh = act(DK), act(DK), act(DV), act(DV)
    i = torch.randn(B, S, NH, generator=g).cuda().transpose(1, 2)
    f = (torch.randn(B, S, NH, generator=g) + 3).cuda().transpose(1, 2)
    pl = ops.MLSTMPlan(q, k, v, i, f, dh)
    n = 5 if pl.family == "simt" else 30
    for _ in range(3):
        pl.forward(); pl.backward()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        pl.forward(); pl.backward()
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / n
    print(f"B{B} NH{NH} S{S} DHqk{DK} DHv{DV}: {pl.family} {pl.variant_fwd}/{pl.variant_bwd} {ms:.3f} ms  {B * S / ms / 1e3:.1f} M tokens/s", flush=True)
