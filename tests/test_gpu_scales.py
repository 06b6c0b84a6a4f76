"""The x-scale ViL layer on the hand-written kernels: the layer tail at the inner dims that are multiples of 256 but do not
divide 2048 (csrc/mlstm_glue.cu), the gate forward on the tensor cores at up to 32 gate outputs (csrc/mlstm_gates_tc.cu),
and a whole x-scale ViLBlockPair (dim 768: inner 1536, NH 12, DH 128) eager and compiled."""
import copy
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float(((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).detach())


# ---------------------------------------------------------------------------------------------------------------------
# Layer tail
# ---------------------------------------------------------------------------------------------------------------------
def tail_reference(h, c, z, w, b, skip, eps):
    B, NH, S, DH = h.shape
    x = h.transpose(1, 2).reshape(B * S, NH * DH)
    n = F.group_norm(x, num_groups=NH, weight=1.0 + w, bias=b, eps=eps).view(B, S, NH * DH)
    return (n + skip * c) * F.silu(z)


@pytest.mark.parametrize("D", [768, 1280, 1536, 1792])
@pytest.mark.parametrize("DH", [64, 128])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_layer_tail_at_new_widths(D, DH, dtype):
    from xlstm_yolo_b200 import ops
    B, S, NH = 2, 203, D // DH
    g = torch.Generator().manual_seed(D + DH)
    h = (torch.randn(B, S, NH, DH, generator=g) * 0.7 + 0.1).to(dtype).cuda().transpose(1, 2)
    c = torch.randn(B, S, D, generator=g).to(dtype).cuda()
    up = torch.randn(B, S, 2 * D, generator=g).to(dtype).cuda()
    w = (torch.randn(D, generator=g) * 0.2).cuda()
    b = (torch.randn(D, generator=g) * 0.2).cuda()
    skip = (1 + torch.randn(D, generator=g) * 0.2).cuda()
    dy = torch.randn(B, S, D, generator=g).to(dtype).cuda()
    assert ops.glue_supported(h, c, up[..., D:])            # z as a column slice with row stride 2 D

    def run():
        leaves = [t.detach().clone().requires_grad_(True) for t in (h, c, up, w, b, skip)]
        y = ops.layer_tail(leaves[0], leaves[1], leaves[2][..., D:], leaves[3], leaves[4], leaves[5], eps=1e-3)
        y.backward(dy)
        return y.detach(), [t.grad for t in leaves]

    y, grads = run()
    ref = [t.detach().double().requires_grad_(True) for t in (h, c, up, w, b, skip)]
    yr = tail_reference(ref[0], ref[1], ref[2][..., D:], ref[3], ref[4], ref[5], 1e-3)
    yr.backward(dy.double())
    ty, tg = (1e-2, 2e-2) if dtype == torch.bfloat16 else (1e-5, 1e-4)
    assert y.shape == (B, S, D) and y.dtype == dtype
    assert rel(y, yr) < ty
    for n, a, r in zip(["dh", "dc", "dup", "dw", "db", "dskip"], grads, ref):
        assert a is not None, n
        assert rel(a, r.grad) < (tg if n in ("dh", "dc", "dup") else 1e-3 if dtype == torch.float32 else 2e-2), n
    y2, grads2 = run()
    assert torch.equal(y2, y)
    for n, a, a2 in zip(["dh", "dc", "dup", "dw", "db", "dskip"], grads, grads2):
        assert torch.equal(a, a2), n                          # fixed-order partial reduction: bit-identical


# ---------------------------------------------------------------------------------------------------------------------
# Gate forward on the tensor cores
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,S,D,NH", [(2, 256, 1024, 8), (2, 400, 1536, 12), (1, 384, 2048, 16), (1, 203, 1536, 12),
                                      (3, 77, 512, 16), (2, 130, 128, 12), (1, 300, 256, 4)])
def test_gate_forward_tensor_cores_wide(B, S, D, NH):
    from xlstm_yolo_b200 import _lib, ops
    g = torch.Generator().manual_seed(D + NH + S)
    q, k, v = ((torch.randn(B, S, D, generator=g) * 0.5).to(torch.bfloat16).cuda() for _ in range(3))
    w_i, w_f = (torch.randn(NH, 3 * D, generator=g).mul(0.05).cuda() for _ in range(2))
    b_i, b_f = (torch.randn(NH, generator=g).cuda() for _ in range(2))
    p = ops._gate_params(q, k, v, w_i, b_i, w_f, b_f, NH)
    streamed = _lib.load().mlstm_b200_gates_fwd_workspace_bytes(p) > 0
    assert streamed == (D >= 512)            # the split weights fit in shared memory at D 128 (16+ outputs) and D 256 (8)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    i, f = ops.gate_proj_fwd_raw(q, k, v, w_i, b_i, w_f, b_f, NH)
    torch.cuda.synchronize()
    assert _lib.launch_count() - n0 == (2 if streamed else 1)      # streamed: the weight split, then the streaming kernel
    x = torch.cat([q, k, v], dim=-1).double()
    ri, rf = F.linear(x, w_i.double(), b_i.double()), F.linear(x, w_f.double(), b_f.double())
    assert i.shape == (B, S, NH) and i.dtype == torch.float32
    assert rel(i, ri) < 2e-6 and rel(f, rf) < 2e-6
    i2, f2 = ops.gate_proj_fwd_raw(q, k, v, w_i, None, w_f, None, NH)
    assert rel(i2, ri - b_i.double()) < 1e-5 and rel(f2, rf - b_f.double()) < 1e-5


# ---------------------------------------------------------------------------------------------------------------------
# x-scale ViLBlockPair
# ---------------------------------------------------------------------------------------------------------------------
def _x_pair(seed=0):
    from xlstm_yolo_b200 import ViLBlockPair
    torch.manual_seed(seed)
    pair = ViLBlockPair(dim=768, chunk_size=64, qkv_block_size=128).cuda()
    with torch.no_grad():
        for p in pair.parameters():
            if p.dim() == 1:
                p.add_(torch.randn_like(p) * 0.1)
    return pair


def _step(m, x, dy, dtype):
    from xlstm_yolo_b200 import _lib
    m.zero_grad(set_to_none=True)
    xx = x.clone().requires_grad_(True)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    with torch.autocast("cuda", dtype=dtype):
        y = m(xx)
    y.backward(dy)
    torch.cuda.synchronize()
    grads = [p.grad for p in m.parameters() if p.requires_grad]
    return [y.detach().float(), xx.grad] + grads, _lib.launch_count() - n0


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_x_scale_pair_kernels_match_the_unfused_layer(dtype):
    pair = _x_pair()
    plain = copy.deepcopy(pair)
    for blk in (plain.rowwise_from_top_left, plain.rowwise_from_bot_right):
        blk.layer.fused_tail = False
        blk.layer.fused_producer = False
        blk.layer.mlstm_cell.fused_gates = False
    g = torch.Generator().manual_seed(1)
    x, dy = (torch.randn(2, 400, 768, generator=g).cuda() for _ in range(2))
    got, _ = _step(pair, x, dy, dtype)
    want, _ = _step(plain, x, dy, dtype)
    assert len(got) == len(want)
    for j, (a, b) in enumerate(zip(got, want)):
        assert (a is None) == (b is None), j       # parameters outside the pair's path (no gradient in either) are skipped
        if b is not None:
            assert torch.isfinite(a).all(), j
            assert rel(a, b) < (2e-2 if j == 0 else 4e-2), (j, rel(a, b))


def test_x_scale_pair_compiles_to_one_graph():
    from functorch.compile import make_boxed_func
    from torch._dynamo.backends.common import aot_autograd
    fw, bw = [], []

    def keep(store):
        def compiler(gm, example_inputs):
            store.append(gm)
            return make_boxed_func(gm.forward)
        return compiler

    pair = _x_pair()
    g = torch.Generator().manual_seed(2)
    x, dy = (torch.randn(2, 400, 768, generator=g).cuda() for _ in range(2))
    want, n_eager = _step(pair, x, dy, torch.bfloat16)
    torch._dynamo.reset()
    comp = torch.compile(pair, backend=aot_autograd(fw_compiler=keep(fw), bw_compiler=keep(bw)), fullgraph=True)
    _step(comp, x, dy, torch.bfloat16)
    got, n_comp = _step(comp, x, dy, torch.bfloat16)
    assert len(fw) == 1 and len(bw) == 1
    tails = [n for n in fw[0].graph.nodes if n.op == "call_function" and str(n.target) == "xlstm_yolo_b200.layer_tail_fwd.default"]
    assert len(tails) == 2
    assert n_comp == n_eager
    for j, (a, b) in enumerate(zip(got, want)):
        assert (a is None) == (b is None), j
        if b is not None:
            assert rel(a, b) < (1e-2 if j == 0 else 2e-2), (j, rel(a, b))


@pytest.mark.skipif(not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "ultralytics")),
                    reason="baseline/_ref (the reference tree) not present")
def test_x_scale_detector_trains_a_few_steps():
    import json
    import subprocess
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench_detector.py"), "--gpus", "1", "--scale", "x", "--batch", "4",
                        "--steps", "3", "--warmup", "1"], cwd=ROOT, capture_output=True, text=True, timeout=1800)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert "unavailable" not in d, d
    assert d["value"] > 0 and d["loss_finite"] is True
