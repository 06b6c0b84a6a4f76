"""torch.compile runs the hand-written layer kernels: the gate projection fused with the cell, the conv + SiLU + q / k / v
producer and the out-norm + skip + SiLU(z) tail are ``torch.library`` custom ops (``xlstm_yolo_b200::*``), so a compiled
``ViLBlockPair`` is one graph that launches what eager mode launches and computes what eager mode computes.

The tests without the ``gpu`` mark trace on CUDA fake tensors, which need no device (only the built library, for its
host-side shape queries)."""
import contextlib

import pytest
import torch
from torch._dynamo.backends.common import aot_autograd
from torch._subclasses.fake_tensor import FakeTensorMode

OPS = ("qkv", "fused_cell", "layer_tail")
BANNED = ("aten.convolution", "aten.native_group_norm", "aten.bmm", "aten.baddbmm")
# (dim, qkv_block_size, S, autocast dtype): the two pairs every whole-layer check runs
PAIRS = [(128, 64, 400, torch.bfloat16), (256, 128, 1600, torch.float16)]


def rel(a, b):
    a, b = a.float(), b.float()
    return ((a - b).abs().max() / b.abs().max().clamp_min(1e-30)).item()


def op_counts(gm):
    """{target name: count} of the call_function nodes of an FX graph."""
    out = {}
    for n in gm.graph.nodes:
        if n.op == "call_function":
            name = str(n.target)
            out[name] = out.get(name, 0) + 1
    return out


def ours(counts, name):
    return counts.get(f"xlstm_yolo_b200.{name}.default", 0)


def banned(counts):
    return [k for k in counts if k.startswith(BANNED)]


def nodes_of(gm, name):
    return [n for n in gm.graph.nodes if n.op == "call_function" and str(n.target) == f"xlstm_yolo_b200.{name}.default"]


class Recorder:
    """An aot_autograd backend that keeps the forward and backward graphs it is handed and runs them as they are."""

    def __init__(self):
        from functorch.compile import make_boxed_func
        self.fw, self.bw = [], []

        def keep(store):
            def compiler(gm, example_inputs):
                store.append(gm)
                return make_boxed_func(gm.forward)
            return compiler

        self.backend = aot_autograd(fw_compiler=keep(self.fw), bw_compiler=keep(self.bw))


@contextlib.contextmanager
def fake_cuda(dtype):
    """Modules and tensors built inside are CUDA fake tensors of ``dtype``."""
    old = torch.get_default_dtype()
    torch.set_default_dtype(dtype)
    try:
        with FakeTensorMode(allow_non_fake_inputs=True), torch.device("cuda"):
            yield
    finally:
        torch.set_default_dtype(old)


def _lib_or_skip():
    from xlstm_yolo_b200 import _lib
    try:
        _lib.load()
    except _lib.LibraryMissing as e:
        pytest.skip(str(e))


# ---------------------------------------------------------------------------------------------------------------------
# Without a device: trace on CUDA fake tensors
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dim,bs,S", [(128, 64, 400), (256, 128, 1600)])
def test_fake_pair_forward_is_one_graph_of_our_ops(dim, bs, S):
    """Forward-only (no_grad): one graph holding two of each forward op and no conv / group norm / bmm; the fused cell
    skips n_row, m_row (save_rows False) and the producer skips silu'(conv(x)) (need_sp False)."""
    _lib_or_skip()
    from xlstm_yolo_b200 import ViLBlockPair
    torch._dynamo.reset()
    rec = Recorder()
    with fake_cuda(torch.bfloat16):
        pair = ViLBlockPair(dim=dim, chunk_size=64, qkv_block_size=bs)
        x = torch.empty(2, S, dim)
        with torch.no_grad():
            y = torch.compile(pair, backend=rec.backend, fullgraph=True)(x)
        assert y.shape == x.shape and y.is_cuda
    assert len(rec.fw) == 1
    counts = op_counts(rec.fw[0])
    assert all(ours(counts, f"{o}_fwd") == 2 for o in OPS), counts
    assert not banned(counts), banned(counts)
    for n in nodes_of(rec.fw[0], "fused_cell_fwd"):
        assert n.args[12] is False          # save_rows
    for n in nodes_of(rec.fw[0], "qkv_fwd"):
        assert n.args[-1] is False          # need_sp


def test_fake_pair_forward_with_dynamic_batch():
    """A symbolic batch size traces into one graph: the chunk-state buffer is sized B times one batch row's bytes."""
    _lib_or_skip()
    from xlstm_yolo_b200 import ViLBlockPair
    torch._dynamo.reset()
    rec = Recorder()
    with fake_cuda(torch.bfloat16):
        pair = ViLBlockPair(dim=128, chunk_size=64, qkv_block_size=64)
        x = torch.empty(3, 400, 128)
        torch._dynamo.mark_dynamic(x, 0)
        with torch.no_grad():
            y = torch.compile(pair, backend=rec.backend, fullgraph=True)(x)
        assert y.shape == x.shape
    assert len(rec.fw) == 1
    counts = op_counts(rec.fw[0])
    assert all(ours(counts, f"{o}_fwd") == 2 for o in OPS), counts
    assert any(isinstance(p, torch.SymInt) for n in nodes_of(rec.fw[0], "fused_cell_fwd")
               for p in n.meta["val"][0].shape)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_state_buffer_bound(dtype):
    """The forward ops get B times the state bytes of one batch row (with a backward following): never less than what
    the library asks for, at any batch size, variant, head dims or forward-only call."""
    _lib_or_skip()
    from xlstm_yolo_b200 import ops
    for NH in (1, 2, 4, 32):
        for S in (16, 100, 400, 1600, 6400):
            for DK, DV in ((64, 64), (128, 128), (256, 256), (16, 16), (32, 64), (64, 128), (192, 192)):
                for B in (1, 2, 3, 8, 17, 32, 100, 257):
                    for save_rows in (True, False):
                        need = ops._state_bytes(B, NH, S, DK, DV, dtype, save_rows)
                        assert need <= ops._states_numel(B, NH, S, DK, DV, dtype), (NH, S, DK, DV, B, save_rows)


def test_trace_time_checks_read_no_address():
    """The support checks decide on shapes, strides and dtypes while tracing: a fake tensor has no data pointer."""
    _lib_or_skip()
    from xlstm_yolo_b200 import ops
    seen = {}

    def f(x, h, c, z):
        seen["qkv"] = ops.qkv_supported(x, 256, 4, 20, 20)
        seen["glue"] = ops.glue_supported(h, c, z)
        seen["gates"] = ops.gates_supported(256)
        return x.sum()

    torch._dynamo.reset()
    with fake_cuda(torch.bfloat16):
        up = torch.empty(2, 400, 512)
        h = torch.empty(2, 400, 4, 64).transpose(1, 2)
        c, z = torch.empty(2, 400, 256), up[..., 256:]
        torch.compile(f, backend="eager", fullgraph=True)(up[..., :256], h, c, z)
    assert seen == {"qkv": True, "glue": True, "gates": True}


# ---------------------------------------------------------------------------------------------------------------------
# On the B200
# ---------------------------------------------------------------------------------------------------------------------
def _pair(dim, bs, seed=0):
    from xlstm_yolo_b200 import ViLBlockPair
    torch.manual_seed(seed)
    pair = ViLBlockPair(dim=dim, chunk_size=64, qkv_block_size=bs).cuda()
    with torch.no_grad():   # non-trivial gates and norms, so every gradient is exercised
        for p in pair.parameters():
            if p.dim() == 1:
                p.add_(torch.randn_like(p) * 0.1)
    return pair


def _step(m, params, x, dy, dtype, dynamic_batch=False):
    """One forward + backward; returns [y, dx, grads of ``params``] and the library launches it took."""
    from xlstm_yolo_b200 import _lib
    for p in params:
        p.grad = None
    xx = x.clone().requires_grad_(True)
    if dynamic_batch:
        torch._dynamo.mark_dynamic(xx, 0)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    with torch.autocast("cuda", dtype=dtype, enabled=dtype is not None):
        y = m(xx)
    y.backward(dy)
    torch.cuda.synchronize()
    n = _lib.launch_count() - n0
    return [y.detach().clone(), xx.grad.clone()] + [None if p.grad is None else p.grad.clone() for p in params], n


def _inputs(B, S, dim, seed=1):
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, S, dim, generator=g).cuda(), torch.randn(B, S, dim, generator=g).cuda()


def _trained_params(m):
    return [p for p in m.parameters() if p.requires_grad]


def _compare(got, want, tag):
    assert len(got) == len(want)
    for j, (a, b) in enumerate(zip(got, want)):
        assert torch.isfinite(a).all(), f"{tag}: output {j} not finite"
        tol = 1e-2 if j == 0 else 2e-2
        assert rel(a, b) < tol, f"{tag}: output {j} rel err {rel(a, b):.3e}"


@pytest.mark.gpu
@pytest.mark.parametrize("dim,bs,S,dtype", PAIRS)
def test_pair_compiles_to_one_graph_of_our_kernels(dim, bs, S, dtype):
    """fullgraph=True; the forward graph holds two of each forward op, the backward graph two of each backward op, and
    neither a convolution, a group norm or a batched GEMM.  The recorded graphs run: launches and results as eager."""
    pair = _pair(dim, bs)
    x, dy = _inputs(2, S, dim)
    want, n_eager = _step(pair, [], x, dy, dtype)
    torch._dynamo.reset()
    rec = Recorder()
    comp = torch.compile(pair, backend=rec.backend, fullgraph=True)
    got, _ = _step(comp, [], x, dy, dtype)
    got, n_comp = _step(comp, [], x, dy, dtype)
    assert len(rec.fw) == 1 and len(rec.bw) == 1
    fw, bw = op_counts(rec.fw[0]), op_counts(rec.bw[0])
    for o in OPS:
        assert ours(fw, f"{o}_fwd") == 2, fw
        assert ours(bw, f"{o}_bwd") == 2, bw
    assert not banned(fw) and not banned(bw), (banned(fw), banned(bw))
    assert n_comp == n_eager, (n_comp, n_eager)
    _compare(got, want, "recorded graphs")


@pytest.mark.gpu
@pytest.mark.parametrize("backend", ["aot_eager", "inductor"])
@pytest.mark.parametrize("dim,bs,S,dtype", PAIRS)
def test_pair_compiled_matches_eager(dim, bs, S, dtype, backend):
    """y, dx and every parameter gradient within the north-star tolerances; the same library launches per step."""
    pair = _pair(dim, bs)
    params = _trained_params(pair)
    x, dy = _inputs(2, S, dim)
    want, n_eager = _step(pair, params, x, dy, dtype)
    torch._dynamo.reset()
    comp = torch.compile(pair, backend=backend)
    _step(comp, params, x, dy, dtype)
    got, n_comp = _step(comp, params, x, dy, dtype)
    assert n_comp == n_eager, (n_comp, n_eager)
    keep = [j for j, g in enumerate(want) if g is not None]
    assert all(got[j] is not None for j in keep)
    _compare([got[j] for j in keep], [want[j] for j in keep], backend)


@pytest.mark.gpu
def test_pair_reduce_overhead_replays_match_eager():
    """mode="reduce-overhead" (CUDA graphs around the compiled step): three replayed steps, each within tolerance."""
    dim, bs, S, dtype = PAIRS[0]
    pair = _pair(dim, bs)
    params = _trained_params(pair)
    x, dy = _inputs(2, S, dim)
    want, _ = _step(pair, params, x, dy, dtype)
    keep = [j for j, g in enumerate(want) if g is not None]
    torch._dynamo.reset()
    comp = torch.compile(pair, mode="reduce-overhead")
    for _ in range(2):    # warm-up and recording
        torch.compiler.cudagraph_mark_step_begin()
        _step(comp, params, x, dy, dtype)
    for r in range(3):
        torch.compiler.cudagraph_mark_step_begin()
        got, _ = _step(comp, params, x, dy, dtype)
        _compare([got[j] for j in keep], [want[j] for j in keep], f"replay {r}")


@pytest.mark.gpu
@pytest.mark.parametrize("input_gate", ["exp", "sigmoid"])
@pytest.mark.parametrize("reverse", [False, True])
def test_fused_cell_compiled_is_bit_identical(input_gate, reverse):
    """MatrixLSTMCell with the fused gate projection, raw output, under aot_eager with fullgraph=True: h, dq, dk, dv and the
    four gate-parameter gradients equal eager bit for bit (deterministic kernels, nothing else in the graph)."""
    from xlstm_yolo_b200 import MatrixLSTMCell
    torch.manual_seed(0)
    cell = MatrixLSTMCell(dim=256, num_heads=4, chunk_size=64, raw_output=True, reverse=reverse, input_gate=input_gate)
    with torch.no_grad():
        cell.igate.weight.normal_(0, 0.05); cell.fgate.weight.normal_(0, 0.05); cell.igate.bias.normal_(0, 1.0)
    cell = cell.cuda()
    assert cell.fused_gates
    g = torch.Generator().manual_seed(1)
    base = [(torch.randn(2, 400, 256, generator=g) * s).bfloat16().cuda() for s in (0.1, 0.1, 1.0)]
    dh = torch.randn(2, 4, 400, 64, generator=g).bfloat16().cuda()
    rec = Recorder()
    torch._dynamo.reset()
    comp = torch.compile(cell, backend=rec.backend, fullgraph=True)
    res = []
    for m in (cell, comp):
        leaves = [t.clone().requires_grad_(True) for t in base]
        cell.zero_grad()
        h = m(*leaves)
        h.backward(dh)
        gates = [cell.igate.weight, cell.igate.bias, cell.fgate.weight, cell.fgate.bias]
        res.append([h.detach()] + [t.grad for t in leaves] + [p.grad.clone() for p in gates])
    assert ours(op_counts(rec.fw[0]), "fused_cell_fwd") == 1 and ours(op_counts(rec.bw[0]), "fused_cell_bwd") == 1
    for a, b in zip(*res):
        assert torch.isfinite(a).all() and torch.equal(a, b)


def _layer_case(case):
    from xlstm_yolo_b200.vil import SequenceTraversal, ViLLayer
    torch.manual_seed(0)
    if case == "block16":
        m, x, dtype = ViLLayer(128, SequenceTraversal.ROWWISE_FROM_BOT_RIGHT, qkv_block_size=16, chunk_size=64), (2, 400, 128), torch.bfloat16
    elif case == "wide_grid":
        m = ViLLayer(128, SequenceTraversal.ROWWISE_FROM_TOP_LEFT, qkv_block_size=64, chunk_size=64, seqlens=[8, 100])
        x, dtype = (2, 800, 128), torch.bfloat16
    else:   # fp32 activations, no autocast
        m, x, dtype = ViLLayer(128, SequenceTraversal.ROWWISE_FROM_BOT_RIGHT, qkv_block_size=64, chunk_size=64), (2, 400, 128), None
    return m.cuda(), x, dtype


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["block16", "wide_grid", "fp32"])
def test_fallbacks_still_fall_back_when_compiled(case):
    """Shapes and dtypes the producer kernel does not take compile to the PyTorch producer (no producer op in the graph)
    and match eager."""
    m, shape, dtype = _layer_case(case)
    params = _trained_params(m)
    x, dy = _inputs(*shape)
    want, _ = _step(m, params, x, dy, dtype)
    torch._dynamo.reset()
    rec = Recorder()
    comp = torch.compile(m, backend=rec.backend)
    got, _ = _step(comp, params, x, dy, dtype)
    assert rec.fw and all(ours(op_counts(gm), "qkv_fwd") == 0 for gm in rec.fw)
    keep = [j for j, g in enumerate(want) if g is not None]
    _compare([got[j] for j in keep], [want[j] for j in keep], case)


@pytest.mark.gpu
def test_misaligned_operands_are_copied_inside_the_ops():
    """A column slice whose start is not 16-byte aligned (row stride still a multiple of 8 elements) reaches the producer
    and the tail inside a compiled function: the ops copy it, and the results equal eager calls on contiguous copies."""
    from xlstm_yolo_b200 import ops
    g = torch.Generator().manual_seed(3)
    B, gh, gw, NH, d = 2, 12, 12, 2, 64
    S, D = gh * gw, NH * d
    big = torch.randn(B, S, 2 * D + 8, generator=g).bfloat16().cuda()
    xs = big[..., 1:1 + D]
    assert xs.data_ptr() % 16 and xs.stride(1) % 8 == 0
    cw, cb = torch.randn(D, 1, 3, 3, generator=g).cuda() * 0.3, torch.randn(D, generator=g).cuda() * 0.1
    ws = [(torch.randn(NH, d, d, generator=g) * d ** -0.5).cuda() for _ in range(3)]
    bs = [(torch.randn(D, generator=g) * 0.1).cuda() for _ in range(3)]
    prod = lambda x: ops.qkv_producer(x, cw, cb, ws[0], bs[0], ws[1], bs[1], ws[2], bs[2], gh, gw, True)
    torch._dynamo.reset()
    with torch.no_grad():
        got = torch.compile(prod, backend="aot_eager", fullgraph=True)(xs)
        want = prod(xs.contiguous())
    for a, b in zip(got, want):
        assert torch.equal(a, b)

    NHt, DH = 4, 64
    Dt = NHt * DH
    h = torch.randn(B, S, NHt, DH, generator=g).bfloat16().cuda().transpose(1, 2)
    wide = torch.randn(B, S, 2 * Dt + 8, generator=g).bfloat16().cuda()
    c, z = wide[..., 1:1 + Dt], torch.randn(B, S, Dt, generator=g).bfloat16().cuda()
    w, b, skip = (torch.randn(Dt, generator=g).cuda() * 0.1 for _ in range(3))
    tail = lambda c_: ops.layer_tail(h, c_, z, w, b, skip)
    torch._dynamo.reset()
    with torch.no_grad():
        got = torch.compile(tail, backend="aot_eager", fullgraph=True)(c)
        want = tail(c.contiguous())
    assert torch.equal(got, want)


@pytest.mark.gpu
def test_inference_graph_skips_saved_rows_and_sp():
    """Under no_grad the compiled forward asks the cell for no n_row / m_row and the producer for no sp."""
    pair = _pair(128, 64)
    x, _ = _inputs(2, 400, 128)
    torch._dynamo.reset()
    rec = Recorder()
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        y = torch.compile(pair, backend=rec.backend, fullgraph=True)(x)
        ye = pair(x)
    assert rel(y, ye) < 1e-2
    cells, prods = nodes_of(rec.fw[0], "fused_cell_fwd"), nodes_of(rec.fw[0], "qkv_fwd")
    assert len(cells) == 2 and len(prods) == 2
    assert all(n.args[12] is False for n in cells) and all(n.args[-1] is False for n in prods)   # save_rows, need_sp


@pytest.mark.gpu
def test_dynamic_batch_compiles_once():
    """torch._dynamo.mark_dynamic(x, 0): batch 2 then 3 compile once, and both match eager."""
    from torch._dynamo.testing import CompileCounterWithBackend
    pair = _pair(128, 64)
    params = _trained_params(pair)
    torch._dynamo.reset()
    cnt = CompileCounterWithBackend("aot_eager")
    comp = torch.compile(pair, backend=cnt)
    for B in (2, 3):
        x, dy = _inputs(B, 400, 128, seed=B)
        want, _ = _step(pair, params, x, dy, torch.bfloat16)
        got, _ = _step(comp, params, x, dy, torch.bfloat16, dynamic_batch=True)
        keep = [j for j, g in enumerate(want) if g is not None]
        _compare([got[j] for j in keep], [want[j] for j in keep], f"B={B}")
    assert cnt.frame_count == 1, cnt.frame_count


# ---------------------------------------------------------------------------------------------------------------------
# torch.library.opcheck on every op (default test_utils, test_aot_dispatch_dynamic included)
# ---------------------------------------------------------------------------------------------------------------------
def _fused_cell_args(DH, gate_mode, reverse, bias):
    g = torch.Generator().manual_seed(11)
    B, S, NH = 2, 160, 2
    D = NH * DH
    q3, k3, v3 = ((torch.randn(B, S, D, generator=g) * s).bfloat16().cuda() for s in (DH ** -0.5, DH ** -0.5, 1.0))
    w_i, w_f = ((torch.randn(NH, 3 * D, generator=g) * 0.02).cuda() for _ in range(2))
    b_i = (torch.randn(NH, generator=g)).cuda() if bias else None
    b_f = (torch.linspace(3, 6, NH)).cuda() if bias else None
    from xlstm_yolo_b200 import ops
    return [q3, k3, v3, w_i, b_i, w_f, b_f, NH, 1e-6, 64, reverse, gate_mode, True,
            ops._states_numel(B, NH, S, DH, DH, torch.bfloat16)]


@pytest.mark.gpu
@pytest.mark.parametrize("DH", [64, 128])
@pytest.mark.parametrize("gate_mode", [0, 1])
@pytest.mark.parametrize("reverse", [False, True])
@pytest.mark.parametrize("bias", [True, False])
def test_opcheck_fused_cell(DH, gate_mode, reverse, bias):
    from xlstm_yolo_b200 import ops  # noqa: F401  (registers the ops)
    args = _fused_cell_args(DH, gate_mode, reverse, bias)
    fwd, bwd = torch.ops.xlstm_yolo_b200.fused_cell_fwd, torch.ops.xlstm_yolo_b200.fused_cell_bwd
    h, i3, f3, n_row, m_row, states = fwd(*args)
    dh = torch.randn_like(h.float()).bfloat16()
    q3, k3, v3, w_i, b_i, w_f, b_f, NH, eps, cs, rev, gm, _, _ = args
    torch.library.opcheck(bwd, (q3, k3, v3, w_i, w_f, i3, f3, h, n_row, m_row, states, dh, NH, eps, cs, rev, gm, bias))
    for j in (0, 1, 2, 3, 5) + ((4, 6) if bias else ()):
        args[j] = args[j].clone().requires_grad_(True)
    torch.library.opcheck(fwd, tuple(args))


def _qkv_args(d, x_dtype, rotate, bias):
    g = torch.Generator().manual_seed(12)
    B, gh, gw, NH = 2, 8, 8, 2
    S, D = gh * gw, NH * d
    up = torch.randn(B, S, 2 * D, generator=g).to(x_dtype).cuda()
    x = up[..., :D]
    cw = (torch.randn(D, 1, 3, 3, generator=g) * 0.3).cuda()
    cb = (torch.randn(D, generator=g) * 0.1).cuda() if bias else None
    ws = [(torch.randn(NH, d, d, generator=g) * d ** -0.5).cuda() for _ in range(3)]
    bs = [(torch.randn(D, generator=g) * 0.1).cuda() if bias else None for _ in range(3)]
    return [x, cw, cb, ws[0], bs[0], ws[1], bs[1], ws[2], bs[2], gh, gw, rotate, True]


@pytest.mark.gpu
@pytest.mark.parametrize("d", [64, 128])
@pytest.mark.parametrize("x_dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("rotate", [False, True])
@pytest.mark.parametrize("bias", [True, False])
def test_opcheck_qkv(d, x_dtype, rotate, bias):
    from xlstm_yolo_b200 import ops  # noqa: F401
    args = _qkv_args(d, x_dtype, rotate, bias)
    fwd, bwd = torch.ops.xlstm_yolo_b200.qkv_fwd, torch.ops.xlstm_yolo_b200.qkv_bwd
    c, q, k, v, sp = fwd(*args)
    assert sp.numel() == c.numel()
    g = torch.Generator().manual_seed(13)
    dc, dq, dk, dv = (torch.randn(c.shape, generator=g).bfloat16().cuda() for _ in range(4))
    x, cw, cb, wq, bq, wk, bk, wv, bv, gh, gw, rot, _ = args
    torch.library.opcheck(bwd, (x, c, cw, cb, wq, wk, wv, sp, dc, dq, dk, dv, gh, gw, rot, bias, bias, bias))
    for j in (0, 1, 3, 5, 7) + ((2, 4, 6, 8) if bias else ()):
        args[j] = args[j].detach().requires_grad_(True)
    torch.library.opcheck(fwd, tuple(args))


@pytest.mark.gpu
@pytest.mark.parametrize("params", [True, False])
def test_opcheck_layer_tail(params):
    from xlstm_yolo_b200 import ops
    g = torch.Generator().manual_seed(14)
    B, S, NH, DH = 2, 96, 4, 64
    D = NH * DH
    h = torch.randn(B, S, NH, DH, generator=g).bfloat16().cuda().transpose(1, 2)
    c, z, dy = (torch.randn(B, S, D, generator=g).bfloat16().cuda() for _ in range(3))
    w, b, skip = ((torch.randn(D, generator=g) * 0.1).cuda() if params else None for _ in range(3))
    fwd, bwd = torch.ops.xlstm_yolo_b200.layer_tail_fwd, torch.ops.xlstm_yolo_b200.layer_tail_bwd
    assert ops.glue_supported(h, c, z)
    torch.library.opcheck(bwd, (h, c, z, w, b, skip, dy, 1e-3))
    leaf = lambda t: None if t is None else t.clone().requires_grad_(True)
    torch.library.opcheck(fwd, (leaf(h.transpose(1, 2)).transpose(1, 2), leaf(c), leaf(z), leaf(w), leaf(b), leaf(skip), 1e-3))


@pytest.mark.gpu
def test_mlstm_op_with_dynamic_batch():
    """The bare cell op (xlstm_yolo_b200::mlstm_fwd / ::mlstm_bwd) with B marked dynamic: batch 2 then 3 compile once and
    equal eager."""
    from torch._dynamo.testing import CompileCounterWithBackend
    from xlstm_yolo_b200 import ops
    cnt = CompileCounterWithBackend("aot_eager")
    torch._dynamo.reset()
    fn = lambda q, k, v, i, f: ops.mlstm(q, k, v, i, f)
    comp = torch.compile(fn, backend=cnt)
    for B in (2, 3):
        g = torch.Generator().manual_seed(B)
        NH, S, DH = 2, 200, 64
        q, k, v = (torch.randn(B, S, NH, DH, generator=g).bfloat16().cuda().transpose(1, 2) * s for s in (0.125, 0.125, 1.0))
        i, f = torch.randn(B, NH, S, generator=g).cuda(), (torch.randn(B, NH, S, generator=g) + 4).cuda()
        dh = torch.randn(B, NH, S, DH, generator=g).bfloat16().cuda()
        res = []
        for m in (fn, comp):
            leaves = [t.detach().clone().requires_grad_(True) for t in (q, k, v, i, f)]
            if m is comp:
                for t in leaves:
                    torch._dynamo.mark_dynamic(t, 0)
            h = m(*leaves)
            h.backward(dh)
            res.append([h.detach()] + [t.grad for t in leaves])
        for a, b in zip(*res):
            assert torch.equal(a, b)
    assert cnt.frame_count == 1, cnt.frame_count
