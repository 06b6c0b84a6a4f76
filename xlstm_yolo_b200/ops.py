"""The mLSTM cell operator on CUDA tensors: a ``torch.autograd.Function`` over the C ABI.

Functional mirror of the reference's backend call (SURVEY.md §8b)::

    h[, (C_last, n_last, m_last)] = mlstm(q, k, v, i, f, c_initial=None, n_initial=None,
                                          m_initial=None, return_last_states=False, ...)

with q,k: (B,NH,S,DHqk), v: (B,NH,S,DHv) — typically strided views of (B,S,NH,DH) storage
(vision_lstm2.py:900-902) — and i,f: (B,NH,S).  PyTorch is plumbing only (allocation,
streams, autograd bookkeeping); all arithmetic happens in ``lib/libmlstm_b200.so``.
CUDA tensors only: there is no CPU or PyTorch fallback here.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import Act, ConvBwdParams, Gate, GateProjParams, GlueParams, Params, QkvBwdParams, QkvParams

_DT = {torch.float32: _lib.MLSTM_F32, torch.bfloat16: _lib.MLSTM_BF16}


def _fail(rc: int, what: str):
    raise RuntimeError(f"mlstm_b200 {what} failed: {_lib.STATUS.get(rc, rc)}: {_lib.last_error()}")


def _act_ok(t: torch.Tensor) -> bool:
    if t.stride(-1) != 1 and t.shape[-1] != 1:
        return False
    if t.dtype == torch.bfloat16:  # TMA: 16-byte aligned base and strides
        if t.data_ptr() % 16 or any(s % 8 for s in t.stride()[:-1]):
            return False
    return True


def _prep_act(t: torch.Tensor) -> torch.Tensor:
    """Keep the caller's strided layout when the kernels can read it, else copy into
    (B,S,NH,DH) storage (the reference's native layout)."""
    if _act_ok(t):
        return t
    B, NH, S, D = t.shape
    out = torch.empty((B, S, NH, D), dtype=t.dtype, device=t.device).transpose(1, 2)
    out.copy_(t)
    return out


def _empty_act(B, NH, S, D, dtype, device) -> torch.Tensor:
    return torch.empty((B, S, NH, D), dtype=dtype, device=device).transpose(1, 2)


def _act(t: Optional[torch.Tensor]) -> Act:
    if t is None:
        return Act(None, 0, 0, 0)
    return Act(t.data_ptr(), t.stride(0), t.stride(1), t.stride(2))


def _gate(t: Optional[torch.Tensor]) -> Gate:
    if t is None:
        return Gate(None, 0, 0, 0)
    return Gate(t.data_ptr(), t.stride(0), t.stride(1), t.stride(2))


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _base_params(q, k, v, i, f, eps, chunk_size, reverse, qk_scale, gate_mode=0) -> Params:
    B, NH, S, DK = q.shape
    p = Params()
    p.abi_version = _lib.ABI_VERSION
    p.B, p.NH, p.S, p.DHQK, p.DHV = B, NH, S, DK, v.shape[-1]
    p.dtype = _DT[q.dtype]
    p.reverse = 1 if reverse else 0
    p.chunk_size = int(chunk_size)
    p.eps = float(eps)
    p.qk_scale = float(qk_scale or 0.0)
    p.gate_mode = int(gate_mode)
    p.q, p.k, p.v = _act(q), _act(k), _act(v)
    p.i, p.f = _gate(i), _gate(f)
    return p


def gate_mode_of(input_gate) -> int:
    if input_gate in (0, "exp", "exponential", None):
        return 0
    if input_gate in (1, "sigmoid", "siging"):
        return 1
    raise ValueError(f"input_gate must be 'exp' or 'sigmoid', got {input_gate!r}")


def kernel_family(q: torch.Tensor, v: torch.Tensor) -> str:
    """'tcgen05' or 'simt' — which kernel family the library would pick for these shapes."""
    p = Params()
    p.abi_version = _lib.ABI_VERSION
    p.B, p.NH, p.S, p.DHQK, p.DHV = q.shape[0], q.shape[1], q.shape[2], q.shape[3], v.shape[3]
    p.dtype = _DT[q.dtype]
    name = _lib.load().mlstm_b200_kernel_name(C.byref(p), 0)
    return name.decode() if name else "none"


def _alloc_states(lib, p, dev, nbytes=None):
    """Per-chunk entry-state buffer of the tcgen05 family (None for SIMT); attaches it to p.  ``nbytes``: a size the caller
    chose (the custom ops, ``_states_numel``), zero-filled so that the bytes the kernels leave unwritten (alignment padding)
    do not differ from call to call; the library checks that it suffices."""
    if nbytes is None:
        with torch.cuda.device(dev):   # size and variant queries see the device the launch will see
            need = lib.mlstm_b200_state_bytes(C.byref(p))
    else:
        need = nbytes
    if not need:
        return None
    states = (torch.empty if nbytes is None else torch.zeros)(need, dtype=torch.uint8, device=dev)
    p.states, p.states_bytes = states.data_ptr(), need
    return states


def mlstm_fwd_raw(q, k, v, i, f, c_initial=None, n_initial=None, m_initial=None, *, eps=1e-6, chunk_size=64,
                  reverse=False, save_rows=True, return_last_states=False, qk_scale=None, gate_mode=0, states_bytes=None):
    """One forward launch through the C ABI.  Inputs must already be CUDA, fp32 or bf16
    (q,k,v same dtype), gates fp32.  Returns (h, n_row, m_row, last_states_or_None, chunk_states)."""
    lib = _lib.load()
    B, NH, S, DK = q.shape
    DV = v.shape[-1]
    dev = q.device
    h = _empty_act(B, NH, S, DV, q.dtype, dev)
    n_row = m_row = None
    if save_rows:
        n_row = torch.empty((B, NH, S), dtype=torch.float32, device=dev)
        m_row = torch.empty((B, NH, S), dtype=torch.float32, device=dev)
    last = None
    if return_last_states:
        last = (torch.empty((B, NH, DK, DV), dtype=torch.float32, device=dev),
                torch.empty((B, NH, DK), dtype=torch.float32, device=dev),
                torch.empty((B, NH, 1), dtype=torch.float32, device=dev))
    p = _base_params(q, k, v, i, f, eps, chunk_size, reverse, qk_scale, gate_mode)
    p.c_initial, p.n_initial, p.m_initial = _ptr(c_initial), _ptr(n_initial), _ptr(m_initial)
    p.h = _act(h)
    p.n_row, p.m_row = _ptr(n_row), _ptr(m_row)
    if last is not None:
        p.c_last, p.n_last, p.m_last = (_ptr(t) for t in last)
    states = _alloc_states(lib, p, dev, states_bytes)
    with torch.cuda.device(dev):
        rc = lib.mlstm_b200_fwd(C.byref(p), _stream())
    if rc:
        _fail(rc, "forward")
    return h, n_row, m_row, last, states


def mlstm_bwd_raw(q, k, v, i, f, h, n_row, m_row, dh, c_initial=None, n_initial=None, m_initial=None, *, eps=1e-6,
                  chunk_size=64, reverse=False, qk_scale=None, states=None, gate_mode=0):
    """One backward call through the C ABI.  Returns (dq, dk, dv, di, df) — dq,dk,dv in the
    layout/dtype of q,k,v; di,df fp32 (B,NH,S)."""
    lib = _lib.load()
    B, NH, S, DK = q.shape
    DV = v.shape[-1]
    dev = q.device
    dq = _empty_act(B, NH, S, DK, q.dtype, dev)
    dk = _empty_act(B, NH, S, DK, q.dtype, dev)
    dv = _empty_act(B, NH, S, DV, q.dtype, dev)
    di = torch.empty((B, S, NH), dtype=torch.float32, device=dev).transpose(1, 2)
    df = torch.empty((B, S, NH), dtype=torch.float32, device=dev).transpose(1, 2)
    p = _base_params(q, k, v, i, f, eps, chunk_size, reverse, qk_scale, gate_mode)
    p.c_initial, p.n_initial, p.m_initial = _ptr(c_initial), _ptr(n_initial), _ptr(m_initial)
    p.h = _act(h)
    p.n_row, p.m_row = _ptr(n_row), _ptr(m_row)
    p.dh = _act(dh)
    p.dq, p.dk, p.dv = _act(dq), _act(dk), _act(dv)
    p.di, p.df = _gate(di), _gate(df)
    if states is not None:
        p.states, p.states_bytes = states.data_ptr(), states.numel()
    with torch.cuda.device(dev):
        need = lib.mlstm_b200_workspace_bytes(C.byref(p), 1)
        ws = None
        if need:
            ws = torch.empty((need + 3) // 4, dtype=torch.float32, device=dev)
            p.workspace, p.workspace_bytes = ws.data_ptr(), ws.numel() * 4
        rc = lib.mlstm_b200_bwd(C.byref(p), _stream())
    if rc:
        _fail(rc, "backward")
    return dq, dk, dv, di, df


class _MLSTMCellFn(torch.autograd.Function):
    """autograd wrapper: saves q,k,v,i,f,h and the per-row (n, m); gates/decay matrices are
    recomputed per chunk in the backward kernels."""

    @staticmethod
    def forward(ctx, q, k, v, i, f, c_initial, n_initial, m_initial, eps, chunk_size, reverse, return_last_states,
                gate_mode=0):
        need_grad = any(t.requires_grad for t in (q, k, v, i, f))
        h, n_row, m_row, last, states = mlstm_fwd_raw(
            q, k, v, i, f, c_initial, n_initial, m_initial, eps=eps, chunk_size=chunk_size, reverse=reverse,
            save_rows=need_grad, return_last_states=return_last_states, gate_mode=gate_mode)
        if need_grad:
            ctx.save_for_backward(q, k, v, i, f, h, n_row, m_row, c_initial, n_initial, m_initial, states)
        ctx.cfg = (eps, chunk_size, reverse, gate_mode)
        if return_last_states:
            ctx.mark_non_differentiable(*last)
            return (h,) + tuple(last)
        return h

    @staticmethod
    def backward(ctx, dh, *dstates):
        q, k, v, i, f, h, n_row, m_row, c0, n0, m0, states = ctx.saved_tensors
        eps, chunk_size, reverse, gate_mode = ctx.cfg
        if dh.dtype != q.dtype:
            dh = dh.to(q.dtype)  # e.g. loss-scaled fp16 -> bf16: no clamping, inf/NaN propagate
        dh = _prep_act(dh)
        dq, dk, dv, di, df = mlstm_bwd_raw(q, k, v, i, f, h, n_row, m_row, dh, c0, n0, m0, eps=eps,
                                           chunk_size=chunk_size, reverse=reverse, states=states, gate_mode=gate_mode)
        return dq, dk, dv, di, df, None, None, None, None, None, None, None, None


# ---------------------------------------------------------------------------------------------
# torch.library registration: the same two C-ABI calls as ``xlstm_yolo_b200::mlstm_fwd`` / ``::mlstm_bwd`` custom ops with
# fake (shape-only) implementations and an autograd formula, so Dynamo / AOT autograd can trace a model that contains the
# cell (the reference compiles its model in debug.py:13).  ``mlstm`` takes this route while torch.compile is tracing and
# the plain autograd.Function otherwise (same kernels, less dispatch overhead per call in eager mode).
# ---------------------------------------------------------------------------------------------
def _states_numel(B, NH, S, DK, DV, dtype):
    """Bytes of the chunk-state buffer the custom ops allocate and their fakes declare: B times what one batch row needs
    with a backward following.  That bounds the library's need at every batch size, variant and forward-only call
    (tests/test_gpu_compile.py), and stays a plain function of a symbolic batch, so a dynamic batch traces into one graph
    (the other sizes specialise)."""
    return B * _state_bytes(1, int(NH), int(S), int(DK), int(DV), dtype, True)


@torch.compiler.assume_constant_result
def _state_bytes(B: int, NH: int, S: int, DK: int, DV: int, dtype: torch.dtype, save_rows: bool) -> int:
    """``mlstm_b200_state_bytes`` for these shapes (a host-side query: no device pointers involved)."""
    p = Params()
    p.abi_version = _lib.ABI_VERSION
    p.B, p.NH, p.S, p.DHQK, p.DHV = B, NH, S, DK, DV
    p.dtype = _DT[dtype]
    if save_rows:
        p.n_row = p.m_row = 0x1000      # "a backward will follow" (only tested for NULL by the query)
    return int(_lib.load().mlstm_b200_state_bytes(C.byref(p)))


@torch.library.custom_op("xlstm_yolo_b200::mlstm_fwd", mutates_args=(), device_types="cuda")
def _mlstm_fwd_op(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, i: torch.Tensor, f: torch.Tensor,
                  c_initial: Optional[torch.Tensor], n_initial: Optional[torch.Tensor], m_initial: Optional[torch.Tensor],
                  eps: float, chunk_size: int, reverse: bool, save_rows: bool, return_last_states: bool,
                  gate_mode: int, states_bytes: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    q, k, v = _prep_act(q), _prep_act(k), _prep_act(v)
    h, n_row, m_row, last, states = mlstm_fwd_raw(q, k, v, i, f, c_initial, n_initial, m_initial, eps=eps, chunk_size=chunk_size,
                                                  reverse=reverse, save_rows=save_rows, return_last_states=return_last_states,
                                                  gate_mode=gate_mode, states_bytes=states_bytes)
    e = lambda dt=torch.float32: torch.empty(0, dtype=dt, device=q.device)
    c_l, n_l, m_l = last if last is not None else (e(), e(), e())
    return (h, n_row if n_row is not None else e(), m_row if m_row is not None else e(),
            states if states is not None else e(torch.uint8), c_l, n_l, m_l)


@_mlstm_fwd_op.register_fake
def _(q, k, v, i, f, c_initial, n_initial, m_initial, eps, chunk_size, reverse, save_rows, return_last_states, gate_mode,
      states_bytes):
    B, NH, S, DK = q.shape
    DV = v.shape[-1]
    dev = q.device
    e = lambda dt=torch.float32: torch.empty(0, dtype=dt, device=dev)
    h = torch.empty((B, S, NH, DV), dtype=q.dtype, device=dev).transpose(1, 2)
    rows = (lambda: torch.empty((B, NH, S), dtype=torch.float32, device=dev)) if save_rows else e
    states = torch.empty(states_bytes, dtype=torch.uint8, device=dev)
    if return_last_states:
        last = (torch.empty((B, NH, DK, DV), dtype=torch.float32, device=dev), torch.empty((B, NH, DK), dtype=torch.float32, device=dev),
                torch.empty((B, NH, 1), dtype=torch.float32, device=dev))
    else:
        last = (e(), e(), e())
    return (h, rows(), rows(), states) + last


@torch.library.custom_op("xlstm_yolo_b200::mlstm_bwd", mutates_args=(), device_types="cuda")
def _mlstm_bwd_op(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, i: torch.Tensor, f: torch.Tensor, h: torch.Tensor,
                  n_row: torch.Tensor, m_row: torch.Tensor, dh: torch.Tensor, c_initial: Optional[torch.Tensor],
                  n_initial: Optional[torch.Tensor], m_initial: Optional[torch.Tensor], states: torch.Tensor, eps: float,
                  chunk_size: int, reverse: bool,
                  gate_mode: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    q, k, v = _prep_act(q), _prep_act(k), _prep_act(v)
    if dh.dtype != q.dtype:
        dh = dh.to(q.dtype)
    return mlstm_bwd_raw(q, k, v, i, f, h, n_row, m_row, _prep_act(dh), c_initial, n_initial, m_initial, eps=eps,
                         chunk_size=chunk_size, reverse=reverse, states=states if states.numel() else None, gate_mode=gate_mode)


@_mlstm_bwd_op.register_fake
def _(q, k, v, i, f, h, n_row, m_row, dh, c_initial, n_initial, m_initial, states, eps, chunk_size, reverse, gate_mode):
    B, NH, S, DK = q.shape
    DV = v.shape[-1]
    act = lambda D: torch.empty((B, S, NH, D), dtype=q.dtype, device=q.device).transpose(1, 2)
    gate = lambda: torch.empty((B, S, NH), dtype=torch.float32, device=q.device).transpose(1, 2)
    return act(DK), act(DK), act(DV), gate(), gate()


def _op_setup_context(ctx, inputs, output):
    q, k, v, i, f, c0, n0, m0, eps, chunk_size, reverse, save_rows, return_last_states, gate_mode, states_bytes = inputs
    h, n_row, m_row, states = output[:4]
    ctx.save_for_backward(q, k, v, i, f, h, n_row, m_row, c0, n0, m0, states)
    ctx.cfg = (eps, chunk_size, reverse, gate_mode)
    ctx.set_materialize_grads(False)


def _op_backward(ctx, dh, *_unused):
    q, k, v, i, f, h, n_row, m_row, c0, n0, m0, states = ctx.saved_tensors
    eps, chunk_size, reverse, gate_mode = ctx.cfg
    if dh is None:
        dh = torch.zeros_like(h)
    dq, dk, dv, di, df = _mlstm_bwd_op(q, k, v, i, f, h, n_row, m_row, dh, c0, n0, m0, states, eps, chunk_size, reverse, gate_mode)
    return dq, dk, dv, di, df, None, None, None, None, None, None, None, None, None, None


_mlstm_fwd_op.register_autograd(_op_backward, setup_context=_op_setup_context)


def _mlstm_traced(q, k, v, i, f, c0, n0, m0, eps, chunk_size, reverse, return_last_states, gate_mode):
    need_grad = torch.is_grad_enabled() and any(t.requires_grad for t in (q, k, v, i, f))
    B, NH, S, DK = q.shape
    nbytes = _states_numel(B, NH, S, DK, v.shape[-1], q.dtype)
    h, _n, _m, _s, c_l, n_l, m_l = _mlstm_fwd_op(q, k, v, i, f, c0, n0, m0, eps, chunk_size, reverse, need_grad,
                                                  return_last_states, gate_mode, nbytes)
    return (h, c_l, n_l, m_l) if return_last_states else h


def mlstm(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, i: torch.Tensor, f: torch.Tensor,
          c_initial: Optional[torch.Tensor] = None, n_initial: Optional[torch.Tensor] = None,
          m_initial: Optional[torch.Tensor] = None, return_last_states: bool = False, *, eps: float = 1e-6,
          chunk_size: int = 64, reverse: bool = False, kernel_dtype: Optional[torch.dtype] = None,
          input_gate: str = "exp"):
    """mLSTM cell on CUDA tensors.

    ``kernel_dtype``: torch.bfloat16 -> tcgen05 kernels (bf16 operands, fp32 accumulation);
    torch.float32 -> fp32 SIMT kernels.  Default: bf16 for bf16/fp16 inputs, fp32 for fp32
    inputs.  The result has the dtype of ``q``.  Initial/last states are fp32 and carry no
    gradient (the reference never differentiates through them).  ``input_gate``: "exp" (exponential input
    gate with max-stabiliser, backends.py:149-263) or "sigmoid" (the "siging" kernels HEAD names on CUDA,
    vision_lstm2.py:835: log-gate logsigmoid(i), no stabiliser, normaliser max(|n|, 1)).
    """
    if not q.is_cuda:
        raise RuntimeError("xlstm_yolo_b200.ops.mlstm needs CUDA tensors (no CPU fallback)")
    in_dtype = q.dtype
    if kernel_dtype is None:
        kernel_dtype = torch.float32 if in_dtype == torch.float32 else torch.bfloat16
    if kernel_dtype not in _DT:
        raise ValueError(f"kernel_dtype must be float32 or bfloat16, got {kernel_dtype}")
    tracing = torch.compiler.is_compiling()
    q, k, v = ((t.to(kernel_dtype) if tracing else _prep_act(t.to(kernel_dtype))) for t in (q, k, v))
    i, f = i.to(torch.float32), f.to(torch.float32)
    c0 = None if c_initial is None else c_initial.detach().to(torch.float32).contiguous()
    n0 = None if n_initial is None else n_initial.detach().to(torch.float32).contiguous()
    m0 = None if m_initial is None else m_initial.detach().to(torch.float32).reshape(q.shape[0], q.shape[1]).contiguous()
    if tracing:   # torch.compile: the registered custom op (layout fix-ups happen inside it)
        out = _mlstm_traced(q, k, v, i, f, c0, n0, m0, float(eps), int(chunk_size), bool(reverse), bool(return_last_states),
                            gate_mode_of(input_gate))
    else:
        out = _MLSTMCellFn.apply(q, k, v, i, f, c0, n0, m0, float(eps), int(chunk_size), bool(reverse),
                                 bool(return_last_states), gate_mode_of(input_gate))
    if return_last_states:
        h, C, n, m = out
        return h.to(in_dtype), (C, n, m)
    return out.to(in_dtype)


# ---------------------------------------------------------------------------------------------
# Fused cell: gate projection + mLSTM as one autograd node (vision_lstm2.py:895-948)
# ---------------------------------------------------------------------------------------------
def _gate_params(q3, k3, v3, w_i, b_i, w_f, b_f, NH) -> GateProjParams:
    B, S, D = q3.shape
    g = GateProjParams()
    g.abi_version = _lib.ABI_VERSION
    g.T, g.D, g.NH = B * S, D, NH
    g.dtype = _DT[q3.dtype]
    g.ld = q3.stride(1)
    g.q, g.k, g.v = q3.data_ptr(), k3.data_ptr(), v3.data_ptr()
    g.w_i, g.w_f = w_i.data_ptr(), w_f.data_ptr()
    g.b_i, g.b_f = _ptr(b_i), _ptr(b_f)
    return g


def _rows_layout_ok(t: torch.Tensor) -> bool:
    """(B,S,D) tensor whose B*S rows are evenly strided (what the gate, tail and producer kernels stream over)."""
    B, S, D = t.shape
    return t.stride(2) == 1 and t.stride(0) == S * t.stride(1) and t.stride(1) % 8 == 0 and D % 8 == 0


def _rows_ok(t: torch.Tensor) -> bool:
    """``_rows_layout_ok`` with a 16-byte aligned base."""
    return _rows_layout_ok(t) and t.data_ptr() % 16 == 0


def _aligned(t: torch.Tensor) -> bool:
    """16-byte aligned base.  A traced tensor has no address: the custom op it reaches copies a misaligned input."""
    return torch.compiler.is_compiling() or t.data_ptr() % 16 == 0


@torch.compiler.assume_constant_result
def gates_supported(D: int, ld: Optional[int] = None) -> bool:
    """Whether csrc/mlstm_gates.cu takes a cell of inner dim D (asks the library: the 8 x 3D fp32 weight tile
    must fit in shared memory, i.e. D <= 2133)."""
    return bool(_lib.load().mlstm_b200_gates_supported(int(D), int(D if ld is None else ld)))


def gate_proj_fwd_raw(q3, k3, v3, w_i, b_i, w_f, b_f, NH):
    """i, f pre-activations (B,S,NH) fp32 from q,k,v (B,S,D) without the cat copy."""
    lib = _lib.load()
    B, S, D = q3.shape
    i = torch.empty((B, S, NH), dtype=torch.float32, device=q3.device)
    f = torch.empty((B, S, NH), dtype=torch.float32, device=q3.device)
    g = _gate_params(q3, k3, v3, w_i, b_i, w_f, b_f, NH)
    g.i, g.f = i.data_ptr(), f.data_ptr()
    need = lib.mlstm_b200_gates_fwd_workspace_bytes(C.byref(g))
    if need:
        ws = torch.empty((need + 15) // 16 * 4, dtype=torch.float32, device=q3.device)
        g.workspace, g.workspace_bytes = ws.data_ptr(), ws.numel() * 4
    with torch.cuda.device(q3.device):
        rc = lib.mlstm_b200_gates_fwd(C.byref(g), _stream())
    if rc:
        _fail(rc, "gate projection forward")
    return i, f


def gate_proj_bwd_raw(q3, k3, v3, w_i, w_f, NH, di, df, dq3, dk3, dv3, need_bias=True):
    """In place: dq3,dk3,dv3 += di W_i + df W_f ; returns (dw_i, db_i, dw_f, db_f)."""
    lib = _lib.load()
    dev = q3.device
    g = _gate_params(q3, k3, v3, w_i, None, w_f, None, NH)
    dw_i, dw_f = torch.empty_like(w_i), torch.empty_like(w_f)
    db_i = torch.empty(NH, dtype=torch.float32, device=dev) if need_bias else None
    db_f = torch.empty(NH, dtype=torch.float32, device=dev) if need_bias else None
    g.di, g.df = di.data_ptr(), df.data_ptr()
    g.dq, g.dk, g.dv = dq3.data_ptr(), dk3.data_ptr(), dv3.data_ptr()
    if not (dq3.stride() == dk3.stride() == dv3.stride()) or dq3.stride(2) != 1 or dq3.stride(0) != dq3.shape[1] * dq3.stride(1):
        raise ValueError("dq3, dk3, dv3 must share one evenly strided (B,S,D) row layout")
    g.ld_d = dq3.stride(1)   # the cell's gradients are dense even when q,k,v are column slices (ld != ld_d)
    g.dw_i, g.dw_f, g.db_i, g.db_f = dw_i.data_ptr(), dw_f.data_ptr(), _ptr(db_i), _ptr(db_f)
    need = lib.mlstm_b200_gates_workspace_bytes(C.byref(g))
    ws = torch.empty(max(1, (need + 3) // 4), dtype=torch.float32, device=dev)
    g.workspace, g.workspace_bytes = ws.data_ptr(), ws.numel() * 4
    with torch.cuda.device(dev):
        rc = lib.mlstm_b200_gates_bwd(C.byref(g), _stream())
    if rc:
        _fail(rc, "gate projection backward")
    return dw_i, db_i, dw_f, db_f


def _cell_rows(q3, k3, v3, rows_ok=None):
    """q, k, v as the gate kernels stream them: evenly strided rows sharing one row stride, else dense copies of all three.
    ``rows_ok`` decides which layouts pass (default ``_rows_ok``; while tracing, the layout half of it)."""
    rows_ok = rows_ok or _rows_ok
    q3, k3, v3 = (t if rows_ok(t) else t.contiguous() for t in (q3, k3, v3))
    if q3.stride(1) != k3.stride(1) or q3.stride(1) != v3.stride(1):
        q3, k3, v3 = q3.contiguous(), k3.contiguous(), v3.contiguous()
    return q3, k3, v3


def fused_cell_fwd_raw(q3, k3, v3, w_i, b_i, w_f, b_f, NH, eps, chunk_size, reverse, gate_mode, save_rows, states_bytes=None):
    """Gate projection + cell forward launches.  q,k,v (B,S,D) as ``_cell_rows`` leaves them, gate weights fp32.
    Returns (h, i3, f3, n_row, m_row, states): h (B,NH,S,DH) view of (B,S,NH,DH) storage, i3, f3 (B,S,NH) fp32;
    n_row, m_row None unless ``save_rows``; states None for the SIMT family."""
    B, S, D = q3.shape
    i3, f3 = gate_proj_fwd_raw(q3, k3, v3, w_i, b_i, w_f, b_f, NH)
    heads = lambda t: t.view(B, S, NH, D // NH).transpose(1, 2)
    h, n_row, m_row, _, states = mlstm_fwd_raw(heads(q3), heads(k3), heads(v3), i3.transpose(1, 2), f3.transpose(1, 2),
                                               eps=eps, chunk_size=chunk_size, reverse=reverse, save_rows=save_rows,
                                               gate_mode=gate_mode, states_bytes=states_bytes)
    return h, i3, f3, n_row, m_row, states


def fused_cell_bwd_raw(q3, k3, v3, w_i, w_f, i3, f3, h, n_row, m_row, states, dh, NH, eps, chunk_size, reverse, gate_mode,
                       has_bias):
    """Cell backward, then one streaming pass that adds the gate path into dq,dk,dv in place and reduces dW, db.
    Returns (dq3, dk3, dv3, dw_i, db_i, dw_f, db_f): dq3.. dense (B,S,D), db_* None unless ``has_bias``."""
    B, S, D = q3.shape
    heads = lambda t: t.view(B, S, NH, D // NH).transpose(1, 2)
    if dh.dtype != q3.dtype:
        dh = dh.to(q3.dtype)
    dh = _prep_act(dh)
    dq, dk, dv, di, df = mlstm_bwd_raw(heads(q3), heads(k3), heads(v3), i3.transpose(1, 2), f3.transpose(1, 2), h,
                                       n_row, m_row, dh, eps=eps, chunk_size=chunk_size, reverse=reverse,
                                       states=states, gate_mode=gate_mode)
    # dq,dk,dv are (B,NH,S,DH) views of fresh (B,S,NH,DH) storage; di,df views of (B,S,NH) storage
    dq3, dk3, dv3 = (t.transpose(1, 2).reshape(B, S, D) for t in (dq, dk, dv))
    dw_i, db_i, dw_f, db_f = gate_proj_bwd_raw(q3, k3, v3, w_i, w_f, NH, di.transpose(1, 2), df.transpose(1, 2),
                                               dq3, dk3, dv3, need_bias=has_bias)
    return dq3, dk3, dv3, dw_i, db_i, dw_f, db_f


class _FusedCellFn(torch.autograd.Function):
    """q,k,v (B,S,D) + gate weights -> h (B,NH,S,DH view of (B,S,NH,DH) storage).  The backward runs
    the cell's kernels, then one streaming pass that adds the gate path into dq,dk,dv in place and
    reduces dW, db — nothing of size (B,S,3D) is ever materialised."""

    @staticmethod
    def forward(ctx, q3, k3, v3, w_i, b_i, w_f, b_f, NH, eps, chunk_size, reverse, gate_mode=0):
        need_grad = any(t is not None and t.requires_grad for t in (q3, k3, v3, w_i, b_i, w_f, b_f))
        h, i3, f3, n_row, m_row, states = fused_cell_fwd_raw(q3, k3, v3, w_i, b_i, w_f, b_f, NH, eps, chunk_size, reverse,
                                                             gate_mode, need_grad)
        if need_grad:
            ctx.save_for_backward(q3, k3, v3, w_i, w_f, i3, f3, h, n_row, m_row, states)
        ctx.cfg = (NH, eps, chunk_size, reverse, gate_mode, b_i is not None)
        return h

    @staticmethod
    def backward(ctx, dh):
        grads = fused_cell_bwd_raw(*ctx.saved_tensors, dh, *ctx.cfg)
        return grads + (None,) * 5


def fused_cell(q3: torch.Tensor, k3: torch.Tensor, v3: torch.Tensor, w_i: torch.Tensor, b_i: Optional[torch.Tensor],
               w_f: torch.Tensor, b_f: Optional[torch.Tensor], num_heads: int, *, eps: float = 1e-6,
               chunk_size: int = 64, reverse: bool = False, kernel_dtype: Optional[torch.dtype] = None,
               input_gate: str = "exp"):
    """``MatrixLSTMCell`` arithmetic up to (not including) the out-norm, on CUDA tensors:
    q,k,v (B,S,D) -> h (B,NH,S,DH).  Gate weights are used in fp32 whatever the autocast state."""
    if not q3.is_cuda:
        raise RuntimeError("xlstm_yolo_b200.ops.fused_cell needs CUDA tensors (no CPU fallback)")
    in_dtype = q3.dtype
    if kernel_dtype is None:
        kernel_dtype = torch.float32 if in_dtype == torch.float32 else torch.bfloat16
    if kernel_dtype not in _DT:
        raise ValueError(f"kernel_dtype must be float32 or bfloat16, got {kernel_dtype}")
    traced = _use_custom_ops()
    # (a traced call cannot see addresses: the op copies a misaligned operand)
    q3, k3, v3 = _cell_rows(*(t.to(kernel_dtype) for t in (q3, k3, v3)), rows_ok=_rows_layout_ok if traced else None)
    f32 = lambda t: None if t is None else t.to(torch.float32).contiguous()
    args = (q3, k3, v3, f32(w_i), f32(b_i), f32(w_f), f32(b_f), int(num_heads), float(eps), int(chunk_size), bool(reverse),
            gate_mode_of(input_gate))
    if traced:
        save_rows = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in args[:7])
        B, S, D = q3.shape
        nbytes = _states_numel(B, num_heads, S, D // num_heads, D // num_heads, kernel_dtype)
        h = _fused_cell_fwd_op(*args, save_rows, nbytes)[0]
    else:
        h = _FusedCellFn.apply(*args)
    return h.to(in_dtype)


# ---------------------------------------------------------------------------------------------
# Fused layer tail: out-norm + learnable skip + SiLU(z) gate (vision_lstm2.py:950, :498-499)
# ---------------------------------------------------------------------------------------------
def glue_supported(h: torch.Tensor, c: torch.Tensor, z: torch.Tensor) -> bool:
    """h (B,NH,S,DH) head-strided view of (B,S,NH,DH) storage; c, z (B,S,D) with evenly strided rows."""
    if not h.is_cuda or h.dtype not in _DT or h.dim() != 4:
        return False
    B, NH, S, DH = h.shape
    D = NH * DH
    if not _glue_lib_ok(int(D), int(NH)):   # the C-side shape gate (D % 256 == 0, D <= 2048, DH | 256)
        return False
    if h.stride() != (S * D, DH, D, 1) or not _aligned(h):
        return False
    return all(t.dtype == h.dtype and t.shape == (B, S, D) and _rows_layout_ok(t) and _aligned(t) for t in (c, z))


@torch.compiler.assume_constant_result
def _glue_lib_ok(D: int, NH: int) -> bool:
    return bool(_lib.load().mlstm_b200_glue_supported(int(D), int(NH)))


def _glue_params(h, c, z, w, b, skip, eps) -> GlueParams:
    B, NH, S, DH = h.shape
    g = GlueParams()
    g.abi_version = _lib.ABI_VERSION
    g.T, g.D, g.NH = B * S, NH * DH, NH
    g.dtype = _DT[h.dtype]
    g.eps = float(eps)
    g.h, g.ld_h = h.data_ptr(), NH * DH
    g.c, g.ld_c = c.data_ptr(), c.stride(1)
    g.z, g.ld_z = z.data_ptr(), z.stride(1)
    g.w, g.b, g.skip = _ptr(w), _ptr(b), _ptr(skip)
    return g


def layer_tail_fwd_raw(h, c, z, w, b, skip, eps):
    """One tail forward launch on operands ``glue_supported`` accepts: y (B,S,D) in h's dtype."""
    lib = _lib.load()
    B, NH, S, DH = h.shape
    y = torch.empty((B, S, NH * DH), dtype=h.dtype, device=h.device)
    g = _glue_params(h, c, z, w, b, skip, eps)
    g.y, g.ld_y = y.data_ptr(), NH * DH
    with torch.cuda.device(h.device):
        rc = lib.mlstm_b200_glue_fwd(C.byref(g), _stream())
    if rc:
        _fail(rc, "layer tail forward")
    return y


def layer_tail_bwd_raw(h, c, z, w, b, skip, dy, eps):
    """One tail backward launch: (dh, dc, dz, dw, db, dskip); dh in h's layout, dc, dz dense, dw, db, dskip fp32 (D)
    or None where the forward had no such parameter."""
    lib = _lib.load()
    B, NH, S, DH = h.shape
    D = NH * DH
    dev = h.device
    if dy.dtype != h.dtype:
        dy = dy.to(h.dtype)
    if not _rows_ok(dy):
        dy = dy.contiguous()
    dh = _empty_act(B, NH, S, DH, h.dtype, dev)
    dc = torch.empty((B, S, D), dtype=h.dtype, device=dev)
    dz = torch.empty((B, S, D), dtype=h.dtype, device=dev)
    dw = torch.empty(D, dtype=torch.float32, device=dev) if w is not None else None
    db = torch.empty(D, dtype=torch.float32, device=dev) if b is not None else None
    dskip = torch.empty(D, dtype=torch.float32, device=dev) if skip is not None else None
    g = _glue_params(h, c, z, w, b, skip, eps)
    g.dy, g.ld_dy = dy.data_ptr(), dy.stride(1)
    g.dh, g.ld_dh = dh.data_ptr(), D
    g.dc, g.ld_dc = dc.data_ptr(), D
    g.dz, g.ld_dz = dz.data_ptr(), D
    g.dw, g.db, g.dskip = _ptr(dw), _ptr(db), _ptr(dskip)
    need = lib.mlstm_b200_glue_workspace_bytes(C.byref(g))
    ws = torch.empty(max(1, (need + 3) // 4), dtype=torch.float32, device=dev)
    g.workspace, g.workspace_bytes = ws.data_ptr(), ws.numel() * 4
    with torch.cuda.device(dev):
        rc = lib.mlstm_b200_glue_bwd(C.byref(g), _stream())
    if rc:
        _fail(rc, "layer tail backward")
    return dh, dc, dz, dw, db, dskip


class _GlueFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, h, c, z, w, b, skip, eps):
        ctx.save_for_backward(h, c, z, w, b, skip)
        ctx.eps = eps
        return layer_tail_fwd_raw(h, c, z, w, b, skip, eps)

    @staticmethod
    def backward(ctx, dy):
        return layer_tail_bwd_raw(*ctx.saved_tensors, dy, ctx.eps) + (None,)


def layer_tail(h: torch.Tensor, conv_act: torch.Tensor, z: torch.Tensor, norm_weight: Optional[torch.Tensor],
               norm_bias: Optional[torch.Tensor], skip: Optional[torch.Tensor], eps: float = 1e-3) -> torch.Tensor:
    """``(LN_head(h) * (1 + w) + b + skip * conv_act) * silu(z)`` -> (B,S,D).  ``h`` is the raw cell output
    (B,NH,S,DH); check ``glue_supported`` first."""
    f32 = lambda t: None if t is None else t.to(torch.float32).contiguous()
    args = (h, conv_act, z, f32(norm_weight), f32(norm_bias), f32(skip), float(eps))
    if _use_custom_ops():
        return _layer_tail_fwd_op(*args)
    return _GlueFn.apply(*args)


# ---------------------------------------------------------------------------------------------------------------
# Producer of the cell's operands: conv + SiLU + block-diagonal q / k / v (csrc/mlstm_qkv.cu; SURVEY.md 8 row f2)
# ---------------------------------------------------------------------------------------------------------------

def qkv_supported(x: torch.Tensor, D: int, NH: int, gh: int, gw: int) -> bool:
    """x: (B,S,D) rows of proj_up's output (a column slice is fine), bf16 or fp16 on CUDA."""
    if not x.is_cuda or x.dtype not in (torch.bfloat16, torch.float16) or x.dim() != 3 or x.shape[1] != gh * gw:
        return False
    if x.stride(2) != 1 or x.stride(0) != x.shape[1] * x.stride(1) or not _aligned(x):
        return False
    return _qkv_lib_ok(int(D), int(NH), int(gh), int(gw), int(x.stride(1)))


@torch.compiler.assume_constant_result
def _qkv_lib_ok(D: int, NH: int, gh: int, gw: int, ld: int) -> bool:
    return bool(_lib.load().mlstm_b200_qkv_supported(D, NH, gh, gw, ld))


def qkv_reference(x, conv_w, conv_b, wq, bq, wk, bk, wv, bv, gh, gw, rotate=False):
    """The four reference ops in plain PyTorch (any device / dtype): returns (c, q, k, v), each (B,S,D).
    conv_w (D,1,3,3); w* (NH,d,d) [out][in]; ``rotate`` convolves with the kernel rotated by 180 degrees."""
    B, S, D = x.shape
    NH, d = wq.shape[0], wq.shape[1]
    w = conv_w.flip(-1, -2) if rotate else conv_w
    img = x.reshape(B, gh, gw, D).permute(0, 3, 1, 2)
    u = torch.nn.functional.conv2d(img, w.to(x.dtype), None if conv_b is None else conv_b.to(x.dtype), padding=1, groups=D)
    c = torch.nn.functional.silu(u).permute(0, 2, 3, 1).reshape(B, S, D)
    hw = lambda t, wt, b: (torch.einsum("bshd,hod->bsho", t.reshape(B, S, NH, d), wt.to(t.dtype)).reshape(B, S, D)
                           + (0 if b is None else b.to(t.dtype)))
    return c, hw(c, wq, bq), hw(c, wk, bk), hw(x, wv, bv)


def colsum(srcs) -> torch.Tensor:
    """Column sums of up to three equally shaped (T, D) bf16 CUDA matrices (evenly strided rows, D % 8 == 0) in one pass:
    (len(srcs), D) fp32, deterministic (csrc/mlstm_qkv.cu).  The projections' bias gradients."""
    lib = _lib.load()
    T, D = srcs[0].shape
    ld = srcs[0].stride(0)
    assert all(t.is_cuda and t.dtype == torch.bfloat16 and t.shape == (T, D) and t.stride() == (ld, 1) for t in srcs)
    dev = srcs[0].device
    out = torch.empty((len(srcs), D), dtype=torch.float32, device=dev)
    need = lib.mlstm_b200_colsum_workspace_bytes(D, len(srcs))
    ws = torch.empty(max(1, need // 4), dtype=torch.float32, device=dev)
    ptrs = (C.c_void_p * len(srcs))(*[t.data_ptr() for t in srcs])
    with torch.cuda.device(dev):
        rc = lib.mlstm_b200_colsum(ptrs, len(srcs), T, D, ld, out.data_ptr(), ws.data_ptr(), ws.numel() * 4, _stream())
    if rc:
        _fail(rc, "column sums")
    return out


def qkv_proj_backward(x, c, wq, wk, wv, dc, dq, dk, dv, need_db=True):
    """The projections' share of the producer's backward as one kernel (csrc/mlstm_qkv.cu, qkv_bwd_kernel): returns
    (dxc, dxv, dWq, dWk, dWv, db) with dxc = dc + dq Wq + dk Wk, dxv = dv Wv (both (B,S,D) bf16), dW* (NH,d,d) fp32,
    db (3, D) fp32 column sums of dq | dk | dv.  x: (B,S,D) bf16 / fp16 rows (column slice allowed); the rest dense bf16."""
    lib = _lib.load()
    B, S, D = x.shape
    NH, d = wq.shape[0], wq.shape[1]
    T, dev = B * S, x.device
    dense = lambda t: None if t is None else (t if (t.dtype == torch.bfloat16 and t.is_contiguous()) else t.to(torch.bfloat16).contiguous())
    c, dq, dk, dv, dc = dense(c), dense(dq), dense(dk), dense(dv), dense(dc)
    kw = [w.detach().to(torch.bfloat16).contiguous() for w in (wq, wk, wv)]
    dxc = torch.empty((B, S, D), dtype=torch.bfloat16, device=dev)
    dxv = torch.empty((B, S, D), dtype=torch.bfloat16, device=dev)
    dws = [torch.empty((NH, d, d), dtype=torch.float32, device=dev) for _ in range(3)]
    db = torch.empty((3, D), dtype=torch.float32, device=dev) if need_db else None
    g = QkvBwdParams()
    g.abi_version = _lib.ABI_VERSION
    g.T, g.D, g.NH, g.x_dtype = T, D, NH, int(x.dtype == torch.float16)
    g.x, g.ld_x = x.data_ptr(), x.stride(1)
    g.c, g.dq, g.dk, g.dv, g.dc = c.data_ptr(), dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), _ptr(dc)
    g.wq, g.wk, g.wv = (w.data_ptr() for w in kw)
    g.dxc, g.dxv = dxc.data_ptr(), dxv.data_ptr()
    g.dwq, g.dwk, g.dwv = (w.data_ptr() for w in dws)
    g.db = _ptr(db)
    need = lib.mlstm_b200_qkv_bwd_workspace_bytes(C.byref(g))
    ws = torch.empty(max(1, (need + 3) // 4), dtype=torch.float32, device=dev)
    g.workspace, g.workspace_bytes = ws.data_ptr(), ws.numel() * 4
    with torch.cuda.device(dev):
        rc = lib.mlstm_b200_qkv_bwd(C.byref(g), _stream())
    if rc:
        _fail(rc, "qkv producer backward")
    return dxc, dxv, dws[0], dws[1], dws[2], db


def conv_silu_backward(x, sp, dxc, dxv, conv_w, need_bias, gh, gw, rotate):
    """Backward of c = silu(conv3x3_depthwise(x)) as one kernel (csrc/mlstm_qkv.cu, conv_bwd_kernel): with du = dxc * sp
    (sp = silu'(conv(x)), saved by the producer's forward) returns (dx, dwc, dbc): dx = conv^T(du) + dxv in x's dtype (B,S,D),
    dwc (D,1,3,3) fp32, dbc (D) fp32 or None."""
    lib = _lib.load()
    B, S, D = x.shape
    dev = x.device
    dense = lambda t: t if (t.dtype == torch.bfloat16 and t.is_contiguous()) else t.to(torch.bfloat16).contiguous()
    dxc, dxv, sp = dense(dxc), dense(dxv), dense(sp)
    cw = conv_w.detach().to(torch.float32).contiguous()
    dx = torch.empty((B, S, D), dtype=x.dtype, device=dev)
    dwc = torch.empty((D, 1, 3, 3), dtype=torch.float32, device=dev)
    dbc = torch.empty(D, dtype=torch.float32, device=dev) if need_bias else None
    g = ConvBwdParams()
    g.abi_version = _lib.ABI_VERSION
    g.B, g.GH, g.GW, g.D = B, gh, gw, D
    g.NH = D // 128 if D % 128 == 0 else D // 64           # channel blocks of the kernel's tiling (independent of the heads)
    g.rotate, g.x_dtype = int(bool(rotate)), int(x.dtype == torch.float16)
    g.x, g.ld_x = x.data_ptr(), x.stride(1)
    g.dxc, g.dxv, g.sp = dxc.data_ptr(), dxv.data_ptr(), sp.data_ptr()
    g.conv_w, g.dx, g.dwc, g.dbc = cw.data_ptr(), dx.data_ptr(), dwc.data_ptr(), _ptr(dbc)
    need = lib.mlstm_b200_conv_bwd_workspace_bytes(C.byref(g))
    ws = torch.empty(max(1, (need + 3) // 4), dtype=torch.float32, device=dev)
    g.workspace, g.workspace_bytes = ws.data_ptr(), ws.numel() * 4
    with torch.cuda.device(dev):
        rc = lib.mlstm_b200_conv_bwd(C.byref(g), _stream())
    if rc:
        _fail(rc, "conv + SiLU backward")
    return dx, dwc, dbc


def _conv_silu_backward(x, conv_w, conv_b, dxc, dxv, gh, gw, rotate):
    """du = dxc * silu'(u) with u = conv(x) recomputed, then the depthwise conv's own backward; dx = conv^T(du) + dxv."""
    B, S, D = x.shape
    w = (conv_w.flip(-1, -2) if rotate else conv_w).to(x.dtype)
    img = x.reshape(B, gh, gw, D).permute(0, 3, 1, 2)
    u = torch.nn.functional.conv2d(img, w, None if conv_b is None else conv_b.to(x.dtype), padding=1, groups=D)
    dxc_img = dxc.reshape(B, gh, gw, D).permute(0, 3, 1, 2)
    du = torch.ops.aten.silu_backward(dxc_img if dxc_img.dtype == u.dtype else dxc_img.to(u.dtype), u)
    dimg, dwc, dbc = torch.ops.aten.convolution_backward(du, img, w, [D] if conv_b is not None else None, [1, 1], [1, 1], [1, 1],
                                                         False, [0, 0], D, [True, True, conv_b is not None])
    if rotate:
        dwc = dwc.flip(-1, -2)
    dx = dimg.permute(0, 2, 3, 1).reshape(B, S, D)
    dx = dx + (dxv if dxv.dtype == dx.dtype else dxv.to(dx.dtype)).reshape(B, S, D)
    return dx, dwc, dbc


def qkv_backward(x, c, conv_w, conv_b, wq, wk, wv, has_bias, dc, dq, dk, dv, gh, gw, rotate, sp=None):
    """Backward of the producer in PyTorch ops (cuBLAS batched GEMMs over the strided head views, cuDNN depthwise conv):
    the saved c replaces everything but the conv pre-activation, which is recomputed.  Works on any device (the CPU
    tests differentiate it against autograd of ``qkv_reference``).  Returns gradients for
    (x, conv_w, conv_b, wq, bq, wk, bk, wv, bv); bias gradients are None where ``has_bias`` says so."""
    B, S, D = x.shape
    NH, d = wq.shape[0], wq.shape[1]
    T = B * S
    if (x.is_cuda and dq.dtype == torch.bfloat16 and c.dtype == torch.bfloat16 and x.dtype in (torch.bfloat16, torch.float16)
            and x.stride(2) == 1 and x.stride(0) == S * x.stride(1) and x.data_ptr() % 16 == 0
            and _lib.load().mlstm_b200_qkv_supported(D, NH, 1, 1, x.stride(1))):
        # the five GEMMs and the bias sums as one tcgen05 kernel; the conv's own backward stays with cuDNN
        dxc, dxv, dwq, dwk, dwv, db = qkv_proj_backward(x, c, wq, wk, wv, dc, dq, dk, dv, need_db=any(has_bias))
        if sp is not None and _lib.load().mlstm_b200_qkv_supported(D, NH, gh, gw, x.stride(1)):
            dx, dwc, dbc = conv_silu_backward(x, sp, dxc, dxv, conv_w, conv_b is not None, gh, gw, rotate)   # one kernel
        else:
            dx, dwc, dbc = _conv_silu_backward(x, conv_w, conv_b, dxc, dxv, gh, gw, rotate)                  # cuDNN
        pick = lambda j: db[j] if has_bias[j] else None
        return (dx, dwc, dbc, dwq, pick(0), dwk, pick(1), dwv, pick(2))
    cd = dq.dtype                                            # compute dtype of the projections' gradients
    heads = lambda t: t.reshape(T, NH, d).transpose(0, 1)   # (NH, T, d) strided view: no copy for evenly strided rows
    dense = lambda t: t if t.is_contiguous() else t.contiguous()
    dqh, dkh, dvh = heads(dense(dq)), heads(dense(dk)), heads(dense(dv))
    ch, xh = heads(c if c.dtype == cd else c.to(cd)), heads(x if x.dtype == cd else x.to(cd))
    # projections: dW = dy^T in, din = dy W
    dwq, dwk, dwv = torch.bmm(dqh.transpose(1, 2), ch), torch.bmm(dkh.transpose(1, 2), ch), torch.bmm(dvh.transpose(1, 2), xh)
    # dxc = dc + dq Wq + dk Wk accumulated by the GEMMs themselves (beta = 1 into the strided head views)
    if dc is not None:
        dxc = dc.reshape(T, D).to(cd, copy=True)
        dxc_h = dxc.view(T, NH, d).transpose(0, 1)
        torch.baddbmm(dxc_h, dqh, wq.to(cd), out=dxc_h)
    else:
        dxc = torch.empty((T, D), dtype=cd, device=x.device)
        dxc_h = dxc.view(T, NH, d).transpose(0, 1)
        torch.bmm(dqh, wq.to(cd), out=dxc_h)
    torch.baddbmm(dxc_h, dkh, wk.to(cd), out=dxc_h)
    # conv + SiLU: u recomputed, du = dxc * silu'(u), then the depthwise conv's own backward and dx = conv^T(du) + dv Wv
    w = (conv_w.flip(-1, -2) if rotate else conv_w).to(x.dtype)
    img = x.reshape(B, gh, gw, D).permute(0, 3, 1, 2)
    u = torch.nn.functional.conv2d(img, w, None if conv_b is None else conv_b.to(x.dtype), padding=1, groups=D)
    dxc_img = dxc.view(B, gh, gw, D).permute(0, 3, 1, 2)
    du = torch.ops.aten.silu_backward(dxc_img if dxc_img.dtype == u.dtype else dxc_img.to(u.dtype), u)
    dimg, dwc, dbc = torch.ops.aten.convolution_backward(du, img, w, [D] if conv_b is not None else None, [1, 1], [1, 1], [1, 1],
                                                         False, [0, 0], D, [True, True, conv_b is not None])
    if rotate:
        dwc = dwc.flip(-1, -2)
    dx = dimg.permute(0, 2, 3, 1).reshape(T, D)
    if dx.dtype == cd and dx.is_contiguous():
        dx_h = dx.view(T, NH, d).transpose(0, 1)
        torch.baddbmm(dx_h, dvh, wv.to(cd), out=dx_h)
    else:
        dx = dx + torch.bmm(dvh, wv.to(cd)).transpose(0, 1).reshape(T, D).to(dx.dtype)
    dx = dx.view(B, S, D)
    if any(has_bias) and dq.is_cuda and cd == torch.bfloat16 and D % 8 == 0:
        cs = colsum([dqh.transpose(0, 1).reshape(T, D), dkh.transpose(0, 1).reshape(T, D), dvh.transpose(0, 1).reshape(T, D)])
        sums = [cs[j] if has_bias[j] else None for j in range(3)]
    else:
        sums = [t.reshape(T, D).sum(0, dtype=torch.float32) if on else None for t, on in zip((dq, dk, dv), has_bias)]
    return (dx, dwc, dbc, dwq, sums[0], dwk, sums[1], dwv, sums[2])


def qkv_fwd_raw(x, conv_w, conv_b, wq, bq, wk, bk, wv, bv, gh, gw, rotate, need_sp):
    """One producer forward launch on an ``x`` that ``qkv_supported`` accepts: (c, q, k, v, sp), each (B,S,D) bf16;
    sp = silu'(conv(x)), which the conv's backward kernel reads, only when ``need_sp`` (else None)."""
    lib = _lib.load()
    B, S, D = x.shape
    NH = wq.shape[0]
    dev = x.device
    f32 = lambda t: None if t is None else t.detach().to(torch.float32).contiguous()
    cw, cb, fbq, fbk, fbv = f32(conv_w), f32(conv_b), f32(bq), f32(bk), f32(bv)
    kq, kk = wq.detach().to(torch.bfloat16).contiguous(), wk.detach().to(torch.bfloat16).contiguous()
    kv = wv.detach().to(x.dtype).contiguous()
    c, q, k, v = (torch.empty((B, S, D), dtype=torch.bfloat16, device=dev) for _ in range(4))
    sp = torch.empty((B, S, D), dtype=torch.bfloat16, device=dev) if need_sp else None
    g = QkvParams()
    g.abi_version = _lib.ABI_VERSION
    g.B, g.GH, g.GW, g.D, g.NH = B, gh, gw, D, NH
    g.rotate, g.x_dtype = int(bool(rotate)), int(x.dtype == torch.float16)
    g.x, g.ld_x = x.data_ptr(), x.stride(1)
    g.conv_w, g.conv_b = cw.data_ptr(), _ptr(cb)
    g.wq, g.wk, g.wv = kq.data_ptr(), kk.data_ptr(), kv.data_ptr()
    g.bq, g.bk, g.bv = _ptr(fbq), _ptr(fbk), _ptr(fbv)
    g.c, g.q, g.k, g.v = c.data_ptr(), q.data_ptr(), k.data_ptr(), v.data_ptr()
    g.sp = _ptr(sp)
    with torch.cuda.device(dev):
        rc = lib.mlstm_b200_qkv_fwd(C.byref(g), _stream())
    if rc:
        _fail(rc, "qkv producer forward")
    return c, q, k, v, sp


def _qkv_grads(x, c, conv_w, conv_b, wq, wk, wv, sp, dc, dq, dk, dv, gh, gw, rotate, has_bias):
    """``qkv_backward`` with each gradient in its input's dtype (the projections' bias gradients stay fp32)."""
    g = qkv_backward(x, c, conv_w, conv_b, wq, wk, wv, has_bias, dc, dq, dk, dv, gh, gw, rotate, sp=sp)
    dx, dwc, dbc, dwq, dbq, dwk, dbk, dwv, dbv = g
    cast = lambda t, like: None if (t is None or like is None) else t.to(like.dtype)
    return dx.to(x.dtype), cast(dwc, conv_w), cast(dbc, conv_b), cast(dwq, wq), dbq, cast(dwk, wk), dbk, cast(dwv, wv), dbv


class _QkvFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, conv_w, conv_b, wq, bq, wk, bk, wv, bv, gh, gw, rotate):
        # silu'(conv(x)) for the conv's backward kernel: only when a backward can follow
        c, q, k, v, sp = qkv_fwd_raw(x, conv_w, conv_b, wq, bq, wk, bk, wv, bv, gh, gw, rotate, any(ctx.needs_input_grad[:9]))
        ctx.save_for_backward(x, c, conv_w, conv_b, wq, wk, wv, sp)
        ctx.meta = (gh, gw, bool(rotate), (bq is not None, bk is not None, bv is not None))
        return c, q, k, v

    @staticmethod
    def backward(ctx, dc, dq, dk, dv):
        x, c, conv_w, conv_b, wq, wk, wv, sp = ctx.saved_tensors
        gh, gw, rotate, has_bias = ctx.meta
        z = lambda t: torch.zeros_like(c) if t is None else t
        return _qkv_grads(x, c, conv_w, conv_b, wq, wk, wv, sp, dc, z(dq), z(dk), z(dv), gh, gw, rotate, has_bias) + (None,) * 3


def qkv_producer(x, conv_w, conv_b, wq, bq, wk, bk, wv, bv, gh: int, gw: int, rotate: bool = False):
    """(c, q, k, v) = (silu(conv(x)), c Wq^T + bq, c Wk^T + bk, x Wv^T + bv), all (B,S,D) bf16, from one kernel
    (csrc/mlstm_qkv.cu).  Check ``qkv_supported`` first.  Backward: ``qkv_backward`` (cuBLAS / cuDNN through PyTorch)."""
    args = (x, conv_w, conv_b, wq, bq, wk, bk, wv, bv, int(gh), int(gw), bool(rotate))
    if _use_custom_ops():
        need_sp = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in args[:9])
        return _qkv_fwd_op(*args, need_sp)[:4]
    return _QkvFn.apply(*args)


class MLSTMPlan:
    """Pre-bound forward+backward call on fixed device buffers (steady-state / benchmark use).

    All outputs and the workspace are allocated once; ``forward()`` / ``backward()`` are then a
    single C-ABI call each (plus the host-side TMA descriptor encode inside the library).
    """

    def __init__(self, q, k, v, i, f, dh, *, eps=1e-6, chunk_size=64, reverse=False, input_gate="exp"):
        self.lib = _lib.load()
        B, NH, S, DK = q.shape
        DV = v.shape[-1]
        dev = q.device
        self.inputs = (q, k, v, i, f, dh)
        self.h = _empty_act(B, NH, S, DV, q.dtype, dev)
        self.n_row = torch.empty((B, NH, S), dtype=torch.float32, device=dev)
        self.m_row = torch.empty((B, NH, S), dtype=torch.float32, device=dev)
        self.dq = _empty_act(B, NH, S, DK, q.dtype, dev)
        self.dk = _empty_act(B, NH, S, DK, q.dtype, dev)
        self.dv = _empty_act(B, NH, S, DV, q.dtype, dev)
        self.di = torch.empty((B, S, NH), dtype=torch.float32, device=dev).transpose(1, 2)
        self.df = torch.empty((B, S, NH), dtype=torch.float32, device=dev).transpose(1, 2)
        p = _base_params(q, k, v, i, f, eps, chunk_size, reverse, None, gate_mode_of(input_gate))
        p.h = _act(self.h)
        p.n_row, p.m_row = _ptr(self.n_row), _ptr(self.m_row)
        p.dh = _act(dh)
        p.dq, p.dk, p.dv = _act(self.dq), _act(self.dk), _act(self.dv)
        p.di, p.df = _gate(self.di), _gate(self.df)
        self.states = _alloc_states(self.lib, p, dev)
        need = self.lib.mlstm_b200_workspace_bytes(C.byref(p), 1)
        self.ws = torch.empty(max(1, (need + 3) // 4), dtype=torch.float32, device=dev)
        p.workspace, p.workspace_bytes = self.ws.data_ptr(), self.ws.numel() * 4
        self.p = p
        self.family = self.lib.mlstm_b200_kernel_name(C.byref(p), 0).decode()
        self.variant_fwd = self.lib.mlstm_b200_kernel_variant(C.byref(p), 0).decode()
        self.variant_bwd = self.lib.mlstm_b200_kernel_variant(C.byref(p), 1).decode()

    def forward(self):
        rc = self.lib.mlstm_b200_fwd(C.byref(self.p), _stream())
        if rc:
            _fail(rc, "forward")
        return self.h

    def backward(self, part: int = -1):
        rc = self.lib.mlstm_b200_bwd_part(C.byref(self.p), part, _stream())
        if rc:
            _fail(rc, "backward")
        return self.dq, self.dk, self.dv, self.di, self.df


# ---------------------------------------------------------------------------------------------------------------
# torch.library registration of the layer kernels: ``xlstm_yolo_b200::fused_cell_fwd`` / ``::fused_cell_bwd``,
# ``::qkv_fwd`` / ``::qkv_bwd`` and ``::layer_tail_fwd`` / ``::layer_tail_bwd`` call the launchers above, so a compiled
# model runs the same kernels as an eager one.  The fakes give the real layouts (Inductor checks the sizes and strides of
# what an op returns).  An absent optional output is an empty tensor, mapped to None in the autograd formulas.  The
# caller sizes the chunk-state buffer (``_states_numel``), so that a dynamic batch needs no data-dependent output size.
# ---------------------------------------------------------------------------------------------------------------
def _use_custom_ops() -> bool:
    """torch.compile traces the custom ops; eager mode calls the autograd.Functions: same launches, less host time.
    Measured on a B200 (1000 W limit, tests/gpu_tools/compile_bench.py), eager ViLBlockPair forward + backward, twelve
    layer-op calls per step: 3.21 ms through the autograd.Functions vs 4.14 ms through the custom ops at dim 128, B 32,
    400 tokens (about 80 us more per call), 3.68 vs 4.19-4.41 ms at dim 256, B 32, 1600 tokens."""
    return torch.compiler.is_compiling()


def _none_to_empty(t: Optional[torch.Tensor], like: torch.Tensor, dtype=torch.float32) -> torch.Tensor:
    return torch.empty(0, dtype=dtype, device=like.device) if t is None else t


def _tail_h(h: torch.Tensor) -> torch.Tensor:
    """h as the tail kernel reads it: a 16-byte aligned (B,NH,S,DH) view of (B,S,NH,DH) storage, else a copy into one."""
    B, NH, S, DH = h.shape
    if h.stride() == (S * NH * DH, DH, NH * DH, 1) and h.data_ptr() % 16 == 0:
        return h
    out = _empty_act(B, NH, S, DH, h.dtype, h.device)
    out.copy_(h)
    return out


def _dense_rows(t: torch.Tensor) -> torch.Tensor:
    return t if _rows_ok(t) else t.contiguous()


@torch.library.custom_op("xlstm_yolo_b200::fused_cell_fwd", mutates_args=(), device_types="cuda")
def _fused_cell_fwd_op(q3: torch.Tensor, k3: torch.Tensor, v3: torch.Tensor, w_i: torch.Tensor, b_i: Optional[torch.Tensor],
                       w_f: torch.Tensor, b_f: Optional[torch.Tensor], num_heads: int, eps: float, chunk_size: int, reverse: bool,
                       gate_mode: int, save_rows: bool,
                       states_bytes: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    q3, k3, v3 = _cell_rows(q3, k3, v3)
    h, i3, f3, n_row, m_row, states = fused_cell_fwd_raw(q3, k3, v3, w_i, b_i, w_f, b_f, num_heads, eps, chunk_size, reverse,
                                                         gate_mode, save_rows, states_bytes)
    return h, i3, f3, _none_to_empty(n_row, h), _none_to_empty(m_row, h), _none_to_empty(states, h, torch.uint8)


@_fused_cell_fwd_op.register_fake
def _(q3, k3, v3, w_i, b_i, w_f, b_f, num_heads, eps, chunk_size, reverse, gate_mode, save_rows, states_bytes):
    B, S, D = q3.shape
    NH, DH, dev = num_heads, D // num_heads, q3.device
    h = torch.empty((B, S, NH, DH), dtype=q3.dtype, device=dev).transpose(1, 2)
    i3, f3 = (torch.empty((B, S, NH), dtype=torch.float32, device=dev) for _ in range(2))
    rows = (lambda: torch.empty((B, NH, S), dtype=torch.float32, device=dev)) if save_rows else \
        (lambda: torch.empty(0, dtype=torch.float32, device=dev))
    states = torch.empty(states_bytes, dtype=torch.uint8, device=dev)
    return h, i3, f3, rows(), rows(), states


@torch.library.custom_op("xlstm_yolo_b200::fused_cell_bwd", mutates_args=(), device_types="cuda")
def _fused_cell_bwd_op(q3: torch.Tensor, k3: torch.Tensor, v3: torch.Tensor, w_i: torch.Tensor, w_f: torch.Tensor,
                       i3: torch.Tensor, f3: torch.Tensor, h: torch.Tensor, n_row: torch.Tensor, m_row: torch.Tensor,
                       states: torch.Tensor, dh: torch.Tensor, num_heads: int, eps: float, chunk_size: int, reverse: bool,
                       gate_mode: int, has_bias: bool) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor,
                                                                torch.Tensor, torch.Tensor, torch.Tensor]:
    q3, k3, v3 = _cell_rows(q3, k3, v3)
    dq3, dk3, dv3, dw_i, db_i, dw_f, db_f = fused_cell_bwd_raw(
        q3, k3, v3, w_i, w_f, i3, f3, _prep_act(h), n_row, m_row, states if states.numel() else None, dh, num_heads, eps,
        chunk_size, reverse, gate_mode, has_bias)
    return dq3, dk3, dv3, dw_i, _none_to_empty(db_i, h), dw_f, _none_to_empty(db_f, h)


@_fused_cell_bwd_op.register_fake
def _(q3, k3, v3, w_i, w_f, i3, f3, h, n_row, m_row, states, dh, num_heads, eps, chunk_size, reverse, gate_mode, has_bias):
    B, S, D = q3.shape
    d3 = lambda: torch.empty((B, S, D), dtype=q3.dtype, device=q3.device)
    db = lambda: torch.empty(num_heads if has_bias else 0, dtype=torch.float32, device=q3.device)
    return d3(), d3(), d3(), torch.empty_like(w_i), db(), torch.empty_like(w_f), db()


def _fused_cell_setup_context(ctx, inputs, output):
    q3, k3, v3, w_i, b_i, w_f, b_f, num_heads, eps, chunk_size, reverse, gate_mode, save_rows, states_bytes = inputs
    h, i3, f3, n_row, m_row, states = output
    ctx.save_for_backward(q3, k3, v3, w_i, w_f, i3, f3, h, n_row, m_row, states)
    ctx.cfg = (num_heads, eps, chunk_size, reverse, gate_mode, b_i is not None)
    ctx.set_materialize_grads(False)


def _fused_cell_backward(ctx, dh, *_unused):
    saved = ctx.saved_tensors
    if dh is None:
        dh = torch.zeros_like(saved[7])
    dq3, dk3, dv3, dw_i, db_i, dw_f, db_f = _fused_cell_bwd_op(*saved, dh, *ctx.cfg)
    has_bias = ctx.cfg[-1]
    return (dq3, dk3, dv3, dw_i, db_i if has_bias else None, dw_f, db_f if has_bias else None) + (None,) * 7


_fused_cell_fwd_op.register_autograd(_fused_cell_backward, setup_context=_fused_cell_setup_context)


@torch.library.custom_op("xlstm_yolo_b200::qkv_fwd", mutates_args=(), device_types="cuda")
def _qkv_fwd_op(x: torch.Tensor, conv_w: torch.Tensor, conv_b: Optional[torch.Tensor], wq: torch.Tensor, bq: Optional[torch.Tensor],
                wk: torch.Tensor, bk: Optional[torch.Tensor], wv: torch.Tensor, bv: Optional[torch.Tensor], gh: int, gw: int,
                rotate: bool, need_sp: bool) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    c, q, k, v, sp = qkv_fwd_raw(_dense_rows(x), conv_w, conv_b, wq, bq, wk, bk, wv, bv, gh, gw, rotate, need_sp)
    return c, q, k, v, _none_to_empty(sp, x, torch.bfloat16)


@_qkv_fwd_op.register_fake
def _(x, conv_w, conv_b, wq, bq, wk, bk, wv, bv, gh, gw, rotate, need_sp):
    act = lambda: torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    return act(), act(), act(), act(), act() if need_sp else torch.empty(0, dtype=torch.bfloat16, device=x.device)


@torch.library.custom_op("xlstm_yolo_b200::qkv_bwd", mutates_args=(), device_types="cuda")
def _qkv_bwd_op(x: torch.Tensor, c: torch.Tensor, conv_w: torch.Tensor, conv_b: Optional[torch.Tensor], wq: torch.Tensor,
                wk: torch.Tensor, wv: torch.Tensor, sp: torch.Tensor, dc: Optional[torch.Tensor], dq: torch.Tensor, dk: torch.Tensor,
                dv: torch.Tensor, gh: int, gw: int, rotate: bool, has_bq: bool, has_bk: bool,
                has_bv: bool) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor,
                                       torch.Tensor, torch.Tensor, torch.Tensor]:
    grads = _qkv_grads(_dense_rows(x), c, conv_w, conv_b, wq, wk, wv, sp if sp.numel() else None, dc, dq, dk, dv, gh, gw,
                       rotate, (has_bq, has_bk, has_bv))
    # outputs own their storage: the projections' bias gradients may be rows of one (3, D) buffer
    return tuple(_none_to_empty(t, x) if t is None else t.clone() if j in (4, 6, 8) else t.contiguous()
                 for j, t in enumerate(grads))


@_qkv_bwd_op.register_fake
def _(x, c, conv_w, conv_b, wq, wk, wv, sp, dc, dq, dk, dv, gh, gw, rotate, has_bq, has_bk, has_bv):
    D, dev = x.shape[2], x.device
    bias = lambda on: torch.empty(D if on else 0, dtype=torch.float32, device=dev)
    return (torch.empty(x.shape, dtype=x.dtype, device=dev), torch.empty(conv_w.shape, dtype=conv_w.dtype, device=dev),
            torch.empty(0, dtype=torch.float32, device=dev) if conv_b is None else torch.empty(D, dtype=conv_b.dtype, device=dev),
            torch.empty(wq.shape, dtype=wq.dtype, device=dev), bias(has_bq), torch.empty(wk.shape, dtype=wk.dtype, device=dev),
            bias(has_bk), torch.empty(wv.shape, dtype=wv.dtype, device=dev), bias(has_bv))


def _qkv_setup_context(ctx, inputs, output):
    x, conv_w, conv_b, wq, bq, wk, bk, wv, bv, gh, gw, rotate, need_sp = inputs
    c, q, k, v, sp = output
    ctx.save_for_backward(x, c, conv_w, conv_b, wq, wk, wv, sp)
    ctx.meta = (gh, gw, rotate, bq is not None, bk is not None, bv is not None)
    ctx.set_materialize_grads(False)


def _qkv_backward(ctx, dc, dq, dk, dv, _dsp):
    x, c, conv_w, conv_b, wq, wk, wv, sp = ctx.saved_tensors
    z = lambda t: torch.zeros_like(c) if t is None else t
    g = _qkv_bwd_op(x, c, conv_w, conv_b, wq, wk, wv, sp, dc, z(dq), z(dk), z(dv), *ctx.meta)
    has_b = (conv_b is not None,) + ctx.meta[3:]
    dx, dwc, dbc, dwq, dbq, dwk, dbk, dwv, dbv = g
    pick = lambda t, on: t if on else None
    return (dx, dwc, pick(dbc, has_b[0]), dwq, pick(dbq, has_b[1]), dwk, pick(dbk, has_b[2]), dwv, pick(dbv, has_b[3]),
            None, None, None, None)


_qkv_fwd_op.register_autograd(_qkv_backward, setup_context=_qkv_setup_context)


@torch.library.custom_op("xlstm_yolo_b200::layer_tail_fwd", mutates_args=(), device_types="cuda")
def _layer_tail_fwd_op(h: torch.Tensor, c: torch.Tensor, z: torch.Tensor, w: Optional[torch.Tensor], b: Optional[torch.Tensor],
                       skip: Optional[torch.Tensor], eps: float) -> torch.Tensor:
    return layer_tail_fwd_raw(_tail_h(h), _dense_rows(c), _dense_rows(z), w, b, skip, eps)


@_layer_tail_fwd_op.register_fake
def _(h, c, z, w, b, skip, eps):
    B, NH, S, DH = h.shape
    return torch.empty((B, S, NH * DH), dtype=h.dtype, device=h.device)


@torch.library.custom_op("xlstm_yolo_b200::layer_tail_bwd", mutates_args=(), device_types="cuda")
def _layer_tail_bwd_op(h: torch.Tensor, c: torch.Tensor, z: torch.Tensor, w: Optional[torch.Tensor], b: Optional[torch.Tensor],
                       skip: Optional[torch.Tensor], dy: torch.Tensor,
                       eps: float) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
    dh, dc, dz, dw, db, dskip = layer_tail_bwd_raw(_tail_h(h), _dense_rows(c), _dense_rows(z), w, b, skip, dy, eps)
    return dh, dc, dz, _none_to_empty(dw, h), _none_to_empty(db, h), _none_to_empty(dskip, h)


@_layer_tail_bwd_op.register_fake
def _(h, c, z, w, b, skip, dy, eps):
    B, NH, S, DH = h.shape
    D, dev = NH * DH, h.device
    d3 = lambda: torch.empty((B, S, D), dtype=h.dtype, device=dev)
    vec = lambda t: torch.empty(0 if t is None else D, dtype=torch.float32, device=dev)
    return _empty_act(B, NH, S, DH, h.dtype, dev), d3(), d3(), vec(w), vec(b), vec(skip)


def _layer_tail_setup_context(ctx, inputs, output):
    h, c, z, w, b, skip, eps = inputs
    ctx.save_for_backward(h, c, z, w, b, skip)
    ctx.eps = eps
    ctx.set_materialize_grads(False)


def _layer_tail_backward(ctx, dy):
    h, c, z, w, b, skip = ctx.saved_tensors
    if dy is None:
        return (None,) * 7
    dh, dc, dz, dw, db, dskip = _layer_tail_bwd_op(h, c, z, w, b, skip, dy, ctx.eps)
    pick = lambda t, like: None if like is None else t
    return dh, dc, dz, pick(dw, w), pick(db, b), pick(dskip, skip), None


_layer_tail_fwd_op.register_autograd(_layer_tail_backward, setup_context=_layer_tail_setup_context)
