"""Drop-in ``MatrixLSTMCell`` (reference: nn/modules/vision_lstm/vision_lstm2.py:802-966).

Same constructor signature, sub-module names (``igate``, ``fgate``, ``outnorm``), parameter
shapes/initialisation and ``forward(q, k, v)`` signature, so state_dicts and pickled
checkpoints interchange and the YAML builders (nn/tasks.py:1212-1214) need no change.

Differences, all deliberate:
  * returns the *intended* ``(B, S, dim)`` (outnorm, heads merged — vision_lstm2.py:950-952,
    commented out at HEAD, which makes ViLLayer.forward fail at :498); ``raw_output=True``
    reproduces HEAD's raw ``(B, NH, S, DH)`` for forensic comparison;
  * the gate projection reads q,k,v in place instead of materialising ``cat[q,k,v]`` (:895): on
    CUDA a hand-written streaming kernel fused with the cell into one autograd node (its backward
    adds the gate path into dq,dk,dv in place), on CPU through weight slices;
  * ``reverse=True`` scans from the last token, replacing the flip pair around the layer
    (:479-480,505-506);
  * ``input_gate="sigmoid"`` selects the sigmoid-input-gate arithmetic that HEAD's CUDA kernel string
    ("chunkwise--triton_xl_chunk_siging", :835,866) names; the default "exp" is the exponential gate
    of the reference's in-tree PyTorch mLSTM (its CPU path, backends.py:149-263);
  * on CUDA the arithmetic is the sm_100a kernel library, not Triton.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F
from torch import nn

from .backend import mLSTMBackend, mLSTMBackendConfig


def bias_linspace_init_(param: torch.Tensor, start: float = 3.4, end: float = 6.0) -> torch.Tensor:
    """Linearly spaced bias (vision_lstm2.py:21-28)."""
    assert param.dim() == 1
    with torch.no_grad():
        param.copy_(torch.linspace(start, end, param.shape[0]))
    return param


class MultiHeadLayerNorm(nn.Module):
    """Per-head layer norm over DH with residual weight ``1 + w`` (vision_lstm2.py:1262-1325)."""

    def __init__(self, ndim: int = -1, weight: bool = True, bias: bool = False, eps: float = 1e-5,
                 residual_weight: bool = True):
        super().__init__()
        self.weight = nn.Parameter(torch.zeros(ndim)) if weight else None
        self.bias = nn.Parameter(torch.zeros(ndim)) if bias else None
        self.eps = eps
        self.residual_weight = residual_weight
        self.ndim = ndim
        self.reset_parameters()

    @property
    def weight_proxy(self):
        if self.weight is None:
            return None
        return 1.0 + self.weight if self.residual_weight else self.weight

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        assert x.ndim == 4, "Input must be 4D tensor (B, NH, S, DH)"
        B, NH, S, DH = x.shape
        y = F.group_norm(x.transpose(1, 2).reshape(B * S, NH * DH), num_groups=NH, weight=self.weight_proxy,
                         bias=self.bias, eps=self.eps)
        return y.view(B, S, NH, DH).transpose(1, 2)

    def reset_parameters(self):
        if self.weight is not None:
            if self.residual_weight:
                nn.init.zeros_(self.weight)
            else:
                nn.init.ones_(self.weight)
        if self.bias is not None:
            nn.init.zeros_(self.bias)


def _fused_gates_ok(dim: int) -> bool:
    from . import ops
    return ops.gates_supported(int(dim))


class MatrixLSTMCell(nn.Module):
    def __init__(self, dim, num_heads, norm_bias=True, eps=1e-6, chunk_size=16, use_autocast=True,
                 autocast_dtype=torch.bfloat16, reverse=False, raw_output=False, input_gate="exp"):
        super().__init__()
        self.dim = dim
        self.num_heads = num_heads
        self.use_autocast = use_autocast
        self.autocast_dtype = autocast_dtype
        self.reverse = reverse
        self.raw_output = raw_output
        self.fused_gates = True   # CUDA: csrc/mlstm_gates.cu instead of three cuBLAS skinny GEMMs
        if input_gate not in ("exp", "sigmoid"):
            raise ValueError(f"input_gate must be 'exp' or 'sigmoid', got {input_gate!r}")
        # "exp": the arithmetic of the reference's in-tree PyTorch mLSTM (its CPU path and our oracle);
        # "sigmoid": what HEAD's CUDA kernel string "...xl_chunk_siging" names (vision_lstm2.py:835,866)
        self.input_gate = input_gate

        self.igate = nn.Linear(3 * dim, num_heads)
        self.fgate = nn.Linear(3 * dim, num_heads)
        self.outnorm = MultiHeadLayerNorm(ndim=dim, weight=True, bias=norm_bias, eps=1e-3)
        self.causal_mask_cache = {}

        kdt = {torch.bfloat16: "bfloat16", torch.float32: "float32", torch.float16: "float16"}[autocast_dtype]
        if not use_autocast:
            kdt = "float32"

        def mk(mode):  # eps = 5e-5: what the reference passes (vision_lstm2.py:827)
            return mLSTMBackend(mLSTMBackendConfig(
                chunkwise_kernel="chunkwise--b200_tcgen05" + ("_siging" if input_gate == "sigmoid" else ""),
                sequence_kernel="native_sequence__native",
                step_kernel="native", chunk_size=int(chunk_size), autocast_kernel_dtype=kdt,
                return_last_states=False, mode=mode, eps=5e-5))

        # the reference keeps four backends (cpu/gpu x train/infer, :819-877); device dispatch
        # lives inside mLSTMBackend here, so two suffice — attribute names kept.
        self.gpu_backend = self.cpu_backend = mk("train")
        self.gpu_backend_infer = self.cpu_backend_infer = mk("train")  # inference: same math, no saved rows
        self.reset_parameters()

    def _gates(self, q, k, v):
        d = self.dim
        wi, wf = self.igate.weight, self.fgate.weight
        w = torch.cat([wi, wf], dim=0)                      # (2NH, 3d) — tiny
        bias = torch.cat([self.igate.bias, self.fgate.bias], dim=0)
        g = F.linear(q, w[:, :d]) + F.linear(k, w[:, d:2 * d]) + F.linear(v, w[:, 2 * d:], bias)
        i, f = g.split(self.num_heads, dim=-1)              # (B,S,NH) each
        return i.transpose(-1, -2), f.transpose(-1, -2)     # (B,NH,S) views

    def forward(self, q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, *, reverse=None, raw_output=None) -> torch.Tensor:
        """``forward(q, k, v)`` is the reference signature (vision_lstm2.py:882).  The keyword-only ``reverse`` /
        ``raw_output`` override the module attributes of the same name for this call only, so a caller (``ViLLayer``)
        never has to mutate the module: the forward stays re-entrant and traceable."""
        reverse = self.reverse if reverse is None else bool(reverse)
        raw_output = self.raw_output if raw_output is None else bool(raw_output)
        B, S, H = q.shape
        if not (q.device == k.device == v.device):
            raise ValueError("All input tensors (q, k, v) must be on the same device.")
        backend = self.gpu_backend if self.training else self.gpu_backend_infer
        with torch.autograd.profiler.record_function("ViLLayer::mlstm_cell"):
            if q.is_cuda and getattr(self, "fused_gates", True) and _fused_gates_ok(H):
                # hand-written gate projection fused with the cell into one autograd node
                h = backend.fused_cell(q, k, v, self.igate, self.fgate, self.num_heads, reverse=reverse)
            else:
                i, f = self._gates(q, k, v)
                qh = q.view(B, S, self.num_heads, -1).transpose(1, 2)
                kh = k.view(B, S, self.num_heads, -1).transpose(1, 2)
                vh = v.view(B, S, self.num_heads, -1).transpose(1, 2)
                h = backend(q=qh, k=kh, v=vh, i=i, f=f, reverse=reverse)  # (B,NH,S,DH)
            if raw_output:
                return h
            h = self.outnorm(h)
            return h.transpose(1, 2).reshape(B, S, -1)

    def reset_parameters(self):
        self.outnorm.reset_parameters()
        torch.nn.init.zeros_(self.fgate.weight)
        bias_linspace_init_(self.fgate.bias, start=3.0, end=6.0)
        torch.nn.init.zeros_(self.igate.weight)
        torch.nn.init.constant_(self.igate.bias, -10)
