"""Drop-in ViL layer stack around the B200 mLSTM cell (SURVEY.md §8 rows a9-a11).

Mirrors, by constructor signature, sub-module names and parameter shapes (so checkpoints load
unchanged), the reference classes in nn/modules/vision_lstm/vision_lstm2.py:

    SequenceTraversal       :16-18
    LinearHeadwiseExpand    :987-1022
    ViLLayer                :386-530
    ViLBlock                :685-735
    ViLBlockPair            :1393-1441
    SequenceConv2d          vision_lstm_util.py:96-129

What is done differently, on purpose:

  * **No flip pair** for ``ROWWISE_FROM_BOT_RIGHT`` (reference flips the whole ``(B,S,dim)``
    tensor twice, :479-480,505-506).  Reversing a row-major token sequence is a 180-degree
    rotation of the H x W grid; every op of the layer except the conv and the cell acts per
    token and commutes with it.  So the layer runs on the un-flipped sequence with (a) the
    depthwise conv using its kernel rotated by 180 degrees and (b) the cell scanning from the
    last token (``reverse=True`` -> the kernels walk chunks backwards, no copy).
    ``flip_free=False`` runs the reference's literal flip formulation (used by the tests to
    prove the two agree).
  * ``ViLBlockPair.forward`` composes ``BR(TL(x))`` — the intended alternating bidirectional
    pair (…checkpoint.py:1406-1408).  HEAD returns the TL output only (:1438-1441);
    ``ViLBlockPair.head_compat = True`` reproduces that.
  * The dense projections stay cuBLAS (``nn.Linear``/einsum) and the depthwise conv stays
    cuDNN, as SURVEY.md §8 a11 prescribes; only the cell is hand-written CUDA.
"""
from __future__ import annotations

import math
from enum import Enum

import torch
import torch.nn.functional as F
from torch import nn

from .cell import MatrixLSTMCell


class SequenceTraversal(Enum):
    ROWWISE_FROM_TOP_LEFT = "rowwise_from_top_left"
    ROWWISE_FROM_BOT_RIGHT = "rowwise_from_bot_right"


def _round_up(x: float, multiple: int) -> int:
    return int(((x + multiple - 1) // multiple) * multiple)


def _grid_height(num_tokens: int, seqlens) -> int:
    if seqlens is not None:
        assert len(seqlens) == 2
        return int(seqlens[0])
    if num_tokens <= 0:
        raise ValueError(f"Input sequence length x.size(1) must be positive, got {num_tokens}")
    side = math.isqrt(num_tokens)
    if side * side != num_tokens:
        raise AssertionError(f"For SequenceConv2d with seqlens=None, the input sequence length x.size(1) "
                             f"(which is {num_tokens}) must be a perfect square.")
    return side


class SequenceConv2d(nn.Conv2d):
    """Conv2d over a row-major token sequence ``(B, H*W, C)`` (vision_lstm_util.py:96-129).

    ``rotate=True`` convolves with the kernel rotated by 180 degrees: on the un-flipped sequence this
    equals flipping the tokens, running the plain conv, and flipping back."""

    def __init__(self, *args, seqlens=None, **kwargs):
        super().__init__(*args, **kwargs)
        self.seqlens = seqlens

    def forward(self, x: torch.Tensor, rotate: bool = False) -> torch.Tensor:
        assert x.ndim == 3
        B, S, C = x.shape
        gh = _grid_height(S, self.seqlens)
        # token-major (B, H*W, C) storage IS the channels-last image: a permuted view, no transpose copy; cuDNN's
        # NHWC depthwise kernels write channels-last, so the way back to (B, S, C) is a view as well
        img = x.reshape(B, gh, S // gh, C).permute(0, 3, 1, 2)
        w = self.weight.flip(-1, -2) if rotate else self.weight
        y = self._conv_forward(img, w, self.bias)
        return y.permute(0, 2, 3, 1).reshape(B, S, C)


class _HeadwiseLinearFn(torch.autograd.Function):
    """Block-diagonal linear on (T, NH*d) rows as ONE strided batched GEMM over the (NH, T, d) view of the
    token-major tensors (lda = ldc = NH*d): it reads and writes the head slices in place — no (NH, T, d)
    transposed copies in either direction, one launch per projection whatever NH is (the reference default
    qkv_block_size=16 gives NH = 32-64), bias fused into the GEMM epilogue."""

    @staticmethod
    def forward(ctx, x2, weight, bias):
        T, D = x2.shape
        NH, d = weight.shape[0], weight.shape[1]
        y = torch.empty((T, D), dtype=x2.dtype, device=x2.device)
        xh, yh = x2.view(T, NH, d).transpose(0, 1), y.view(T, NH, d).transpose(0, 1)   # (NH, T, d) strided views
        wt = weight.transpose(1, 2)                                                      # (NH, d_in, d_out) view
        if bias is None:
            torch.bmm(xh, wt, out=yh)
        else:
            torch.baddbmm(bias.view(NH, 1, d), xh, wt, out=yh)
        ctx.save_for_backward(x2, weight)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        x2, weight = ctx.saved_tensors
        NH, d = weight.shape[0], weight.shape[1]
        T = x2.shape[0]
        if dy.stride(1) != 1 or dy.stride(0) != NH * d:
            dy = dy.contiguous()
        dyh = dy.view(T, NH, d).transpose(0, 1)
        dx = dw = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty((T, NH * d), dtype=x2.dtype, device=x2.device)
            torch.bmm(dyh, weight, out=dx.view(T, NH, d).transpose(0, 1))
        if ctx.needs_input_grad[1]:
            dw = torch.bmm(dyh.transpose(1, 2), x2.view(T, NH, d).transpose(0, 1))
        db = dy.sum(0) if ctx.has_bias and ctx.needs_input_grad[2] else None
        return dx, dw, db


class LinearHeadwiseExpand(nn.Module):
    """Block-diagonal projection: one ``(d, d)`` matrix per head (vision_lstm2.py:987-1022)."""

    def __init__(self, dim, num_heads, bias=False):
        super().__init__()
        assert dim % num_heads == 0
        self.dim = dim
        self.num_heads = num_heads
        d = dim // num_heads
        self.weight = nn.Parameter(torch.empty(num_heads, d, d))
        self.bias = nn.Parameter(torch.empty(dim)) if bias else None
        self.reset_parameters()

    def reset_parameters(self):
        nn.init.normal_(self.weight.data, mean=0.0, std=math.sqrt(2 / 5 / self.weight.shape[-1]))
        if self.bias is not None:
            nn.init.zeros_(self.bias.data)

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        lead = x.shape[:-1]
        x2 = x.reshape(-1, self.dim)
        if x2.stride(1) != 1:
            x2 = x2.contiguous()
        bias = None if self.bias is None else self.bias.to(x2.dtype)
        return _HeadwiseLinearFn.apply(x2, self.weight.to(x2.dtype), bias).view(*lead, self.dim)

    def extra_repr(self):
        return f"dim={self.dim}, num_heads={self.num_heads}, bias={self.bias is not None}, "


class FeedForward(nn.Module):
    """Gated FFN the reference builds inside every ViLLayer but never calls (vision_lstm2.py:159-217);
    kept so state_dicts carry the same keys."""

    def __init__(self, embedding_dim, ffn_proj_factor=2.6667, ffn_round_up_to_multiple_of=64, use_bias=True,
                 weight_mode="fused", num_blocks=15):
        super().__init__()
        self.embedding_dim = embedding_dim
        self.weight_mode = weight_mode
        self.num_blocks = num_blocks
        self.up_proj_dim = _round_up(embedding_dim * ffn_proj_factor, ffn_round_up_to_multiple_of)
        if weight_mode == "single":
            self.proj_up_gate = nn.Linear(embedding_dim, self.up_proj_dim, bias=use_bias)
            self.proj_up = nn.Linear(embedding_dim, self.up_proj_dim, bias=use_bias)
        elif weight_mode == "fused":
            self.proj_up_gate_z = nn.Linear(embedding_dim, 2 * self.up_proj_dim, bias=use_bias)
        else:
            raise ValueError(f"unknown weight_mode {weight_mode!r}")
        self.proj_down = nn.Linear(self.up_proj_dim, embedding_dim, bias=use_bias)
        self.act_fn = nn.SiLU()

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if self.weight_mode == "single":
            return self.proj_down(self.act_fn(self.proj_up_gate(x)) * self.proj_up(x))
        gate, z = self.proj_up_gate_z(x).split(self.up_proj_dim, dim=-1)
        return self.proj_down(self.act_fn(gate) * z)


class ViLLayer(nn.Module):
    def __init__(self, dim, direction, expansion=2, qkv_block_size=4, proj_bias=True, norm_bias=True,
                 conv_bias=True, conv_kernel_size=3, conv_kind="2d", init_weights="original-fixed", seqlens=None,
                 num_blocks=15, gate_soft_cap=15.0, ffn_proj_factor=2.6667, ffn_round_up_to_multiple_of=64,
                 weight_mode="fused", chunk_size=64, flip_free=True):
        super().__init__()
        assert dim % qkv_block_size == 0, "dim must be divisible by qkv_block_size"
        if conv_kind != "2d":
            raise NotImplementedError("Only 2d convolution is implemented")
        assert conv_kernel_size % 2 == 1, "conv_kernel_size must be odd"
        self.dim = dim
        self.direction = direction
        self.expansion = expansion
        self.qkv_block_size = qkv_block_size
        self.gate_soft_cap = gate_soft_cap
        self.weight_mode = weight_mode
        self.num_blocks = num_blocks
        self.flip_free = flip_free
        self.fused_tail = True    # CUDA: csrc/mlstm_glue.cu for out-norm + skip + SiLU(z)
        self.fused_producer = True   # CUDA, bf16 / fp16 activations: csrc/mlstm_qkv.cu for conv + SiLU + q / k / v

        inner_dim = expansion * dim
        num_heads = inner_dim // qkv_block_size
        self.proj_up = nn.Linear(dim, 2 * inner_dim, bias=proj_bias)
        self.q_proj = LinearHeadwiseExpand(dim=inner_dim, num_heads=num_heads, bias=proj_bias)
        self.k_proj = LinearHeadwiseExpand(dim=inner_dim, num_heads=num_heads, bias=proj_bias)
        self.v_proj = LinearHeadwiseExpand(dim=inner_dim, num_heads=num_heads, bias=proj_bias)
        self.conv = SequenceConv2d(inner_dim, inner_dim, kernel_size=conv_kernel_size, padding=conv_kernel_size // 2,
                                   groups=inner_dim, bias=conv_bias, seqlens=seqlens)
        self.mlstm_cell = MatrixLSTMCell(dim=inner_dim, num_heads=num_heads, norm_bias=norm_bias, chunk_size=chunk_size)
        self.learnable_skip = nn.Parameter(torch.ones(inner_dim))
        self.proj_down = nn.Linear(inner_dim, dim, bias=proj_bias)
        self.norm = nn.RMSNorm(dim, eps=1e-6, elementwise_affine=norm_bias)
        self.ffn_norm = nn.RMSNorm(dim, eps=1e-6, elementwise_affine=norm_bias)
        self.ffn = FeedForward(embedding_dim=dim, ffn_proj_factor=ffn_proj_factor,
                               ffn_round_up_to_multiple_of=ffn_round_up_to_multiple_of, use_bias=proj_bias,
                               weight_mode=weight_mode, num_blocks=num_blocks or 1)
        self.reset_parameters()

    @property
    def backwards(self) -> bool:
        return self.direction == SequenceTraversal.ROWWISE_FROM_BOT_RIGHT

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """``(B, S, dim)`` -> ``(B, S, dim)``; token order is never physically reversed when flip_free."""
        anti = self.backwards and self.flip_free
        literal_flip = self.backwards and not self.flip_free
        y = self.norm(x)
        if literal_flip:
            y = y.flip(dims=[1])
        x_mlstm, z = self.proj_up(y).chunk(2, dim=-1)
        cell = self.mlstm_cell
        conv_act = None
        if (x.is_cuda and getattr(self, "fused_producer", True)
                and self.conv.kernel_size == (3, 3) and self.conv.padding == (1, 1) and self.conv.stride == (1, 1)
                and self.conv.dilation == (1, 1) and self.conv.groups == self.conv.in_channels == self.conv.out_channels):
            # conv + SiLU + the three block-diagonal projections as one kernel (vision_lstm2.py:482-491 are four
            # round trips over (B,S,inner)); bf16 outputs, which is what the cell kernels read
            from . import ops
            gh = _grid_height(x_mlstm.shape[1], self.conv.seqlens)
            gw = x_mlstm.shape[1] // gh
            if ops.qkv_supported(x_mlstm, x_mlstm.shape[2], self.q_proj.num_heads, gh, gw):
                conv_act, q, k, v = ops.qkv_producer(x_mlstm, self.conv.weight, self.conv.bias, self.q_proj.weight, self.q_proj.bias,
                                                     self.k_proj.weight, self.k_proj.bias, self.v_proj.weight, self.v_proj.bias,
                                                     gh, gw, rotate=anti)
        if conv_act is None:
            conv_act = F.silu(self.conv(x_mlstm, rotate=anti))
            q, k, v = self.q_proj(conv_act), self.k_proj(conv_act), self.v_proj(x_mlstm)
        y = None
        if x.is_cuda and getattr(self, "fused_tail", True) and not cell.raw_output:
            # out-norm + skip + SiLU(z) gate as one streaming kernel over the raw cell output
            # (vision_lstm2.py:950, :498-499 are four separate (B,S,inner) round trips).  Direction and output
            # form are call arguments: no module state is touched, so the forward is re-entrant.
            from . import ops
            h_raw = cell(q, k, v, reverse=anti, raw_output=True)                 # (B,NH,S,DH)
            # (each on its own: the producer already hands conv_act over in the cell's dtype, z keeps the autocast / model dtype)
            conv_act_k = conv_act if conv_act.dtype == h_raw.dtype else conv_act.to(h_raw.dtype)
            z_k = z if z.dtype == h_raw.dtype else z.to(h_raw.dtype)
            if ops.glue_supported(h_raw, conv_act_k, z_k):
                y = ops.layer_tail(h_raw, conv_act_k, z_k, cell.outnorm.weight, cell.outnorm.bias, self.learnable_skip,
                                   eps=cell.outnorm.eps)
            else:
                y = (cell.outnorm(h_raw).transpose(1, 2).reshape(x.shape[0], x.shape[1], -1)
                     + self.learnable_skip * conv_act) * F.silu(z)
        if y is None:
            h = cell(q, k, v, reverse=anti)
            y = (h + self.learnable_skip * conv_act) * F.silu(z)
        if y.dtype != self.proj_down.weight.dtype and not torch.is_autocast_enabled():
            y = y.to(self.proj_down.weight.dtype)   # model.half() inference around the bf16 kernels (engine/validator.py:117-119)
        y = self.proj_down(y)
        if literal_flip:
            y = y.flip(dims=[1])
        return x + y

    def reset_parameters(self):
        nn.init.xavier_uniform_(self.proj_up.weight)
        if self.proj_up.bias is not None:
            nn.init.zeros_(self.proj_up.bias)
        for proj in (self.q_proj, self.k_proj, self.v_proj):
            proj.reset_parameters()
        nn.init.xavier_uniform_(self.proj_down.weight)
        if self.proj_down.bias is not None:
            nn.init.zeros_(self.proj_down.bias)
        nn.init.ones_(self.learnable_skip)
        self.mlstm_cell.reset_parameters()
        self.norm.reset_parameters()
        self.ffn_norm.reset_parameters()


class ViLBlock(nn.Module):
    def __init__(self, dim, direction, drop_path=0.0, conv_kind="2d", conv_kernel_size=3, proj_bias=True,
                 norm_bias=True, seqlens=None, num_blocks=None, init_weights="original", chunk_size=256,
                 qkv_block_size=4):
        super().__init__()
        self.dim = dim
        self.direction = direction
        self.norm_bias = norm_bias
        self.drop_path = nn.Identity()           # reference: DropPath(drop_prob=0.0), never applied (:716,731)
        self.norm = nn.RMSNorm(dim, eps=1e-3)    # present in the state_dict, unused in forward (:728)
        # like the reference (:718-730) the inner layer gets fixed conv/bias settings and seqlens=None
        self.layer = ViLLayer(dim, direction, qkv_block_size=qkv_block_size, proj_bias=True, norm_bias=True,
                              conv_bias=True, conv_kernel_size=3, conv_kind="2d", init_weights="original",
                              seqlens=None, num_blocks=None, chunk_size=chunk_size)
        self.reset_parameters()

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        return self.layer(x)

    def reset_parameters(self):
        self.layer.reset_parameters()
        self.norm.reset_parameters()


class ViLBlockPair(nn.Module):
    head_compat = False   # True: return the top-left block's output only, as HEAD does (:1438-1441)

    def __init__(self, dim, drop_path=0.0, conv_kind="2d", conv_kernel_size=3, proj_bias=True, norm_bias=True,
                 seqlens=None, num_blocks=15, init_weights="original", chunk_size=256, qkv_block_size=4):
        super().__init__()
        common = dict(dim=dim, drop_path=drop_path, conv_kind=conv_kind, conv_kernel_size=conv_kernel_size,
                      proj_bias=proj_bias, norm_bias=norm_bias, seqlens=seqlens, num_blocks=num_blocks,
                      init_weights=init_weights, chunk_size=chunk_size, qkv_block_size=qkv_block_size)
        self.rowwise_from_top_left = ViLBlock(direction=SequenceTraversal.ROWWISE_FROM_TOP_LEFT, **common)
        self.rowwise_from_bot_right = ViLBlock(direction=SequenceTraversal.ROWWISE_FROM_BOT_RIGHT, **common)

    def forward(self, x: torch.Tensor, seqlens=None) -> torch.Tensor:
        out = self.rowwise_from_top_left(x)
        if self.head_compat:
            return out
        return self.rowwise_from_bot_right(out)
