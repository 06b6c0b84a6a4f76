"""CPU-side checks: the C-ABI library loads and exports every symbol the header declares, the
ctypes mirror matches the C struct layout, argument validation works without a GPU, and the
host-side mirrors of the reference interface (mLSTMBackend seam, MatrixLSTMCell) behave."""
import copy
import ctypes as C
import inspect
import itertools
import os
import pickle
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
from oracle import mlstm_oracle as O  # noqa: E402
from xlstm_yolo_b200 import MatrixLSTMCell, _lib, build, mLSTMBackend, mLSTMBackendConfig  # noqa: E402


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _lib.load()


def test_library_exports_every_declared_symbol(lib):
    hdr = open(os.path.join(ROOT, "include", "mlstm_b200.h")).read()
    declared = set(re.findall(r"\b(mlstm_b200_\w+)\s*\(", hdr))
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.mlstm_b200_abi_version() == _lib.ABI_VERSION


@pytest.mark.parametrize("cname,ctype", [("mlstm_params", _lib.Params), ("mlstm_gate_proj_params", _lib.GateProjParams),
                                         ("mlstm_glue_params", _lib.GlueParams), ("mlstm_qkv_params", _lib.QkvParams),
                                         ("mlstm_qkv_bwd_params", _lib.QkvBwdParams), ("mlstm_conv_bwd_params", _lib.ConvBwdParams)])
def test_ctypes_struct_matches_c_layout(tmp_path, cname, ctype):
    fields = [n for n, _ in ctype._fields_]
    src = tmp_path / "layout.c"
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{ROOT}/include/mlstm_b200.h"', "int main(void){",
             f'printf("%zu\\n", sizeof({cname}));']
    lines += [f'printf("%zu\\n", offsetof({cname}, {f}));' for f in fields]
    lines += ["return 0;}"]
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-o", str(exe), str(src)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    assert int(out[0]) == C.sizeof(ctype)
    for f, off in zip(fields, out[1:]):
        assert getattr(ctype, f).offset == int(off), f


def test_gate_projection_validation_needs_no_gpu(lib):
    g = _lib.GateProjParams()
    assert lib.mlstm_b200_gates_fwd(None, None) == -1
    g.abi_version, g.T, g.D, g.NH, g.dtype, g.ld = _lib.ABI_VERSION, 16, 60, 4, _lib.MLSTM_BF16, 60
    assert lib.mlstm_b200_gates_fwd(C.byref(g), None) == -2 and b"multiples of 8" in lib.mlstm_b200_last_error()
    g.D = g.ld = 64
    assert lib.mlstm_b200_gates_fwd(C.byref(g), None) == -1          # null pointers
    assert lib.mlstm_b200_gates_workspace_bytes(C.byref(g)) == 4 * 1 * (8 * 192 + 8)   # one token range of 16
    g.T = 51200
    slabs = 1
    assert lib.mlstm_b200_gates_workspace_bytes(C.byref(g)) == 4 * (4 * 148 // slabs) * (8 * 192 + 8)
    g.T = 0
    assert lib.mlstm_b200_gates_fwd(C.byref(g), None) == 0           # empty input: nothing to do


def _params(**kw):
    p = _lib.Params()
    p.abi_version = _lib.ABI_VERSION
    p.B, p.NH, p.S, p.DHQK, p.DHV = 2, 2, 64, 64, 64
    p.dtype = _lib.MLSTM_BF16
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def test_validation_errors_need_no_gpu(lib):
    assert lib.mlstm_b200_fwd(None, None) == -1
    p = _params()
    assert lib.mlstm_b200_fwd(C.byref(p), None) == -1 and b"null" in lib.mlstm_b200_last_error()
    p = _params(abi_version=99)
    assert lib.mlstm_b200_fwd(C.byref(p), None) == -1 and b"abi_version" in lib.mlstm_b200_last_error()
    p = _params(dtype=7)
    assert lib.mlstm_b200_fwd(C.byref(p), None) == -2
    p = _params(DHQK=0)
    assert lib.mlstm_b200_bwd(C.byref(p), None) == -1
    # empty inputs are a successful no-op
    p = _params(S=0)
    assert lib.mlstm_b200_fwd(C.byref(p), None) == 0
    p = _params(B=0)
    assert lib.mlstm_b200_bwd(C.byref(p), None) == 0


def test_kernel_family_and_workspace(lib):
    p = _params()
    assert lib.mlstm_b200_kernel_name(C.byref(p), 0) == b"tcgen05"
    rows, items = 2 * 2 * 64, 2 * 2 * 1
    assert lib.mlstm_b200_workspace_bytes(C.byref(p), 1) >= 9 * 4 * rows + items * (64 * 64 * 2 + 64 * 4)   # dn, R/K partials, dCs, dns
    assert lib.mlstm_b200_workspace_bytes(C.byref(p), 0) == 0
    assert lib.mlstm_b200_state_bytes(C.byref(p)) == 0   # forward-only call (no saved rows): the single-pass forward keeps its states on chip
    p.n_row = p.m_row = 0x1000                             # a backward will follow
    assert lib.mlstm_b200_state_bytes(C.byref(p)) >= 2 * 2 * 1 * (64 * 64 * 2 + 64 * 4 + 4)   # per-chunk entry states
    p = _params(DHQK=8, DHV=8)
    assert lib.mlstm_b200_kernel_name(C.byref(p), 0) == b"simt"
    assert lib.mlstm_b200_state_bytes(C.byref(p)) == 0
    p = _params(dtype=_lib.MLSTM_F32, DHQK=16, DHV=16)
    assert lib.mlstm_b200_kernel_name(C.byref(p), 0) == b"simt"
    p = _params(dtype=_lib.MLSTM_F32, DHQK=128, DHV=128)
    assert lib.mlstm_b200_kernel_name(C.byref(p), 0) == b"simt"
    p = _params(DHQK=256, DHV=256)   # bf16: the slice-streaming tcgen05 family (mlstm_tc_256.cu), always chunk-parallel
    assert lib.mlstm_b200_kernel_name(C.byref(p), 0) == b"tcgen05"
    assert lib.mlstm_b200_kernel_variant(C.byref(p), 0) == b"two_phase" and lib.mlstm_b200_kernel_variant(C.byref(p), 1) == b"chunk_parallel"
    assert lib.mlstm_b200_state_bytes(C.byref(p)) >= items * (256 * 256 * 2 + 256 * 4 + 4)
    assert lib.mlstm_b200_workspace_bytes(C.byref(p), 1) >= 4 * rows * (1 + 2 * 8) + items * (256 * 256 * 2 + 256 * 4 + 4 * 4)
    p = _params(dtype=_lib.MLSTM_F32, DHQK=256, DHV=256)   # fp32: value-sliced SIMT kernels: dn per slice + R + fp32 dq/dk accumulators
    assert lib.mlstm_b200_kernel_name(C.byref(p), 0) == b"simt"
    assert lib.mlstm_b200_workspace_bytes(C.byref(p), 1) == 4 * (rows * 5 + 2 * rows * 256)
    # bf16 head dims the tcgen05 kernels are not written for — DHqk != DHv (mLSTMLayerVision's qk_dim_factor = 0.5), DH = 16
    # (the reference's default qkv_block_size), 32, 192 — run them zero-padded to 64 / 128 / 256 (mlstm_api.cu): the padded
    # q, k, v, h and initial / last states ride behind the chunk states, padded dh, dq, dk, dv behind the workspace
    p = _params(DHQK=64, DHV=128)
    assert lib.mlstm_b200_kernel_name(C.byref(p), 0) == b"tcgen05"
    assert lib.mlstm_b200_kernel_variant(C.byref(p), 0) in (b"single_pass", b"two_phase")
    sq = _params(DHQK=128, DHV=128)
    st_extra = 2 * (2 * 2 * 128 * 128 * 4) + 2 * (2 * 2 * 128 * 4)       # padded initial / last C and n
    # padded width 64 / 128: the kernels run on the caller's narrow tensors (TMA supplies the zero columns): no room for copies
    assert lib.mlstm_b200_state_bytes(C.byref(p)) >= lib.mlstm_b200_state_bytes(C.byref(sq)) + st_extra
    assert lib.mlstm_b200_state_bytes(C.byref(p)) < lib.mlstm_b200_state_bytes(C.byref(sq)) + st_extra + 2 * 64 * 2 * 128 * 2
    assert lib.mlstm_b200_workspace_bytes(C.byref(p), 1) < lib.mlstm_b200_workspace_bytes(C.byref(sq), 1) + 1024
    for dk, dv in ((16, 16), (32, 32), (192, 192), (128, 64), (24, 40)):
        assert lib.mlstm_b200_kernel_name(C.byref(_params(DHQK=dk, DHV=dv)), 0) == b"tcgen05", (dk, dv)
    # padded width 256 (the slice-streaming family reads rows with plain loads): four padded copies on either side
    w, sq = _params(DHQK=192, DHV=192), _params(DHQK=256, DHV=256)
    w.n_row = w.m_row = sq.n_row = sq.m_row = 0x1000
    act = 2 * 64 * 2 * 256 * 2                                           # B S NH DP bf16
    assert lib.mlstm_b200_state_bytes(C.byref(w)) >= lib.mlstm_b200_state_bytes(C.byref(sq)) + 4 * act
    assert lib.mlstm_b200_workspace_bytes(C.byref(w), 1) >= lib.mlstm_b200_workspace_bytes(C.byref(sq), 1) + 4 * act
    assert lib.mlstm_b200_kernel_name(C.byref(_params(DHQK=20, DHV=64)), 0) == b"simt"      # rows must be 16-byte multiples
    assert lib.mlstm_b200_kernel_name(C.byref(_params(DHQK=264, DHV=264)), 0) is None       # nothing to pad to, too wide for SIMT
    assert lib.mlstm_b200_kernel_name(C.byref(_params(dtype=_lib.MLSTM_F32, DHQK=64, DHV=128)), 0) == b"simt"
    p = _params(DHQK=512, DHV=512)
    assert lib.mlstm_b200_kernel_name(C.byref(p), 0) is None
    assert lib.mlstm_b200_kernel_variant(C.byref(p), 1) is None
    assert lib.mlstm_b200_kernel_variant(C.byref(_params()), 0) in (b"single_pass", b"two_phase")
    # The dispatch table of the tensor-core family (the host library sees no device, so it sizes for 148 SMs): the forward
    # is two-phase for head dim 256, and otherwise when 2 B NH <= 148 with >= 4 chunks; the backward is the fused walk iff
    # the (padded) head dim is 64 or 128 and 2 B NH > 148.  The states buffer holds the chunk states unless a single-pass
    # forward is called without saved rows; a padded head dim adds the padded initial / last states and, at DP = 256, the
    # padded copies of q, k, v, h.
    al = lambda x: (x + 255) & ~255
    for (B, NH), S, DH in itertools.product([(1, 4), (8, 4), (37, 2), (32, 4), (75, 1)], [64, 384, 512, 1600],
                                            [64, 128, 256, 16, 192]):
        DP = 64 if DH <= 64 else (128 if DH <= 128 else 256)
        two_phase = DP == 256 or (2 * B * NH <= 148 and S > 3 * 128)
        fused = DP != 256 and 2 * B * NH > 148
        items = B * NH * -(-S // 128)
        for n_row in (None, 0x1000):
            p = _params(B=B, NH=NH, S=S, DHQK=DH, DHV=DH)
            p.n_row = p.m_row = n_row
            assert lib.mlstm_b200_kernel_variant(C.byref(p), 0) == (b"two_phase" if two_phase else b"single_pass")
            assert lib.mlstm_b200_kernel_variant(C.byref(p), 1) == (b"fused_walk" if fused else b"chunk_parallel")
            states = al(items * (DP * DP * 2 + DP * 4 + 4)) if two_phase or n_row else 0
            if DP != DH:
                states += (4 * al(B * S * NH * DP * 2) if DP == 256 else 0) + 2 * al(B * NH * DP * DP * 4) + 2 * al(B * NH * DP * 4)
            assert lib.mlstm_b200_state_bytes(C.byref(p)) == states, (B, NH, S, DH, n_row)


def test_layer_tail_validation_needs_no_gpu(lib):
    g = _lib.GlueParams()
    assert lib.mlstm_b200_glue_fwd(None, None) == -1
    g.abi_version, g.T, g.D, g.NH, g.dtype, g.eps = _lib.ABI_VERSION, 64, 192, 4, _lib.MLSTM_BF16, 1e-3
    assert lib.mlstm_b200_glue_fwd(C.byref(g), None) == -2 and b"multiple of 256" in lib.mlstm_b200_last_error()
    g.D = 512
    g.ld_h = g.ld_c = g.ld_y = 512
    g.ld_z = 1024
    assert lib.mlstm_b200_glue_fwd(C.byref(g), None) == -1          # null pointers
    assert lib.mlstm_b200_glue_workspace_bytes(C.byref(g)) == 4 * 3 * 512 * 4   # 128 (token, segment) units / 32 per CTA
    g.T = 0
    assert lib.mlstm_b200_glue_fwd(C.byref(g), None) == 0


def test_operand_producer_validation_needs_no_gpu(lib):
    """Shape gates, error codes and workspace sizes of the producer entry points (ABI 5) without a device."""
    assert lib.mlstm_b200_qkv_supported(512, 4, 40, 40, 1024) == 1 and lib.mlstm_b200_qkv_supported(256, 4, 20, 20, 256) == 1
    assert lib.mlstm_b200_qkv_supported(512, 4, 100, 100, 1024) == 0      # grid wider than the staged halo
    assert lib.mlstm_b200_qkv_supported(64, 4, 20, 20, 64) == 0           # block size 16
    assert lib.mlstm_b200_qkv_supported(512, 4, 40, 40, 1020) == 0        # row stride not a multiple of 8
    q = _lib.QkvParams()
    assert lib.mlstm_b200_qkv_fwd(None, None) == -1
    q.abi_version, q.B, q.GH, q.GW, q.D, q.NH, q.ld_x = _lib.ABI_VERSION, 2, 20, 20, 64, 4, 64
    assert lib.mlstm_b200_qkv_fwd(C.byref(q), None) == -2 and b"64 or 128" in lib.mlstm_b200_last_error()
    q.D = q.ld_x = 256
    assert lib.mlstm_b200_qkv_fwd(C.byref(q), None) == -1                 # null pointers
    q.B = 0
    assert lib.mlstm_b200_qkv_fwd(C.byref(q), None) == 0                  # empty batch: nothing to do
    q.abi_version = 4
    assert lib.mlstm_b200_qkv_fwd(C.byref(q), None) == -1 and b"abi_version" in lib.mlstm_b200_last_error()
    b = _lib.QkvBwdParams()
    b.abi_version, b.T, b.D, b.NH, b.ld_x = _lib.ABI_VERSION, 51200, 512, 4, 1024
    # 37 CTAs per block (148 / 4), per CTA three d x d fp32 weight-gradient partials + three bias rows
    assert lib.mlstm_b200_qkv_bwd_workspace_bytes(C.byref(b)) == 4 * 37 * 4 * (3 * 128 * 128 + 3 * 128)
    assert lib.mlstm_b200_qkv_bwd(C.byref(b), None) == -1                 # null pointers
    b.T = 100
    assert lib.mlstm_b200_qkv_bwd_workspace_bytes(C.byref(b)) == 4 * 1 * 4 * (3 * 128 * 128 + 3 * 128)   # one tile: one CTA per block
    c = _lib.ConvBwdParams()
    c.abi_version, c.B, c.GH, c.GW, c.D, c.NH, c.ld_x = _lib.ABI_VERSION, 32, 40, 40, 512, 4, 1024
    assert lib.mlstm_b200_conv_bwd_workspace_bytes(C.byref(c)) == 4 * 37 * 4 * 10 * 128
    assert lib.mlstm_b200_conv_bwd(C.byref(c), None) == -1
    c.GW = 128
    assert lib.mlstm_b200_conv_bwd(C.byref(c), None) == -2
    assert lib.mlstm_b200_colsum_workspace_bytes(512, 3) == 4 * 296 * 3 * 512
    assert lib.mlstm_b200_colsum(None, 3, 10, 512, 512, None, None, 0, None) == -1


def test_cuda_op_refuses_cpu_tensors():
    from xlstm_yolo_b200 import ops
    x = torch.randn(1, 2, 8, 16)
    g = torch.randn(1, 2, 8)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.mlstm(x, x, x, g, g)


# ---- MatrixLSTMCell drop-in contract (reference: vision_lstm2.py:802-966) ---------------------

def test_cell_constructor_signature_matches_reference():
    sig = inspect.signature(MatrixLSTMCell.__init__)
    names = list(sig.parameters)[1:8]
    assert names == ["dim", "num_heads", "norm_bias", "eps", "chunk_size", "use_autocast", "autocast_dtype"]
    d = {k: v.default for k, v in sig.parameters.items()}
    assert d["norm_bias"] is True and d["eps"] == 1e-6 and d["chunk_size"] == 16 and d["use_autocast"] is True
    assert d["autocast_dtype"] == torch.bfloat16
    fwd = inspect.signature(MatrixLSTMCell.forward).parameters
    assert list(fwd)[:4] == ["self", "q", "k", "v"]                 # the reference's positional signature (vision_lstm2.py:882)
    # anything beyond it is keyword-only with a default: per-call overrides instead of mutated module state
    assert all(p.kind is inspect.Parameter.KEYWORD_ONLY and p.default is None for p in list(fwd.values())[4:])


def test_cell_state_dict_and_init():
    cell = MatrixLSTMCell(dim=256, num_heads=4)
    sd = cell.state_dict()
    assert {k: tuple(v.shape) for k, v in sd.items()} == {
        "igate.weight": (4, 768), "igate.bias": (4,), "fgate.weight": (4, 768), "fgate.bias": (4,),
        "outnorm.weight": (256,), "outnorm.bias": (256,)}
    assert torch.all(sd["igate.weight"] == 0) and torch.all(sd["fgate.weight"] == 0)
    assert torch.all(sd["igate.bias"] == -10)                      # vision_lstm2.py:965
    assert torch.allclose(sd["fgate.bias"], torch.tensor([3.0, 4.0, 5.0, 6.0]))   # :962
    assert torch.all(sd["outnorm.weight"] == 0) and cell.outnorm.eps == 1e-3       # :812
    assert "outnorm.bias" not in MatrixLSTMCell(dim=64, num_heads=4, norm_bias=False).state_dict()
    # no persistent buffers, survives pickle / deepcopy / half / float (EMA + checkpoints)
    assert len(list(cell.buffers())) == 0
    c2 = pickle.loads(pickle.dumps(cell))
    c3 = copy.deepcopy(cell).half().float()
    for k in sd:
        assert torch.equal(c2.state_dict()[k], sd[k]) and torch.allclose(c3.state_dict()[k], sd[k], atol=1e-2)


@pytest.mark.parametrize("reverse", [False, True])
def test_cell_cpu_forward_matches_oracle(reverse):
    torch.manual_seed(0)
    cell = MatrixLSTMCell(dim=64, num_heads=4, chunk_size=16, reverse=reverse)
    with torch.no_grad():
        cell.igate.weight.normal_(0, 0.05)
        cell.fgate.weight.normal_(0, 0.05)
        cell.igate.bias.fill_(0.0)
        cell.outnorm.weight.normal_(0, 0.1)
    q, k, v = (torch.randn(2, 50, 64) for _ in range(3))
    y = cell(q, k, v)
    want = O.cell_forward(q, k, v, 4, cell.igate.weight, cell.igate.bias, cell.fgate.weight, cell.fgate.bias,
                          cell.outnorm.weight, cell.outnorm.bias, chunk_size=16, eps=5e-5, reverse=reverse)
    assert y.shape == (2, 50, 64)
    assert (y - want).abs().max() < 1e-4
    y.square().mean().backward()
    assert cell.igate.weight.grad.abs().sum() > 0 and cell.fgate.bias.grad.abs().sum() > 0
    # HEAD's raw (B,NH,S,DH) output is still reachable
    assert MatrixLSTMCell(dim=64, num_heads=4, raw_output=True)(q, k, v).shape == (2, 4, 50, 16)


def test_backend_seam_cpu():
    g = torch.Generator().manual_seed(1)
    q, k, v = (torch.randn(2, 3, 40, 8, generator=g) for _ in range(3))
    i, f = torch.randn(2, 3, 40, generator=g), 3 + torch.randn(2, 3, 40, generator=g)
    # the kernel string HEAD configures on CUDA names the sigmoid-input-gate arithmetic (vision_lstm2.py:835)
    sig = mLSTMBackend(mLSTMBackendConfig(chunkwise_kernel="chunkwise--triton_xl_chunk_siging", sequence_kernel="native_sequence__triton",
                                          step_kernel="triton", chunk_size=16, autocast_kernel_dtype="bfloat16",
                                          return_last_states=False, mode="train", eps=5e-5))
    assert sig.input_gate == "sigmoid"
    assert (sig(q=q, k=k, v=v, i=i, f=f) - O.mlstm_siging_parallel(q, k, v, i, f, eps=5e-5)).abs().max() < 1e-5
    C0s, n0s = torch.randn(2, 3, 8, 8, generator=g), torch.randn(2, 3, 8, generator=g)
    hs, (Cs, ns, ms) = sig(q, k, v, i, f, c_initial=C0s, n_initial=n0s, return_last_states=True)
    ws_, (Cws, nws, _) = O.mlstm_siging_recurrent(q, k, v, i, f, C0s, n0s, eps=5e-5, return_last_states=True)
    assert (hs - ws_).abs().max() < 1e-5 and (Cs - Cws).abs().max() < 1e-4 and (ns - nws).abs().max() < 1e-4 and ms.abs().max() == 0
    # the kernel string of the reference's CPU path: exponential input gate
    be = mLSTMBackend(mLSTMBackendConfig(chunkwise_kernel="chunkwise--native_autograd", sequence_kernel="native_sequence__native",
                                         step_kernel="native", chunk_size=16, autocast_kernel_dtype="bfloat16",
                                         return_last_states=False, mode="train", eps=5e-5))
    assert be.input_gate == "exp"
    h = be(q=q, k=k, v=v, i=i, f=f)
    want = O.mlstm_chunkwise(q, k, v, i, f, chunk_size=16, eps=5e-5)
    assert (h - want).abs().max() < 1e-5
    C0, n0, m0 = torch.randn(2, 3, 8, 8, generator=g), torch.randn(2, 3, 8, generator=g), torch.randn(2, 3, 1, generator=g)
    h2, (C1, n1, m1) = be(q, k, v, i, f, c_initial=C0, n_initial=n0, m_initial=m0, return_last_states=True, mode="inference")
    w2, (Cw, nw, mw) = O.mlstm_chunkwise(q, k, v, i, f, C0, n0, m0, chunk_size=16, eps=5e-5, return_last_states=True)
    assert (h2 - w2).abs().max() < 1e-5 and (C1 - Cw).abs().max() < 1e-4 and (m1 - mw).abs().max() < 1e-5
    assert be.config.mode == "train"          # read by mlstm_large.py:305-306
    with pytest.raises(ValueError):
        be(q, k, v, i[:, :, :-1], f)
    with pytest.raises(ValueError):
        mLSTMBackendConfig(mode="nope")


def test_mlstm_kernels_shim_exports_what_the_reference_imports():
    from xlstm_yolo_b200 import compat
    compat.install()
    from mlstm_kernels.torch.backend_module import (BackendModeType, ChunkwiseKernelType, DtypeType,  # noqa: F401
                                                    SequenceKernelType, StepKernelType, mLSTMBackend as B2,
                                                    mLSTMBackendConfig as C2)
    from mlstm_kernels.torch.chunkwise.triton_xl_chunk import mlstm_chunkwise__xl_chunk  # noqa: F401
    assert B2 is mLSTMBackend and C2 is mLSTMBackendConfig


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "xlstm_yolo_b200")
    for dirpath, _, files in os.walk(pkg):
        for fn in files:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dirpath, fn)).read()
                assert "import oracle" not in txt and "from oracle" not in txt, fn


def test_three_way_bf16_split_reproduces_fp32_weights():
    """Numerics claim of the tensor-core gate forward (csrc/mlstm_gates_tc.cu): an fp32 weight split as hi = bf16(w),
    mid = bf16(w - hi), lo = bf16(w - hi - mid) is recovered by hi + mid + lo to fp32 rounding (each part carries 8 significant
    bits, three of them cover the 24 of fp32), so one N = 3 x outputs MMA with fp32 accumulation computes the fp32-weight product."""
    import torch
    g = torch.Generator().manual_seed(0)
    w = torch.randn(1 << 16, generator=g) * torch.logspace(-6, 3, 1 << 16)
    hi = w.bfloat16().float()
    mid = (w - hi).bfloat16().float()
    lo = (w - hi - mid).bfloat16().float()
    rec = hi.double() + mid.double() + lo.double()
    assert float(((rec - w.double()).abs() / w.double().abs().clamp_min(1e-30)).max()) <= 2.0 ** -23
    two = hi.double() + mid.double()     # two parts only: ~2^-16, the reason the third row block exists
    assert float(((two - w.double()).abs() / w.double().abs().clamp_min(1e-30)).max()) > 2.0 ** -18
