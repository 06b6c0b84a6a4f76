"""Every kernel variant against the oracle: the parity sweep of test_gpu_parity.py re-run in a child
process with the dispatch pinned (MLSTM_FORCE_VARIANT is read once per process): single-pass or two-phase forward
(first digit 1 / 2) with the chunk-parallel or the fused single-walk backward (second digit 2 / 3; DH = 256 has no fused
walk and falls through to the chunk-parallel kernels), whatever the shape would pick — the oracle cases are small
batches, which the automatic dispatch would never send to the wide-batch kernels the bench runs."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["12", "22", "13", "23"])
def test_parity_sweep_with_pinned_variant(variant):
    env = dict(os.environ, MLSTM_FORCE_VARIANT=variant)
    select = "(test_cuda_matches_oracle or test_initial_and_last_states or sigmoid_input_gate)"
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.join(ROOT, "tests", "test_gpu_parity.py"), "-m", "gpu", "-q",
                        "-x", "-k", select, "-p", "no:cacheprovider"],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]


@pytest.mark.gpu
@pytest.mark.parametrize("B,NH,S,DH,reverse", [(8, 4, 1600, 128, False), (2, 4, 1000, 64, True), (3, 2, 700, 128, False)])
def test_whole_backward_call_matches_the_two_parts(B, NH, S, DH, reverse):
    """With 2*B*NH <= #SM the whole-backward call runs the adjoint-state walk and the dq kernel in ONE launch
    (tc_bwd_sa_kernel, dn from tc_dn_kernel; csrc/mlstm_tc_bwd.cu) while `mlstm_b200_bwd_part(0)` + `(1)` launch them one
    after the other.  Same arithmetic up to the summation order of dn_t = dnf_t (dh_t . h_t): dq is bit-identical (kernel A
    keeps its own dn), the rest agrees to fp32 rounding; the merged call is deterministic."""
    import torch
    from xlstm_yolo_b200 import ops
    g = torch.Generator().manual_seed(11)
    def act():
        return (torch.randn(B, S, NH, DH, generator=g) * 0.5).to(torch.bfloat16).cuda().transpose(1, 2)
    q, k, v, dh = act(), act(), act(), act()
    i = torch.randn(B, S, NH, generator=g).cuda().transpose(1, 2)
    f = (torch.randn(B, S, NH, generator=g) + 3.0).cuda().transpose(1, 2)
    pl = ops.MLSTMPlan(q, k, v, i, f, dh, chunk_size=64, reverse=reverse)
    if pl.variant_bwd != "chunk_parallel":
        pytest.skip(f"dispatch picked {pl.variant_bwd}")
    pl.forward()
    pl.backward(0)
    pl.backward(1)
    torch.cuda.synchronize()
    parts = [t.clone() for t in (pl.dq, pl.dk, pl.dv, pl.di, pl.df)]
    pl.backward()
    torch.cuda.synchronize()
    whole = [t.clone() for t in (pl.dq, pl.dk, pl.dv, pl.di, pl.df)]
    pl.backward()
    torch.cuda.synchronize()
    assert torch.equal(whole[0], parts[0])
    for a, b_ in zip(whole[1:], parts[1:]):
        scale = float(b_.float().abs().max())
        # bf16 outputs: one ulp of the largest element; di / df (fp32): R - K cancels, so dn's last-bit differences show up
        # amplified — between 1e-5 and 1e-3 of the largest element on these cases, against the 2e-2 the oracle comparison allows
        tol = 1e-2 if a.dtype == torch.bfloat16 else 1e-3
        err = float((a.float() - b_.float()).abs().max())
        assert err <= tol * scale, (err, scale)
    for a, t in zip(whole, (pl.dq, pl.dk, pl.dv, pl.di, pl.df)):
        assert torch.equal(a, t)
