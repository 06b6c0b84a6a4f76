"""The l and x detector scales without a GPU: the layer-tail and gate-projection shape rules at their inner dims, the
workspace sizes the library reports for them, and the two YAMLs."""
import ctypes as C
import os
import re
import subprocess
import sys

import pytest
import yaml

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
YAMLS = os.path.join(ROOT, "xlstm_yolo_b200", "compat", "yamls")


@pytest.fixture(scope="module")
def lib():
    from xlstm_yolo_b200 import _lib
    try:
        return _lib.load()
    except _lib.LibraryMissing as e:
        pytest.skip(str(e))


@pytest.mark.parametrize("D", [256, 512, 768, 1024, 1280, 1536, 1792, 2048])
@pytest.mark.parametrize("DH", [64, 128])
def test_layer_tail_takes_every_multiple_of_256_up_to_2048(lib, D, DH):
    assert lib.mlstm_b200_glue_supported(D, D // DH) == 1


@pytest.mark.parametrize("D,NH", [(640, 5), (640, 10), (2304, 18), (2304, 9)])
def test_layer_tail_refuses_other_widths(lib, D, NH):
    assert lib.mlstm_b200_glue_supported(D, NH) == 0


def _glue_grid(T, D):
    """The backward's CTA count: (8 // nseg) * nseg warps per CTA, >= 4 (token, segment) units per warp, <= 296 CTAs."""
    nseg = D // 256
    wpc = (8 // nseg) * nseg
    return max(1, min(296, -(-T * nseg // (wpc * 4))))


@pytest.mark.parametrize("D", [256, 768, 1280, 1536, 1792, 2048])
@pytest.mark.parametrize("T", [1, 37, 3200, 51200])
def test_layer_tail_workspace_follows_the_cta_size(lib, D, T):
    from xlstm_yolo_b200 import _lib
    g = _lib.GlueParams()
    g.abi_version, g.T, g.D, g.NH = _lib.ABI_VERSION, T, D, D // 128
    assert lib.mlstm_b200_glue_workspace_bytes(C.byref(g)) == 4 * 3 * D * _glue_grid(T, D)


def test_layer_tail_validation_accepts_the_new_widths(lib):
    """Past the shape rule, a forward at D 1536 stops at its NULL pointers; D 2304 stops at the shape rule."""
    from xlstm_yolo_b200 import _lib
    g = _lib.GlueParams()
    g.abi_version, g.T, g.NH, g.dtype = _lib.ABI_VERSION, 16, 12, 1
    g.ld_h = g.ld_c = g.ld_z = g.ld_y = 1536
    g.D = 1536
    assert lib.mlstm_b200_glue_fwd(C.byref(g), None) == -1
    g.D, g.NH = 2304, 18
    g.ld_h = g.ld_c = g.ld_z = g.ld_y = 2304
    assert lib.mlstm_b200_glue_fwd(C.byref(g), None) == -2 and b"multiple of 256" in lib.mlstm_b200_last_error()


def _gate_params(T, D, NH, dtype=1, addr=1 << 20):
    from xlstm_yolo_b200 import _lib
    g = _lib.GateProjParams()
    g.abi_version, g.T, g.D, g.NH, g.dtype, g.ld = _lib.ABI_VERSION, T, D, NH, dtype, D
    g.q, g.k, g.v = addr, addr, addr
    return g


@pytest.mark.parametrize("D,NH,rows", [(512, 8, 48), (1024, 4, 32), (1024, 8, 48), (1536, 12, 96), (2048, 16, 96),
                                       (512, 12, 96)])
def test_gate_forward_workspace_holds_the_streamed_split_weights(lib, D, NH, rows):
    """bf16 tensor-core forward whose split B operand does not fit in shared memory: (3 D / 64) slices of [rows][64] bf16,
    rows = hi | mid | lo of 8, 16 or 32 padded outputs."""
    assert lib.mlstm_b200_gates_fwd_workspace_bytes(C.byref(_gate_params(1000, D, NH))) == (3 * D // 64) * rows * 128


@pytest.mark.parametrize("D,NH", [(256, 4), (512, 4), (256, 8), (128, 6), (64, 8), (128, 12)])
def test_gate_forward_with_resident_weights_needs_no_workspace(lib, D, NH):
    """The shapes whose split weights fit in shared memory (among them every shape the tensor cores took at ABI 5) run
    with no workspace, as before."""
    assert lib.mlstm_b200_gates_fwd_workspace_bytes(C.byref(_gate_params(1000, D, NH))) == 0


@pytest.mark.parametrize("case", ["fp32", "33 outputs", "D % 64", "unaligned", "empty", "D > 2133", "ld < D"])
def test_gate_forward_on_simt_or_refused_needs_no_workspace(lib, case):
    g = {"fp32": lambda: _gate_params(1000, 1536, 12, dtype=0), "33 outputs": lambda: _gate_params(1000, 512, 32),
         "D % 64": lambda: _gate_params(1000, 520, 4), "unaligned": lambda: _gate_params(1000, 1536, 12, addr=(1 << 20) + 8),
         "empty": lambda: _gate_params(0, 1536, 12), "D > 2133": lambda: _gate_params(1000, 2176, 4),
         "ld < D": lambda: _gate_params(1000, 1536, 12)}[case]()
    if case == "ld < D":
        g.ld = 1024
    assert lib.mlstm_b200_gates_fwd_workspace_bytes(C.byref(g)) == 0


def test_gate_forward_refuses_an_abi5_caller(lib):
    """ABI 6 added the forward workspace: a caller built for ABI 5 (no workspace) is refused by the version check."""
    from xlstm_yolo_b200 import _lib
    assert _lib.ABI_VERSION == 6 and lib.mlstm_b200_abi_version() == 6
    g = _gate_params(1000, 1536, 12)
    wi = (C.c_float * 1)()
    g.w_i = g.w_f = g.i = g.f = C.cast(wi, C.c_void_p).value
    g.abi_version = 5
    assert lib.mlstm_b200_gates_fwd(C.byref(g), None) == -1 and b"ABI version" in lib.mlstm_b200_last_error()


def test_gate_forward_refuses_a_missing_workspace(lib):
    from xlstm_yolo_b200 import _lib
    g = _gate_params(1000, 1536, 12)
    wi = (C.c_float * 1)()
    g.w_i = g.w_f = C.cast(wi, C.c_void_p).value
    g.i = g.f = C.cast(wi, C.c_void_p).value
    assert lib.mlstm_b200_gates_fwd(C.byref(g), None) == -3 and b"workspace" in lib.mlstm_b200_last_error()


def _vil_rows(scale):
    cfg = yaml.safe_load(open(os.path.join(YAMLS, f"xlstm-yolo-{scale}.yaml")))
    text = open(os.path.join(YAMLS, f"xlstm-yolo-{scale}.yaml")).read().splitlines()
    rows = [(row, next(l for l in text if "ViLFusionBlock" in l and f"seqlens: {row[3][2]['seqlens']}".replace("'", "") in l))
            for row in cfg["backbone"] if row[2] == "ViLFusionBlock"]
    return cfg, rows


@pytest.mark.parametrize("scale,hidden,S", [("l", 512, (1600, 400)), ("x", 768, (1600, 400))])
def test_scale_yamls_state_their_vil_shapes(scale, hidden, S):
    cfg, rows = _vil_rows(scale)
    assert set(cfg["scales"]) == {"n", "s", "m", "l", "x"}
    assert cfg["scales"]["l"] == [1.00, 1.00, 512] and cfg["scales"]["x"] == [1.00, 1.50, 512]
    assert len(rows) == 2
    for (row, line), s in zip(rows, S):
        c_in, hid, kw = row[3]
        assert c_in == hid == hidden and kw["qkv_block_size"] == 128
        assert kw["seqlens"][0] * kw["seqlens"][1] == s
        inner, DH = 2 * hid, kw["qkv_block_size"]
        m = re.search(r"S=(\d+) at 640\^2, inner (\d+), NH (\d+), DH (\d+)", line)
        assert m and [int(v) for v in m.groups()] == [s, inner, inner // DH, DH], line


def test_vil_widths_follow_the_scale_table():
    """The ViL rows carry min(c, max_channels) * width of the Conv that feeds them, for every scale."""
    for scale in ("n", "s", "m", "l", "x"):
        cfg = yaml.safe_load(open(os.path.join(YAMLS, f"xlstm-yolo-{scale}.yaml")))
        _, width, max_ch = cfg["scales"][scale]
        bb = cfg["backbone"]
        for i, row in enumerate(bb):
            if row[2] == "ViLFusionBlock":
                conv_c = bb[i - 1][3][0]
                assert row[3][0] == row[3][1] == int(min(conv_c, max_ch) * width), (scale, i)


@pytest.mark.skipif(not os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "ultralytics")),
                    reason="baseline/_ref (the reference tree) not present")
@pytest.mark.parametrize("scale", ["l", "x"])
def test_reference_parse_model_builds_the_scale(scale, tmp_path):
    code = f"""
import os, sys, yaml
sys.path.insert(0, {ROOT!r})
from xlstm_yolo_b200.compat import reference_loader as RL
RL.import_reference(os.path.join({ROOT!r}, "baseline", "_ref"))
from ultralytics.nn.tasks import DetectionModel
cfg = yaml.safe_load(open(os.path.join({YAMLS!r}, "xlstm-yolo-{scale}.yaml")))
cfg["scale"] = "{scale}"
m = DetectionModel(cfg, ch=3, nc=80, verbose=False)
print("VIL", sorted({{type(x).__name__ for x in m.modules() if "ViL" in type(x).__name__}}))
"""
    env = dict(os.environ, YOLO_CONFIG_DIR=str(tmp_path))
    r = subprocess.run([sys.executable, "-c", code], cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    assert "ViLFusionBlock" in r.stdout
