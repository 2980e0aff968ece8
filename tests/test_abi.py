"""CPU: the C-ABI library builds, loads, exports every symbol include/b200unet.h declares, and the ctypes binding
agrees with the header (argument count and kind). No compute calls (no GPU here)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g

    g.build()
    from unet_torch_b200 import _lib

    return _lib


def header_decls():
    h = open(os.path.join(ROOT, "include", "b200unet.h")).read()
    h = re.sub(r"/\*.*?\*/", "", h, flags=re.S)
    return re.findall(r"\b(?:int|int64_t|const char\*)\s+(b200unet_\w+)\s*\(([^;]*?)\)\s*;", h, flags=re.S)


def test_every_declared_symbol_is_exported_and_bound(lib):
    decls = header_decls()
    assert len(decls) >= 30
    cdll = ctypes.CDLL(lib.LIB_PATH)
    for name, args in decls:
        assert hasattr(cdll, name), f"{name} declared in include/b200unet.h but not exported"
        assert name in lib.SIGNATURES, f"{name} has no ctypes binding"
        arglist = [a.strip() for a in args.split(",") if a.strip() and a.strip() != "void"]
        bound = lib.SIGNATURES[name][1]
        assert len(arglist) == len(bound), name
        for a, ct in zip(arglist, bound):
            is_ptr = "*" in a or "b200_stream_t" in a
            want = "c_void_p" if is_ptr else "c_double" if a.startswith("double") else "c_float" if a.startswith(
                "float") else "c_long" if "int64_t" in a else "c_int"
            assert ct.__name__ == want, (name, a, ct.__name__)
    assert set(lib.SIGNATURES) == {n for n, _ in decls}


def test_host_only_queries(lib):
    assert lib.query("b200unet_version") >= 100
    assert (lib.query("b200unet_tile_h"), lib.query("b200unet_tile_w")) == (8, 16)
    # split-K workspace: splits * Cout * 9 * Cin floats, at least one split
    ws = lib.query("b200unet_conv3x3_wgrad_workspace_floats", 16, 512, 512, 64, 64)
    assert ws % (64 * 9 * 64) == 0 and ws >= 64 * 9 * 64
    # deep layer: 192 base CTAs -> 3 pixel splits fill 3.9 waves of 148 SMs instead of 1.3
    assert lib.query("b200unet_conv3x3_wgrad_workspace_floats", 16, 32, 32, 1024, 1024) == 3 * 1024 * 9 * 1024
    # statistics rows: one per persistent CTA for the resident-weight kernel (Cin <= 128), one per 8x16 tile otherwise
    assert lib.query("b200unet_conv3x3_stat_rows", 16, 512, 512, 64, 64) == 148
    assert lib.query("b200unet_conv3x3_stat_rows", 16, 64, 64, 512, 512) > 0
    assert lib.query("b200unet_launch_count") == 0
    # attention gates: one statistics row per 8x16 tile for the 1x1 GEMM, four (one per (i,j)) for the ConvTranspose2d; gate
    # kernels: one row per block, at most 148 x 8; reduction workspace = 148 x 8 rows of 4C + 8 floats
    assert lib.query("b200unet_conv1x1_stat_rows", 16, 512, 512) == 16 * 64 * 32
    assert lib.query("b200unet_convt2x2_stat_rows", 16, 256, 256) == 4 * 16 * 32 * 16
    assert lib.query("b200unet_gate_stat_rows", 16 * 512 * 512, 32) == 148 * 8 and lib.query("b200unet_gate_stat_rows", 64, 32) == 1
    assert lib.query("b200unet_gate_workspace_floats", 256) == 148 * 8 * (4 * 256 + 8)
    assert lib.query("b200unet_conv1x1_wgrad_workspace_floats", 16, 512, 512, 64, 64) % (64 * 64) == 0


def test_bad_shapes_are_errors_not_fallbacks(lib):
    # no GPU needed: argument validation happens before anything touches the device
    with pytest.raises(RuntimeError, match="multiples of 64"):
        lib.call("b200unet_conv3x3_igemm", None, 48, None, None, 64, None, 1, 8, 16, 48, 64, None)
    with pytest.raises(RuntimeError, match="n_classes"):
        lib.call("b200unet_head_fprop", None, 64, None, None, None, 1, 8, 8, 64, 9, None)
    assert "n_classes" in lib.last_error()
    with pytest.raises(RuntimeError, match="32, 64, 128 or 256"):   # gate kernels: hidden widths of a width-64 network only
        lib.call("b200unet_gate_psi_fwd", None, 512, None, 512, None, None, None, None, None, None, None, None, 64, 512, None)
    with pytest.raises(RuntimeError, match="multiples of 64"):
        lib.call("b200unet_conv1x1_fprop", 1, 32, 1, None, 1, 64, None, 64, 1, 8, 16, 32, 64, None)
    with pytest.raises(RuntimeError, match="empty problem"):
        lib.call("b200unet_sgemm_strided", 1, 1, 1, None, 0, 4, 4, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, None)


def test_bn_statistics_entry_points_validate_before_launch(lib):
    # a BatchNorm built with track_running_stats=False has no running buffers: eval mode has no affine to compute
    with pytest.raises(RuntimeError, match="null running statistics"):
        lib.call("b200unet_bn_eval_affine", 1, 1, None, None, 1e-5, 1, 1, 64, None)
    with pytest.raises(RuntimeError, match="null running statistics"):
        lib.call("b200unet_bn_eval_affine", 1, 1, 1, None, 1e-5, 1, 1, 64, None)
    with pytest.raises(RuntimeError, match="null argument"):
        lib.call("b200unet_bn_eval_stats", None, None, 1e-5, 1, 1, 64, None)
    # fold_rows: the column width of a block is a power of two <= 256 or a multiple of 256
    for ncols in (192, 384):
        with pytest.raises(RuntimeError, match=f"ncols={ncols}"):
            lib.call("b200unet_fold_rows", 1, 5000, ncols, 1, 296, None)
    with pytest.raises(RuntimeError, match="bad arguments"):
        lib.call("b200unet_fold_rows", 1, 100, 64, 1, 296, None)    # more output rows than input rows
    with pytest.raises(RuntimeError, match="bad column range"):
        lib.call("b200unet_partial_colsum", 1, 8, 64, 40, 25, 1, None)


def test_bn_relu_backward_passes_validate_the_pool_arguments_before_launch(lib):
    """Both BatchNorm+ReLU backward passes refuse a call without a gradient source, and a pooled gradient without window
    positions or with an odd H or W: the kernels read pool_idx and the 2x2 windows of y unchecked."""
    launches = lib.query("b200unet_launch_count")

    def reduce_rows(g1, g_pool, pool_idx, h, w, c=64):
        lib.call("b200unet_bn_relu_bwd_reduce_rows", g1, c, g_pool, pool_idx, 1, c, 1, 1, 1, 1, 1, 1, 2, h, w, c, None)

    def apply(g1, g_pool, pool_idx, h, w, c=64):
        lib.call("b200unet_bn_relu_bwd_apply", g1, c, g_pool, pool_idx, 1, c, 1, 1, 1, 1, 1, 1, 8.0, None, 1, c, 1, 1, 2, h, w,
                 c, None)

    for fn, name in ((reduce_rows, "bn_relu_bwd_reduce"), (apply, "bn_relu_bwd_apply")):
        with pytest.raises(RuntimeError, match=f"{name}: C=96 must be a power of two"):
            fn(1, None, None, 4, 4, c=96)
        with pytest.raises(RuntimeError, match=f"{name}: no gradient source"):
            fn(None, None, None, 4, 4)
        with pytest.raises(RuntimeError, match=rf"{name}\(pool\): bad arguments"):
            fn(1, 1, None, 4, 4)            # pooled gradient without window positions
        for h, w in ((3, 4), (4, 5)):
            with pytest.raises(RuntimeError, match=rf"{name}\(pool\): bad arguments"):
                fn(1, 1, 1, h, w)
    assert lib.query("b200unet_launch_count") == launches


def test_header_is_plain_c_and_a_c_host_links_the_library(lib, tmp_path):
    """The boundary is a C ABI: include/b200unet.h must compile as C99 (no C++ in the signatures), and a C host program
    must link libb200unet.so and reach the host-only entry points (what a cgo / JNI / FFI binding does)."""
    import shutil
    import subprocess

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    hdr = os.path.join(ROOT, "include", "b200unet.h")
    r = subprocess.run([gcc, "-std=c99", "-Wall", "-Wextra", "-Werror", "-fsyntax-only", "-x", "c", hdr],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    src = tmp_path / "host.c"
    src.write_text(
        '#include <stdio.h>\n#include "b200unet.h"\n'
        "int main(void) {\n"
        '  printf("%d %d %d %lld\\n", b200unet_version(), b200unet_tile_h(), b200unet_tile_w(),\n'
        "         (long long)b200unet_conv3x3_wgrad_workspace_floats(16, 32, 32, 1024, 1024));\n"
        "  /* attention-gate entry points: host-only size queries, and argument validation before any launch */\n"
        '  printf("%d %lld\\n", b200unet_gate_stat_rows(64, 32), (long long)b200unet_gate_workspace_floats(256));\n'
        "  if (b200unet_gate_dx(0, 64, 0, 0, 0, 0, 64, 1, 64, 0) == 0) return 2;\n"
        "  /* a bad shape is an error code + message, never a fallback */\n"
        "  int rc = b200unet_head_fprop(0, 64, 0, 0, 0, 1, 8, 8, 64, 9, 0);\n"
        '  printf("%d %s\\n", rc, b200unet_last_error());\n'
        "  return rc == 0;\n}\n")
    exe = tmp_path / "host"
    libdir = os.path.dirname(lib.LIB_PATH)
    r = subprocess.run([gcc, "-std=c99", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe), "-L", libdir,
                        "-l:libb200unet.so", f"-Wl,-rpath,{libdir}"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, (r.stdout, r.stderr)
    first, gate, second = r.stdout.strip().splitlines()
    v, th, tw, ws = first.split()
    assert int(v) >= 100 and (int(th), int(tw)) == (8, 16) and int(ws) == 3 * 1024 * 9 * 1024
    assert gate.split() == ["1", str(148 * 8 * (4 * 256 + 8))]
    assert second.split()[0] != "0" and "n_classes" in second
