"""CPU-side checks of the drop-in boundary: the C-ABI library loads without a GPU and exports every symbol
include/crf_sm100.h declares; host-side argument validation returns errors instead of crashing."""
import ctypes
import os
import re

import pytest

from monocular_depth_estimation_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    src = open(os.path.join(ROOT, "include", "crf_sm100.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(crf_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("extension not built (run __graft_entry__.build())")
    lib = ctypes.CDLL(_lib.LIB_PATH)
    declared = _header_symbols()
    assert declared, "no declarations parsed"
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/crf_sm100.h but not exported"
    assert sorted(_lib.EXPORTED_SYMBOLS) == declared, "python binding list and header disagree"


def test_version_and_error_reporting_without_gpu():
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("extension not built")
    lib = _lib.lib()
    assert lib.crf_abi_version() == 4
    d = _lib.BlockDesc()
    d.B, d.H, d.W, d.C, d.num_heads, d.window, d.shift = 1, 7, 7, 96, 3, 7, 0   # C not a multiple of 64
    s = ctypes.c_size_t()
    assert lib.crf_block_sizes(ctypes.byref(d), ctypes.byref(s), None, None) != 0
    assert b"multiple of 64" in lib.crf_last_error()
    d.C, d.num_heads, d.shift = 128, 4, 7
    assert lib.crf_block_sizes(ctypes.byref(d), ctypes.byref(s), None, None) != 0
    assert b"shift_size must in 0-window_size" in lib.crf_last_error()
    d.shift = 3
    assert lib.crf_block_sizes(ctypes.byref(d), ctypes.byref(s), None, None) == 0 and s.value > 0


def test_struct_sizes_match_header_layout():
    # 12 int32 + 7 int64 + 2 int32 ; 13 pointers + 2 floats + pointer + 2 int32 ; 13 pointers
    assert ctypes.sizeof(_lib.BlockDesc) == 12 * 4 + 7 * 8 + 8
    assert ctypes.sizeof(_lib.BlockParams) == 13 * 8 + 8 + 8 + 8
    assert ctypes.sizeof(_lib.BlockGrads) == 13 * 8


def test_ctypes_structs_match_the_c_header_field_by_field(tmp_path):
    """Compile a tiny C program against include/crf_sm100.h (gcc) that prints sizeof and every offsetof, and compare
    with the ctypes mirrors in _lib.py -- a silent mismatch here would corrupt arguments at the drop-in boundary."""
    import shutil
    import subprocess
    if shutil.which("gcc") is None:
        pytest.skip("gcc not available")
    structs = {"crf_block_desc": _lib.BlockDesc, "crf_block_params": _lib.BlockParams,
               "crf_block_grads": _lib.BlockGrads, "crf_layer_args": _lib.LayerArgs, "crf_gemm_args": _lib.GemmArgs,
               "crf_adam_tensor": _lib.AdamTensor, "crf_mlp_args": _lib.MlpArgs}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "crf_sm100.h"', 'int main(void) {']
    for cname, cls in structs.items():
        lines.append(f'  printf("{cname} %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname}.{fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines) + "\n")
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = dict(ln.split() for ln in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    for cname, cls in structs.items():
        assert int(out[cname]) == ctypes.sizeof(cls), cname
        for fname, _ in cls._fields_:
            assert int(out[f"{cname}.{fname}"]) == getattr(cls, fname).offset, f"{cname}.{fname}"



def _sizes(lib, d):
    s, f, b = ctypes.c_size_t(), ctypes.c_size_t(), ctypes.c_size_t()
    rc = lib.crf_block_sizes(ctypes.byref(d), ctypes.byref(s), ctypes.byref(f), ctypes.byref(b))
    return rc, s.value, f.value, b.value


def test_buffer_sizes_host_side():
    """crf_block_sizes / crf_layer_sizes are pure host arithmetic: check them without a GPU -- 256-byte granularity,
    inference < training, growth with the problem, and the figure DESIGN.md quotes for the 1/4 scale of config 2."""
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("extension not built")
    from monocular_depth_estimation_b200 import ops
    lib = _lib.lib()
    d = ops.make_desc(8, 120, 160, 128, 4, 3, device=0)
    rc, saved, _, ws = _sizes(lib, d)
    assert rc == 0 and saved % 256 == 0 and ws % 256 == 0
    T, C = 8 * 120 * 160, 128
    # xn1, qk(2C), vb, attn_o, xn2 bf16 + x1 fp32 + pre, act (4C bf16 each) + bf16 weights + stats / lse
    floor = T * C * (2 + 4 + 2 + 2 + 2 + 4 + 8 + 8)
    assert floor <= saved <= int(floor * 1.1) + (1 << 20), (saved, floor)
    assert 0.55e9 < saved < 0.80e9            # "about 0.75 GB per block" (DESIGN.md section 2)
    d_inf = ops.make_desc(8, 120, 160, 128, 4, 3, device=0, training=0)
    assert _sizes(lib, d_inf)[1] < saved       # no pre-activation kept for inference
    small = ops.make_desc(2, 60, 80, 128, 4, 3, device=0)
    assert _sizes(lib, small)[1] < saved and _sizes(lib, small)[3] < ws
    # layer level: two blocks + shared v + intermediate outputs; more than two stand-alone blocks' saved areas minus v
    sb, wb = ctypes.c_size_t(), ctypes.c_size_t()
    assert lib.crf_layer_sizes(ctypes.byref(d), 2, 1, ctypes.byref(sb), ctypes.byref(wb)) == 0
    assert sb.value > 2 * (saved - T * C * 2 - 4096) and wb.value >= ws
    assert lib.crf_layer_sizes(ctypes.byref(d), 0, 0, ctypes.byref(sb), ctypes.byref(wb)) != 0
    assert b"depth" in lib.crf_last_error()


def test_head_width_validation():
    """head_dim 16 / 32 / 64 / 128 are accepted; anything else is rejected with a message, not a crash."""
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("extension not built")
    from monocular_depth_estimation_b200 import ops
    lib = _lib.lib()
    for C, nH, ok in [(128, 4, True), (128, 8, True), (128, 2, True), (128, 1, True), (64, 1, True), (512, 4, True),
                      (64, 8, False), (128, 3, False), (256, 1, False), (192, 4, False)]:
        rc = _sizes(lib, ops.make_desc(1, 7, 7, C, nH, 0, device=0))[0]
        assert (rc == 0) == ok, (C, nH)
        if not ok:
            assert b"head_dim must be 16, 32, 64 or 128" in lib.crf_last_error()
    # every width in [64, 1024] that is a multiple of 64, with every supported head width that divides it
    for C in range(64, 1025, 64):
        for hd in (16, 32, 64, 128):
            if C % hd == 0:
                rc = _sizes(lib, ops.make_desc(1, 7, 7, C, C // hd, 0, device=0))[0]
                assert rc == 0, (C, hd, lib.crf_last_error())
    for C in (32, 96, 1088):
        assert _sizes(lib, ops.make_desc(1, 7, 7, C, 1, 0, device=0))[0] != 0, C
        assert b"multiple of 64" in lib.crf_last_error(), C
