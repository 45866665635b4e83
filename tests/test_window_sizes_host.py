"""Window sizes 2..8 on the host (no GPU).

1. `WindowGeom` and the relative-position index helpers of csrc/crf_window.cuh, compiled with g++, equal the oracle's
   index maps (source slots, region ids, the mask derived from them, relative_position_index) for every window size
   the kernels implement, both shifts, every H, W <= 24 and the decoder's feature maps.
2. The oracle's closed forms equal a literal transcription of the reference's tensor code (window_partition /
   window_reverse, pad + roll + crop, the img_mask slicing of the shifted-window mask, the relative-position index)
   beyond window 7, where the golden fixtures (all window 7) do not reach.
3. fast_div (the attention kernels' float-reciprocal division) is exact for every divisor these geometries produce.
4. The modules build the reference's state_dict shapes at every supported window and refuse the others; the library
   refuses windows 1 and 9 with a message naming the range.
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import crf_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "monocular_depth_estimation_b200", "csrc")
WINDOWS = range(2, 9)

SHIM = r"""
#define __host__
#define __device__
#include "crf_window.cuh"
extern "C" void window_maps(int H, int W, int ws, int shift, int* dims, int* src, int* region) {
  crf::WindowGeom g(H, W, ws, shift);
  dims[0] = g.Hp; dims[1] = g.Wp; dims[2] = g.nWw; dims[3] = g.nW;
  if (!src) return;
  for (int w = 0; w < g.nW; ++w)
    for (int p = 0; p < ws * ws; ++p) {
      src[w * ws * ws + p] = g.source(w, p);
      region[w * ws * ws + p] = g.region(w, p);
    }
}
// rel[i][j] from rel_position_index and from rpb_base - rpb_col; returns the table size (-1: no such window)
extern "C" int rel_index(int ws, int* rel, int* split) {
  return crf::with_window(ws, [&](auto w) {
    constexpr int WS = decltype(w)::value;
    for (int i = 0; i < WS * WS; ++i)
      for (int j = 0; j < WS * WS; ++j) {
        rel[i * WS * WS + j] = crf::rel_position_index<WS>(i, j);
        split[i * WS * WS + j] = crf::rpb_base<WS>(i) - crf::rpb_col<WS>(j);
      }
    return crf::rpb_table_size(WS);
  });
}
"""


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    d = tmp_path_factory.mktemp("geom_ws")
    src, so = d / "shim.cpp", d / "libgeom_ws.so"
    src.write_text(SHIM)
    subprocess.run(["g++", "-std=c++17", "-O1", "-shared", "-fPIC", "-x", "c++", "-I", CSRC, str(src), "-o", str(so)],
                   check=True)
    lib = ctypes.CDLL(str(so))
    ip = ctypes.POINTER(ctypes.c_int)
    lib.window_maps.argtypes = [ctypes.c_int] * 4 + [ip, ip, ip]
    lib.window_maps.restype = None
    lib.rel_index.argtypes = [ctypes.c_int, ip, ip]
    lib.rel_index.restype = ctypes.c_int
    return lib


def _ip(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int))


def _maps(lib, H, W, ws, shift):
    dims = np.zeros(4, dtype=np.int32)
    lib.window_maps(H, W, ws, shift, _ip(dims), None, None)
    n = int(dims[3]) * ws * ws
    src, reg = np.empty(n, dtype=np.int32), np.empty(n, dtype=np.int32)
    lib.window_maps(H, W, ws, shift, _ip(dims), _ip(src), _ip(reg))
    return dims, src.reshape(-1, ws * ws), reg.reshape(-1, ws * ws)


DECODER_MAPS = [(15, 20), (30, 40), (60, 80), (120, 160), (240, 320)]
GEOMS = [(H, W) for H in range(1, 25) for W in range(1, 25)] + DECODER_MAPS


@pytest.mark.parametrize("ws", WINDOWS)
def test_window_geom_matches_oracle_maps(shim, ws):
    for (H, W) in GEOMS:
        for shift in (0, ws // 2):
            dims, src, reg = _maps(shim, H, W, ws, shift)
            Hp, Wp = O.padded_size(H, ws), O.padded_size(W, ws)
            assert dims.tolist() == [Hp, Wp, Wp // ws, (Hp // ws) * (Wp // ws)], (H, W, ws)
            assert np.array_equal(src, O.window_source_index(H, W, ws, shift)), (H, W, ws, shift)
            if shift:
                assert np.array_equal(reg, O.window_region_ids(H, W, ws, shift)), (H, W, ws, shift)
                mask = np.where(reg[:, :, None] == reg[:, None, :], 0.0, -100.0).astype(np.float32)
                assert np.array_equal(mask, O.shift_mask(H, W, ws, shift)), (H, W, ws, shift)


@pytest.mark.parametrize("ws", WINDOWS)
def test_relative_position_index_helpers_match_oracle(shim, ws):
    n = ws * ws
    rel, split = np.empty(n * n, dtype=np.int32), np.empty(n * n, dtype=np.int32)
    assert shim.rel_index(ws, _ip(rel), _ip(split)) == (2 * ws - 1) ** 2
    ref = O.relative_position_index(ws)
    assert np.array_equal(rel.reshape(n, n), ref)
    assert np.array_equal(split.reshape(n, n), ref)
    assert ref.min() == 0 and ref.max() == (2 * ws - 1) ** 2 - 1


def test_with_window_refuses_other_sizes(shim):
    buf = np.empty(81 * 81, dtype=np.int32)
    for ws in (0, 1, 9, 12):
        assert shim.rel_index(ws, _ip(buf), _ip(buf)) == -1


@pytest.mark.parametrize("ws", WINDOWS)
def test_every_token_has_exactly_one_window_slot(shim, ws):
    for (H, W) in [(1, 1), (ws, ws), (ws + 1, 2 * ws - 1), (8, 13), (9, 10), (23, 17)] + DECODER_MAPS:
        for shift in (0, ws // 2):
            _, src, _ = _maps(shim, H, W, ws, shift)
            real = src[src >= 0]
            assert real.size == H * W and np.array_equal(np.sort(real), np.arange(H * W)), (H, W, ws, shift)


def _fast_div(a, d):
    """numpy restatement of fast_div(a, d, 1.0f / d) in fp32 (csrc/crf_attn_async.cu)."""
    rd = np.float32(1.0) / np.float32(d)
    q = np.trunc((a.astype(np.float32) + np.float32(0.5)) * rd).astype(np.int64)
    r = a - q * d
    return np.where(r < 0, q - 1, np.where(r >= d, q + 1, q))


def test_float_reciprocal_division_is_exact_for_every_window():
    """Domain 0 <= a < 2^22 (the kernels' limit on B * nW).  A rounding error of the reciprocal shows first next to a
    multiple of d, so every multiple of d with its two neighbours is checked, plus 2^16 random points."""
    top = 1 << 22
    divisors = set()
    for ws in WINDOWS:
        for (H, W) in GEOMS + [(480, 640), (960, 1280)]:
            Hp, Wp = O.padded_size(H, ws), O.padded_size(W, ws)
            divisors.update({Wp // ws, (Hp // ws) * (Wp // ws)})
    rnd = np.random.default_rng(0).integers(0, top, 1 << 16)
    for d in sorted(divisors):
        k = np.arange(0, top, d, dtype=np.int64)
        a = np.concatenate([k - 1, k, k + 1, rnd])
        a = a[(a >= 0) & (a < top)]
        assert np.array_equal(_fast_div(a, d), a // d), d


# ---------------------------------------------------------------------------------------------------------------------
# The reference's tensor code, transcribed literally (newcrf_layers.py:30-59, :90-99, :212-249, :332-350)
# ---------------------------------------------------------------------------------------------------------------------
def ref_window_partition(x, window_size):
    B, H, W, C = x.shape
    x = x.view(B, H // window_size, window_size, W // window_size, window_size, C)
    windows = x.permute(0, 1, 3, 2, 4, 5).contiguous().view(-1, window_size, window_size, C)
    return windows


def ref_window_reverse(windows, window_size, H, W):
    B = int(windows.shape[0] / (H * W / window_size / window_size))
    x = windows.view(B, H // window_size, W // window_size, window_size, window_size, -1)
    x = x.permute(0, 1, 3, 2, 4, 5).contiguous().view(B, H, W, -1)
    return x


def ref_pad_roll_partition(x, window_size, shift_size):
    B, H, W, C = x.shape
    pad_l = pad_t = 0
    pad_r = (window_size - W % window_size) % window_size
    pad_b = (window_size - H % window_size) % window_size
    x = F.pad(x, (0, 0, pad_l, pad_r, pad_t, pad_b))
    if shift_size > 0:
        shifted_x = torch.roll(x, shifts=(-shift_size, -shift_size), dims=(1, 2))
    else:
        shifted_x = x
    x_windows = ref_window_partition(shifted_x, window_size)
    return x_windows.view(-1, window_size * window_size, C)


def ref_reverse_roll_crop(windows, B, H, W, window_size, shift_size):
    C = windows.shape[-1]
    pad_r = (window_size - W % window_size) % window_size
    pad_b = (window_size - H % window_size) % window_size
    Hp, Wp = H + pad_b, W + pad_r
    windows = windows.view(-1, window_size, window_size, C)
    shifted_x = ref_window_reverse(windows, window_size, Hp, Wp)
    if shift_size > 0:
        x = torch.roll(shifted_x, shifts=(shift_size, shift_size), dims=(1, 2))
    else:
        x = shifted_x
    if pad_r > 0 or pad_b > 0:
        x = x[:, :H, :W, :].contiguous()
    return x


def ref_attn_mask(H, W, window_size, shift_size):
    Hp = int(np.ceil(H / window_size)) * window_size
    Wp = int(np.ceil(W / window_size)) * window_size
    img_mask = torch.zeros((1, Hp, Wp, 1))
    h_slices = (slice(0, -window_size), slice(-window_size, -shift_size), slice(-shift_size, None))
    w_slices = (slice(0, -window_size), slice(-window_size, -shift_size), slice(-shift_size, None))
    cnt = 0
    for h in h_slices:
        for w in w_slices:
            img_mask[:, h, w, :] = cnt
            cnt += 1
    mask_windows = ref_window_partition(img_mask, window_size)
    mask_windows = mask_windows.view(-1, window_size * window_size)
    attn_mask = mask_windows.unsqueeze(1) - mask_windows.unsqueeze(2)
    attn_mask = attn_mask.masked_fill(attn_mask != 0, float(-100.0)).masked_fill(attn_mask == 0, float(0.0))
    return attn_mask


def ref_relative_position_index(window_size):
    window_size = (window_size, window_size)
    coords_h = torch.arange(window_size[0])
    coords_w = torch.arange(window_size[1])
    coords = torch.stack(torch.meshgrid([coords_h, coords_w], indexing="ij"))
    coords_flatten = torch.flatten(coords, 1)
    relative_coords = coords_flatten[:, :, None] - coords_flatten[:, None, :]
    relative_coords = relative_coords.permute(1, 2, 0).contiguous()
    relative_coords[:, :, 0] += window_size[0] - 1
    relative_coords[:, :, 1] += window_size[1] - 1
    relative_coords[:, :, 0] *= 2 * window_size[1] - 1
    return relative_coords.sum(-1)


@pytest.mark.parametrize("ws", WINDOWS)
def test_oracle_closed_forms_equal_the_reference_tensor_code(ws):
    gen = torch.Generator().manual_seed(ws)
    assert np.array_equal(O.relative_position_index(ws), ref_relative_position_index(ws).numpy())
    for (H, W) in [(1, 1), (ws - 1 or 1, ws + 1), (ws, ws), (9, 10), (15, 20), (2 * ws + 1, 3 * ws - 1), (30, 40)]:
        x = torch.randn(2, H, W, 3, generator=gen)
        for shift in (0, ws // 2):
            got = O.window_gather(x, ws, shift)
            want = ref_pad_roll_partition(x, ws, shift)
            assert torch.equal(got, want), (H, W, ws, shift)
            back = O.window_scatter(want, 2, H, W, ws, shift)
            assert torch.equal(back, ref_reverse_roll_crop(want, 2, H, W, ws, shift)), (H, W, ws, shift)
            assert torch.equal(back, x)
            if shift:
                assert torch.equal(torch.from_numpy(O.shift_mask(H, W, ws, shift)), ref_attn_mask(H, W, ws, shift))


# ---------------------------------------------------------------------------------------------------------------------
# Modules and the library's argument checks
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ws", WINDOWS)
def test_modules_build_the_reference_state_dict_at_every_window(ws):
    import monocular_depth_estimation_b200 as pkg
    layer = pkg.BasicCRFLayer(dim=64, depth=2, num_heads=2, v_dim=64, window_size=ws)
    assert [b.shift_size for b in layer.blocks] == [0, ws // 2]
    sd = layer.state_dict()
    for i in range(2):
        assert tuple(sd[f"blocks.{i}.attn.relative_position_bias_table"].shape) == ((2 * ws - 1) ** 2, 2)
        idx = sd[f"blocks.{i}.attn.relative_position_index"]
        assert tuple(idx.shape) == (ws * ws, ws * ws)
        assert np.array_equal(idx.numpy(), O.relative_position_index(ws))
    blk = pkg.CRFBlock(64, 2, 64, window_size=ws, shift_size=ws // 2)
    assert tuple(blk.attn.relative_position_bias_table.shape) == ((2 * ws - 1) ** 2, 2)


@pytest.mark.parametrize("ws", [1, 9, 12])
def test_modules_refuse_unsupported_windows(ws):
    import monocular_depth_estimation_b200 as pkg
    with pytest.raises(NotImplementedError, match="window_size"):
        pkg.CRFBlock(64, 2, 64, window_size=ws)
    with pytest.raises(NotImplementedError, match="window_size"):
        pkg.BasicCRFLayer(dim=64, depth=2, num_heads=2, v_dim=64, window_size=ws)
    with pytest.raises(NotImplementedError, match="window_size"):
        pkg.NewCRF(input_dim=64, embed_dim=64, v_dim=64, window_size=ws, num_heads=2)


def test_library_window_range():
    from monocular_depth_estimation_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        pytest.skip("extension not built (run __graft_entry__.build())")
    lib = _lib.lib()
    d = _lib.BlockDesc()
    d.B, d.H, d.W, d.C, d.num_heads = 1, 15, 20, 128, 4
    s = ctypes.c_size_t()
    for ws, ok in ((1, False), (2, True), (5, True), (7, True), (8, True), (9, False)):
        for prec in (_lib.PREC_BF16, _lib.PREC_FP32):
            d.window, d.shift, d.precision = ws, ws // 2, prec
            rc = lib.crf_block_sizes(ctypes.byref(d), ctypes.byref(s), None, None)
            if ok:
                assert rc == 0 and s.value > 0, (ws, lib.crf_last_error())
            else:
                assert rc != 0 and b"window must be in [2, 8]" in lib.crf_last_error(), ws
            rc = lib.crf_layer_sizes(ctypes.byref(d), 2, 1, ctypes.byref(s), None)
            assert (rc == 0) == ok, (ws, lib.crf_last_error())
