// Closed-form window index maps shared by device kernels and host code.
//
// Restates (without materialising anything) the composition the reference performs with tensors:
//   F.pad to (Hp, Wp)  ->  torch.roll(-shift, -shift)  ->  window_partition      (newcrf_layers.py:212-233, :30-42)
// and its inverse window_reverse -> torch.roll(+shift) -> crop (:239-249, :45-59), plus the region ids the
// shifted-window attention mask is built from (:332-350), and the relative-position index (:90-99).
#pragma once
#include <stdint.h>

#include <type_traits>

namespace crf {

// Window sizes the attention kernels implement: N = ws * ws tokens must fit the 64-row half of a 128-row pair tile.
constexpr int kMinWindow = 2;
constexpr int kMaxWindow = 8;

// relative_position_index[i][j] = (yi - yj + ws-1) * (2ws-1) + (xi - xj + ws-1) = rpb_base<ws>(i) - rpb_col<ws>(j)
// (newcrf_layers.py:90-99), token i = (yi, xi) = (i / ws, i % ws).  The bias table has (2ws-1)^2 rows.
// (Templates: the kernels are instantiated per window size and see these constants from the start.)
__host__ __device__ constexpr int rpb_table_size(int ws) { return (2 * ws - 1) * (2 * ws - 1); }
template <int WS>
__host__ __device__ constexpr int rpb_col(int j) { return (j / WS) * (2 * WS - 1) + (j % WS); }
template <int WS>
__host__ __device__ constexpr int rpb_base(int i) { return (i / WS) * (2 * WS - 1) + (i % WS) + (WS - 1) * (2 * WS); }
template <int WS>
__host__ __device__ constexpr int rel_position_index(int i, int j) {
  return (i / WS - j / WS + (WS - 1)) * (2 * WS - 1) + (i % WS - j % WS + (WS - 1));
}
// floats a kernel reserves for one head's table column (rounded up to 32 bytes: 176 at ws 7)
__host__ __device__ constexpr int rpb_table_padded(int ws) { return (rpb_table_size(ws) + 7) / 8 * 8; }

// Calls f(std::integral_constant<int, WS>()) for a supported window size ws (the kernels are instantiated per window)
// and returns its result; returns -1 for any other ws.
template <typename F>
int with_window(int ws, F&& f) {
  switch (ws) {
    case 2: return f(std::integral_constant<int, 2>());
    case 3: return f(std::integral_constant<int, 3>());
    case 4: return f(std::integral_constant<int, 4>());
    case 5: return f(std::integral_constant<int, 5>());
    case 6: return f(std::integral_constant<int, 6>());
    case 7: return f(std::integral_constant<int, 7>());
    case 8: return f(std::integral_constant<int, 8>());
    default: return -1;
  }
}

struct WindowGeom {
  int H, W;      // feature map
  int ws;        // window size (kMinWindow..kMaxWindow in the attention kernels)
  int shift;     // 0 or ws/2
  int Hp, Wp;    // padded to multiples of ws
  int nWw, nW;   // windows per row / per image
  __host__ __device__ WindowGeom() {}
  __host__ __device__ WindowGeom(int H_, int W_, int ws_, int shift_) : H(H_), W(W_), ws(ws_), shift(shift_) {
    Hp = (H + ws - 1) / ws * ws;
    Wp = (W + ws - 1) / ws * ws;
    nWw = Wp / ws;
    nW = (Hp / ws) * nWw;
  }
  // Token (h*W + w) feeding position p (0..ws*ws-1) of window `win` of an image, or -1 for a zero-pad position.
  __host__ __device__ int source(int win, int p) const {
    const int wh = win / nWw, ww = win - wh * nWw;
    const int i = p / ws, j = p - i * ws;
    int h = wh * ws + i + shift;
    int w = ww * ws + j + shift;
    if (h >= Hp) h -= Hp;
    if (w >= Wp) w -= Wp;
    return (h < H && w < W) ? h * W + w : -1;
  }
  // Region id (0..8) of position p of window `win` on the shifted, padded grid (only meaningful if shift > 0).
  __host__ __device__ int region(int win, int p) const {
    const int wh = win / nWw, ww = win - wh * nWw;
    const int i = p / ws, j = p - i * ws;
    const int h = wh * ws + i, w = ww * ws + j;
    const int rh = h < Hp - ws ? 0 : (h < Hp - shift ? 1 : 2);
    const int rw = w < Wp - ws ? 0 : (w < Wp - shift ? 1 : 2);
    return rh * 3 + rw;
  }
};

}  // namespace crf
