// K3 (bicubic upsample + argmax, models.py:38-41 and 270) as a kernel template over a per-pixel sink, shared by the
// predict path (head.cu: K3Mask, the mask only) and the batched evaluation (eval.cu: a sink that also scores every
// full-resolution pixel against its label, so the f32 logits at full resolution are never written).
#pragma once
#include "cubic.cuh"

namespace nbc {

__device__ __forceinline__ float cubic_sample(const float* __restrict__ plane, int w, const int (&iy)[4],
                                              const float (&wy)[4], const int (&ix)[4], const float (&wx)[4]) {
  float out = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float* r = plane + (int64_t)iy[i] * w;
    float inner = __fmul_rn(__ldg(r + ix[0]), wx[0]);
    inner = __fadd_rn(inner, __fmul_rn(__ldg(r + ix[1]), wx[1]));
    inner = __fadd_rn(inner, __fmul_rn(__ldg(r + ix[2]), wx[2]));
    inner = __fadd_rn(inner, __fmul_rn(__ldg(r + ix[3]), wx[3]));
    const float term = __fmul_rn(inner, wy[i]);
    out = (i == 0) ? term : __fadd_rn(out, term);
  }
  return out;
}

// The predict path's sink: nothing beyond the mask.
struct K3Mask {
  struct Acc {};
  __device__ __forceinline__ void pixel(Acc&, int, int, int, int, const float (&)[3], int) const {}
  __device__ __forceinline__ void flush(Acc&, int) const {}
};

// Ragged batch: image n has H_n valid rows in a canvas of Hc rows; its logits occupy ceil(H_n/8) rows of the hc-row
// logits canvas -- per-image in / out heights (scale = h_n / H_n), otherwise the arithmetic of upsample_kernel<true>.
// K3 with the x pass SHARED by the output rows of a group.  An output pixel is a 4 x 4 cubic sample of each class plane:
// the inner (x) sums depend on (source row, X) only, and kRows = 8 consecutive output rows of an 8x upsample touch at
// most 6 distinct source rows -- so a thread (one X) computes the <= 6 x 3 inner sums once, keeps them in its own column
// of shared memory (no synchronisation: a thread only reads what it wrote) and finishes its 8 outputs from them: 9
// global loads per output pixel instead of 48.  Exactly the arithmetic of cubic_sample (same operations, same order), so
// the mask is bit-identical; a group that would need more than kSrc source rows (upscaling by less than ~2x) takes the
// per-pixel path.  heights == nullptr: dense batch (every image H rows, h logits rows).
constexpr int kK3Rows = 8, kK3Src = 6;
template <class Sink>
__device__ __forceinline__ void upsample_argmax_rows(const float* __restrict__ logits, int hc, int w, int Hc, int W, int h_dense,
                                                     float scale_x, const int* __restrict__ heights, uint8_t* __restrict__ mask,
                                                     const Sink& sink, typename Sink::Acc& acc) {
  __shared__ float s_inner[3][kK3Src][256];
  const int X = blockIdx.x * blockDim.x + threadIdx.x;
  const int Y0 = blockIdx.y * kK3Rows;
  const int n = blockIdx.z;
  const int H = heights != nullptr ? min(max(__ldg(heights + n), 1), Hc) : Hc;
  if (X >= W || Y0 >= H) return;
  const int h = heights != nullptr ? ((((H - 1) / 2 + 1) - 1) / 2 + 1 - 1) / 2 + 1 : h_dense;
  const float scale_y = __fdiv_rn((float)h, (float)H);
  const int rows = min(kK3Rows, H - Y0);
  int ix[4];
  float wx[4];
  cubic_taps(X, scale_x, w, ix, wx);
  int iy[4];
  float wy[4];
  cubic_taps(Y0, scale_y, h, iy, wy);
  const int r_min = iy[0];
  cubic_taps(Y0 + rows - 1, scale_y, h, iy, wy);
  const int nsrc = iy[3] - r_min + 1;      // tap rows are non-decreasing in Y and in k
  const int64_t plane = (int64_t)hc * w;
  const float* base = logits + (int64_t)n * 3 * plane;
  uint8_t* out = mask + ((int64_t)n * Hc + Y0) * W + X;
  if (nsrc > kK3Src) {
    for (int y = 0; y < rows; ++y) {
      cubic_taps(Y0 + y, scale_y, h, iy, wy);
      float best = 0.f, vs[3];
      int arg = 0;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float v = cubic_sample(base + c * plane, w, iy, wy, ix, wx);
        vs[c] = v;
        if (c == 0 || v > best) best = v, arg = c;
      }
      out[(int64_t)y * W] = (uint8_t)arg;
      sink.pixel(acc, n, H, Y0 + y, X, vs, arg);
    }
    return;
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    for (int r = 0; r < nsrc; ++r) {
      const float* rp = base + c * plane + (int64_t)(r_min + r) * w;
      float inner = __fmul_rn(__ldg(rp + ix[0]), wx[0]);
      inner = __fadd_rn(inner, __fmul_rn(__ldg(rp + ix[1]), wx[1]));
      inner = __fadd_rn(inner, __fmul_rn(__ldg(rp + ix[2]), wx[2]));
      inner = __fadd_rn(inner, __fmul_rn(__ldg(rp + ix[3]), wx[3]));
      s_inner[c][r][threadIdx.x] = inner;
    }
  }
  for (int y = 0; y < rows; ++y) {
    cubic_taps(Y0 + y, scale_y, h, iy, wy);
    float best = 0.f, vs[3];
    int arg = 0;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      float v = __fmul_rn(s_inner[c][iy[0] - r_min][threadIdx.x], wy[0]);
#pragma unroll
      for (int k = 1; k < 4; ++k) v = __fadd_rn(v, __fmul_rn(s_inner[c][iy[k] - r_min][threadIdx.x], wy[k]));
      vs[c] = v;
      if (c == 0 || v > best) best = v, arg = c;
    }
    out[(int64_t)y * W] = (uint8_t)arg;
    sink.pixel(acc, n, H, Y0 + y, X, vs, arg);
  }
}

template <class Sink>
__global__ void __launch_bounds__(256) upsample_argmax_rows_kernel(const float* __restrict__ logits, int hc, int w, int Hc, int W,
                                                                   int h_dense, float scale_x, const int* __restrict__ heights,
                                                                   uint8_t* __restrict__ mask, Sink sink) {
  typename Sink::Acc acc{};
  upsample_argmax_rows(logits, hc, w, Hc, W, h_dense, scale_x, heights, mask, sink, acc);
  sink.flush(acc, blockIdx.z);     // every thread of the block gets here (the body's returns leave the body only)
}

}  // namespace nbc
