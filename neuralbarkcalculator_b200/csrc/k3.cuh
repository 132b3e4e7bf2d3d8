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

// The predict path's sink: nothing beyond the mask.  kMask: K3 writes the argmax mask (a sink without it passes no mask).
struct K3Mask {
  static constexpr bool kMask = true;
  struct Acc {};
  __device__ __forceinline__ void pixel(Acc&, int, int, int, int, const float (&)[3], int) const {}
  __device__ __forceinline__ void flush(Acc&, int) const {}
};

// The view set of flip test-time augmentation: up to kK3MaxViews logits canvases [N,3,hc,w], each the network's output for
// a mirrored copy of the batch (nbc_flip_ragged_u8), with its flip flags (1 = columns, 2 = the image's own rows [0, H_n)).
// Passed by value.  A single view with flag 0 is plain K3.
constexpr int kK3MaxViews = 4;
struct K3Views {
  const float* logits[kK3MaxViews];
  int flip[kK3MaxViews];
};
__host__ __device__ inline K3Views k3_one(const float* logits) { return K3Views{{logits, nullptr, nullptr, nullptr}, {0, 0, 0, 0}}; }

// Ragged batch: image n has H_n valid rows in a canvas of Hc rows; its logits occupy ceil(H_n/8) rows of the hc-row
// logits canvas -- per-image in / out heights (scale = h_n / H_n), otherwise the arithmetic of upsample_kernel<true>.
// K3 with the x pass SHARED by the output rows of a group.  An output pixel is a 4 x 4 cubic sample of each class plane:
// the inner (x) sums depend on (source row, X) only, and kRows = 8 consecutive output rows of an 8x upsample touch at
// most 6 distinct source rows -- so a thread (one X) computes the <= 6 x 3 inner sums once, keeps them in its own column
// of shared memory (no synchronisation: a thread only reads what it wrote) and finishes its 8 outputs from them: 9
// global loads per output pixel instead of 48.  Exactly the arithmetic of cubic_sample (same operations, same order), so
// the mask is bit-identical; a group that would need more than kSrc source rows (upscaling by less than ~2x) takes the
// per-pixel path.  heights == nullptr: dense batch (every image H rows, h logits rows).
// kV views (1, 2 or 4): view v's value at output pixel (Y, X) is its K3 value at the mirrored pixel (vflip ? H-1-Y : Y,
// hflip ? W-1-X : X).  Under a row flip the group's 8 output rows are a contiguous mirrored range of view rows, so the
// shared x pass and the <= kSrc criterion apply per view, one view after another through the same s_inner column.  A
// thread keeps its rows x 3 running sums in registers, adds the views in order (((L0 + L1) + L2) + L3) and scales by
// 1/kV (exact) before the argmax; with kV = 1 nothing is added or scaled and the body is plain K3.
constexpr int kK3Rows = 8, kK3Src = 6;
template <int kV, class Sink>
__device__ __forceinline__ void upsample_argmax_rows(const K3Views& views, int hc, int w, int Hc, int W, int h_dense,
                                                     float scale_x, const int* __restrict__ heights, uint8_t* __restrict__ mask,
                                                     const Sink& sink, typename Sink::Acc& acc) {
  static_assert(kV == 1 || kV == 2 || kV == 4, "K3 takes 1, 2 or 4 views");
  __shared__ float s_inner[3][kK3Src][256];
  const int X = blockIdx.x * blockDim.x + threadIdx.x;
  const int Y0 = blockIdx.y * kK3Rows;
  const int n = blockIdx.z;
  const int H = heights != nullptr ? min(max(__ldg(heights + n), 1), Hc) : Hc;
  if (X >= W || Y0 >= H) return;
  const int h = heights != nullptr ? ((((H - 1) / 2 + 1) - 1) / 2 + 1 - 1) / 2 + 1 : h_dense;
  const float scale_y = __fdiv_rn((float)h, (float)H);
  const int rows = min(kK3Rows, H - Y0);
  const int64_t plane = (int64_t)hc * w;
  uint8_t* out = Sink::kMask ? mask + ((int64_t)n * Hc + Y0) * W + X : nullptr;
  float sum[kV > 1 ? kK3Rows : 1][3];     // running sums over the views (registers: every index below is unrolled)
  // one output value of view v: add it to the running sum, or finish the pixel after the last view
  auto take = [&](int v, int y, float (&vs)[3]) {
    if constexpr (kV > 1) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        if (v > 0) vs[c] = __fadd_rn(sum[y][c], vs[c]);
        sum[y][c] = vs[c];
      }
      if (v < kV - 1) return;
#pragma unroll
      for (int c = 0; c < 3; ++c) vs[c] = __fmul_rn(vs[c], 1.f / kV);
    }
    float best = 0.f;
    int arg = 0;
#pragma unroll
    for (int c = 0; c < 3; ++c)
      if (c == 0 || vs[c] > best) best = vs[c], arg = c;      // ties -> lowest index (torch.argmax)
    if constexpr (Sink::kMask) out[(int64_t)y * W] = (uint8_t)arg;
    sink.pixel(acc, n, H, Y0 + y, X, vs, arg);
  };
#pragma unroll
  for (int v = 0; v < kV; ++v) {
    const int flip = kV > 1 ? views.flip[v] : 0;
    const bool vflip = (flip & 2) != 0;
    const float* base = views.logits[v] + (int64_t)n * 3 * plane;
    int ix[4];
    float wx[4];
    cubic_taps((flip & 1) ? W - 1 - X : X, scale_x, w, ix, wx);
    int iy[4];
    float wy[4];
    const int ylo = vflip ? H - Y0 - rows : Y0;     // the group's view rows: [ylo, ylo + rows)
    cubic_taps(ylo, scale_y, h, iy, wy);
    const int r_min = iy[0];
    cubic_taps(ylo + rows - 1, scale_y, h, iy, wy);
    const int nsrc = iy[3] - r_min + 1;      // tap rows are non-decreasing in Y and in k
    if (nsrc > kK3Src) {
#pragma unroll(kV > 1 ? kK3Rows : 1)
      for (int y = 0; y < (kV > 1 ? kK3Rows : rows); ++y) {
        if (kV > 1 && y >= rows) continue;
        cubic_taps(vflip ? H - 1 - (Y0 + y) : Y0 + y, scale_y, h, iy, wy);
        float vs[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) vs[c] = cubic_sample(base + c * plane, w, iy, wy, ix, wx);
        take(v, y, vs);
      }
      continue;
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
#pragma unroll(kV > 1 ? kK3Rows : 1)
    for (int y = 0; y < (kV > 1 ? kK3Rows : rows); ++y) {
      if (kV > 1 && y >= rows) continue;
      cubic_taps(vflip ? H - 1 - (Y0 + y) : Y0 + y, scale_y, h, iy, wy);
      float vs[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        float val = __fmul_rn(s_inner[c][iy[0] - r_min][threadIdx.x], wy[0]);
#pragma unroll
        for (int k = 1; k < 4; ++k) val = __fadd_rn(val, __fmul_rn(s_inner[c][iy[k] - r_min][threadIdx.x], wy[k]));
        vs[c] = val;
      }
      take(v, y, vs);
    }
  }
}

template <class Sink, int kV = 1>
__global__ void __launch_bounds__(256) upsample_argmax_rows_kernel(K3Views views, int hc, int w, int Hc, int W, int h_dense,
                                                                   float scale_x, const int* __restrict__ heights,
                                                                   uint8_t* __restrict__ mask, Sink sink) {
  typename Sink::Acc acc{};
  upsample_argmax_rows<kV>(views, hc, w, Hc, W, h_dense, scale_x, heights, mask, sink, acc);
  sink.flush(acc, blockIdx.z);     // every thread of the block gets here (the body's returns leave the body only)
}

// The view set of a C-ABI call: logits_host / flips_host are HOST arrays of V entries.  Refuses V other than 1, 2, 4,
// a missing canvas and flip flags outside 0..3.
inline int k3_views_args(const float* const* logits_host, const int32_t* flips_host, int V, K3Views& views, const char* what) {
  NBC_REQUIRE(logits_host && flips_host, "%s: null view array", what);
  NBC_REQUIRE(V == 1 || V == 2 || V == 4, "%s: the view set has 1, 2 or 4 views (got %d)", what, V);
  views = K3Views{};
  for (int v = 0; v < V; ++v) {
    NBC_REQUIRE(logits_host[v], "%s: view %d has no logits", what, v);
    NBC_REQUIRE(flips_host[v] >= 0 && flips_host[v] <= 3, "%s: view %d has flip flags %d, outside 0..3", what, v, flips_host[v]);
    views.logits[v] = logits_host[v];
    views.flip[v] = flips_host[v];
  }
  return 0;
}

// The K3 launch of a view set: grid (W / 256, Hc / 8, N); V is 1, 2 or 4 (the caller has checked it).
template <class Sink>
void launch_k3(int V, const K3Views& views, int N, int hc, int w, int Hc, int W, int h_dense, const int* heights, uint8_t* mask,
               const Sink& sink, cudaStream_t stream) {
  const dim3 grid(ceil_div(W, 256), ceil_div(Hc, kK3Rows), N);
  const float sx = (float)w / (float)W;
  if (V == 4)
    upsample_argmax_rows_kernel<Sink, 4><<<grid, 256, 0, stream>>>(views, hc, w, Hc, W, h_dense, sx, heights, mask, sink);
  else if (V == 2)
    upsample_argmax_rows_kernel<Sink, 2><<<grid, 256, 0, stream>>>(views, hc, w, Hc, W, h_dense, sx, heights, mask, sink);
  else
    upsample_argmax_rows_kernel<Sink, 1><<<grid, 256, 0, stream>>>(views, hc, w, Hc, W, h_dense, sx, heights, mask, sink);
}

}  // namespace nbc
