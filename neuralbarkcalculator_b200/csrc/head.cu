// Head tail + K3.
//  * nbc_head_1x1: Dropout (identity in eval) + Conv2d(512, 3, 1) with bias (models.py:113-124) on the bf16
//    NHWC features, f32 weights, f32 planar logits [N,3,h*w].  HBM-bound: one warp per pixel, 32 B per lane.
//  * nbc_upsample_argmax / nbc_upsample_bicubic: F.interpolate(mode='bicubic', align_corners=False)
//    (models.py:38-41) fused with torch.argmax(dim=1) (models.py:270).  The 12.6 MB f32 full-resolution logits
//    are never written in the argmax variant.  Index / weight arithmetic follows torch's upsample_bicubic2d in
//    f32 with explicit IEEE operations (no fma contraction) in the order of oracle/model.py
//    ``upsample_bicubic_restated`` so the result is bit-identical to that restatement.
#include "common.cuh"
#include "k3.cuh"

namespace nbc {

// kIters = Cin / 256: every lane owns 8 consecutive channels of each 256-channel slab and keeps its 3 x 8 x kIters
// weights in registers, so the inner loop is one 16-byte load + 24 FMAs per slab.
template <int kIters>
__global__ void __launch_bounds__(256) head1x1_kernel(const __nv_bfloat16* __restrict__ x, int P, int N, int Cin,
                                                      const float* __restrict__ w, const float* __restrict__ bias,
                                                      float* __restrict__ logits, int f16, const int* __restrict__ valid_h,
                                                      int row_w) {
  const int lane = threadIdx.x & 31;
  // 32-bit pixel indices (the host checks N * P < 2^31): the first version's 64-bit divisions per pixel cost more than the
  // 48 FMAs of the pixel
  const int warp_global = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
  const int nwarps = (int)((gridDim.x * blockDim.x) >> 5);
  const int M = N * P;
  const float b0 = __ldg(bias), b1 = __ldg(bias + 1), b2 = __ldg(bias + 2);
  float wr[kIters][3][8];
#pragma unroll
  for (int it = 0; it < kIters; ++it)
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
      for (int e = 0; e < 8; ++e) wr[it][k][e] = __ldg(w + k * Cin + it * 256 + lane * 8 + e);
  // kPix pixels per warp and iteration: their loads are all issued before the first FMA (one pixel at a time left the
  // kernel at 1.5 TB/s -- too little memory-level parallelism)
  constexpr int kPix = 4;
  for (int m0 = warp_global; m0 < M; m0 += nwarps * kPix) {
    uint4 v[kPix][kIters];
    bool on[kPix];
#pragma unroll
    for (int j = 0; j < kPix; ++j) {
      const int m = m0 + j * nwarps;
      on[j] = m < M;
      if (on[j] && valid_h != nullptr) {   // ragged batch: rows at or below an image's last valid one feed nothing (K3 clamps its taps)
        const int img = m / P;
        on[j] = (m - img * P) / row_w < __ldg(valid_h + img);
      }
      if (on[j]) {
        const __nv_bfloat16* xr = x + (int64_t)m * Cin + lane * 8;
#pragma unroll
        for (int it = 0; it < kIters; ++it) v[j][it] = __ldg(reinterpret_cast<const uint4*>(xr + it * 256));
      }
    }
#pragma unroll
    for (int j = 0; j < kPix; ++j) {
      if (!on[j]) continue;      // warp-uniform
      const int m = m0 + j * nwarps;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f;
#pragma unroll
      for (int it = 0; it < kIters; ++it) {
        const uint32_t u[4] = {v[j][it].x, v[j][it].y, v[j][it].z, v[j][it].w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float f0 = lo16(u[k], f16), f1 = hi16(u[k], f16);
          a0 = fmaf(f0, wr[it][0][2 * k], a0), a0 = fmaf(f1, wr[it][0][2 * k + 1], a0);
          a1 = fmaf(f0, wr[it][1][2 * k], a1), a1 = fmaf(f1, wr[it][1][2 * k + 1], a1);
          a2 = fmaf(f0, wr[it][2][2 * k], a2), a2 = fmaf(f1, wr[it][2][2 * k + 1], a2);
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        a0 += __shfl_xor_sync(0xffffffffu, a0, o);
        a1 += __shfl_xor_sync(0xffffffffu, a1, o);
        a2 += __shfl_xor_sync(0xffffffffu, a2, o);
      }
      if (lane == 0) {
        const int img = m / P, pix = m - img * P;
        float* o = logits + (int64_t)img * 3 * P + pix;
        o[0] = a0 + b0;
        o[P] = a1 + b1;
        o[2 * P] = a2 + b2;
      }
    }
  }
}

template <bool kArgmax>
__global__ void __launch_bounds__(256) upsample_kernel(const float* __restrict__ logits, int N, int C, int h, int w,
                                                       int H, int W, float scale_y, float scale_x,
                                                       uint8_t* __restrict__ mask, float* __restrict__ out) {
  const int X = blockIdx.x * blockDim.x + threadIdx.x;
  const int Y = blockIdx.y;
  const int n = blockIdx.z;
  if (X >= W) return;
  int ix[4], iy[4];
  float wx[4], wy[4];
  cubic_taps(X, scale_x, w, ix, wx);
  cubic_taps(Y, scale_y, h, iy, wy);
  const int64_t plane = (int64_t)h * w;
  if (kArgmax) {
    float best = 0.f;
    int arg = 0;
    for (int c = 0; c < C; ++c) {
      const float v = cubic_sample(logits + ((int64_t)n * C + c) * plane, w, iy, wy, ix, wx);
      if (c == 0 || v > best) best = v, arg = c;  // ties -> lowest index (torch.argmax)
    }
    mask[((int64_t)n * H + Y) * W + X] = (uint8_t)arg;
  } else {
    for (int c = 0; c < C; ++c)
      out[(((int64_t)n * C + c) * H + Y) * W + X] =
          cubic_sample(logits + ((int64_t)n * C + c) * plane, w, iy, wy, ix, wx);
  }
}

__global__ void heights_kernel(const int* __restrict__ first_last, int N, int* __restrict__ heights) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n < N) heights[n] = first_last[2 * n + 1] - first_last[2 * n];
}

}  // namespace nbc

using namespace nbc;

extern "C" int nbc_heights_from_first_last(const int32_t* first_last, int N, int32_t* heights, void* stream) {
  NBC_REQUIRE(first_last && heights && N > 0, "nbc_heights_from_first_last: bad argument");
  heights_kernel<<<ceil_div(N, 128), 128, 0, reinterpret_cast<cudaStream_t>(stream)>>>(first_last, N, heights);
  NBC_CHECK_LAUNCH();
  return 0;
}

extern "C" int nbc_upsample_argmax_ragged(const float* logits, int N, int hc, int w, int Hc, int W, const int32_t* heights,
                                          uint8_t* mask, void* stream) {
  NBC_REQUIRE(logits && heights && mask, "nbc_upsample_argmax_ragged: null pointer");
  NBC_REQUIRE(N > 0 && hc > 0 && w > 0 && Hc > 0 && W > 0 && Hc <= 65535 && N <= 65535, "nbc_upsample_argmax_ragged: bad shape");
  launch_k3(1, k3_one(logits), N, hc, w, Hc, W, 0, heights, mask, K3Mask(), reinterpret_cast<cudaStream_t>(stream));
  NBC_CHECK_LAUNCH();
  return 0;
}

namespace nbc {
// The full-resolution logits sink of the view set: f32 [N,3,Hc,W], rows [0, H_n) of image n.
struct K3Logits {
  static constexpr bool kMask = false;
  struct Acc {};
  float* __restrict__ out;
  int Hc, W;
  __device__ __forceinline__ void pixel(Acc&, int n, int, int Y, int X, const float (&v)[3], int) const {
    const int64_t plane = (int64_t)Hc * W, at = (int64_t)n * 3 * plane + (int64_t)Y * W + X;
#pragma unroll
    for (int c = 0; c < 3; ++c) out[at + c * plane] = v[c];
  }
  __device__ __forceinline__ void flush(Acc&, int) const {}
};

// dst image n = src image n mirrored within its rows [0, H_n) (flags & 2) and the W columns (flags & 1); rows H_n..Hc-1
// of dst are zero.  One block per (canvas row, image); bytes of a row are independent, so threads stride over them.
__global__ void __launch_bounds__(256) flip_ragged_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, int Hc, int W,
                                                          const int* __restrict__ heights, int flags) {
  const int y = blockIdx.x, n = blockIdx.y;
  const int H = min(max(__ldg(heights + n), 1), Hc);
  const int64_t row = 3ll * W;
  uint8_t* d = dst + ((int64_t)n * Hc + y) * row;
  if (y >= H) {
    for (int i = threadIdx.x; i < (int)row; i += blockDim.x) d[i] = 0;
    return;
  }
  const uint8_t* s = src + ((int64_t)n * Hc + ((flags & 2) ? H - 1 - y : y)) * row;
  for (int i = threadIdx.x; i < (int)row; i += blockDim.x) {
    const int x = i / 3, ch = i - 3 * x;
    d[i] = __ldg(s + ((flags & 1) ? 3 * (W - 1 - x) + ch : i));
  }
}

}  // namespace nbc

extern "C" int nbc_flip_ragged_u8(const uint8_t* src, uint8_t* dst, int N, int Hc, int W, const int32_t* heights, int flags,
                                  void* stream) {
  NBC_REQUIRE(src && dst && heights, "nbc_flip_ragged_u8: null pointer");
  NBC_REQUIRE(src != dst, "nbc_flip_ragged_u8: src and dst must not be the same canvas");
  NBC_REQUIRE(N > 0 && Hc > 0 && W > 0 && N <= 65535 && 3ll * W < (1ll << 31), "nbc_flip_ragged_u8: bad shape N=%d Hc=%d W=%d",
              N, Hc, W);
  NBC_REQUIRE(flags >= 0 && flags <= 3, "nbc_flip_ragged_u8: flags is 1 (columns), 2 (rows) or 3 (both), got %d", flags);
  flip_ragged_kernel<<<dim3(Hc, N), 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(src, dst, Hc, W, heights, flags);
  NBC_CHECK_LAUNCH();
  return 0;
}

extern "C" int nbc_upsample_argmax_views_ragged(const float* const* logits, const int32_t* flips, int V, int N, int hc, int w, int Hc,
                                                int W, const int32_t* heights, uint8_t* mask, void* stream) {
  K3Views views;
  const int rc = k3_views_args(logits, flips, V, views, "nbc_upsample_argmax_views_ragged");
  if (rc != 0) return rc;
  NBC_REQUIRE(heights && mask, "nbc_upsample_argmax_views_ragged: null pointer");
  NBC_REQUIRE(N > 0 && hc > 0 && w > 0 && Hc > 0 && W > 0 && Hc <= 65535 * kK3Rows && N <= 65535,
              "nbc_upsample_argmax_views_ragged: bad shape");
  launch_k3(V, views, N, hc, w, Hc, W, 0, heights, mask, K3Mask(), reinterpret_cast<cudaStream_t>(stream));
  NBC_CHECK_LAUNCH();
  return 0;
}

extern "C" int nbc_upsample_bicubic_views_ragged(const float* const* logits, const int32_t* flips, int V, int N, int hc, int w,
                                                 int Hc, int W, const int32_t* heights, float* out, void* stream) {
  K3Views views;
  const int rc = k3_views_args(logits, flips, V, views, "nbc_upsample_bicubic_views_ragged");
  if (rc != 0) return rc;
  NBC_REQUIRE(heights && out, "nbc_upsample_bicubic_views_ragged: null pointer");
  NBC_REQUIRE(N > 0 && hc > 0 && w > 0 && Hc > 0 && W > 0 && Hc <= 65535 * kK3Rows && N <= 65535,
              "nbc_upsample_bicubic_views_ragged: bad shape");
  K3Logits sink;
  sink.out = out, sink.Hc = Hc, sink.W = W;
  launch_k3(V, views, N, hc, w, Hc, W, 0, heights, nullptr, sink, reinterpret_cast<cudaStream_t>(stream));
  NBC_CHECK_LAUNCH();
  return 0;
}

namespace nbc {
int head_1x1(const void* x_bf16, int64_t pixels_per_image, int N, int Cin, const float* w3xC, const float* bias3,
             float* logits_planar, int f16, cudaStream_t stream, const int* valid_h, int row_w) {
  NBC_REQUIRE(x_bf16 && w3xC && bias3 && logits_planar, "nbc_head_1x1: null pointer");
  NBC_REQUIRE((Cin == 256 || Cin == 512 || Cin == 1024) && N > 0 && pixels_per_image > 0,
              "nbc_head_1x1: Cin must be 256, 512 or 1024 (got %d)", Cin);
  const int64_t M = (int64_t)N * pixels_per_image;
  NBC_REQUIRE(M < (1ll << 31) - (1 << 24), "nbc_head_1x1: N * pixels_per_image must be < 2^31");
  const int64_t want = ceil_div64(M, 8 * 4);
  const int blocks = (int)(want < 148 * 8 ? (want < 1 ? 1 : want) : 148 * 8);
  const __nv_bfloat16* xb = reinterpret_cast<const __nv_bfloat16*>(x_bf16);
  if (Cin == 256)
    head1x1_kernel<1><<<blocks, 256, 0, stream>>>(xb, (int)pixels_per_image, N, Cin, w3xC, bias3, logits_planar, f16, valid_h, row_w);
  else if (Cin == 512)
    head1x1_kernel<2><<<blocks, 256, 0, stream>>>(xb, (int)pixels_per_image, N, Cin, w3xC, bias3, logits_planar, f16, valid_h, row_w);
  else
    head1x1_kernel<4><<<blocks, 256, 0, stream>>>(xb, (int)pixels_per_image, N, Cin, w3xC, bias3, logits_planar, f16, valid_h, row_w);
  NBC_CHECK_LAUNCH();
  return 0;
}
}  // namespace nbc

extern "C" int nbc_head_1x1(const void* x_bf16, int64_t pixels_per_image, int N, int Cin, int f16, const float* w3xC,
                            const float* bias3, float* logits_planar, void* stream) {
  return head_1x1(x_bf16, pixels_per_image, N, Cin, w3xC, bias3, logits_planar, f16 ? 1 : 0,
                  reinterpret_cast<cudaStream_t>(stream), nullptr, 1);
}

static int upsample_common(const float* logits, int N, int C, int h, int w, int H, int W, uint8_t* mask, float* out,
                           cudaStream_t stream) {
  NBC_REQUIRE(logits && (mask || out), "nbc_upsample: null pointer");
  NBC_REQUIRE(N > 0 && C > 0 && h > 0 && w > 0 && H > 0 && W > 0 && H <= 65535 && N <= 65535, "nbc_upsample: bad shape");
  const float sy = (float)h / (float)H, sx = (float)w / (float)W;  // IEEE f32 division, as torch
  dim3 grid(ceil_div(W, 256), H, N);
  if (mask && C == 3)
    launch_k3(1, k3_one(logits), N, h, w, H, W, h, nullptr, mask, K3Mask(), stream);
  else if (mask)
    upsample_kernel<true><<<grid, 256, 0, stream>>>(logits, N, C, h, w, H, W, sy, sx, mask, nullptr);
  else
    upsample_kernel<false><<<grid, 256, 0, stream>>>(logits, N, C, h, w, H, W, sy, sx, nullptr, out);
  NBC_CHECK_LAUNCH();
  return 0;
}

extern "C" int nbc_upsample_argmax(const float* logits, int N, int h, int w, int H, int W, uint8_t* mask,
                                   void* stream) {
  NBC_REQUIRE(mask, "nbc_upsample_argmax: null mask");
  return upsample_common(logits, N, 3, h, w, H, W, mask, nullptr, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int nbc_upsample_bicubic(const float* logits, int N, int C, int h, int w, int H, int W, float* out,
                                    void* stream) {
  NBC_REQUIRE(out, "nbc_upsample_bicubic: null out");
  return upsample_common(logits, N, C, h, w, H, W, nullptr, out, reinterpret_cast<cudaStream_t>(stream));
}
