// Training-path kernels, part 2: maxpool backward, stem weight gradient, dropout, classifier (1x1) backward, the
// adjoint of the bicubic upsample, zero insertion for stride-2 data gradients, and Adam.
#include "common.cuh"
#include "cubic.cuh"
#include "train.h"

namespace nbc {

static int grid_for2(int64_t n) {
  const int64_t b = ceil_div64(n, 256);
  return (int)(b < 1 ? 1 : (b > 148 * 16 ? 148 * 16 : b));
}

// ------------------------------------------------------------------------------------------------ maxpool (training)
// Forward that also records, per output element, WHICH of the 9 window positions held the first maximum (row-major
// scan, torch's rule); the backward then needs no comparisons: dx[h,w] = sum of dy over the (<= 4) windows whose
// recorded position is (h,w).  One thread = 8 channels (16 bytes) of one pixel.
__global__ void __launch_bounds__(256) maxpool_fwd_idx_kernel(const uint4* __restrict__ x, int N, int H, int W, int C8, int Ho,
                                                              int Wo, uint4* __restrict__ y, uint2* __restrict__ idx) {
  const int64_t total = (int64_t)N * Ho * Wo * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C8);
    int64_t t = i / C8;
    const int wo = (int)(t % Wo);
    t /= Wo;
    const int ho = (int)(t % Ho);
    const int n = (int)(t / Ho);
    float best[8];
    uint32_t pos[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) best[e] = -INFINITY, pos[e] = 0;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int h = 2 * ho - 1 + ky;
      if (h < 0 || h >= H) continue;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int w = 2 * wo - 1 + kx;
        if (w < 0 || w >= W) continue;
        const uint4 q = __ldg(x + (((int64_t)n * H + h) * W + w) * C8 + c);
        const uint32_t u[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float a = bf16lo(u[k]), b = bf16hi(u[k]);
          if (a > best[2 * k]) best[2 * k] = a, pos[2 * k] = ky * 3 + kx;
          if (b > best[2 * k + 1]) best[2 * k + 1] = b, pos[2 * k + 1] = ky * 3 + kx;
        }
      }
    }
    y[i] = make_uint4(pack_bf16x2(best[0], best[1]), pack_bf16x2(best[2], best[3]), pack_bf16x2(best[4], best[5]),
                      pack_bf16x2(best[6], best[7]));
    idx[i] = make_uint2(pos[0] | (pos[1] << 8) | (pos[2] << 16) | (pos[3] << 24),
                        pos[4] | (pos[5] << 8) | (pos[6] << 16) | (pos[7] << 24));
  }
}

__global__ void __launch_bounds__(256) maxpool_bwd_idx_kernel(const uint4* __restrict__ dy, const uint2* __restrict__ idx, int N,
                                                              int H, int W, int C8, int Ho, int Wo, uint4* __restrict__ dx) {
  const int64_t total = (int64_t)N * H * W * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C8);
    int64_t t = i / C8;
    const int w = (int)(t % W);
    t /= W;
    const int h = (int)(t % H);
    const int n = (int)(t / H);
    float g[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) g[e] = 0.f;
    // windows (ho, wo) with 2*ho-1 <= h <= 2*ho+1
    for (int ho = h / 2; ho <= min(Ho - 1, (h + 1) / 2); ++ho) {
      const uint32_t ky = (uint32_t)(h - (2 * ho - 1));
      for (int wo = w / 2; wo <= min(Wo - 1, (w + 1) / 2); ++wo) {
        const uint32_t me = ky * 3 + (uint32_t)(w - (2 * wo - 1));
        const int64_t o = (((int64_t)n * Ho + ho) * Wo + wo) * C8 + c;
        const uint2 ix = __ldg(idx + o);
        const uint4 q = __ldg(dy + o);
        const uint32_t u[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint32_t word = k < 2 ? ix.x : ix.y;
          const uint32_t p0 = (word >> (16 * (k & 1))) & 0xFFu, p1 = (word >> (16 * (k & 1) + 8)) & 0xFFu;
          if (p0 == me) g[2 * k] += bf16lo(u[k]);
          if (p1 == me) g[2 * k + 1] += bf16hi(u[k]);
        }
      }
    }
    dx[i] = make_uint4(pack_bf16x2(g[0], g[1]), pack_bf16x2(g[2], g[3]), pack_bf16x2(g[4], g[5]), pack_bf16x2(g[6], g[7]));
  }
}

int maxpool_forward_idx(const void* x, int N, int H, int W, int C, void* y, void* idx, cudaStream_t stream) {
  NBC_REQUIRE(C % 8 == 0, "maxpool: C must be a multiple of 8");
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  maxpool_fwd_idx_kernel<<<grid_for2((int64_t)N * Ho * Wo * (C / 8)), 256, 0, stream>>>(
      reinterpret_cast<const uint4*>(x), N, H, W, C / 8, Ho, Wo, reinterpret_cast<uint4*>(y), reinterpret_cast<uint2*>(idx));
  NBC_CHECK_LAUNCH();
  return 0;
}

int maxpool_backward(const void* dy, const void* idx, int N, int H, int W, int C, void* dx, cudaStream_t stream) {
  NBC_REQUIRE(C % 8 == 0, "maxpool: C must be a multiple of 8");
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  maxpool_bwd_idx_kernel<<<grid_for2((int64_t)N * H * W * (C / 8)), 256, 0, stream>>>(
      reinterpret_cast<const uint4*>(dy), reinterpret_cast<const uint2*>(idx), N, H, W, C / 8, Ho, Wo,
      reinterpret_cast<uint4*>(dx));
  NBC_CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------------------------------------ stem weight gradient
// dW[oc][ky][kx][c] += sum_p dz[p][oc] * padded[n][2ho+ky][2wo+kx][c]   (padded = the bf16 staging image of the stem)
// block = 64 output pixels; thread (oc = tid & 63, g = tid >> 6) accumulates the taps t = g, g+4, ... (37 of 147)
__global__ void __launch_bounds__(256) stem_wgrad_kernel(const __nv_bfloat16* __restrict__ dz, const uint2* __restrict__ padded,
                                                         int N, int Ho, int Wo, int Hp, int Wp, float* __restrict__ dw) {
  __shared__ float s_in[8][16][4];   // input patch rows ky..: 7 rows x (2*? ) -- one output pixel at a time (see below)
  __shared__ float s_dz[64];
  const int tid = threadIdx.x, oc = tid & 63, g = tid >> 6;
  float acc[37];
  int off[37];   // smem offset of tap tp = g + 4 i : ((ky * 16 + kx) * 4 + c)
#pragma unroll
  for (int i = 0; i < 37; ++i) {
    acc[i] = 0.f;
    const int tp = min(g + 4 * i, 146), c = tp % 3, kk = tp / 3;
    off[i] = ((kk / 7) * 16 + (kk % 7)) * 4 + c;
  }
  const float* s_flat = &s_in[0][0][0];
  const int64_t M = (int64_t)N * Ho * Wo;
  const int64_t per_block = ceil_div64(M, gridDim.x);
  const int64_t m0 = (int64_t)blockIdx.x * per_block, m1 = min(M, m0 + per_block);
  for (int64_t m = m0; m < m1; ++m) {
    const int wo = (int)(m % Wo);
    const int64_t t = m / Wo;
    const int ho = (int)(t % Ho);
    const int n = (int)(t / Ho);
    __syncthreads();
    if (tid < 64) s_dz[tid] = __bfloat162float(dz[m * 64 + tid]);
    if (tid >= 64 && tid < 64 + 56) {   // 7 rows x 8 pixels of the padded image (the 8th pixel is never used)
      const int k = tid - 64, ky = k >> 3, kx = k & 7;
      const uint2 v = __ldg(padded + ((int64_t)n * Hp + 2 * ho + ky) * Wp + 2 * wo + kx);
      s_in[ky][kx][0] = bf16lo(v.x), s_in[ky][kx][1] = bf16hi(v.x), s_in[ky][kx][2] = bf16lo(v.y), s_in[ky][kx][3] = 0.f;
    }
    __syncthreads();
    const float d = s_dz[oc];
#pragma unroll
    for (int i = 0; i < 37; ++i) acc[i] = fmaf(d, s_flat[off[i]], acc[i]);   // tap index (ky*7 + kx)*3 + c
  }
#pragma unroll
  for (int i = 0; i < 37; ++i) {
    const int tp = g + 4 * i;
    if (tp < 147) atomicAdd(dw + oc * 147 + tp, acc[i]);
  }
}

int stem_wgrad(const void* dz, const void* padded, int N, int Ho, int Wo, float* dw, cudaStream_t stream) {
  stem_wgrad_kernel<<<148 * 8, 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(dz),
                                                 reinterpret_cast<const uint2*>(padded), N, Ho, Wo, 2 * Ho + 5, 2 * Wo + 6, dw);
  NBC_CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------------------------------------ dropout
// keep(i) = hash(seed, i) >= p, scaled by 1/(1-p); the same hash gives the backward mask, nothing is stored
__device__ __forceinline__ float hash_uniform(uint64_t seed, uint64_t i) {
  uint64_t z = seed + 0x9E3779B97F4A7C15ull * (i + 1);
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z = z ^ (z >> 31);
  return (float)(z >> 40) * (1.0f / 16777216.0f);
}
__global__ void __launch_bounds__(256) dropout_kernel(const __nv_bfloat16* __restrict__ x, int64_t n, float p, uint64_t seed,
                                                      __nv_bfloat16* __restrict__ y) {
  const float scale = 1.f / (1.f - p);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float v = __bfloat162float(x[i]);
    y[i] = __float2bfloat16_rn(hash_uniform(seed, (uint64_t)i) >= p ? v * scale : 0.f);
  }
}
int dropout_apply(const void* x, int64_t n, float p, uint64_t seed, void* y, cudaStream_t stream) {
  dropout_kernel<<<grid_for2(n), 256, 0, stream>>>(reinterpret_cast<const __nv_bfloat16*>(x), n, p, seed,
                                                   reinterpret_cast<__nv_bfloat16*>(y));
  NBC_CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------------------------------------ classifier backward
// dlow f32 [N][3][P];  x bf16 [N*P][C] (after dropout);  w f32 [3][C]
// dx[p][k] = sum_c dlow[c][p] * w[c][k]  (then through the dropout mask);  dW[c][k] += sum_p dlow[c][p] x[p][k]; db[c] += sum_p
// Each block stores its pixel slab's dW and db to partial[block][3C + 3]; cls_finalize_kernel adds the blocks in a fixed
// order, so the gradient does not depend on the order the blocks finish.
constexpr int kClsBlocks = 148 * 4;
size_t cls_partial_bytes(int C) { return (size_t)kClsBlocks * (3 * C + 3) * sizeof(float); }

__global__ void __launch_bounds__(256) cls_bwd_kernel(const float* __restrict__ dlow, const __nv_bfloat16* __restrict__ x,
                                                      const float* __restrict__ w, int N, int64_t P, int C, float drop_p,
                                                      uint64_t seed, __nv_bfloat16* __restrict__ dx, float* __restrict__ partial) {
  // thread owns channels k = tid, tid + 256, ...; block owns a slab of pixels
  const int64_t M = (int64_t)N * P;
  const int64_t per_block = ceil_div64(M, gridDim.x);
  const int64_t m0 = (int64_t)blockIdx.x * per_block, m1 = min(M, m0 + per_block);
  const float scale = 1.f / (1.f - drop_p);
  float* part = partial + (int64_t)blockIdx.x * (3 * C + 3);
  for (int k = threadIdx.x; k < C; k += blockDim.x) {
    const float w0 = w[k], w1 = w[C + k], w2 = w[2 * C + k];
    float a0 = 0.f, a1 = 0.f, a2 = 0.f;
    for (int64_t m = m0; m < m1; ++m) {
      const int64_t n = m / P, pix = m - n * P;
      const float* d = dlow + n * 3 * P + pix;
      const float d0 = __ldg(d), d1 = __ldg(d + P), d2 = __ldg(d + 2 * P);
      const float xv = __bfloat162float(x[m * C + k]);
      a0 = fmaf(d0, xv, a0), a1 = fmaf(d1, xv, a1), a2 = fmaf(d2, xv, a2);
      float g = d0 * w0 + d1 * w1 + d2 * w2;
      if (drop_p > 0.f) g = hash_uniform(seed, (uint64_t)(m * C + k)) >= drop_p ? g * scale : 0.f;
      dx[m * C + k] = __float2bfloat16_rn(g);
    }
    part[k] = a0, part[C + k] = a1, part[2 * C + k] = a2;
  }
  if (threadIdx.x < 3) {
    float s = 0.f;
    for (int64_t m = m0; m < m1; ++m) {
      const int64_t n = m / P, pix = m - n * P;
      s += dlow[n * 3 * P + threadIdx.x * P + pix];
    }
    part[3 * C + threadIdx.x] = s;
  }
}
// one warp per output: lane l adds blocks l, l + 32, ... in order, then a fixed butterfly over the lanes; one writer
__global__ void __launch_bounds__(256) cls_finalize_kernel(const float* __restrict__ partial, int C, int blocks, float* __restrict__ dw,
                                                           float* __restrict__ db) {
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int n = 3 * C + 3;
  if (i >= n) return;
  float s = 0.f;
  for (int b = lane; b < blocks; b += 32) s += partial[(int64_t)b * n + i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) {
    float* d = i < 3 * C ? dw + i : db + (i - 3 * C);
    *d += s;
  }
}
int cls_backward(const float* dlow, const void* x, const float* w, int N, int64_t P, int C, float drop_p, uint64_t seed,
                 void* dx, float* dw, float* db, void* partial, cudaStream_t stream) {
  float* part = reinterpret_cast<float*>(partial);
  cls_bwd_kernel<<<kClsBlocks, 256, 0, stream>>>(dlow, reinterpret_cast<const __nv_bfloat16*>(x), w, N, P, C, drop_p, seed,
                                                 reinterpret_cast<__nv_bfloat16*>(dx), part);
  NBC_CHECK_LAUNCH();
  cls_finalize_kernel<<<ceil_div((3 * C + 3) * 32, 256), 256, 0, stream>>>(part, C, kClsBlocks, dw, db);
  NBC_CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------------------------------------ upsample backward
// adjoint of F.interpolate(mode='bicubic', align_corners=False): dlow[n,c,i,j] = sum_{Y,X} wy(Y,i) wx(X,j) dup[n,c,Y,X],
// separable: first over X (-> T[n,c,Y,j]), then over Y.  taps tables idx/wt: [out][4]
__global__ void taps_table_kernel(int in_size, int out_size, float scale, int* __restrict__ idx, float* __restrict__ wt) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= out_size) return;
  int ix[4];
  float w[4];
  cubic_taps(d, scale, in_size, ix, w);
#pragma unroll
  for (int k = 0; k < 4; ++k) idx[4 * d + k] = ix[k], wt[4 * d + k] = w[k];
}
// Band table of the adjoint along one dimension: for low-res index j, band[j][t] = sum_k [idx(d,k) == j] * wt(d,k) with
// d = lo[j] + t -- the (dense, short) column j of the interpolation matrix.  kAdjBand bounds the band length.
constexpr int kAdjBand = 64;
__global__ void adjoint_band_kernel(int in_size /*lo-res*/, int out_size /*hi-res*/, float inv_scale, const int* __restrict__ idx,
                                    const float* __restrict__ wt, int* __restrict__ lo_out, float* __restrict__ band) {
  const int j = blockIdx.x;
  int lo = (int)floorf(((float)j - 2.5f) * inv_scale) - 2, hi = (int)ceilf(((float)j + 2.5f) * inv_scale) + 2;
  if (j == 0) lo = 0;
  if (j == in_size - 1) hi = out_size - 1;
  lo = max(lo, 0), hi = min(hi, out_size - 1);
  if (threadIdx.x == 0) lo_out[2 * j] = lo, lo_out[2 * j + 1] = hi - lo + 1;
  for (int t = threadIdx.x; t < kAdjBand; t += blockDim.x) {
    const int d = lo + t;
    float a = 0.f;
    if (d <= hi) {
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (idx[4 * d + k] == j) a += wt[4 * d + k];
    }
    band[j * kAdjBand + t] = a;
  }
}
// out[r][j] = sum_t band[j][t] * in[r][lo[j] + t] along the LAST dim; one thread = one j for 4 consecutive rows
__global__ void __launch_bounds__(256) adjoint_last_kernel(const float* __restrict__ in, int64_t rows, int out_size /*hi-res*/,
                                                           int in_size /*lo-res*/, const int* __restrict__ lo_cnt,
                                                           const float* __restrict__ band, float* __restrict__ out) {
  const int64_t groups = (rows + 3) / 4;
  const int64_t total = groups * in_size;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int j = (int)(i % in_size);
    const int64_t r0 = (i / in_size) * 4;
    const int lo = __ldg(lo_cnt + 2 * j), cnt = __ldg(lo_cnt + 2 * j + 1);
    const float* bw = band + j * kAdjBand;
    const float* src = in + r0 * out_size + lo;
    const int nr = (int)min((int64_t)4, rows - r0);
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int t = 0; t < cnt; ++t) {
      const float w = __ldg(bw + t);
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (q < nr) acc[q] = fmaf(w, __ldg(src + (int64_t)q * out_size + t), acc[q]);
    }
    for (int q = 0; q < nr; ++q) out[(r0 + q) * in_size + j] = acc[q];
  }
}
// same along the second-to-last dim: in [R][H][w] -> out [R][h][w]
__global__ void __launch_bounds__(256) adjoint_rows_kernel(const float* __restrict__ in, int64_t R, int H, int h, int w,
                                                           float inv_scale, const int* __restrict__ idx,
                                                           const float* __restrict__ wt, float* __restrict__ out) {
  const int64_t total = R * h * w;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int x = (int)(i % w);
    int64_t t = i / w;
    const int j = (int)(t % h);
    const int64_t r = t / h;
    int lo = (int)floorf(((float)j - 2.5f) * inv_scale) - 2, hi = (int)ceilf(((float)j + 2.5f) * inv_scale) + 2;
    if (j == 0) lo = 0;
    if (j == h - 1) hi = H - 1;
    lo = max(lo, 0), hi = min(hi, H - 1);
    const float* src = in + r * H * w + x;
    float acc = 0.f;
    for (int d = lo; d <= hi; ++d) {
      const float v = __ldg(src + (int64_t)d * w);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (__ldg(idx + 4 * d + k) == j) acc = fmaf(__ldg(wt + 4 * d + k), v, acc);
    }
    out[i] = acc;
  }
}
size_t upsample_bwd_workspace_bytes(int N, int C, int h, int w, int H, int W) {
  return align_up((size_t)N * C * H * w * 4, 256) + align_up((size_t)(H + W) * 4 * 8, 256) +
         align_up((size_t)w * (kAdjBand + 2) * 4, 256);
}
int upsample_backward(const float* dup, int N, int C, int h, int w, int H, int W, float* dlow, void* workspace,
                      cudaStream_t stream) {
  char* ws = reinterpret_cast<char*>(workspace);
  float* T = reinterpret_cast<float*>(ws);
  char* tb = ws + align_up((size_t)N * C * H * w * 4, 256);
  int* idx_x = reinterpret_cast<int*>(tb);
  float* wt_x = reinterpret_cast<float*>(tb + (size_t)W * 16);
  int* idx_y = reinterpret_cast<int*>(tb + (size_t)W * 32);
  float* wt_y = reinterpret_cast<float*>(tb + (size_t)W * 32 + (size_t)H * 16);
  const float sx = (float)w / (float)W, sy = (float)h / (float)H;
  taps_table_kernel<<<ceil_div(W, 128), 128, 0, stream>>>(w, W, sx, idx_x, wt_x);
  NBC_CHECK_LAUNCH();
  taps_table_kernel<<<ceil_div(H, 128), 128, 0, stream>>>(h, H, sy, idx_y, wt_y);
  NBC_CHECK_LAUNCH();
  // the band of hi-res positions that touch one low-res column must fit the table
  NBC_REQUIRE((int)ceilf(5.f * (float)W / (float)w) + 6 <= kAdjBand, "upsample_backward: scale %d/%d too large", W, w);
  char* bt = tb + align_up((size_t)(H + W) * 4 * 8, 256);
  int* lo_cnt = reinterpret_cast<int*>(bt);
  float* band = reinterpret_cast<float*>(bt + (size_t)w * 8);
  adjoint_band_kernel<<<w, 64, 0, stream>>>(w, W, (float)W / (float)w, idx_x, wt_x, lo_cnt, band);
  NBC_CHECK_LAUNCH();
  adjoint_last_kernel<<<grid_for2(((int64_t)N * C * H + 3) / 4 * w), 256, 0, stream>>>(dup, (int64_t)N * C * H, W, w, lo_cnt, band, T);
  NBC_CHECK_LAUNCH();
  adjoint_rows_kernel<<<grid_for2((int64_t)N * C * h * w), 256, 0, stream>>>(T, (int64_t)N * C, H, h, w, (float)H / (float)h,
                                                                           idx_y, wt_y, dlow);
  NBC_CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------------------------------------ zero insertion
// up[n, 2h, 2w, :] = dz[n, h, w, :], zero elsewhere  (data gradient of a stride-2 conv = stride-1 conv of this)
__global__ void __launch_bounds__(256) zero_insert_kernel(const uint4* __restrict__ dz, int N, int Ho, int Wo, int H, int W, int C8,
                                                          uint4* __restrict__ up) {
  const int64_t total = (int64_t)N * H * W * C8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % C8);
    int64_t t = i / C8;
    const int w = (int)(t % W);
    t /= W;
    const int h = (int)(t % H);
    const int n = (int)(t / H);
    uint4 v = make_uint4(0, 0, 0, 0);
    if ((h & 1) == 0 && (w & 1) == 0 && (h >> 1) < Ho && (w >> 1) < Wo)
      v = __ldg(dz + (((int64_t)n * Ho + (h >> 1)) * Wo + (w >> 1)) * C8 + c);
    up[i] = v;
  }
}
int zero_insert(const void* dz, int N, int Ho, int Wo, int H, int W, int C, void* up, cudaStream_t stream) {
  zero_insert_kernel<<<grid_for2((int64_t)N * H * W * (C / 8)), 256, 0, stream>>>(reinterpret_cast<const uint4*>(dz), N, Ho, Wo,
                                                                               H, W, C / 8, reinterpret_cast<uint4*>(up));
  NBC_CHECK_LAUNCH();
  return 0;
}

// ------------------------------------------------------------------------------------------------ Adam
// torch.optim.Adam (amsgrad=False, L2 weight decay added to the gradient), one fused pass over the flat buffers
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                   float* __restrict__ v, int64_t n, float lr, float b1, float b2, float eps,
                                                   float wd, float bc1, float bc2_sqrt, float grad_scale) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float gi = g[i] * grad_scale;
    const float pi = p[i];
    gi = fmaf(wd, pi, gi);
    const float mi = m[i] + (1.f - b1) * (gi - m[i]);          // lerp, as torch
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi, v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] = pi - (lr / bc1) * (mi / denom);
  }
}
int adam_step(float* p, const float* g, float* m, float* v, int64_t n, float lr, float b1, float b2, float eps, float wd,
              int step, float grad_scale, cudaStream_t stream) {
  const float bc1 = 1.f - powf(b1, (float)step), bc2 = 1.f - powf(b2, (float)step);
  adam_kernel<<<grid_for2(n), 256, 0, stream>>>(p, g, m, v, n, lr, b1, b2, eps, wd, bc1, sqrtf(bc2), grad_scale);
  NBC_CHECK_LAUNCH();
  return 0;
}

}  // namespace nbc
