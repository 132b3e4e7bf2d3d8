// Device arithmetic shared by the per-call losses (wce.cu, lovasz.cu) and the batched evaluation (eval.cu).  Each
// function is the one definition of its expression: a caller that inlines it computes bit for bit what the others do.
#pragma once
#include "common.cuh"

namespace nbc {

constexpr int kLvThreads = 256;
constexpr int kWceBlocks = 148 * 8;      // grid cap of the K4 reduction

struct LovaszHeader {
  int gts[3];        // pixels per label
  int pad;
  float loss[3];     // per-class loss (only meaningful where gts > 0)
  float pad2;
};

struct FgOf {
  __host__ __device__ __forceinline__ uint32_t operator()(const uint32_t& v) const { return v >> 31; }
};

__device__ __forceinline__ void softmax3(float a, float b, float c, float (&p)[3]) {
  const float m = fmaxf(a, fmaxf(b, c));
  const float ea = expf(a - m), eb = expf(b - m), ec = expf(c - m);
  const float s = ea + eb + ec;
  p[0] = ea / s, p[1] = eb / s, p[2] = ec / s;
}

// the error whose descending order drives the Lovasz extension: |[t == c] - p_c| (lovasz_losses.py:204-212)
__device__ __forceinline__ float lovasz_error(float p, bool fg) { return fabsf((fg ? 1.f : 0.f) - p); }

// K4's per-pixel term: CE(l, t) * weights[max(argmax l, t)] (utils.py:151-165).  e0..e2, s feed the gradient.
__device__ __forceinline__ float wce_term(float l0, float l1, float l2, int t, float w0, float w1, float w2, float& e0,
                                          float& e1, float& e2, float& s, float& w) {
  int am = 0;
  float mx = l0;
  if (l1 > mx) mx = l1, am = 1;
  if (l2 > mx) mx = l2, am = 2;
  e0 = expf(l0 - mx), e1 = expf(l1 - mx), e2 = expf(l2 - mx);
  s = e0 + e1 + e2;
  const float lse = mx + logf(s);
  const float lt = (t == 0) ? l0 : (t == 1 ? l1 : l2);
  const int mc = max(am, t);
  w = (mc == 0) ? w0 : (mc == 1 ? w1 : w2);
  return (lse - lt) * w;
}

// sum of a 256-thread block's double values: warp butterflies, then the 8 warp sums in order (valid on thread 0)
__device__ __forceinline__ double wce_block_sum(double local, double* s_part /* [8] shared */) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = local;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int k = 0; k < 8; ++k) s += s_part[k];
  return s;
}

// the loss from the block partials, summed in block order
__device__ __forceinline__ float wce_partials_mean(const double* __restrict__ partial, int n, double inv_total) {
  double s = 0.0;
  for (int i = 0; i < n; ++i) s += partial[i];
  return (float)(s * inv_total);
}

// Lovasz gradient at rank i of a class with G labelled pixels, cf = cumsum(fg) up to and including rank i, fg = the
// indicator at rank i: exactly the reference's f32 expression 1 - intersection / union, differenced (lovasz_losses.py:19-31)
__device__ __forceinline__ float lovasz_rank_grad(int G, int64_t i, uint32_t cf, uint32_t fg) {
  const float gts = (float)G;
  const float inter = gts - (float)cf;
  const float uni = gts + (float)((uint32_t)(i + 1) - cf);
  float g = 1.f - inter / uni;
  if (i > 0) {
    const uint32_t cfp = cf - fg;
    const float inter_p = gts - (float)cfp;
    const float uni_p = gts + (float)((uint32_t)i - cfp);
    g = g - (1.f - inter_p / uni_p);
  }
  return g;
}

// f32 sum of a kLvThreads block's contributions: warp butterflies, then the warp sums in order (valid on thread 0)
__device__ __forceinline__ float lovasz_block_sum(float contrib, float* s_part /* [kLvThreads / 32] shared */) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) contrib += __shfl_xor_sync(0xffffffffu, contrib, o);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = contrib;
  __syncthreads();
  float s = 0.f;
  if (threadIdx.x == 0)
    for (int w = 0; w < kLvThreads / 32; ++w) s += s_part[w];
  return s;
}

// one class's loss from its block partials: double, 256 threads, fixed order (valid on thread 0)
__device__ __forceinline__ float lovasz_partials_sum(const float* __restrict__ partial, int nblocks, double* s /* [256] shared */) {
  double a = 0.0;
  for (int i = threadIdx.x; i < nblocks; i += 256) a += (double)partial[i];
  s[threadIdx.x] = a;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) s[threadIdx.x] += s[threadIdx.x + o];
    __syncthreads();
  }
  return (float)s[0];
}

// mean() of lovasz_losses.py:258-276 over the present classes: acc / n, 0 when none is present
__device__ __forceinline__ float lovasz_present_mean(const int (&gts)[3], const float (&loss)[3]) {
  int np = 0;
  float acc = 0.f;
  for (int c = 0; c < 3; ++c)
    if (gts[c] > 0) acc += loss[c], ++np;
  return np > 0 ? acc / (float)np : 0.f;
}

}  // namespace nbc
