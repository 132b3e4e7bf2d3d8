// Weight gradient of a convolution on the tcgen05 tensor cores (training path, row a14: the backward of every
// nn.Conv2d of the reference's FCN-ResNet50, __main__.py:231-269).
//
//   dW[co][ky][kx][ci] += sum over output pixels p of  dz[p][co] * x[p * stride + tap offset][ci]
//
// GEMM view per tap:  D[M = co, N = ci] = A[M, K = pixels] * B[N, K = pixels]^T.  Both operands are NHWC
// activations, i.e. the GEMM-K index (the pixel) is the SLOW dimension in memory: they are "MN-major" operands.
// A TMA box {64 channels, tw, th, 1} lands in shared memory as one 128-byte row per pixel (128B swizzle, 8-pixel
// atoms of 1024 B) -- exactly the canonical MN-major SWIZZLE_128B layout of the UMMA descriptor, with
// LBO = distance between two 64-channel blocks and SBO = 1024 (8 pixels).  No transposition anywhere.
//   * one CTA = one (co tile of 128, ci tile of BN, tap, pixel range): split-K over the pixels fills the 148 SMs
//   * K block = 64 pixels (a tw x th rectangle of the output); x is read through the same shifted / parity-lattice
//     tensor maps as the forward operand (zero fill outside the image = the conv padding)
//   * f32 accumulator in TMEM.  Epilogue: with one split, dw += acc (this CTA is the element's only writer); with
//     several, plain 16-byte stores of the partial tile to its scratch slot [item][split][128][BN], and
//     wgrad_reduce_kernel then adds the splits in a fixed order, dw = dw + sum_s partial[s], one writer per element.
//     The result depends on the shape and the SM count only, never on the order in which the CTAs finish.
// Warp roles: 0 = TMA producer, 1 = MMA issuer + TMEM owner, 2..5 = epilogue.
#include <algorithm>

#include "common.cuh"
#include "conv.h"
#include "train.h"

namespace nbc {

struct WgradTcParams {
  CUtensorMap tmDz;     // dz [N][Ho][Wo][Cout], box {64, tw, th, 1}
  CUtensorMap tmX[4];   // x  [N][H][W][Cin] (stride 1) or its four parity lattices (stride 2), box {64, tw, th, 1}
  float* dw;            // [Cout][taps][Cin]
  float* partial;       // splits > 1: scratch [grid][128][BN], slot blockIdx.x = item * splits + split; else null
  int Cout, Cin, taps;
  int tw_log2, th, tw, tiles_w, tiles_h;
  int num_pix_tiles;    // N * tiles_h * tiles_w
  int tiles_per_split, splits;
  int ci_tiles, co_tiles;
  int8_t tap_map[9];
  int16_t tap_dh[9];
  int16_t tap_dw[9];
};

constexpr int kWgThreads = 192;
constexpr int kWgPix = 64;                      // pixels (GEMM K) per pipeline stage
constexpr int kWgBlockBytes = kWgPix * 128;     // one 64-channel block of a stage: 64 pixels x 128 B

// BN == 32 is the stem: its B operand is the zero-padded staging image of the forward stem (stem.cu),
// [N][Hp][Wp][4] bf16, read as "32 channels" = 8 consecutive pixels x 4 channels per output pixel (64-byte rows,
// 64B swizzle), one tap row ky per CTA -- the same overlapping-window tensor maps as the forward implicit GEMM.
template <int BN>
struct WgCfg {
  static constexpr bool kStem = (BN == 32);
  static constexpr int kABytes = 2 * kWgBlockBytes;            // 128 co
  static constexpr int kBBytes = kStem ? kWgPix * 64 : (BN / 64) * kWgBlockBytes;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStages = (BN == 256) ? 4 : (BN == 128 ? 6 : 8);
  static constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*barriers*/ + 1024 /*align slack*/;
};

// MN-major operand, 128B swizzle: rows of 128 B = 64 channels of one pixel, 8-pixel atoms (SBO = 1024 B),
// 64-channel blocks LBO bytes apart.  Same bit layout as umma_desc_kmajor (common.cuh).
// kSwizzleBytes = 64: rows of 64 B = 32 "channels", 8-pixel atoms of 512 B, layout type 4.
template <uint32_t kSwizzleBytes = 128>
__device__ __forceinline__ uint64_t umma_desc_mnmajor(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((8 * kSwizzleBytes) >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)(kSwizzleBytes == 128 ? 2 : 4) << 61;
  return d;
}
// kind::f16 instruction descriptor with both operands MN-major (bits 15 / 16)
__host__ __device__ constexpr uint32_t umma_idesc_bf16_mn(int M, int N) {
  return umma_idesc_bf16(M, N) | (1u << 15) | (1u << 16);
}

template <int BN>
__global__ void __launch_bounds__(kWgThreads, 1) wgrad_tc_kernel(const __grid_constant__ WgradTcParams p) {
  using Cfg = WgCfg<BN>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + Cfg::kStages * Cfg::kStageBytes);
  uint64_t* empty_bar = full_bar + Cfg::kStages;
  uint64_t* tfull_bar = empty_bar + Cfg::kStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tfull_bar + 1);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;

  // work item of this CTA
  int item = blockIdx.x;
  const int split = item % p.splits;
  item /= p.splits;
  const int tap = item % p.taps;
  item /= p.taps;
  const int ci_tile = item % p.ci_tiles;
  const int co_tile = item / p.ci_tiles;
  const int t_begin = split * p.tiles_per_split;
  const int t_end = min(p.num_pix_tiles, t_begin + p.tiles_per_split);
  const int kblocks = t_end - t_begin;

  if (threadIdx.x == 0) {
    for (int i = 0; i < Cfg::kStages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    mbar_init(tfull_bar, 1);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, BN);
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmDz);
    tma_prefetch_desc(&p.tmX[p.tap_map[tap]]);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);

  if (kblocks > 0) {
    if (warp == 0) {
      // ================================ TMA producer ================================
      if (elect_one()) {
        const CUtensorMap* mX = &p.tmX[p.tap_map[tap]];
        const int dh = p.tap_dh[tap], dw_ = p.tap_dw[tap];
        uint32_t stage = 0, phase = 0;
        for (int t = t_begin; t < t_end; ++t) {
          const int tw_i = t % p.tiles_w;
          const int r = t / p.tiles_w;
          const int th_i = r % p.tiles_h;
          const int img = r / p.tiles_h;
          const int w0 = tw_i << p.tw_log2, h0 = th_i * p.th;
          mbar_wait(&empty_bar[stage], phase ^ 1u, 100 + (int)stage);
          uint8_t* s = smem + stage * Cfg::kStageBytes;
          mbar_expect_tx(&full_bar[stage], Cfg::kStageBytes);
#pragma unroll
          for (int i = 0; i < 2; ++i) tma_load_4d(s + i * kWgBlockBytes, &p.tmDz, &full_bar[stage], co_tile * 128 + i * 64, w0, h0, img);
          if (Cfg::kStem) {
            tma_load_4d(s + Cfg::kABytes, mX, &full_bar[stage], 0, w0 + dw_, h0 + dh, img);
          } else {
#pragma unroll
            for (int j = 0; j < BN / 64; ++j)
              tma_load_4d(s + Cfg::kABytes + j * kWgBlockBytes, mX, &full_bar[stage], ci_tile * BN + j * 64, w0 + dw_, h0 + dh, img);
          }
          if (++stage == Cfg::kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      // ================================ MMA issuer ================================
      if (elect_one()) {
        constexpr uint32_t idesc = umma_idesc_bf16_mn(128, BN);
        uint32_t stage = 0, phase = 0;
        for (int kb = 0; kb < kblocks; ++kb) {
          mbar_wait(&full_bar[stage], phase, 200 + (int)stage);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + stage * Cfg::kStageBytes);
          const uint32_t b_addr = a_addr + Cfg::kABytes;
#pragma unroll
          for (int k = 0; k < kWgPix / 16; ++k) {
            // 16 pixels = two 8-pixel atoms = 2048 B further down both operands
            const uint64_t bdesc = Cfg::kStem ? umma_desc_mnmajor<64>(b_addr + k * 1024, 0)
                                              : umma_desc_mnmajor<128>(b_addr + k * 2048, kWgBlockBytes);
            umma_bf16(tmem_base, umma_desc_mnmajor<128>(a_addr + k * 2048, kWgBlockBytes), bdesc, idesc,
                      (uint32_t)((kb | k) != 0));
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == Cfg::kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        umma_commit(tfull_bar);
      }
      __syncwarp();
    } else {
      // ================================ epilogue (warps 2..5) ================================
      const int q = warp & 3;   // TMEM lane quarter of this warp
      const int co = co_tile * 128 + q * 32 + lane;
      mbar_wait(tfull_bar, 0, 400);
      tc_fence_after();
      const bool row_ok = co < p.Cout;
      float* prow = p.partial ? p.partial + ((int64_t)blockIdx.x * 128 + q * 32 + lane) * BN : nullptr;
      float* drow = p.dw + ((int64_t)co * p.taps + tap) * p.Cin + ci_tile * BN;
#pragma unroll 1
      for (int c = 0; c < BN; c += 32) {
        uint32_t r[32];
        tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + c, r);
        tmem_ld_wait();
        if (!row_ok) continue;
        if (prow != nullptr) {
#pragma unroll
          for (int i = 0; i < 32; i += 4)
            *reinterpret_cast<float4*>(prow + c + i) =
                make_float4(__uint_as_float(r[i]), __uint_as_float(r[i + 1]), __uint_as_float(r[i + 2]), __uint_as_float(r[i + 3]));
        } else if (Cfg::kStem) {
          // column = kx * 4 + c of tap row ky = tap; the stem gradient is f32 [64][7][7][3]
          float* d = p.dw + ((int64_t)co * 49 + tap * 7) * 3;
#pragma unroll
          for (int kx = 0; kx < 7; ++kx)
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) d[kx * 3 + ch] += __uint_as_float(r[kx * 4 + ch]);
        } else {
#pragma unroll
          for (int i = 0; i < 32; i += 4) {
            float4* d = reinterpret_cast<float4*>(drow + c + i);
            float4 v = *d;
            v.x += __uint_as_float(r[i]), v.y += __uint_as_float(r[i + 1]), v.z += __uint_as_float(r[i + 2]),
                v.w += __uint_as_float(r[i + 3]);
            *d = v;
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, BN);
}

bool wgrad_tc_supported(const ConvGeom& g) {
  if (g.Cin % 64 != 0 || g.Cout % 64 != 0) return false;
  if (g.kh * g.kw > 9) return false;
  if (g.stride != 1 && g.stride != 2) return false;
  if (g.stride == 2 && (g.H < 2 || g.W < 2)) return false;
  return g.Ho() >= 1 && g.Wo() >= 1;
}

static int floordiv2(int a) { return (a >= 0) ? a / 2 : -((-a + 1) / 2); }

// Fixed-order sum of the split partials into dw.  A block covers 32 elements (float4 columns of a tile row, or single
// stem taps) x 8 groups of splits: group g adds splits [g * per, (g + 1) * per) in index order, then the group sums are
// added in group order and dw = dw + sum is stored by one thread.  The order is a function of `splits` alone.
struct WgReduceParams {
  const float* partial;
  float* dw;
  int64_t n;            // elements: float4 columns of the partial tiles, or stem gradient entries
  int splits, BN, taps, ci_tiles, Cout, Cin;
};
constexpr int kRedLanes = 32, kRedGroups = 8;

__device__ __forceinline__ float4 add4(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }

template <bool kStem>
__global__ void __launch_bounds__(kRedLanes * kRedGroups) wgrad_reduce_kernel(const WgReduceParams r) {
  __shared__ float4 part[kRedGroups][kRedLanes];
  const int lane = threadIdx.x, grp = threadIdx.y;
  const int64_t e = (int64_t)blockIdx.x * kRedLanes + lane;
  bool valid = e < r.n;
  int64_t src = 0;   // floats: the element in split 0
  float* dst = nullptr;
  if (valid) {
    if (kStem) {
      // e = (tap * 64 + co) * 21 + kx * 3 + ch; partial column kx * 4 + ch of row co in slot tap * splits + s
      const int j = (int)(e % 21);
      const int t = (int)(e / 21), co = t % 64, tap = t / 64;
      src = ((int64_t)tap * r.splits * 128 + co) * 32 + (j / 3) * 4 + j % 3;
      dst = r.dw + (co * 49 + tap * 7) * 3 + j;
    } else {
      const int vpr = r.BN / 4;
      const int c4 = (int)(e % vpr);
      const int64_t t = e / vpr;
      const int row = (int)(t % 128);
      const int64_t item = t / 128;
      const int tap = (int)(item % r.taps), ci_tile = (int)((item / r.taps) % r.ci_tiles), co_tile = (int)(item / r.taps / r.ci_tiles);
      const int co = co_tile * 128 + row;
      valid = co < r.Cout;
      src = (item * r.splits * 128 + row) * r.BN + c4 * 4;
      dst = r.dw + ((int64_t)co * r.taps + tap) * r.Cin + ci_tile * r.BN + c4 * 4;
    }
  }
  const int64_t slot = (int64_t)128 * r.BN;
  const int per = ceil_div(r.splits, kRedGroups);
  const int s0 = grp * per, s1 = min(r.splits, s0 + per);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (valid && s0 < s1) {
    if (kStem) {
      float a = r.partial[src + s0 * slot];
      for (int s = s0 + 1; s < s1; ++s) a += r.partial[src + s * slot];
      acc.x = a;
    } else {
      acc = *reinterpret_cast<const float4*>(r.partial + src + s0 * slot);
#pragma unroll 4
      for (int s = s0 + 1; s < s1; ++s) acc = add4(acc, *reinterpret_cast<const float4*>(r.partial + src + s * slot));
    }
  }
  part[grp][lane] = acc;
  __syncthreads();
  if (grp != 0 || !valid) return;
  float4 sum = part[0][lane];
  for (int g = 1; g * per < r.splits; ++g) sum = add4(sum, part[g][lane]);
  if (kStem) {
    *dst += sum.x;
  } else {
    float4* d = reinterpret_cast<float4*>(dst);
    *d = add4(*d, sum);
  }
}

// output tiling (64-pixel rectangles) and the split-K of the pixel tiles; shapes only, no pointers
static void wg_tiling(WgradTcParams& p, int N, int Ho, int Wo) {
  // 64-pixel output rectangle: fewest tiles, widest on ties
  int best_tw = 64, best_tiles = INT32_MAX;
  for (int tw = 64; tw >= 8; tw >>= 1) {
    const int tiles = ceil_div(Wo, tw) * ceil_div(Ho, 64 / tw);
    if (tiles < best_tiles) best_tiles = tiles, best_tw = tw;
  }
  p.tw = best_tw, p.th = 64 / best_tw;
  p.tw_log2 = 0;
  while ((1 << p.tw_log2) < p.tw) ++p.tw_log2;
  p.tiles_w = ceil_div(Wo, p.tw), p.tiles_h = ceil_div(Ho, p.th);
  p.num_pix_tiles = N * p.tiles_w * p.tiles_h;
}
// each split with at least 16 K blocks; splits recomputed so that none is empty
static void wg_split(WgradTcParams& p, int splits) {
  const int max_splits = ceil_div(p.num_pix_tiles, 16);
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  p.tiles_per_split = ceil_div(p.num_pix_tiles, splits);
  p.splits = ceil_div(p.num_pix_tiles, p.tiles_per_split);
}
static int wg_bn(const ConvGeom& g) {
  const int bn = (g.Cin % 256 == 0) ? 256 : (g.Cin % 128 == 0 ? 128 : 64);
  return bn;
}
// one wave: as many splits as fit the SMs once.  More, smaller splits balance better but every split adds a full tile
// of f32 partials to reduce (with the former atomics, 4x oversubscription cost 6 % of the training step)
static void wg_geometry(WgradTcParams& p, const ConvGeom& g) {
  wg_tiling(p, g.N, g.Ho(), g.Wo());
  p.Cout = g.Cout, p.Cin = g.Cin, p.taps = g.kh * g.kw;
  p.ci_tiles = g.Cin / wg_bn(g);
  p.co_tiles = ceil_div(g.Cout, 128);
  const int base_items = p.co_tiles * p.ci_tiles * p.taps;
  int splits = std::max(1, sm_count() / base_items);
  wg_split(p, splits);
}
static void wg_stem_geometry(WgradTcParams& p, int N, int Ho, int Wo) {
  wg_tiling(p, N, Ho, Wo);
  p.Cout = 64, p.Cin = 32, p.taps = 7;
  p.ci_tiles = 1, p.co_tiles = 1;
  int splits = ceil_div(sm_count() * 2, 7);
  wg_split(p, splits);
}
static size_t wg_scratch_bytes(const WgradTcParams& p, int bn) {
  return p.splits > 1 ? (size_t)p.co_tiles * p.ci_tiles * p.taps * p.splits * 128 * bn * sizeof(float) : 0;
}

size_t wgrad_tc_scratch_bytes(const ConvGeom& g) {
  if (!wgrad_tc_supported(g)) return 0;
  WgradTcParams p;
  memset(&p, 0, sizeof(p));
  wg_geometry(p, g);
  return wg_scratch_bytes(p, wg_bn(g));
}
size_t stem_wgrad_tc_scratch_bytes(int N, int Ho, int Wo) {
  WgradTcParams p;
  memset(&p, 0, sizeof(p));
  wg_stem_geometry(p, N, Ho, Wo);
  return wg_scratch_bytes(p, 32);
}

// scratch == null: one split (dw += acc in the epilogue).  Otherwise the shape's split-K, then the reduction.
template <int BN>
static int launch_wgrad(WgradTcParams& p, void* scratch, size_t scratch_bytes, cudaStream_t stream) {
  static bool attr_set = false;
  if (!attr_set) {
    NBC_CUDA(cudaFuncSetAttribute(wgrad_tc_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, WgCfg<BN>::kSmemBytes));
    attr_set = true;
  }
  if (scratch == nullptr) wg_split(p, 1);
  const size_t need = wg_scratch_bytes(p, BN);
  if (need > scratch_bytes) {
    set_error("wgrad_tc: scratch %zu < %zu bytes", scratch_bytes, need);
    return NBC_ERR_WORKSPACE;
  }
  p.partial = need > 0 ? reinterpret_cast<float*>(scratch) : nullptr;
  const int grid = p.co_tiles * p.ci_tiles * p.taps * p.splits;
  wgrad_tc_kernel<BN><<<grid, kWgThreads, WgCfg<BN>::kSmemBytes, stream>>>(p);
  NBC_CHECK_LAUNCH();
  if (p.partial == nullptr) return 0;
  WgReduceParams r;
  r.partial = p.partial, r.dw = p.dw;
  r.splits = p.splits, r.BN = BN, r.taps = p.taps, r.ci_tiles = p.ci_tiles, r.Cout = p.Cout, r.Cin = p.Cin;
  constexpr bool kStem = WgCfg<BN>::kStem;
  r.n = kStem ? (int64_t)7 * 64 * 21 : (int64_t)p.co_tiles * p.ci_tiles * p.taps * 128 * (BN / 4);
  wgrad_reduce_kernel<kStem><<<(unsigned)ceil_div64(r.n, kRedLanes), dim3(kRedLanes, kRedGroups), 0, stream>>>(r);
  NBC_CHECK_LAUNCH();
  return 0;
}

int wgrad_tc(const ConvGeom& g, const void* dz, const void* x, float* dw, void* scratch, size_t scratch_bytes,
             cudaStream_t stream) {
  if (!wgrad_tc_supported(g)) {
    set_error("wgrad_tc: unsupported shape Cin=%d Cout=%d k=%dx%d stride=%d", g.Cin, g.Cout, g.kh, g.kw, g.stride);
    return NBC_ERR_INVALID;
  }
  NBC_REQUIRE((reinterpret_cast<uintptr_t>(dw) & 15) == 0, "wgrad_tc: dw must be 16-byte aligned");
  NBC_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 15) == 0, "wgrad_tc: scratch must be 16-byte aligned");
  WgradTcParams p;
  memset(&p, 0, sizeof(p));
  wg_geometry(p, g);
  const int Ho = g.Ho(), Wo = g.Wo();
  p.dw = dw;
  const int bn = wg_bn(g);

  const uint64_t eb = 2;
  int rc = conv_encode_act_map(&p.tmDz, dz, (uint64_t)g.Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)g.N, (uint64_t)g.Cout * eb,
                               (uint64_t)Wo * g.Cout * eb, (uint64_t)Ho * Wo * g.Cout * eb, p.tw, p.th);
  if (rc) return rc;
  const char* xb = reinterpret_cast<const char*>(x);
  if (g.stride == 1) {
    rc = conv_encode_act_map(&p.tmX[0], xb, (uint64_t)g.Cin, (uint64_t)g.W, (uint64_t)g.H, (uint64_t)g.N, (uint64_t)g.Cin * eb,
                             (uint64_t)g.W * g.Cin * eb, (uint64_t)g.H * g.W * g.Cin * eb, p.tw, p.th);
    if (rc) return rc;
    for (int ky = 0; ky < g.kh; ++ky)
      for (int kx = 0; kx < g.kw; ++kx) {
        const int t = ky * g.kw + kx;
        p.tap_map[t] = 0;
        p.tap_dh[t] = (int16_t)(ky * g.dil - g.pad);
        p.tap_dw[t] = (int16_t)(kx * g.dil - g.pad);
      }
  } else {
    bool used[4] = {false, false, false, false};
    for (int ky = 0; ky < g.kh; ++ky)
      for (int kx = 0; kx < g.kw; ++kx) {
        const int t = ky * g.kw + kx;
        const int oy = ky * g.dil - g.pad, ox = kx * g.dil - g.pad;
        const int py = ((oy % 2) + 2) % 2, px = ((ox % 2) + 2) % 2;
        p.tap_map[t] = (int8_t)(py * 2 + px);
        p.tap_dh[t] = (int16_t)floordiv2(oy);
        p.tap_dw[t] = (int16_t)floordiv2(ox);
        used[py * 2 + px] = true;
      }
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px) {
        if (!used[py * 2 + px]) continue;
        const uint64_t Wd = (uint64_t)(g.W - px + 1) / 2, Hd = (uint64_t)(g.H - py + 1) / 2;
        const char* base = xb + ((uint64_t)py * g.W + px) * g.Cin * eb;
        rc = conv_encode_act_map(&p.tmX[py * 2 + px], base, (uint64_t)g.Cin, Wd, Hd, (uint64_t)g.N, 2ull * g.Cin * eb,
                                 2ull * g.W * g.Cin * eb, (uint64_t)g.H * g.W * g.Cin * eb, p.tw, p.th);
        if (rc) return rc;
      }
  }
  switch (bn) {
    case 256: return launch_wgrad<256>(p, scratch, scratch_bytes, stream);
    case 128: return launch_wgrad<128>(p, scratch, scratch_bytes, stream);
    default: return launch_wgrad<64>(p, scratch, scratch_bytes, stream);
  }
}

// stem: dW f32 [64][7][7][3] += dz^T * padded image (the bf16 staging buffer [N][Hp = 2Ho+5][Wp = 2Wo+6][4] of stem.cu)
int stem_wgrad_tc(const void* dz, const void* padded, int N, int Ho, int Wo, float* dw, void* scratch, size_t scratch_bytes,
                  cudaStream_t stream) {
  NBC_REQUIRE((reinterpret_cast<uintptr_t>(scratch) & 15) == 0, "stem_wgrad_tc: scratch must be 16-byte aligned");
  WgradTcParams p;
  memset(&p, 0, sizeof(p));
  wg_stem_geometry(p, N, Ho, Wo);
  p.dw = dw;
  const int Hp = 2 * Ho + 5, Wp = 2 * Wo + 6;
  int rc = conv_encode_act_map(&p.tmDz, dz, 64, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N, 128, (uint64_t)Wo * 128,
                               (uint64_t)Ho * Wo * 128, p.tw, p.th);
  if (rc) return rc;
  const char* base = reinterpret_cast<const char*>(padded);
  const uint64_t row_bytes = (uint64_t)Wp * 8;
  for (int py = 0; py < 2; ++py) {
    rc = conv_encode_act_map(&p.tmX[py], base + py * row_bytes, 32, (uint64_t)Wo, (uint64_t)(Hp - py + 1) / 2, (uint64_t)N, 16,
                             2 * row_bytes, (uint64_t)Hp * row_bytes, p.tw, p.th, 32);
    if (rc) return rc;
  }
  for (int ky = 0; ky < 7; ++ky) p.tap_map[ky] = (int8_t)(ky & 1), p.tap_dh[ky] = (int16_t)(ky >> 1), p.tap_dw[ky] = 0;
  return launch_wgrad<32>(p, scratch, scratch_bytes, stream);
}

}  // namespace nbc
