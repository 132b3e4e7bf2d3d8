// K2 -- implicit-GEMM convolution on the 5th-gen tensor cores (tcgen05.mma, TMEM accumulators, TMA operands).
//
// Replaces every nn.Conv2d + BatchNorm2d (+ReLU, +residual add) of the reference's FCN-ResNet50
// (models.py:113-139 FCNHead / fcn_resnet50; torchvision Bottleneck) for Cin % 64 == 0, Cout % 64 == 0.
//
// GEMM view:  D[M = N*Ho*Wo pixels, Cout] = A[M, K = taps*Cin] * W[Cout, K]^T   (bf16 x bf16 -> f32)
//   * M tile  = a th x tw rectangle of 128 output pixels of one image.  For tap (ky,kx) and channel block c the A
//     operand is ONE 4-D TMA box {64 ch, tw, th, 1} of the NHWC input shifted by the tap offset; out-of-bounds
//     coordinates (the conv zero padding, ragged image edges) are zero-filled by the TMA unit.
//   * stride-2 convs read one of four "parity lattices" of the input (tensor maps with doubled strides), so the
//     box stays dense; the tap table says which lattice and which shift.
//   * B operand = TMA box {64 k, BLOCK_N} of the packed weights [Cout][kh][kw][Cin] (BN scale folded in).
//   * both land in 128B-swizzled K-major smem and are consumed by tcgen05.mma (M=128, N=BLOCK_N, K=16) issued
//     by one thread; the f32 accumulator lives in TMEM, double buffered so the epilogue of tile i overlaps the
//     main loop of tile i+1.
//   * epilogue (8 warps): tcgen05.ld -> + bias (+ residual) -> ReLU -> bf16 -> 128B-swizzled staging buffer in
//     shared memory -> TMA store.  The residual group is prefetched INTO the staging buffer by TMA and updated in
//     place, so residual reads and output writes are full 128-byte lines issued by the copy engine, not by the LSU.
//
// One skeleton, four kernels.  Every kernel is a persistent CTA (one per SM) with the same warp roles:
//   warp 0 = operand producer, warp 1 = MMA issuer + TMEM owner, warps 2..9 = epilogue (epilogue_role),
//   warp 10 = output / residual TMA (output_role).
// tc_prologue / tc_teardown (shared memory layout, barriers, TMEM, programmatic dependent launch, ragged map) and the
// two output-side roles are shared; a kernel only writes its producer and MMA issuer, and names the tile walk its
// roles follow (CtaWalk: one CTA per tile; PairWalk: a CTA pair per two tiles).
//   conv_tc_kernel        the general case: one shifted TMA box per (tap, channel block), cta_group::1.
//   conv_tc_pair_kernel   clusters of 2 CTAs, one M = 256 cta_group::2 MMA over both SMs, half a weight tile per CTA;
//                         want_pair() holds the measured rule that picks it.
//   conv_tc_stem_kernel   the stem's 128 x 1 tiles out of 7 bulk-copied input rows, weights resident.
//   conv_tc_halo3_kernel  layer1's 64 -> 64 3x3 out of one halo box per 128 x 1 tile, weights resident.
// Consecutive conv launches are chained by programmatic dependent launch.
#include "common.cuh"
#include "conv.h"

namespace nbc {

struct ConvTcParams {
  CUtensorMap tmA[4];
  CUtensorMap tmB;
  CUtensorMap tmOut;  // output [N][Ho][Wo][Cout], box {64 ch, tw, th, 1}: one 64-channel group of a tile per TMA store
  CUtensorMap tmRes;  // residual, same geometry (RES kernels only)
  const float* bias;
  const __nv_bfloat16* residual;
  __nv_bfloat16* out;
  int N, Ho, Wo, Cout;
  int tw_log2, th, tw, tiles_w, tiles_h;
  int num_m_tiles, num_n_tiles;
  int n_taps, cblocks;
  // optional SECOND operand source accumulated into the same tile (a 1x1 convolution of another tensor: the
  // downsample branch of a bottleneck fused into its conv3): cblocks2 K blocks read through tmA[map2] at the tile's own
  // pixel coordinates, after the taps of the main source; its weights follow the main ones along K.  0 = none.
  int cblocks2, map2;
  int relu;
  int f16;  // operand / output format: 0 bf16, 1 fp16
  // ragged batches: valid_h[img] = number of valid OUTPUT rows of image img (nullptr: all rows valid).  Rows at or
  // beyond it are written as zeros (at least kRaggedHalo of them: the zero padding the next layer reads); tiles
  // that start beyond the halo are skipped.
  const int* valid_h;
  int8_t tap_map[9];
  int16_t tap_dh[9];
  int16_t tap_dw[9];
  // stem only (conv_tc_stem_kernel): the zero-padded staging image [N][stem_hp][stem_wp][4] (see stem.cu)
  const uint8_t* stem_src;
  int stem_hp, stem_wp;
};

constexpr int kRaggedHalo = 4;   // >= the largest padding / dilation of any consumer (layer4: dilation 4)
constexpr int kTcThreads = 352;  // warp 0 TMA operands, warp 1 MMA, warps 2..9 epilogue, warp 10 output / residual TMA
constexpr int kOutBufBytes = 128 * 64 * 2;  // 128 pixels x 64 channels x 16 bit: one output group of a tile
constexpr int kSmemLimit = 232448;          // 227 KB of dynamic shared memory per CTA on sm_100
constexpr int kMaxRaggedImages = 64;
constexpr int kMapBytes = 512;   // ragged tile map (see ragged_map_setup): behind the 256-byte barrier block

// Shared memory of every conv kernel, in this order from a 1024-aligned base: STAGES operand stages of STAGE_BYTES,
// W_BYTES of resident weights (halo kernels; 0 otherwise), OB output staging buffers of 16 KB, the barrier block, the
// ragged map.  BN = output channels per tile; PAIR = a CTA of conv_tc_pair_kernel.
constexpr int tc_fixed_bytes(int w_bytes, int ob) { return w_bytes + ob * kOutBufBytes + 256 /*barriers*/ + kMapBytes + 1024 /*align slack*/; }
constexpr int tc_stages(int stage_bytes, int fixed_bytes, int max_stages) {
  return (kSmemLimit - fixed_bytes) / stage_bytes < max_stages ? (kSmemLimit - fixed_bytes) / stage_bytes : max_stages;
}
template <int STAGES, int STAGE_BYTES, int W_BYTES, int BN, int OB, bool PAIR>
struct TcLayout {
  static constexpr int kStages = STAGES;
  static constexpr int kStageBytes = STAGE_BYTES;
  static constexpr int kWBytes = W_BYTES;
  static constexpr int kOB = OB;
  static constexpr bool kPair = PAIR;
  static constexpr int kUsedBytes = STAGES * STAGE_BYTES + tc_fixed_bytes(W_BYTES, OB);
  // > half an SM's shared memory keeps one CTA (one TMEM owner) per SM
  static constexpr int kSmemBytes = kUsedBytes < 120 * 1024 ? 120 * 1024 : kUsedBytes;
  static constexpr int kTmemCols = 2 * BN;                  // two accumulator buffers
  static constexpr int kSteps = BN / 64;                    // 64-channel output groups ("steps") per tile
  static constexpr int kWarpsPerStep = (BN == 64) ? 8 : 4;  // epilogue warps that fill one staging buffer
  static_assert(STAGES >= 2 && kUsedBytes <= kSmemLimit, "shared memory budget");
  static_assert((STAGES * STAGE_BYTES) % 1024 == 0 && W_BYTES % 1024 == 0, "staging buffers 1024-aligned");
  static_assert((2 * STAGES + 4 + 2 * OB + 1) * 8 + 4 <= 256, "barrier block");
};

// conv_tc_kernel.  KBLK = K elements per pipeline stage: 64 (128-byte swizzle) for the bottleneck / head convs, 32
// (64-byte swizzle) for the per-window stem, whose K block is one 7-tap row of 8 pixels x 4 channels.
// OB = output staging buffers: 4 when the epilogue sets the pace (residual layers, K <= 512), 2 (and a deeper operand
// ring) when the MMA main loop does.
template <int BN, int KBLK, int OB>
struct TcCfg : TcLayout<tc_stages(128 * KBLK * 2 + BN * KBLK * 2, tc_fixed_bytes(0, OB), BN == 256 ? 4 : (BN == 128 ? 6 : 8)),
                        128 * KBLK * 2 + BN * KBLK * 2, 0, BN, OB, false> {
  static constexpr int kABytes = 128 * KBLK * 2;        // 128 pixels x KBLK bf16
  static constexpr uint32_t kSwizzleBytes = KBLK * 2;   // 128 or 64
};
// conv_tc_pair_kernel: each CTA stages its 128 pixels of A and HALF of the weight tile
template <int BN, int OB>
struct TcCfgPair : TcLayout<tc_stages(128 * 64 * 2 + (BN / 2) * 64 * 2, tc_fixed_bytes(0, OB), 8), 128 * 64 * 2 + (BN / 2) * 64 * 2,
                            0, BN, OB, true> {
  static constexpr int kABytes = 128 * 64 * 2;
  static_assert(BN == 128 || BN == 256, "pair kernel: BN = 128 or 256");
};

struct TileCoord {
  int img, h0, w0, n_tile;
};
__device__ __forceinline__ TileCoord tile_coord(const ConvTcParams& p, int tile) {
  TileCoord t;
  t.n_tile = tile % p.num_n_tiles;
  int m_tile = tile / p.num_n_tiles;
  const int tw_i = m_tile % p.tiles_w;
  m_tile /= p.tiles_w;
  const int th_i = m_tile % p.tiles_h;
  t.img = m_tile / p.tiles_h;
  t.w0 = tw_i << p.tw_log2;
  t.h0 = th_i * p.th;
  return t;
}
// Ragged batches: the CTAs walk a COMPACT enumeration of the M tiles -- per image only the tiles that start above row
// valid_h + kRaggedHalo (live tiles, then the few zero-halo tiles) -- so that the static round-robin over the persistent
// CTAs stays balanced.  (Walking the dense numbering and skipping dead tiles left some CTAs with up to 20 % more live
// tiles than others: the network pass of a real chunk, mean 610 of 1024 rows, took 5.9 ms against 4.9 ms for a dense
// batch of the same work.)  s_map[i] = enumerated M tiles of the images before i, s_map[N] = their total; a virtual M
// index maps back to the dense m_tile the rest of the kernel works with.  The map holds kMaxRaggedImages images; larger
// ragged batches walk the dense numbering and skip dead tiles.
static_assert((kMaxRaggedImages + 1) * 4 <= kMapBytes, "ragged map");
__host__ __device__ __forceinline__ bool ragged_mapped(const ConvTcParams& p) {
  return p.valid_h != nullptr && p.N <= kMaxRaggedImages;
}
__device__ __forceinline__ bool ragged_map_setup(const ConvTcParams& p, int* s_map) {
  const bool mapped = ragged_mapped(p);   // uniform over the grid
  if (mapped) {
    if (threadIdx.x == 0) {
      int acc = 0;
      for (int i = 0; i < p.N; ++i) {
        s_map[i] = acc;
        const int rows = min(max(__ldg(p.valid_h + i), 0) + kRaggedHalo, p.Ho);
        acc += min((rows + p.th - 1) / p.th, p.tiles_h) * p.tiles_w;
      }
      s_map[p.N] = acc;
    }
    __syncthreads();
  }
  return mapped;
}
// dense m_tile of virtual M index vm (num_m_tiles = "beyond the last": a phantom for the pair kernel).  `hint` is the
// caller's cursor (the image of its previous lookup): every walker visits its tiles in increasing order, so the search
// is one or two shared-memory reads, not a scan -- this runs once per tile in single threads that pace the pipeline.
__device__ __forceinline__ int ragged_real_m(const ConvTcParams& p, const int* s_map, int vm, int& hint) {
  if (s_map == nullptr) return vm;
  if (vm >= s_map[p.N]) return p.num_m_tiles;
  int img = (s_map[hint] <= vm) ? hint : 0;
  while (s_map[img + 1] <= vm) ++img;
  hint = img;
  return img * p.tiles_h * p.tiles_w + (vm - s_map[img]);
}
__device__ __forceinline__ bool mtile_dead(const ConvTcParams& p, int m_tile) {
  if (m_tile >= p.num_m_tiles) return true;
  if (p.valid_h == nullptr) return false;
  const int mt = m_tile / p.tiles_w;
  return (mt % p.tiles_h) * p.th >= __ldg(p.valid_h + mt / p.tiles_h);
}

// ------------------------------------------------------------------------------------------------------------
// Tile walks.  Each role of a CTA visits the tiles i = first(), first() + step(), ... < total in order and asks at(i, hint)
// for this CTA's tile: its coordinates and "dead" (starts at or below the last valid row of its image: no loads, no
// MMA).  Every role keeps its own hint, so each does one ragged-map lookup per tile.
// ------------------------------------------------------------------------------------------------------------
struct Tile {
  TileCoord t;
  bool dead;
};
// one CTA per tile, over the (virtual, see ragged_map_setup) tiles
struct CtaWalk {
  const int* s_map;
  int total;
  __device__ __forceinline__ CtaWalk(const ConvTcParams& p, const int* map)
      : s_map(map), total((map ? map[p.N] : p.num_m_tiles) * p.num_n_tiles) {}
  __device__ __forceinline__ int first() const { return blockIdx.x; }
  __device__ __forceinline__ int step() const { return gridDim.x; }
  __device__ __forceinline__ Tile at(const ConvTcParams& p, int vt, int& hint) const {
    int tile = vt;
    if (s_map != nullptr) {
      const int vm = vt / p.num_n_tiles;
      tile = ragged_real_m(p, s_map, vm, hint) * p.num_n_tiles + (vt - vm * p.num_n_tiles);
    }
    Tile v;
    v.t = tile_coord(p, tile);
    v.dead = p.valid_h != nullptr && v.t.h0 >= __ldg(p.valid_h + v.t.img);
    return v;
  }
  __device__ __forceinline__ static bool phantom(const ConvTcParams&, const TileCoord&) { return false; }
  // the epilogue warps hand accumulator buffer `bar` back to the MMA warp
  __device__ __forceinline__ static void release_acc(uint64_t* bar) { mbar_arrive(bar); }
};
// CTA pairs: pair tiles are numbered over (virtual) M pairs; the two M tiles of a pair need not be neighbours.  CTA
// `rank` gets its own tile of the pair, "dead" only when BOTH tiles of the pair are.  An M tile beyond the last one
// (odd tile count) is a phantom: its loads are zero-filled and its stores dropped by the TMA unit.
struct PairWalk {
  const int* s_map;
  int cluster_id, num_clusters, total, rank;
  __device__ __forceinline__ PairWalk(const ConvTcParams& p, const int* map)
      : s_map(map), cluster_id(blockIdx.x >> 1), num_clusters(gridDim.x >> 1),
        total((((map ? map[p.N] : p.num_m_tiles) + 1) >> 1) * p.num_n_tiles), rank((int)cluster_ctarank()) {}
  __device__ __forceinline__ int first() const { return cluster_id; }
  __device__ __forceinline__ int step() const { return num_clusters; }
  __device__ __forceinline__ Tile at(const ConvTcParams& p, int pt, int& hint) const {
    const int mp = pt / p.num_n_tiles, n = pt - mp * p.num_n_tiles;
    const int m0 = ragged_real_m(p, s_map, 2 * mp, hint);
    const int m1 = ragged_real_m(p, s_map, 2 * mp + 1, hint);
    Tile r;
    r.dead = mtile_dead(p, m0) && mtile_dead(p, m1);
    r.t = tile_coord(p, (rank ? m1 : m0) * p.num_n_tiles + n);
    return r;
  }
  __device__ __forceinline__ static bool phantom(const ConvTcParams& p, const TileCoord& t) { return t.img >= p.N; }
  // "accumulator empty" lives in the leader: both CTAs' epilogue warps arrive there
  __device__ __forceinline__ static void release_acc(uint64_t* bar) { mbar_arrive_cluster(mapa_shared(smem_u32(bar), 0)); }
};

// ------------------------------------------------------------------------------------------------------------
// Prologue and teardown
// ------------------------------------------------------------------------------------------------------------
struct TcShared {
  uint8_t* stages;         // operand ring
  uint8_t* wres;           // resident weights
  uint8_t* obuf;           // output staging buffers
  uint64_t* full_bar;      // operand stage landed (pair: in the leader, both producers' bytes)
  uint64_t* empty_bar;     // operand stage consumed by the MMAs
  uint64_t* tfull_bar;     // accumulator buffer complete
  uint64_t* tempty_bar;    // accumulator buffer read out by the epilogue (pair: in the leader, both epilogues)
  uint64_t* bufready_bar;  // staging buffer may be used by the epilogue (residual landed / store drained)
  uint64_t* outready_bar;  // staging buffer holds a finished output group
  uint64_t* w_bar;         // resident weights landed
  const int* s_map;        // ragged tile map, nullptr: dense numbering
  uint32_t tmem_base;
};

// a_map: the operand map the producer prefetches (nullptr: none); res: the kernel reads a residual
template <class Cfg>
__device__ __forceinline__ TcShared tc_prologue(const ConvTcParams& p, int warp, const CUtensorMap* a_map, bool res) {
  extern __shared__ uint8_t smem_raw[];
  // in a pair the dynamic shared window starts at the same offset in both CTAs (same kernel, no static shared memory),
  // so the aligned buffers and barriers sit at identical offsets -- which cta_group::2 MMA descriptors and multicast
  // commits need
  TcShared s;
  s.stages = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  s.wres = s.stages + Cfg::kStages * Cfg::kStageBytes;
  s.obuf = s.wres + Cfg::kWBytes;
  s.full_bar = reinterpret_cast<uint64_t*>(s.obuf + Cfg::kOB * kOutBufBytes);
  s.empty_bar = s.full_bar + Cfg::kStages;
  s.tfull_bar = s.empty_bar + Cfg::kStages;
  s.tempty_bar = s.tfull_bar + 2;
  s.bufready_bar = s.tempty_bar + 2;
  s.outready_bar = s.bufready_bar + Cfg::kOB;
  s.w_bar = s.outready_bar + Cfg::kOB;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(s.w_bar + 1);

  if (threadIdx.x == 0) {
    for (int i = 0; i < Cfg::kStages; ++i) {
      mbar_init(&s.full_bar[i], Cfg::kPair ? 2 : 1);
      mbar_init(&s.empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s.tfull_bar[i], 1);
      mbar_init(&s.tempty_bar[i], Cfg::kPair ? 16 : 8);
    }
    for (int i = 0; i < Cfg::kOB; ++i) {
      mbar_init(&s.bufready_bar[i], 1);
      mbar_init(&s.outready_bar[i], Cfg::kWarpsPerStep);
    }
    if (Cfg::kWBytes > 0) mbar_init(s.w_bar, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    if (Cfg::kPair)
      tmem_alloc_pair(tmem_slot, Cfg::kTmemCols);
    else
      tmem_alloc(tmem_slot, Cfg::kTmemCols);
  }
  const int lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    if (a_map != nullptr) tma_prefetch_desc(a_map);
    tma_prefetch_desc(&p.tmB);
  }
  if (warp == 10 && lane == 0) {
    tma_prefetch_desc(&p.tmOut);
    if (res) tma_prefetch_desc(&p.tmRes);
  }
  tc_fence_before();
  if (Cfg::kPair)
    cluster_sync_all();
  else
    __syncthreads();
  tc_fence_after();
  s.tmem_base = *reinterpret_cast<volatile uint32_t*>(tmem_slot);
  // programmatic dependent launch: everything above overlapped the tail of the previous kernel; its output (our
  // input / residual) may only be touched from here on
  pdl_launch_dependents();
  pdl_wait();

  int* s_map = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(s.full_bar) + 256);
  s.s_map = ragged_map_setup(p, s_map) ? s_map : nullptr;
  return s;
}

template <class Cfg>
__device__ __forceinline__ void tc_teardown(int warp, uint32_t tmem_base) {
  // neither CTA of a pair may leave while the other can still touch its shared memory / barriers / TMEM
  tc_fence_before();
  if (Cfg::kPair)
    cluster_sync_all();
  else
    __syncthreads();
  if (warp == 1) {
    if (Cfg::kPair)
      tmem_dealloc_pair(tmem_base, Cfg::kTmemCols);
    else
      tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

// output group handled by local step j of a tile (see the epilogue): half 0 of the epilogue warps owns the even
// steps, half 1 the odd ones; each half walks its own contiguous range of channels
template <int STEPS>
__device__ __forceinline__ int step_group(int j) {
  return STEPS == 1 ? 0 : (j & 1) * (STEPS / 2) + (j >> 1);
}

// ------------------------------------------------------------------------------------------------------------
// Output / residual TMA (warp 10, each CTA its own tiles).  One thread walks the (live tile, output group) steps in
// order.  RES: the residual group of step s + OB - 1 is fetched into its staging buffer while the epilogue warps work
// on step s; the epilogue adds the accumulator IN PLACE and the same buffer then leaves through a TMA store (full
// 128-byte lines, no partial-sector writes).
// ------------------------------------------------------------------------------------------------------------
template <int BN, int OB, bool RES, class Walk>
__device__ __forceinline__ void output_role(const ConvTcParams& p, const TcShared& s, const Walk& walk) {
  if (elect_one()) {
    constexpr int kSteps = BN / 64;
    constexpr int kAhead = RES ? OB - 1 : 0;
    // two cursors over this CTA's live tiles: ld (residual prefetch, runs ahead) and st (output stores)
    int ld_tile = walk.first(), st_tile = walk.first(), ld_hint = 0, st_hint = 0, ld_j = 0, st_j = 0;
    TileCoord ld_t{}, st_t{};
    auto seek = [&](int& i, int& hint, TileCoord& t) {
      for (; i < walk.total; i += walk.step()) {
        const Tile v = walk.at(p, i, hint);
        t = v.t;
        if (!v.dead) break;
      }
    };
    if (RES) seek(ld_tile, ld_hint, ld_t);
    seek(st_tile, st_hint, st_t);
    uint32_t ld_s = 0, st_s = 0;
    auto issue_load = [&]() {
      const uint32_t b = ld_s % OB;
      mbar_expect_tx(&s.bufready_bar[b], kOutBufBytes);
      tma_load_4d(s.obuf + b * kOutBufBytes, &p.tmRes, &s.bufready_bar[b], ld_t.n_tile * BN + step_group<kSteps>(ld_j) * 64,
                  ld_t.w0, ld_t.h0, ld_t.img);
      ++ld_s;
      if (++ld_j == kSteps) {
        ld_j = 0;
        ld_tile += walk.step();
        seek(ld_tile, ld_hint, ld_t);
      }
    };
    if (RES) {
      for (int i = 0; i < kAhead && ld_tile < walk.total; ++i) issue_load();
    }
    while (st_tile < walk.total) {
      if (RES && ld_tile < walk.total) {
        tma_store_wait_read<0>();   // the buffer of step ld_s - OB (= st_s - 1) has been read by its store
        issue_load();
      }
      const uint32_t b = st_s % OB;
      mbar_wait(&s.outready_bar[b], (st_s / OB) & 1u, 500 + (int)b);
      tma_store_4d(&p.tmOut, s.obuf + b * kOutBufBytes, st_t.n_tile * BN + step_group<kSteps>(st_j) * 64, st_t.w0, st_t.h0,
                   st_t.img);
      tma_store_commit();
      if (!RES) {
        tma_store_wait_read<0>();
        mbar_arrive(&s.bufready_bar[b]);
      }
      ++st_s;
      if (++st_j == kSteps) {
        st_j = 0;
        st_tile += walk.step();
        seek(st_tile, st_hint, st_t);
      }
    }
    tma_store_wait_all();
  }
  __syncwarp();
}

// ------------------------------------------------------------------------------------------------------------
// Epilogue (warps 2..9, each CTA its own 128 TMEM lanes).  TMEM gives each thread one pixel row of the accumulator.  The
// thread adds bias (+ the residual it finds in the staging buffer), applies ReLU, packs to 16 bit and writes its row
// into the 128B-swizzled staging buffer -- the layout TMA expects -- at the very address the residual came from.
// 16-byte unit u of row r lives at r * 128 + ((u ^ (r & 7)) << 4): the 8 lanes of a quarter-warp hit 8 different
// units, i.e. all 32 banks.  RES / RELU / F16 are compile-time so the inner loop carries no runtime branches: on the
// low-K layers the epilogue, not the MMA, sets the pace.
// ------------------------------------------------------------------------------------------------------------
template <int BN, int OB, bool RES, bool RELU, bool F16, class Walk>
__device__ __forceinline__ void epilogue_role(const ConvTcParams& p, const TcShared& s, const Walk& walk) {
  constexpr int kSteps = BN / 64;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ew = warp - 2;
  const int q = warp & 3;          // TMEM lane quarter this warp may access
  const int half = ew >> 2;        // BN >= 128: which steps of the tile; BN == 64: which 32 of the 64 columns
  constexpr int kUnits = (BN == 64) ? 4 : 8;            // 16-byte units (8 channels) per row this warp handles per step
  constexpr int kMySteps = (BN == 64) ? 1 : kSteps / 2;  // steps per tile of this warp
  const int row = q * 32 + lane;                         // pixel of the tile == TMEM lane == staging row
  const uint32_t row_off = (uint32_t)row * 128u;
  const uint32_t rsw = (uint32_t)(row & 7);
  const int u0 = (BN == 64) ? half * 4 : 0;
  uint32_t acc = 0, acc_phase = 0, live_tiles = 0;
  int hint = 0;
  for (int vt = walk.first(); vt < walk.total; vt += walk.step()) {
    const Tile v = walk.at(p, vt, hint);
    const TileCoord t = v.t;
    const bool phantom = Walk::phantom(p, t);
    const int vh = phantom ? 0 : (p.valid_h != nullptr ? __ldg(p.valid_h + t.img) : INT_MAX);
    const int h = t.h0 + (row >> p.tw_log2), w = t.w0 + (row & (p.tw - 1));
    if (v.dead) {
      // dead tile: no MMA was issued for it; only the zero halo is written (plain stores, rare)
      if (!phantom && t.h0 < vh + kRaggedHalo && w < p.Wo && h < p.Ho && h < vh + kRaggedHalo) {
        constexpr int kColsZ = BN / 2;
        __nv_bfloat16* o = p.out + (((int64_t)t.img * p.Ho + h) * p.Wo + w) * p.Cout + t.n_tile * BN + half * kColsZ;
        for (int c = 0; c < kColsZ; c += 8) *reinterpret_cast<uint4*>(o + c) = make_uint4(0u, 0u, 0u, 0u);
      }
      continue;
    }
    const bool live = h < vh;
    mbar_wait(&s.tfull_bar[acc], acc_phase, 400 + (int)acc);
    tc_fence_after();
#pragma unroll
    for (int i = 0; i < kMySteps; ++i) {
      const int j = (BN == 64) ? 0 : half + 2 * i;
      const int grp = step_group<kSteps>(j);
      const uint32_t st = live_tiles * kSteps + j;
      const uint32_t b = st % OB;
      const int col0 = grp * 64 + u0 * 8;    // first column (within the BN tile) of this warp's units
      uint32_t a[kUnits * 8];
      const uint32_t t_addr = s.tmem_base + ((uint32_t)(q * 32) << 16) + acc * BN + col0;
#pragma unroll
      for (int k = 0; k < kUnits / 4; ++k) tmem_ld32(t_addr + 32 * k, reinterpret_cast<uint32_t(&)[32]>(a[32 * k]));
      const float* bptr = p.bias + t.n_tile * BN + col0;
      mbar_wait(&s.bufready_bar[b], RES ? ((st / OB) & 1u) : (((st / OB) & 1u) ^ 1u), 600 + (int)b);
      tmem_ld_wait();
      if (i == kMySteps - 1) {
        // the accumulator is in registers: hand the TMEM buffer back to the MMA warp
        tc_fence_before();
        __syncwarp();
        if (lane == 0) Walk::release_acc(&s.tempty_bar[acc]);
      }
      uint8_t* rowp = s.obuf + b * kOutBufBytes + row_off;
#pragma unroll
      for (int u = 0; u < kUnits; ++u) {
        const float4 b0 = __ldg(reinterpret_cast<const float4*>(bptr + u * 8));
        const float4 b1 = __ldg(reinterpret_cast<const float4*>(bptr + u * 8 + 4));
        uint4* sp = reinterpret_cast<uint4*>(rowp + ((((uint32_t)(u0 + u)) ^ rsw) << 4));
        float v8[8] = {__uint_as_float(a[u * 8 + 0]) + b0.x, __uint_as_float(a[u * 8 + 1]) + b0.y,
                       __uint_as_float(a[u * 8 + 2]) + b0.z, __uint_as_float(a[u * 8 + 3]) + b0.w,
                       __uint_as_float(a[u * 8 + 4]) + b1.x, __uint_as_float(a[u * 8 + 5]) + b1.y,
                       __uint_as_float(a[u * 8 + 6]) + b1.z, __uint_as_float(a[u * 8 + 7]) + b1.w};
        if (RES) {
          const uint4 r4 = *sp;
          const uint32_t rv[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) v8[2 * k] += lo16(rv[k], F16), v8[2 * k + 1] += hi16(rv[k], F16);
        }
        if (RELU) {
#pragma unroll
          for (int k = 0; k < 8; ++k) v8[k] = fmaxf(v8[k], 0.f);
        }
        uint4 o = make_uint4(pack16x2(v8[0], v8[1], F16), pack16x2(v8[2], v8[3], F16), pack16x2(v8[4], v8[5], F16),
                             pack16x2(v8[6], v8[7], F16));
        if (!live) o = make_uint4(0u, 0u, 0u, 0u);   // rows below the image in a ragged batch: the next layer's zero padding
        *sp = o;
      }
      fence_proxy_async();   // make this thread's staging writes visible to the TMA (async proxy) store
      __syncwarp();
      if (lane == 0) mbar_arrive(&s.outready_bar[b]);
    }
    ++live_tiles;
    acc ^= 1u;
    if (acc == 0) acc_phase ^= 1u;
  }
}

// ------------------------------------------------------------------------------------------------------------
// conv_tc_kernel: one CTA per tile, cta_group::1
// ------------------------------------------------------------------------------------------------------------
template <int BN, int KBLK, int OB, bool RES, bool RELU, bool F16>
__global__ void __launch_bounds__(kTcThreads, 1) conv_tc_kernel(const __grid_constant__ ConvTcParams p) {
  using Cfg = TcCfg<BN, KBLK, OB>;
  constexpr int kABytes = Cfg::kABytes;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const TcShared s = tc_prologue<Cfg>(p, warp, &p.tmA[0], RES);
  const CtaWalk walk(p, s.s_map);
  const int kblocks = p.n_taps * p.cblocks + p.cblocks2;

  if (warp == 0) {
    // ================================ TMA producer ================================
    if (elect_one()) {
      uint32_t stage = 0, phase = 0;
      int hint = 0;
      for (int vt = walk.first(); vt < walk.total; vt += walk.step()) {
        const Tile v = walk.at(p, vt, hint);
        if (v.dead) continue;
        const TileCoord t = v.t;
        const int n0 = t.n_tile * BN;
        for (int tap = 0; tap < p.n_taps; ++tap) {
          const CUtensorMap* mA = &p.tmA[p.tap_map[tap]];
          const int cw = t.w0 + p.tap_dw[tap], ch = t.h0 + p.tap_dh[tap];
          for (int cb = 0; cb < p.cblocks; ++cb) {
            mbar_wait(&s.empty_bar[stage], phase ^ 1u, 100 + (int)stage);
            uint8_t* sA = s.stages + stage * Cfg::kStageBytes;
            mbar_expect_tx(&s.full_bar[stage], Cfg::kStageBytes);
            tma_load_4d(sA, mA, &s.full_bar[stage], cb * KBLK, cw, ch, t.img);
            tma_load_2d(sA + kABytes, &p.tmB, &s.full_bar[stage], (tap * p.cblocks + cb) * KBLK, n0);
            if (++stage == Cfg::kStages) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
        for (int cb = 0; cb < p.cblocks2; ++cb) {   // second source (fused downsample branch)
          mbar_wait(&s.empty_bar[stage], phase ^ 1u, 100 + (int)stage);
          uint8_t* sA = s.stages + stage * Cfg::kStageBytes;
          mbar_expect_tx(&s.full_bar[stage], Cfg::kStageBytes);
          tma_load_4d(sA, &p.tmA[p.map2], &s.full_bar[stage], cb * KBLK, t.w0, t.h0, t.img);
          tma_load_2d(sA + kABytes, &p.tmB, &s.full_bar[stage], (p.n_taps * p.cblocks + cb) * KBLK, n0);
          if (++stage == Cfg::kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================================ MMA issuer ================================
    if (elect_one()) {
      constexpr uint32_t idesc = F16 ? umma_idesc_f16(128, BN) : umma_idesc_bf16(128, BN);
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      int hint = 0;
      for (int vt = walk.first(); vt < walk.total; vt += walk.step()) {
        if (walk.at(p, vt, hint).dead) continue;
        mbar_wait(&s.tempty_bar[acc], acc_phase ^ 1u, 300 + (int)acc);
        tc_fence_after();
        const uint32_t d_tmem = s.tmem_base + acc * BN;
        for (int kb = 0; kb < kblocks; ++kb) {
          mbar_wait(&s.full_bar[stage], phase, 200 + (int)stage);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(s.stages + stage * Cfg::kStageBytes);
          const uint32_t b_addr = a_addr + kABytes;
#pragma unroll
          for (int k = 0; k < KBLK / 16; ++k) {
            umma_bf16(d_tmem, umma_desc_kmajor<Cfg::kSwizzleBytes>(a_addr + k * 32),
                      umma_desc_kmajor<Cfg::kSwizzleBytes>(b_addr + k * 32), idesc, (uint32_t)((kb | k) != 0));
          }
          umma_commit(&s.empty_bar[stage]);
          if (++stage == Cfg::kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        umma_commit(&s.tfull_bar[acc]);
        acc ^= 1u;
        if (acc == 0) acc_phase ^= 1u;
      }
    }
    __syncwarp();
  } else if (warp == 10) {
    output_role<BN, OB, RES>(p, s, walk);
  } else {
    epilogue_role<BN, OB, RES, RELU, F16>(p, s, walk);
  }
  tc_teardown<Cfg>(warp, s.tmem_base);
}

// ------------------------------------------------------------------------------------------------------------
// CTA-pair variant (cluster of 2, tcgen05 cta_group::2).  One MMA of M = 256 spans the two SMs of a TPC: CTA r of the
// pair owns M tile 2*m_pair + r (its own 128 pixels of A, its own 128 TMEM lanes, its own epilogue / output TMA) and
// stages only HALF of the weight tile (BN/2 rows of B) -- 32 KB instead of 48 KB of shared-memory fill per K block
// at BN = 256, so the same shared memory holds 6 operand stages instead of 4.  The leader (rank 0) issues every MMA;
// "stage full" barriers live in the leader (both CTAs' TMA loads count their bytes there), "stage empty" and
// "accumulator full" are multicast by tcgen05.commit to both CTAs, "accumulator empty" is arrived remotely by the
// peer's epilogue warps (PairWalk::release_acc).  A pair is skipped in a ragged batch only when BOTH of its tiles are
// dead (see PairWalk).
// ------------------------------------------------------------------------------------------------------------
template <int BN, int OB, bool RES, bool RELU, bool F16>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kTcThreads, 1)
    conv_tc_pair_kernel(const __grid_constant__ ConvTcParams p) {
  using Cfg = TcCfgPair<BN, OB>;
  constexpr int kABytes = Cfg::kABytes;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const TcShared s = tc_prologue<Cfg>(p, warp, &p.tmA[0], RES);
  const PairWalk walk(p, s.s_map);
  const bool leader = walk.rank == 0;
  const int kblocks = p.n_taps * p.cblocks + p.cblocks2;

  if (warp == 0) {
    // ================================ TMA producer (both CTAs) ================================
    if (elect_one()) {
      uint32_t stage = 0, phase = 0;
      const uint32_t full0 = mapa_shared(smem_u32(&s.full_bar[0]), 0);   // the leader's full barriers
      int hint = 0;
      for (int pt = walk.first(); pt < walk.total; pt += walk.step()) {
        const Tile pr = walk.at(p, pt, hint);
        if (pr.dead) continue;
        const TileCoord t = pr.t;
        const int n0 = t.n_tile * BN + walk.rank * (BN / 2);
        for (int kb = 0; kb < kblocks; ++kb) {
          const CUtensorMap* mA;
          int c0, cw, ch;
          if (kb < p.n_taps * p.cblocks) {
            const int tap = kb / p.cblocks, cb = kb - tap * p.cblocks;
            mA = &p.tmA[p.tap_map[tap]];
            c0 = cb * 64, cw = t.w0 + p.tap_dw[tap], ch = t.h0 + p.tap_dh[tap];
          } else {   // second source (fused downsample branch)
            mA = &p.tmA[p.map2];
            c0 = (kb - p.n_taps * p.cblocks) * 64, cw = t.w0, ch = t.h0;
          }
          mbar_wait(&s.empty_bar[stage], phase ^ 1u, 100 + (int)stage);
          uint8_t* sA = s.stages + stage * Cfg::kStageBytes;
          const uint32_t fb = full0 + stage * 8u;
          if (leader)
            mbar_expect_tx(&s.full_bar[stage], 2 * Cfg::kStageBytes);
          else
            mbar_arrive_cluster(fb);
          tma_load_4d_pair(sA, mA, fb, c0, cw, ch, t.img);
          tma_load_2d_pair(sA + kABytes, &p.tmB, fb, kb * 64, n0);
          if (++stage == Cfg::kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================================ MMA issuer (leader only) ================================
    if (leader && elect_one()) {
      constexpr uint32_t idesc = F16 ? umma_idesc_f16(256, BN) : umma_idesc_bf16(256, BN);
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      int hint = 0;
      for (int pt = walk.first(); pt < walk.total; pt += walk.step()) {
        if (walk.at(p, pt, hint).dead) continue;
        mbar_wait(&s.tempty_bar[acc], acc_phase ^ 1u, 300 + (int)acc);
        tc_fence_after();
        const uint32_t d_tmem = s.tmem_base + acc * BN;
        for (int kb = 0; kb < kblocks; ++kb) {
          mbar_wait(&s.full_bar[stage], phase, 200 + (int)stage);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(s.stages + stage * Cfg::kStageBytes);
          const uint32_t b_addr = a_addr + kABytes;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            umma_bf16_pair(d_tmem, umma_desc_kmajor<128>(a_addr + k * 32), umma_desc_kmajor<128>(b_addr + k * 32), idesc,
                           (uint32_t)((kb | k) != 0));
          }
          umma_commit_pair(&s.empty_bar[stage], 3);
          if (++stage == Cfg::kStages) {
            stage = 0;
            phase ^= 1u;
          }
        }
        umma_commit_pair(&s.tfull_bar[acc], 3);
        acc ^= 1u;
        if (acc == 0) acc_phase ^= 1u;
      }
    }
    __syncwarp();
  } else if (warp == 10) {
    output_role<BN, OB, RES>(p, s, walk);
  } else {
    epilogue_role<BN, OB, RES, RELU, F16>(p, s, walk);
  }
  tc_teardown<Cfg>(warp, s.tmem_base);
}

// ------------------------------------------------------------------------------------------------------------
// Stem variant with a HALO tile (128 x 1 tiles).  conv_tc_kernel<64, 32> fetches the stem's A operand as 7 boxes of
// 128 rows x 64 bytes per tile -- 896 L2 requests of 1.4 sectors each, and ncu shows the launch bound by that request
// rate (12 % tensor-pipe activity).  The windows of neighbouring outputs overlap: tap row ky of output wo is the 64
// bytes (8 pixels x 4 channels) at padded pixel 2*wo, i.e. 16 bytes after the window of output wo - 1.  16 bytes is
// exactly the row pitch of a NO-SWIZZLE K-major UMMA core matrix (8 rows x 16 bytes, rows 16 bytes apart): with LBO =
// 16 B (next 16 bytes of K) and SBO = 128 B (next 8 rows) a descriptor reads the 128 overlapping windows of a tile
// straight out of one contiguous input row.  So a 128 x 1 output tile needs 7 bulk copies of 2 096 bytes (one per tap
// row) instead of 896 small requests, and the 28 KB of stem weights stay resident in shared memory for the whole
// kernel.  Epilogue / output path as in conv_tc_kernel<64, ...>.
// ------------------------------------------------------------------------------------------------------------
constexpr int kStemRowBytes = 2112;                 // (2 * 127 + 8) pixels x 8 B = 2 096, rounded up to a multiple of 64
constexpr int kStemStageBytes = 7 * kStemRowBytes + 64;      // 14 848 = 116 x 128
using StemCfg = TcLayout<6, kStemStageBytes, 7 * 64 * 64 /*7 tap rows x 64 output channels x 32 k, 64B-swizzled*/, 64, 4, false>;
static_assert(StemCfg::kUsedBytes > 120 * 1024, "stem halo kernel: shared memory budget");

__device__ __forceinline__ void bulk_load_1d(void* smem, const void* gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem)),
               "l"(reinterpret_cast<uint64_t>(gmem)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// K-major operand WITHOUT swizzle: 8-row x 16-byte core matrices, rows 16 bytes apart (fixed by the hardware),
// LBO = distance between the two 16-byte K halves of one MMA, SBO = distance between 8-row groups
__device__ __forceinline__ uint64_t umma_desc_kmajor_noswizzle(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)(lbo_bytes >> 4) << 16;
  d |= (uint64_t)(sbo_bytes >> 4) << 32;
  d |= (uint64_t)1 << 46;
  return d;      // layout type 0 = no swizzle
}

template <bool RELU, bool F16>
__global__ void __launch_bounds__(kTcThreads, 1) conv_tc_stem_kernel(const __grid_constant__ ConvTcParams p) {
  using Cfg = StemCfg;
  constexpr int BN = 64;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const TcShared s = tc_prologue<Cfg>(p, warp, nullptr, false);
  const CtaWalk walk(p, s.s_map);      // one N tile: all 64 output channels

  if (warp == 0) {
    // ================================ producer: weights once, then 7 input rows per tile ================================
    if (elect_one()) {
      mbar_expect_tx(s.w_bar, Cfg::kWBytes);
      for (int ky = 0; ky < 7; ++ky) tma_load_2d(s.wres + ky * 4096, &p.tmB, s.w_bar, ky * 32, 0);
      uint32_t stage = 0, phase = 0;
      const int64_t row_bytes = (int64_t)p.stem_wp * 8;
      int hint = 0;
      for (int vt = walk.first(); vt < walk.total; vt += walk.step()) {
        const Tile v = walk.at(p, vt, hint);
        if (v.dead) continue;
        const TileCoord t = v.t;      // tw = 128, th = 1: h0 = output row, w0 = first output column
        // what is left of the padded row from pixel 2 * w0 on (a multiple of 16 bytes); beyond it lie outputs >= Wo
        const uint32_t len = (uint32_t)min((int64_t)(2 * 127 + 8) * 8, row_bytes - (int64_t)t.w0 * 16);
        mbar_wait(&s.empty_bar[stage], phase ^ 1u, 100 + (int)stage);
        uint8_t* sA = s.stages + stage * Cfg::kStageBytes;
        mbar_expect_tx(&s.full_bar[stage], 7 * len);
        const uint8_t* src = p.stem_src + ((int64_t)t.img * p.stem_hp + 2 * t.h0) * row_bytes + (int64_t)t.w0 * 16;
        for (int ky = 0; ky < 7; ++ky) bulk_load_1d(sA + ky * kStemRowBytes, src + ky * row_bytes, len, &s.full_bar[stage]);
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
      constexpr uint32_t idesc = F16 ? umma_idesc_f16(128, BN) : umma_idesc_bf16(128, BN);
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      mbar_wait(s.w_bar, 0, 700);
      const uint32_t w_addr = smem_u32(s.wres);
      int hint = 0;
      for (int vt = walk.first(); vt < walk.total; vt += walk.step()) {
        if (walk.at(p, vt, hint).dead) continue;
        mbar_wait(&s.tempty_bar[acc], acc_phase ^ 1u, 300 + (int)acc);
        mbar_wait(&s.full_bar[stage], phase, 200 + (int)stage);
        tc_fence_after();
        const uint32_t d_tmem = s.tmem_base + acc * BN;
        const uint32_t a_addr = smem_u32(s.stages + stage * Cfg::kStageBytes);
#pragma unroll
        for (int ky = 0; ky < 7; ++ky) {
#pragma unroll
          for (int k = 0; k < 2; ++k) {      // K = 32 per tap row = two MMAs of K = 16 (32 bytes)
            umma_bf16(d_tmem, umma_desc_kmajor_noswizzle(a_addr + ky * kStemRowBytes + k * 32, 16, 128),
                      umma_desc_kmajor<64>(w_addr + ky * 4096 + k * 32), idesc, (uint32_t)((ky | k) != 0));
          }
        }
        umma_commit(&s.empty_bar[stage]);
        umma_commit(&s.tfull_bar[acc]);
        if (++stage == Cfg::kStages) {
          stage = 0;
          phase ^= 1u;
        }
        acc ^= 1u;
        if (acc == 0) acc_phase ^= 1u;
      }
    }
    __syncwarp();
  } else if (warp == 10) {
    output_role<BN, Cfg::kOB, false>(p, s, walk);
  } else {
    epilogue_role<BN, Cfg::kOB, false, RELU, F16>(p, s, walk);
  }
  tc_teardown<Cfg>(warp, s.tmem_base);
}

// ------------------------------------------------------------------------------------------------------------
// 3x3 HALO kernel for the 64 -> 64 convolutions of layer1 (stride 1, dilation 1, pad 1; 128 x 1 output tiles).
// conv_tc_kernel fetches the A operand of every tap as its own shifted 128-pixel box: nine L2 fetches of every input
// byte, and ncu shows those launches bound by that request rate (24.7 % tensor-pipe activity at 0.9 TB/s of DRAM traffic).
// Here ONE TMA box per tile -- {64 ch, 130 px, 3 rows} of the NHWC input starting one pixel up and left of the tile, the
// conv padding zero-filled by the TMA unit -- lands as 390 rows of 128 bytes in the 128-byte-swizzled K-major layout, and
// tap (ky, kx) is the very same tile read through a descriptor whose start address is advanced by (130 ky + kx) rows of
// 128 bytes -- i.e. to an address that is NOT a multiple of the 1024-byte swizzle atom.  Measured on B200 (round 2, GPU
// call 13): that works as is, with the descriptor's base-offset field left 0 -- the tensor core applies the 128-byte
// swizzle to the absolute shared-memory address (bits [4,7) ^= bits [7,10)), exactly as the TMA unit did when it wrote
// the tile; setting base offset = (start >> 7) & 7 gives wrong results.  The nine 8 KB weight slabs stay resident in
// shared memory for the whole kernel.  Epilogue / output path as in conv_tc_kernel<64, ...>.
// layer1 conv2: 0.049 -> 0.033 ms per [8,624,1024] pass (480 -> 715 TFLOP/s).
// ------------------------------------------------------------------------------------------------------------
constexpr int kHaloW = 130;
// 3 x 130 x 128 B = 49 920 per stage, rounded up to 49 x 1024; 9 taps x 64 output channels x 64 input channels x 2 B of weights
using Halo3Cfg = TcLayout<2, 50176, 9 * 64 * 128, 64, 3, false>;
static_assert(Halo3Cfg::kUsedBytes > 120 * 1024, "3x3 halo kernel: shared memory budget");

template <bool RELU, bool F16>
__global__ void __launch_bounds__(kTcThreads, 1) conv_tc_halo3_kernel(const __grid_constant__ ConvTcParams p) {
  using Cfg = Halo3Cfg;
  constexpr int BN = 64;
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const TcShared s = tc_prologue<Cfg>(p, warp, &p.tmA[1], false);
  const CtaWalk walk(p, s.s_map);      // one N tile: all 64 output channels

  if (warp == 0) {
    // ================================ producer: weights once, then one halo box per tile ================================
    if (elect_one()) {
      mbar_expect_tx(s.w_bar, Cfg::kWBytes);
      for (int t = 0; t < 9; ++t) tma_load_2d(s.wres + t * 8192, &p.tmB, s.w_bar, t * 64, 0);
      uint32_t stage = 0, phase = 0;
      int hint = 0;
      for (int vt = walk.first(); vt < walk.total; vt += walk.step()) {
        const Tile v = walk.at(p, vt, hint);
        if (v.dead) continue;
        mbar_wait(&s.empty_bar[stage], phase ^ 1u, 100 + (int)stage);
        mbar_expect_tx(&s.full_bar[stage], 3 * kHaloW * 128);
        tma_load_4d(s.stages + stage * Cfg::kStageBytes, &p.tmA[1], &s.full_bar[stage], 0, v.t.w0 - 1, v.t.h0 - 1, v.t.img);
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
      constexpr uint32_t idesc = F16 ? umma_idesc_f16(128, BN) : umma_idesc_bf16(128, BN);
      uint32_t stage = 0, phase = 0, acc = 0, acc_phase = 0;
      mbar_wait(s.w_bar, 0, 700);
      const uint32_t w_addr = smem_u32(s.wres);
      int hint = 0;
      for (int vt = walk.first(); vt < walk.total; vt += walk.step()) {
        if (walk.at(p, vt, hint).dead) continue;
        mbar_wait(&s.tempty_bar[acc], acc_phase ^ 1u, 300 + (int)acc);
        mbar_wait(&s.full_bar[stage], phase, 200 + (int)stage);
        tc_fence_after();
        const uint32_t d_tmem = s.tmem_base + acc * BN;
        const uint32_t a_addr = smem_u32(s.stages + stage * Cfg::kStageBytes);
#pragma unroll
        for (int t = 0; t < 9; ++t) {
          const uint32_t a_tap = a_addr + (uint32_t)((t / 3) * kHaloW + (t % 3)) * 128u;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            umma_bf16(d_tmem, umma_desc_kmajor<128>(a_tap + k * 32), umma_desc_kmajor<128>(w_addr + t * 8192 + k * 32), idesc,
                      (uint32_t)((t | k) != 0));
          }
        }
        umma_commit(&s.empty_bar[stage]);
        umma_commit(&s.tfull_bar[acc]);
        if (++stage == Cfg::kStages) {
          stage = 0;
          phase ^= 1u;
        }
        acc ^= 1u;
        if (acc == 0) acc_phase ^= 1u;
      }
    }
    __syncwarp();
  } else if (warp == 10) {
    output_role<BN, Cfg::kOB, false>(p, s, walk);
  } else {
    epilogue_role<BN, Cfg::kOB, false, RELU, F16>(p, s, walk);
  }
  tc_teardown<Cfg>(warp, s.tmem_base);
}

// ------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------
static int encode_act_map(CUtensorMap* m, const void* base, uint64_t C, uint64_t Wd, uint64_t Hd, uint64_t Nd,
                          uint64_t strideW, uint64_t strideH, uint64_t strideN, uint32_t boxW, uint32_t boxH,
                          uint32_t boxC = 64) {
  encode_tiled_fn enc = get_encode_tiled();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
    return NBC_ERR_DEVICE;
  }
  cuuint64_t dims[4] = {C, Wd, Hd, Nd};
  cuuint64_t strides[3] = {strideW, strideH, strideN};
  cuuint32_t box[4] = {boxC, boxW, boxH, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, boxC == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(activation) failed: %d (C=%llu W=%llu H=%llu N=%llu box=%ux%u)", (int)r,
              (unsigned long long)C, (unsigned long long)Wd, (unsigned long long)Hd, (unsigned long long)Nd, boxW, boxH);
    return NBC_ERR_CUDA;
  }
  return 0;
}

static int encode_weight_map(CUtensorMap* m, const void* base, uint64_t K, uint64_t Cout, uint32_t boxN,
                             uint32_t boxK = 64) {
  encode_tiled_fn enc = get_encode_tiled();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
    return NBC_ERR_DEVICE;
  }
  cuuint64_t dims[2] = {K, Cout};
  cuuint64_t strides[1] = {K * 2};
  cuuint32_t box[2] = {boxK, boxN};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, boxK == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(weights) failed: %d (K=%llu Cout=%llu)", (int)r, (unsigned long long)K,
              (unsigned long long)Cout);
    return NBC_ERR_CUDA;
  }
  return 0;
}

int conv_encode_act_map(CUtensorMap* m, const void* base, uint64_t C, uint64_t Wd, uint64_t Hd, uint64_t Nd, uint64_t strideW,
                        uint64_t strideH, uint64_t strideN, uint32_t boxW, uint32_t boxH, uint32_t boxC) {
  return encode_act_map(m, base, C, Wd, Hd, Nd, strideW, strideH, strideN, boxW, boxH, boxC);
}

bool conv_tc_supported(const ConvGeom& g) {
  if (g.Cin % 64 != 0 || g.Cout % 64 != 0) return false;
  if (g.kh * g.kw > 9) return false;
  if (g.stride != 1 && g.stride != 2) return false;
  if (g.Ho() < 1 || g.Wo() < 1) return false;
  if (g.stride == 2 && (g.H < 2 || g.W < 2)) return false;
  return true;
}

static int floordiv(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }

struct ConvTcLaunch {
  ConvTcParams p;
  int block_n;
  int kblk;
  int grid;
  int out_bufs;
  int pair;   // 1: conv_tc_pair_kernel (clusters of 2, cta_group::2 MMA)
  int stem_halo;   // 1: conv_tc_stem_kernel (128 x 1 stem tiles)
  int halo3;       // 1: conv_tc_halo3_kernel (64 -> 64 3x3 out of one halo box per tile)
};

// Which launches run on CTA pairs (conv_tc_pair_kernel).  Measured per layer class on B200 (profiles/r01s_*): pairs win
// where the operand pipeline or the MMA sets the pace -- Cout % 256 == 0 without a residual and K >= 512 (the 1x1
// reductions out of wide tensors, the 3x3 convs of layer3 / layer4 / the head, conv3 + downsample of layer3 / layer4) --
// and lose on the residual layers (epilogue / HBM bound), on BN = 128 and on very short K.
static int want_pair(bool residual, int bn, int kblocks) { return (!residual && bn == 256 && kblocks >= 8) ? 1 : 0; }
// the persistent conv kernels occupy every SM (DESIGN §8: leaving some to the side streams never paid)
static void set_grid(ConvTcLaunch* L) {
  const ConvTcParams& p = L->p;
  const int sms = sm_count();
  if (L->pair) {
    const int pairs = ((p.num_m_tiles + 1) / 2) * p.num_n_tiles;
    L->grid = 2 * (pairs < sms / 2 ? pairs : sms / 2);
  } else {
    const int total = p.num_m_tiles * p.num_n_tiles;
    L->grid = total < sms ? total : sms;
  }
}

// output (and residual) as [N][Ho][Wo][Cout] with the box of one 64-channel group of a tile
static int encode_out_maps(ConvTcParams* p, int N, int Ho, int Wo, int Cout, const void* y, const void* residual) {
  const uint64_t eb = 2;
  int rc = encode_act_map(&p->tmOut, y, (uint64_t)Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N, (uint64_t)Cout * eb,
                          (uint64_t)Wo * Cout * eb, (uint64_t)Ho * Wo * Cout * eb, p->tw, p->th);
  if (rc) return rc;
  if (residual != nullptr)
    rc = encode_act_map(&p->tmRes, residual, (uint64_t)Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N, (uint64_t)Cout * eb,
                        (uint64_t)Wo * Cout * eb, (uint64_t)Ho * Wo * Cout * eb, p->tw, p->th);
  else
    p->tmRes = p->tmOut;
  return rc;
}

// 128-pixel output rectangle: fewest tiles, widest on ties
static void choose_tile(int Ho, int Wo, ConvTcParams* p) {
  int best_tw = 128, best_tiles = INT32_MAX;
  for (int tw = 128; tw >= 8; tw >>= 1) {
    const int th = 128 / tw;
    const int tiles = ceil_div(Wo, tw) * ceil_div(Ho, th);
    if (tiles < best_tiles) best_tiles = tiles, best_tw = tw;
  }
  p->tw = best_tw;
  p->th = 128 / best_tw;
  p->tw_log2 = 0;
  while ((1 << p->tw_log2) < p->tw) ++p->tw_log2;
  p->tiles_w = ceil_div(Wo, p->tw);
  p->tiles_h = ceil_div(Ho, p->th);
}

static int build_launch(const ConvGeom& g, const void* x, const void* w, const float* bias, const void* residual,
                        void* y, ConvTcLaunch* L) {
  ConvTcParams& p = L->p;
  memset(&p, 0, sizeof(p));
  const int Ho = g.Ho(), Wo = g.Wo();
  choose_tile(Ho, Wo, &p);
  p.N = g.N, p.Ho = Ho, p.Wo = Wo, p.Cout = g.Cout;
  p.num_m_tiles = g.N * p.tiles_w * p.tiles_h;
  const int bn = (g.Cout % 256 == 0) ? 256 : (g.Cout % 128 == 0 ? 128 : 64);
  L->block_n = bn;
  L->kblk = 64;
  p.num_n_tiles = g.Cout / bn;
  p.n_taps = g.kh * g.kw;
  p.cblocks = g.Cin / 64;
  p.relu = g.relu;
  p.f16 = g.f16;
  p.bias = bias;
  p.residual = reinterpret_cast<const __nv_bfloat16*>(residual);
  p.out = reinterpret_cast<__nv_bfloat16*>(y);

  const uint64_t eb = 2;  // bytes per element
  const char* xb = reinterpret_cast<const char*>(x);
  if (g.stride == 1) {
    int rc = encode_act_map(&p.tmA[0], xb, g.Cin, g.W, g.H, g.N, (uint64_t)g.Cin * eb, (uint64_t)g.W * g.Cin * eb,
                            (uint64_t)g.H * g.W * g.Cin * eb, p.tw, p.th);
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
        p.tap_dh[t] = (int16_t)floordiv(oy, 2);
        p.tap_dw[t] = (int16_t)floordiv(ox, 2);
        used[py * 2 + px] = true;
      }
    for (int py = 0; py < 2; ++py)
      for (int px = 0; px < 2; ++px) {
        if (!used[py * 2 + px]) continue;
        const uint64_t Wd = (uint64_t)(g.W - px + 1) / 2, Hd = (uint64_t)(g.H - py + 1) / 2;
        const char* base = xb + ((uint64_t)py * g.W + px) * g.Cin * eb;
        int rc = encode_act_map(&p.tmA[py * 2 + px], base, g.Cin, Wd, Hd, g.N, 2ull * g.Cin * eb,
                                2ull * g.W * g.Cin * eb, (uint64_t)g.H * g.W * g.Cin * eb, p.tw, p.th);
        if (rc) return rc;
      }
    // the prefetch in the kernel touches tmA[0]; make sure it is a valid map
    if (!used[0]) p.tmA[0] = p.tmA[p.tap_map[0]];
  }
  L->stem_halo = 0;
  // 3x3 halo kernel for layer1's 64 -> 64 convolutions; other tiles of that shape take the nine-box path
  L->halo3 = (g.Cin == 64 && g.Cout == 64 && g.kh == 3 && g.kw == 3 && g.stride == 1 && g.dil == 1 && g.pad == 1 &&
              residual == nullptr && p.tw == 128 && p.th == 1)
                 ? 1
                 : 0;
  if (L->halo3) {
    int rc = encode_act_map(&p.tmA[1], xb, g.Cin, g.W, g.H, g.N, (uint64_t)g.Cin * eb, (uint64_t)g.W * g.Cin * eb,
                            (uint64_t)g.H * g.W * g.Cin * eb, kHaloW, 3);
    if (rc) return rc;
  }
  L->pair = L->halo3 ? 0 : want_pair(residual != nullptr, bn, p.n_taps * p.cblocks);
  int rc = encode_weight_map(&p.tmB, w, (uint64_t)p.n_taps * g.Cin, g.Cout, L->pair ? bn / 2 : bn);
  if (rc) return rc;
  rc = encode_out_maps(&p, g.N, Ho, Wo, g.Cout, y, residual);
  if (rc) return rc;
  L->out_bufs = (residual != nullptr || p.n_taps * p.cblocks <= 8) ? 4 : 2;
  set_grid(L);
  return 0;
}

// One launch helper for every conv kernel.  Programmatic dependent launch: the prologue of a conv kernel -- barrier
// init, TMEM allocation, descriptor prefetch -- runs while the previous kernel of the stream drains (see pdl_wait()).
// The pair kernel's __cluster_dims__(2, 1, 1) makes its grid a whole number of pairs.
template <void (*Kernel)(ConvTcParams), int SMEM>
static int launch_tc(const ConvTcLaunch& L, cudaStream_t stream) {
  static bool attr_set = false;
  if (!attr_set) {
    NBC_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM));
    attr_set = true;
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)L.grid);
  cfg.blockDim = dim3(kTcThreads);
  cfg.dynamicSmemBytes = (size_t)SMEM;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  NBC_CUDA(cudaLaunchKernelEx(&cfg, Kernel, L.p));
  count_launch();
  return 0;
}

static int no_kernel(const char* family, const ConvTcLaunch& L) {
  set_error("conv_tc: no %s kernel for block_n=%d out_bufs=%d residual=%d relu=%d f16=%d", family, L.block_n, L.out_bufs,
            L.p.residual != nullptr ? 1 : 0, L.p.relu, L.p.f16);
  return NBC_ERR_INVALID;
}

// Kernel families.  Family::run<OB, RES, RELU, F16> launches the family's kernel for one variant key, or refuses a
// combination that no selection rule produces: no kernel is compiled for it.
template <int BN>
struct CtaKernels {   // conv_tc_kernel with 64-element K blocks: every combination
  template <int OB, bool RES, bool RELU, bool F16>
  static int run(const ConvTcLaunch& L, cudaStream_t stream) {
    return launch_tc<conv_tc_kernel<BN, 64, OB, RES, RELU, F16>, TcCfg<BN, 64, OB>::kSmemBytes>(L, stream);
  }
};
struct StemKernels {   // the per-window stem, conv_tc_kernel<64, 32>: 4 staging buffers, no residual
  template <int OB, bool RES, bool RELU, bool F16>
  static int run(const ConvTcLaunch& L, cudaStream_t stream) {
    if constexpr (OB != 4 || RES)
      return no_kernel("per-window stem", L);
    else
      return launch_tc<conv_tc_kernel<64, 32, 4, false, RELU, F16>, TcCfg<64, 32, 4>::kSmemBytes>(L, stream);
  }
};
struct PairKernels {   // conv_tc_pair_kernel<256>: no residual (want_pair)
  template <int OB, bool RES, bool RELU, bool F16>
  static int run(const ConvTcLaunch& L, cudaStream_t stream) {
    if constexpr (RES)
      return no_kernel("CTA-pair", L);
    else
      return launch_tc<conv_tc_pair_kernel<256, OB, false, RELU, F16>, TcCfgPair<256, OB>::kSmemBytes>(L, stream);
  }
};
// the halo kernels have a fixed staging depth; out_bufs only describes the launch
struct StemHaloKernels {
  template <int OB, bool RES, bool RELU, bool F16>
  static int run(const ConvTcLaunch& L, cudaStream_t stream) {
    if constexpr (RES)
      return no_kernel("stem halo", L);
    else
      return launch_tc<conv_tc_stem_kernel<RELU, F16>, StemCfg::kSmemBytes>(L, stream);
  }
};
struct Halo3Kernels {
  template <int OB, bool RES, bool RELU, bool F16>
  static int run(const ConvTcLaunch& L, cudaStream_t stream) {
    if constexpr (RES)
      return no_kernel("3x3 halo", L);
    else
      return launch_tc<conv_tc_halo3_kernel<RELU, F16>, Halo3Cfg::kSmemBytes>(L, stream);
  }
};

// variant key of a launch: 8 = residual (always with 4 staging buffers), 4 = 4 staging buffers, 2 = ReLU, 1 = fp16
template <class Family>
static int launch_variant(const ConvTcLaunch& L, cudaStream_t stream) {
  const int key = (L.p.residual != nullptr ? 8 : (L.out_bufs == 4 ? 4 : 0)) | (L.p.relu ? 2 : 0) | (L.p.f16 ? 1 : 0);
  switch (key) {
    case 0: return Family::template run<2, false, false, false>(L, stream);
    case 1: return Family::template run<2, false, false, true>(L, stream);
    case 2: return Family::template run<2, false, true, false>(L, stream);
    case 3: return Family::template run<2, false, true, true>(L, stream);
    case 4: return Family::template run<4, false, false, false>(L, stream);
    case 5: return Family::template run<4, false, false, true>(L, stream);
    case 6: return Family::template run<4, false, true, false>(L, stream);
    case 7: return Family::template run<4, false, true, true>(L, stream);
    case 8: return Family::template run<4, true, false, false>(L, stream);
    case 9: return Family::template run<4, true, false, true>(L, stream);
    case 10: return Family::template run<4, true, true, false>(L, stream);
    case 11: return Family::template run<4, true, true, true>(L, stream);
    default: return no_kernel("conv_tc", L);
  }
}

// Stem as an implicit GEMM (see stem.cu): A = the zero-padded, normalised bf16 image [N][Hp][Wp][4]; one K block is
// tap row ky = 8 consecutive pixels x 4 channels (32 elements, 64 B) starting at padded pixel (2*ho + ky, 2*wo).
// The windows of neighbouring outputs overlap (stride 16 B, extent 64 B): the tensor map simply describes that
// address function.  Even / odd padded rows are two lattices, exactly like the stride-2 convolutions.
int conv_tc_prepare_stem(int N, int Ho, int Wo, int Hp, int Wp, const void* padded, const void* w224, const float* bias,
                         void* y, ConvTcPrepared* out, const int* valid_h, int f16, int relu) {
  ConvTcLaunch* L = reinterpret_cast<ConvTcLaunch*>(out->storage);
  ConvTcParams& p = L->p;
  memset(&p, 0, sizeof(p));
  p.f16 = f16;
  choose_tile(Ho, Wo, &p);
  p.N = N, p.Ho = Ho, p.Wo = Wo, p.Cout = 64;
  p.num_m_tiles = N * p.tiles_w * p.tiles_h;
  p.num_n_tiles = 1;
  p.n_taps = 7, p.cblocks = 1, p.relu = relu;
  p.bias = bias, p.residual = nullptr, p.out = reinterpret_cast<__nv_bfloat16*>(y);
  p.valid_h = valid_h;
  L->block_n = 64, L->kblk = 32;
  const char* base = reinterpret_cast<const char*>(padded);
  const uint64_t row_bytes = (uint64_t)Wp * 8;
  for (int py = 0; py < 2; ++py) {
    int rc = encode_act_map(&p.tmA[py], base + py * row_bytes, 32, (uint64_t)Wo, (uint64_t)(Hp - py + 1) / 2, (uint64_t)N,
                            16, 2 * row_bytes, (uint64_t)Hp * row_bytes, p.tw, p.th, 32);
    if (rc) return rc;
  }
  for (int ky = 0; ky < 7; ++ky) p.tap_map[ky] = (int8_t)(ky & 1), p.tap_dh[ky] = (int16_t)(ky >> 1), p.tap_dw[ky] = 0;
  int rc = encode_weight_map(&p.tmB, w224, 224, 64, 64, 32);
  if (rc) return rc;
  rc = encode_out_maps(&p, N, Ho, Wo, 64, y, nullptr);
  if (rc) return rc;
  L->out_bufs = 4;
  L->pair = 0;
  L->halo3 = 0;
  // halo kernel (conv_tc_stem_kernel): 128 x 1 tiles (the production geometry, Wo = 512; stem 0.180 -> 0.105 ms per
  // [8,624,1024] pass on B200); other tile shapes take the per-window kernel conv_tc_kernel<64, 32>
  p.stem_src = reinterpret_cast<const uint8_t*>(padded);
  p.stem_hp = Hp, p.stem_wp = Wp;
  L->stem_halo = (p.tw == 128 && p.th == 1 && (reinterpret_cast<uintptr_t>(padded) & 15) == 0) ? 1 : 0;
  set_grid(L);
  return 0;
}

int conv_tc_prepare(const ConvGeom& g, const void* x, const void* w, const float* bias, const void* residual, void* y,
                    ConvTcPrepared* out, const int* valid_h) {
  static_assert(sizeof(ConvTcLaunch) <= sizeof(out->storage), "ConvTcPrepared::storage too small");
  if (!conv_tc_supported(g)) {
    set_error("conv_tc: unsupported shape Cin=%d Cout=%d k=%dx%d stride=%d", g.Cin, g.Cout, g.kh, g.kw, g.stride);
    return NBC_ERR_INVALID;
  }
  if ((reinterpret_cast<uintptr_t>(bias) & 15) != 0) {
    set_error("conv_tc: bias must be 16-byte aligned");
    return NBC_ERR_INVALID;
  }
  ConvTcLaunch* L = reinterpret_cast<ConvTcLaunch*>(out->storage);
  int rc = build_launch(g, x, w, bias, residual, y, L);
  L->p.valid_h = valid_h;
  return rc;
}

// y = act(conv(x; w[:, :K1]) + conv1x1(x2; w[:, K1:]) + bias): g is the main convolution (stride 1), g2 a 1x1 convolution
// (stride 1 or 2, no padding) of a second tensor with the same output geometry; w = the two packed weight matrices
// concatenated along K per output channel.  One accumulator, one epilogue, no intermediate tensor.
int conv_tc_prepare_dual(const ConvGeom& g, const void* x, const ConvGeom& g2, const void* x2, const void* w_cat,
                         const float* bias, void* y, ConvTcPrepared* out, const int* valid_h) {
  if (!conv_tc_supported(g) || !conv_tc_supported(g2) || g.stride != 1 || g2.kh != 1 || g2.kw != 1 || g2.pad != 0 ||
      g2.Cout != g.Cout || g2.N != g.N || g2.Ho() != g.Ho() || g2.Wo() != g.Wo()) {
    set_error("conv_tc_prepare_dual: unsupported pair (main %dx%d k%d s%d, second Cin=%d k%d s%d)", g.Cin, g.Cout, g.kh, g.stride,
              g2.Cin, g2.kh, g2.stride);
    return NBC_ERR_INVALID;
  }
  if ((reinterpret_cast<uintptr_t>(bias) & 15) != 0) {
    set_error("conv_tc: bias must be 16-byte aligned");
    return NBC_ERR_INVALID;
  }
  ConvTcLaunch* L = reinterpret_cast<ConvTcLaunch*>(out->storage);
  int rc = build_launch(g, x, w_cat, bias, nullptr, y, L);
  if (rc) return rc;
  ConvTcParams& p = L->p;
  p.valid_h = valid_h;
  const uint64_t eb = 2;
  const char* xb = reinterpret_cast<const char*>(x2);
  p.map2 = 1;        // the main source is a stride-1 convolution: it only uses tmA[0]
  p.cblocks2 = g2.Cin / 64;
  if (g2.stride == 1)
    rc = encode_act_map(&p.tmA[1], xb, g2.Cin, g2.W, g2.H, g2.N, (uint64_t)g2.Cin * eb, (uint64_t)g2.W * g2.Cin * eb,
                        (uint64_t)g2.H * g2.W * g2.Cin * eb, p.tw, p.th);
  else   // stride 2, no padding: the even / even lattice of the input
    rc = encode_act_map(&p.tmA[1], xb, g2.Cin, (uint64_t)(g2.W + 1) / 2, (uint64_t)(g2.H + 1) / 2, g2.N, 2ull * g2.Cin * eb,
                        2ull * g2.W * g2.Cin * eb, (uint64_t)g2.H * g2.W * g2.Cin * eb, p.tw, p.th);
  if (rc) return rc;
  L->pair = want_pair(false, L->block_n, p.n_taps * p.cblocks + p.cblocks2);
  rc = encode_weight_map(&p.tmB, w_cat, (uint64_t)p.n_taps * g.Cin + g2.Cin, g.Cout, L->pair ? L->block_n / 2 : L->block_n);
  if (rc) return rc;
  L->out_bufs = (p.n_taps * p.cblocks + p.cblocks2 <= 8) ? 4 : 2;
  set_grid(L);
  return 0;
}

int conv_tc_run(const ConvTcPrepared* prep, cudaStream_t stream) {
  const ConvTcLaunch& L = *reinterpret_cast<const ConvTcLaunch*>(prep->storage);
  if (L.stem_halo) return launch_variant<StemHaloKernels>(L, stream);
  if (L.halo3) return launch_variant<Halo3Kernels>(L, stream);
  if (L.kblk == 32) return launch_variant<StemKernels>(L, stream);
  if (L.pair) return L.block_n == 256 ? launch_variant<PairKernels>(L, stream) : no_kernel("CTA-pair", L);
  switch (L.block_n) {
    case 256: return launch_variant<CtaKernels<256>>(L, stream);
    case 128: return launch_variant<CtaKernels<128>>(L, stream);
    case 64: return launch_variant<CtaKernels<64>>(L, stream);
    default: return no_kernel("conv_tc_kernel", L);
  }
}

void conv_tc_describe(const ConvTcPrepared* prep, ConvTcVariant* v) {
  const ConvTcLaunch* L = reinterpret_cast<const ConvTcLaunch*>(prep->storage);
  v->pair = L->pair, v->halo3 = L->halo3, v->stem_halo = L->stem_halo, v->dual = L->p.cblocks2 > 0;
  v->block_n = L->block_n, v->kblk = L->kblk, v->out_bufs = L->out_bufs;
  v->ragged_map = L->p.valid_h == nullptr ? -1 : (ragged_mapped(L->p) ? 1 : 0);
}

int conv_tc(const ConvGeom& g, const void* x, const void* w, const float* bias, const void* residual, void* y,
            cudaStream_t stream) {
  ConvTcPrepared prep;
  int rc = conv_tc_prepare(g, x, w, bias, residual, y, &prep);
  if (rc) return rc;
  return conv_tc_run(&prep, stream);
}

}  // namespace nbc
