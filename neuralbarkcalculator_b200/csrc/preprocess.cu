// K1 -- 4x cubic resize (4096^2 -> 1024^2) + dark-band trim, all in integer arithmetic on u8.
//
// Replaces Preprocessor._preprocess_image (models.py:191-203: skimage resize order=3 + trim_black + imsave's
// float->u8) and trim_black (models.py:157-166).  At exactly 4x the cubic (Catmull-Rom) sample point sits at
// 4i+1.5, i.e. a separable 4-tap filter [-1, 9, 9, -1]/16 over the pixel's own 4x4 block, so
//     S = sum_{p,q} w_p w_q * in[4i+p, 4j+q]   (exact int, = 256 * resized value)
//     out = clamp((S + 128) >> 8, min(in), max(in))        -- skimage clips to the input range, then u8 rounding
//     nondark(i,j) = sum_c clip(S_c) / (256*255) > 1e-3   <=>  min(in) >= 1  or  sum_c max(S_c, 0) >= 66
// Pass 1 reads the raw image once (16-byte loads, 48 B per thread per row), writes (S+128)>>8 saturated to u8
// (coalesced 16-byte stores through shared memory), and reduces the input min / max and the per-row non-dark counts.
// A one-block kernel turns the counts into the [first, last) rows (keep a row iff > 85 % of its pixels are non-dark).
// Pass 2 clamps to the input range and compacts the rows.
// The BMP pixel array (bottom-up, BGR) is consumed directly: flags bit0 = BGR, bit1 = bottom-up.
#include <algorithm>
#include <vector>

#include "common.cuh"

namespace nbc {

struct PreHeader {
  int inv_min;  // 255 - min(in), reduced with atomicMax so a zero-filled header is the identity
  int max;
  int pad[2];
};

// One launch handles up to kPreBatch scans (blockIdx.z = scan): a chunk of the engine's ragged batch goes through K1 in
// three launches instead of three per scan (the small trim / clamp kernels are launch-latency bound: 5 us each for
// microseconds of work).  Scan z reads raw[z] (memory rows [lo[z], hi[z]) are really there, the rest are zero by
// definition), uses the workspace slice z (header, row counts, the saturated u8 intermediate) and writes result z.
constexpr int kPreBatch = 16;
struct PreBatch {
  const uint8_t* raw[kPreBatch];
  int lo[kPreBatch], hi[kPreBatch];
};

__device__ __forceinline__ int byte_of(uint32_t v, int i) { return (v >> (8 * i)) & 0xFF; }

// The 48 source bytes of 4 output pixels on each of the 4 source rows of output row ho (zero where the thread is idle)
template <bool kAligned>
__device__ __forceinline__ void pass1_load(const uint8_t* __restrict__ raw, int H, int64_t pitch, int flags, int ho, int wo0,
                                           int npx, uint32_t (&words)[4][12]) {
  const int nbytes = npx * 12;
#pragma unroll
  for (int pr = 0; pr < 4; ++pr) {
    const int r = 4 * ho + pr;
    const int64_t rr = (flags & 2) ? (int64_t)(H - 1 - r) : (int64_t)r;
    const uint8_t* src = raw + rr * pitch + (int64_t)wo0 * 12;
    if (kAligned && npx == 4) {
      const uint4* s4 = reinterpret_cast<const uint4*>(src);
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        const uint4 v = __ldg(s4 + i);
        words[pr][4 * i] = v.x, words[pr][4 * i + 1] = v.y, words[pr][4 * i + 2] = v.z, words[pr][4 * i + 3] = v.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 12; ++i) {
        uint32_t v = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          const int idx = 4 * i + b;
          // replicate the first byte into the padding so it does not disturb min / max
          const uint32_t byte = (idx < nbytes) ? src[idx] : src[0];
          v |= byte << (8 * b);
        }
        words[pr][i] = v;
      }
    }
  }
}

// One block = one output row (256 threads x 4 output pixels).  The results leave as u8 SATURATED to [0, 255] -- pass 2
// clamps to the input range [lo, hi], a sub-interval, so clamp(clamp(v, 0, 255), lo, hi) == clamp(v, lo, hi) -- staged
// through shared memory so that a warp's 384 output bytes go out as 24 coalesced 16-byte stores instead of 384 two-byte
// ones (the partial-sector writes of the first version cost more than the 50 MB of reads).
// span_lo / span_hi: the memory rows [span_lo, span_hi) are the ones `raw` really holds (multiples of 4); every other row
// is all zero BY DEFINITION (the host found the scan's dark bands, nbc_host_zero_row_span, and copied only the rows in
// between) -- such a group of four rows is never dereferenced and contributes min = max = 0, S = 0.
// The body of one pass-1 block for one scan; resize4x_pass1 (uniform chunk) and mixed_resize4x_pass1 (mixed chunk) only
// differ in where they find the scan's pointers, span, pitch and flags.
template <bool kAligned>
__device__ __forceinline__ void resize4x_pass1_block(const uint8_t* __restrict__ raw, int span_lo, int span_hi, int H, int W,
                                                     int64_t pitch, int flags, PreHeader* hdr, int* __restrict__ rowcount,
                                                     uint8_t* __restrict__ r8) {
  __shared__ __align__(16) uint32_t s_out[8][96];   // per warp: 32 threads x 12 bytes
  const int Wo = W >> 2;
  const int groups = (Wo + 3) >> 2;  // 4 output pixels per thread
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  const int ho = blockIdx.y;
  const bool active = g < groups;
  const int wo0 = g << 2;
  const int npx = active ? min(4, Wo - wo0) : 0;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int mem_row = 4 * ((flags & 2) ? (H >> 2) - 1 - ho : ho);     // first memory row of this output row's group
  const bool zero_rows = mem_row < span_lo || mem_row >= span_hi;
  uint32_t mn2 = 0xFFFFFFFFu, mx2 = 0u;   // min / max as two 16-bit fields
  int nondark = 0;
  uint32_t packed[3] = {0u, 0u, 0u};      // the thread's 12 output bytes (4 pixels x RGB)
  if (active && zero_rows) mn2 = 0u;
  if (active && !zero_rows) {
    uint32_t cur[4][12];
    pass1_load<kAligned>(raw, H, pitch, flags, ho, wo0, npx, cur);
    // Vertical pass on PACKED 16-bit fields: each word (4 bytes of one row) is widened to two words of two 16-bit
    // fields (PRMT), so that min / max are one min.u16x2 / max.u16x2 each and the 4-tap column filter is plain 32-bit
    // integer arithmetic on two columns at once:  V' = 9 (r1 + r2) + 1020 - (r0 + r3)  in [0, 5610] -- no carry
    // between fields, never negative.  Horizontal pass: S = -V'[b] + 9 V'[b+3] + 9 V'[b+6] - V'[b+9] - 16 * 1020.
    uint32_t Vp[24];   // field f (byte column f of the 48) lives in Vp[f >> 1], bits 16 * (f & 1)
#pragma unroll
    for (int i = 0; i < 12; ++i) {
      uint32_t e[4][2];
#pragma unroll
      for (int pr = 0; pr < 4; ++pr) {
        e[pr][0] = __byte_perm(cur[pr][i], 0u, 0x4140);   // bytes 0, 1 -> fields
        e[pr][1] = __byte_perm(cur[pr][i], 0u, 0x4342);   // bytes 2, 3 -> fields
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          asm("min.u16x2 %0, %0, %1;" : "+r"(mn2) : "r"(e[pr][k]));
          asm("max.u16x2 %0, %0, %1;" : "+r"(mx2) : "r"(e[pr][k]));
        }
      }
#pragma unroll
      for (int k = 0; k < 2; ++k)
        Vp[2 * i + k] = 9u * (e[1][k] + e[2][k]) + (0x03FC03FCu - (e[0][k] + e[3][k]));   // 0x03FC = 1020 in both fields
    }
    auto field = [&](int f) { return (int)((Vp[f >> 1] >> (16 * (f & 1))) & 0xFFFFu); };
#pragma unroll
    for (int px = 0; px < 4; ++px) {
      if (px < npx) {
        int Sp[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int b = px * 12 + c;     // byte column of tap 0; taps are 3 columns apart
          Sp[c] = -field(b) + 9 * field(b + 3) + 9 * field(b + 6) - field(b + 9) - 16 * 1020;
        }
        nondark += (max(Sp[0], 0) + max(Sp[1], 0) + max(Sp[2], 0)) >= 66 ? 1 : 0;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          const int sc = (flags & 1) ? Sp[2 - c] : Sp[c];                  // BGR -> RGB
          const uint32_t v = (uint32_t)min(max((sc + 128) >> 8, 0), 255);
          const int byte = px * 3 + c;
          packed[byte >> 2] |= v << (8 * (byte & 3));
        }
      }
    }
  }
  // output: the warp's 32 x 12 bytes are contiguous in the row; stage them and store 16 bytes per lane
  s_out[wid][lane * 3] = packed[0], s_out[wid][lane * 3 + 1] = packed[1], s_out[wid][lane * 3 + 2] = packed[2];
  __syncwarp();
  {
    const int wo_warp = (blockIdx.x * blockDim.x + wid * 32) << 2;        // first output pixel of this warp
    const int valid_bytes = max(0, min(128, Wo - wo_warp)) * 3;           // bytes of the row this warp owns
    uint8_t* dst = r8 + ((int64_t)ho * Wo + wo_warp) * 3;
    const bool vec = ((reinterpret_cast<uintptr_t>(dst) & 15) == 0);
    int tail = 0;                                                         // first byte the byte loop has to store
    if (vec) {
      if (lane * 16 + 16 <= valid_bytes) reinterpret_cast<uint4*>(dst)[lane] = reinterpret_cast<const uint4*>(s_out[wid])[lane];
      tail = valid_bytes & ~15;
    }
    const uint8_t* sb = reinterpret_cast<const uint8_t*>(s_out[wid]);
    for (int i = tail + lane; i < valid_bytes; i += 32) dst[i] = sb[i];      // unaligned rows / the ragged end of a row
  }
  // reductions: warp, then one (min, max, count) per block; the two range atomics all land on the same address, so
  // they are skipped when they cannot change it (the values only grow, a stale read just means one redundant atomic)
  int mn = (int)min(mn2 & 0xFFFFu, mn2 >> 16), mx = (int)max(mx2 & 0xFFFFu, mx2 >> 16);
  if (!active) mn = 255, mx = 0;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    nondark += __shfl_xor_sync(0xffffffffu, nondark, o);
  }
  __shared__ int s_mn[8], s_mx[8], s_nd[8];
  if (lane == 0) s_mn[wid] = mn, s_mx[wid] = mx, s_nd[wid] = nondark;
  __syncthreads();
  if (threadIdx.x == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    for (int i = 1; i < nw; ++i) mn = min(mn, s_mn[i]), mx = max(mx, s_mx[i]), nondark += s_nd[i];
    if (255 - mn > __ldcg(&hdr->inv_min)) atomicMax(&hdr->inv_min, 255 - mn);
    if (mx > __ldcg(&hdr->max)) atomicMax(&hdr->max, mx);
    if (nondark) atomicAdd(&rowcount[ho], nondark);
  }
}

template <bool kAligned>
__global__ void __launch_bounds__(256) resize4x_pass1(const __grid_constant__ PreBatch batch, int H, int W, int64_t pitch,
                                                      int flags, uint8_t* __restrict__ hdrs, size_t hdr_stride,
                                                      uint8_t* __restrict__ r8s, size_t r8_stride) {
  const int z = blockIdx.z;
  resize4x_pass1_block<kAligned>(batch.raw[z], batch.lo[z], batch.hi[z], H, W, pitch, flags,
                                 reinterpret_cast<PreHeader*>(hdrs + z * hdr_stride),
                                 reinterpret_cast<int*>(hdrs + z * hdr_stride + sizeof(PreHeader)), r8s + z * r8_stride);
}

// rows of a u8 image that needs no resize: nondark <=> any channel non-zero (sum/255 > 1e-3)
__global__ void __launch_bounds__(256) rowcount_u8(const uint8_t* __restrict__ img, int H, int W,
                                                    int* __restrict__ rowcount) {
  const int h = blockIdx.x;
  int cnt = 0;
  for (int w = threadIdx.x; w < W; w += blockDim.x) {
    const uint8_t* p = img + ((int64_t)h * W + w) * 3;
    cnt += ((int)p[0] + p[1] + p[2]) >= 1 ? 1 : 0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&rowcount[h], cnt);
}

// trim_black row rule (models.py:160-164): keep[r] = count/W > 0.85; first = argmax(keep);
// last = H - argmax(keep[::-1]); nothing kept -> (0, H).  all_nondark: min(in) >= 1 makes every pixel non-dark.
// One block per scan: block z reads the row counts / header `ws_stride` bytes after those of block z - 1 (0 for a single
// scan) and writes first_last + 2 z.
__device__ __forceinline__ void trim_rows_block(const int* __restrict__ rowcount, const PreHeader* hdr, int Ho, int Wo, int square,
                                                int32_t* first_last) {
  __shared__ int s_first, s_last_from_end;
  if (threadIdx.x == 0) s_first = INT_MAX, s_last_from_end = INT_MAX;
  __syncthreads();
  const bool all_nondark = hdr && (255 - hdr->inv_min) >= 1;
  for (int r = threadIdx.x; r < Ho; r += blockDim.x) {
    const int c = all_nondark ? Wo : rowcount[r];
    const bool keep = ((double)c / (double)Wo) > 0.85;
    if (keep) {
      atomicMin(&s_first, r);
      atomicMin(&s_last_from_end, Ho - 1 - r);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    int first = 0, last = Ho;
    if (square && s_first != INT_MAX) {
      first = s_first;
      last = Ho - s_last_from_end;
    }
    first_last[0] = first;
    first_last[1] = last;
  }
}

__global__ void __launch_bounds__(1024) trim_rows_kernel(const int* __restrict__ rowcount, const PreHeader* hdr,
                                                         int Ho, int Wo, int square, int32_t* first_last, size_t ws_stride = 0) {
  rowcount = reinterpret_cast<const int*>(reinterpret_cast<const char*>(rowcount) + blockIdx.x * ws_stride);
  if (hdr) hdr = reinterpret_cast<const PreHeader*>(reinterpret_cast<const char*>(hdr) + blockIdx.x * ws_stride);
  trim_rows_block(rowcount, hdr, Ho, Wo, square, first_last + 2 * blockIdx.x);
}

__global__ void __launch_bounds__(256) resize4x_pass2(const uint8_t* __restrict__ hdrs, size_t hdr_stride,
                                                      const uint8_t* __restrict__ r8s, size_t r8_stride, int Wo,
                                                      const int32_t* __restrict__ first_last_all,
                                                      uint8_t* __restrict__ out_all, int64_t out_stride) {
  const int z = blockIdx.y;
  const uint8_t* __restrict__ r8 = r8s + z * r8_stride;
  const PreHeader* hdr = reinterpret_cast<const PreHeader*>(hdrs + z * hdr_stride);
  const int32_t* first_last = first_last_all + 2 * z;
  uint8_t* __restrict__ out = out_all + z * out_stride;
  const int first = first_last[0], last = first_last[1];
  const uint32_t lo = (uint32_t)(255 - hdr->inv_min), hi = (uint32_t)hdr->max;
  const uint32_t lo4 = lo * 0x01010101u, hi4 = hi * 0x01010101u;
  const int64_t total = (int64_t)(last - first) * Wo * 3;
  const uint8_t* src = r8 + (int64_t)first * Wo * 3;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * 16;
  const bool vec = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16; i < total; i += stride) {
    if (vec && i + 16 <= total) {
      uint4 v = __ldg(reinterpret_cast<const uint4*>(src + i));
      v.x = __vminu4(__vmaxu4(v.x, lo4), hi4), v.y = __vminu4(__vmaxu4(v.y, lo4), hi4);
      v.z = __vminu4(__vmaxu4(v.z, lo4), hi4), v.w = __vminu4(__vmaxu4(v.w, lo4), hi4);
      *reinterpret_cast<uint4*>(out + i) = v;
    } else {
      for (int64_t j = i; j < min(i + 16, total); ++j) out[j] = (uint8_t)min(max((uint32_t)src[j], lo), hi);
    }
  }
}

__global__ void __launch_bounds__(256) copy_rows_u8(const uint8_t* __restrict__ img, int W,
                                                    const int32_t* __restrict__ first_last, uint8_t* __restrict__ out) {
  const int first = first_last[0], last = first_last[1];
  const int64_t total = (int64_t)(last - first) * W * 3;
  const uint8_t* src = img + (int64_t)first * W * 3;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = src[i];
}

static size_t pre_header_bytes(int Ho) { return align_up(sizeof(PreHeader) + (size_t)Ho * sizeof(int), 256); }

// ------------------------------------------------------------------------------------------------------------
// General-ratio resize: any H x W image whose larger side exceeds the target becomes target x target
// (models.py:194-198: skimage.transform.resize(image, (1024, 1024), order=3, mode='reflect', anti_aliasing=False)).
// Restated as in oracle/preprocess.py::resize_general_f64 -- float64, separable Catmull-Rom cubic convolution
// (columns first, then rows), source coordinate (dst + 0.5) * (n_in / n_out) - 0.5, taps floor(src) - 1 .. + 2 reflected
// symmetrically at the border, result clipped to the input's global [min, max], u8 = floor(v + 0.5), non-dark iff
// (v0/255 + v1/255) + v2/255 > 1e-3 -- with every operation written as an explicitly rounded f64 intrinsic in the
// oracle's order (no FMA contraction), so that the bytes match the restatement.  Not a bandwidth kernel: one thread per
// output pixel gathers 4 x 4 x 3 input bytes; the 4x path above stays the one for the scanner's 4096^2 images.
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void minmax_block(const uint8_t* __restrict__ raw, int H, int W, int64_t pitch, PreHeader* hdr) {
  int mn = 255, mx = 0;
  const int64_t rowb = (int64_t)W * 3;
  for (int r = blockIdx.x; r < H; r += gridDim.x) {
    const uint8_t* p = raw + (int64_t)r * pitch;
    for (int64_t i = threadIdx.x; i < rowb; i += blockDim.x) {
      const int v = p[i];
      mn = min(mn, v), mx = max(mx, v);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMax(&hdr->inv_min, 255 - mn);
    atomicMax(&hdr->max, mx);
  }
}

__global__ void __launch_bounds__(256) minmax_u8(const uint8_t* __restrict__ raw, int H, int W, int64_t pitch, PreHeader* hdr) {
  minmax_block(raw, H, W, pitch, hdr);
}

struct CubicTaps {
  int idx[4];
  double t;
};
__device__ __forceinline__ CubicTaps cubic_taps(int n_in, int n_out, int o) {
  CubicTaps c;
  const double scale = __ddiv_rn((double)n_in, (double)n_out);
  const double src = __dsub_rn(__dmul_rn(__dadd_rn((double)o, 0.5), scale), 0.5);
  const double fl = floor(src);
  c.t = __dsub_rn(src, fl);
  const int i0 = (int)fl;
  const int period = 2 * n_in;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    int id = (i0 + k - 1) % period;
    if (id < 0) id += period;
    c.idx[k] = id >= n_in ? period - 1 - id : id;      // numpy 'symmetric': d c b a | a b c d | d c b a
  }
  return c;
}
// f1 + 0.5 x (f2 - f0 + x (2 f0 - 5 f1 + 4 f2 - f3 + x (3 (f1 - f2) + f3 - f0))), evaluated left to right as numpy does
__device__ __forceinline__ double cubic_f64(double f0, double f1, double f2, double f3, double x) {
  const double a = __dsub_rn(__dadd_rn(__dmul_rn(3.0, __dsub_rn(f1, f2)), f3), f0);
  const double b = __dadd_rn(
      __dsub_rn(__dadd_rn(__dsub_rn(__dmul_rn(2.0, f0), __dmul_rn(5.0, f1)), __dmul_rn(4.0, f2)), f3), __dmul_rn(x, a));
  const double c = __dadd_rn(__dsub_rn(f2, f0), __dmul_rn(x, b));
  return __dadd_rn(f1, __dmul_rn(__dmul_rn(0.5, x), c));
}

__device__ __forceinline__ void resize_general_block(const uint8_t* __restrict__ raw, int H, int W, int64_t pitch, int flags,
                                                     int Ho, int Wo, const PreHeader* __restrict__ hdr, uint8_t* __restrict__ r8,
                                                     int* __restrict__ rowcount) {
  const int ho = blockIdx.y;
  const int wo = blockIdx.x * blockDim.x + threadIdx.x;
  int nondark = 0;
  if (wo < Wo) {
    const CubicTaps rt = cubic_taps(H, Ho, ho), ct = cubic_taps(W, Wo, wo);
    const double lo = (double)(255 - hdr->inv_min), hi = (double)hdr->max;
    double v[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const int cs = (flags & 1) ? 2 - c : c;      // BGR source
      double col[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int r = rt.idx[k];
        const uint8_t* p = raw + ((flags & 2) ? (int64_t)(H - 1 - r) : (int64_t)r) * pitch + cs;
        col[k] = cubic_f64((double)p[(int64_t)ct.idx[0] * 3], (double)p[(int64_t)ct.idx[1] * 3], (double)p[(int64_t)ct.idx[2] * 3],
                           (double)p[(int64_t)ct.idx[3] * 3], ct.t);
      }
      double o = cubic_f64(col[0], col[1], col[2], col[3], rt.t);
      o = fmin(fmax(o, lo), hi);      // np.clip(out, img.min(), img.max())
      v[c] = o;
      r8[((int64_t)ho * Wo + wo) * 3 + c] = (uint8_t)(int)floor(__dadd_rn(o, 0.5));
    }
    const double s = __dadd_rn(__dadd_rn(__ddiv_rn(v[0], 255.0), __ddiv_rn(v[1], 255.0)), __ddiv_rn(v[2], 255.0));
    nondark = s > 1e-3 ? 1 : 0;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) nondark += __shfl_xor_sync(0xffffffffu, nondark, o);
  if ((threadIdx.x & 31) == 0 && nondark) atomicAdd(&rowcount[ho], nondark);
}

__global__ void __launch_bounds__(256) resize_general_kernel(const uint8_t* __restrict__ raw, int H, int W, int64_t pitch,
                                                             int flags, int Ho, int Wo, const PreHeader* __restrict__ hdr,
                                                             uint8_t* __restrict__ r8, int* __restrict__ rowcount) {
  resize_general_block(raw, H, W, pitch, flags, Ho, Wo, hdr, r8, rowcount);
}

// ------------------------------------------------------------------------------------------------------------
// Mixed chunk: raw images of any size in one call (nbc_preprocess_mixed_batch_u8), each routed as Preprocessor.preprocess_array
// routes it.  The per-image geometry lives in a device table at the start of the workspace; every kernel family runs once
// for the chunk with blockIdx.z = the z-th image of its kind (the table's per-kind index lists), and each image has its own
// header (global min / max, row counts), intermediate and {first,last}.  The blocks run the same device code as the
// per-image entries, so every image's bytes equal theirs.
// ------------------------------------------------------------------------------------------------------------
enum MixedKind { kMixed4x = 0, kMixedGeneral = 1, kMixedTrim = 2, kMixedCopy = 3 };

struct MixedImage {
  const uint8_t* raw;   // memory row r of the pixel array is at raw + r * pitch (rows outside [lo, hi) are never read)
  int64_t pitch;
  int H, W, flags, kind;
  int lo, hi;           // memory rows the buffer really holds (the zero-band span of a 4x scan; [0, H) otherwise)
  int Ho, Wo;           // processed size before the trim
};

struct MixedTable {
  const MixedImage* img;
  const int* list[4];   // per kind: the images of that kind, in chunk order
  uint8_t* hdrs;        // per image: PreHeader + row counts
  size_t hdr_stride;
  uint8_t* r8s;         // per image: the untrimmed processed image, Ho x Wo x 3
  size_t r8_stride;
};

template <bool kAligned>
__global__ void __launch_bounds__(256) mixed_resize4x_pass1(const __grid_constant__ MixedTable t, int H, int W) {
  const int i = t.list[kMixed4x][blockIdx.z];
  const MixedImage& m = t.img[i];
  uint8_t* hdr = t.hdrs + i * t.hdr_stride;
  resize4x_pass1_block<kAligned>(m.raw, m.lo, m.hi, H, W, m.pitch, m.flags, reinterpret_cast<PreHeader*>(hdr),
                                 reinterpret_cast<int*>(hdr + sizeof(PreHeader)), t.r8s + i * t.r8_stride);
}

__global__ void __launch_bounds__(256) mixed_minmax(const __grid_constant__ MixedTable t) {
  const int i = t.list[kMixedGeneral][blockIdx.z];
  const MixedImage& m = t.img[i];
  minmax_block(m.raw, m.H, m.W, m.pitch, reinterpret_cast<PreHeader*>(t.hdrs + i * t.hdr_stride));
}

__global__ void __launch_bounds__(256) mixed_resize_general(const __grid_constant__ MixedTable t) {
  const int i = t.list[kMixedGeneral][blockIdx.z];
  const MixedImage& m = t.img[i];
  uint8_t* hdr = t.hdrs + i * t.hdr_stride;
  resize_general_block(m.raw, m.H, m.W, m.pitch, m.flags, m.Ho, m.Wo, reinterpret_cast<const PreHeader*>(hdr),
                       t.r8s + i * t.r8_stride, reinterpret_cast<int*>(hdr + sizeof(PreHeader)));
}

// images that need no resize: one block per row turns the raw row (pitch, BGR, bottom-up) into RGB top-down in the
// intermediate and, for those that are trimmed, counts its non-dark pixels as rowcount_u8 does (any channel non-zero)
__global__ void __launch_bounds__(256) mixed_small_rows(const __grid_constant__ MixedTable t, int kind) {
  const int i = t.list[kind][blockIdx.z];
  const MixedImage& m = t.img[i];
  const int h = blockIdx.x;
  if (h >= m.H) return;
  const uint8_t* src = m.raw + ((m.flags & 2) ? (int64_t)(m.H - 1 - h) : (int64_t)h) * m.pitch;
  uint8_t* dst = t.r8s + i * t.r8_stride + (int64_t)h * m.W * 3;
  const bool bgr = m.flags & 1;
  int cnt = 0;
  for (int w = threadIdx.x; w < m.W; w += blockDim.x) {
    const uint8_t c0 = src[w * 3], c1 = src[w * 3 + 1], c2 = src[w * 3 + 2];
    dst[w * 3] = bgr ? c2 : c0, dst[w * 3 + 1] = c1, dst[w * 3 + 2] = bgr ? c0 : c2;
    cnt += ((int)c0 + c1 + c2) >= 1 ? 1 : 0;
  }
  if (kind != kMixedTrim) return;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(reinterpret_cast<int*>(t.hdrs + i * t.hdr_stride + sizeof(PreHeader)) + h, cnt);
}

// {first,last} of every image (block z = image z): trim_black on the square results, [0, H) for the untouched ones.
// Resized images pass their header, as the per-image entries do (min(in) >= 1 makes every pixel non-dark).
__global__ void __launch_bounds__(1024) mixed_trim_rows(const __grid_constant__ MixedTable t, int32_t* first_last) {
  const int i = blockIdx.x;
  const MixedImage& m = t.img[i];
  const uint8_t* hdr = t.hdrs + i * t.hdr_stride;
  const bool resized = m.kind == kMixed4x || m.kind == kMixedGeneral;
  trim_rows_block(reinterpret_cast<const int*>(hdr + sizeof(PreHeader)), resized ? reinterpret_cast<const PreHeader*>(hdr) : nullptr,
                  m.Ho, m.Wo, m.kind != kMixedCopy ? 1 : 0, first_last + 2 * i);
}

// rows [first, last) of every image to out + z * out_stride; the 4x intermediate is saturated to [0, 255] and is clamped to
// the input range here (resize4x_pass2), the others are final already (copy_rows_u8)
__global__ void __launch_bounds__(256) mixed_store(const __grid_constant__ MixedTable t, const int32_t* __restrict__ first_last,
                                                   uint8_t* __restrict__ out_all, int64_t out_stride) {
  const int i = blockIdx.y;
  const MixedImage& m = t.img[i];
  const PreHeader* hdr = reinterpret_cast<const PreHeader*>(t.hdrs + i * t.hdr_stride);
  const bool clamp = m.kind == kMixed4x;
  const uint32_t lo = clamp ? (uint32_t)(255 - hdr->inv_min) : 0u, hi = clamp ? (uint32_t)hdr->max : 255u;
  const uint32_t lo4 = lo * 0x01010101u, hi4 = hi * 0x01010101u;
  const int first = first_last[2 * i], last = first_last[2 * i + 1];
  const int64_t total = (int64_t)(last - first) * m.Wo * 3;
  const uint8_t* src = t.r8s + i * t.r8_stride + (int64_t)first * m.Wo * 3;
  uint8_t* __restrict__ out = out_all + i * out_stride;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x * 16;
  const bool vec = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(out)) & 15) == 0;
  for (int64_t j = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 16; j < total; j += stride) {
    if (vec && j + 16 <= total) {
      uint4 v = __ldg(reinterpret_cast<const uint4*>(src + j));
      v.x = __vminu4(__vmaxu4(v.x, lo4), hi4), v.y = __vminu4(__vmaxu4(v.y, lo4), hi4);
      v.z = __vminu4(__vmaxu4(v.z, lo4), hi4), v.w = __vminu4(__vmaxu4(v.w, lo4), hi4);
      *reinterpret_cast<uint4*>(out + j) = v;
    } else {
      for (int64_t k = j; k < min(j + 16, total); ++k) out[k] = (uint8_t)min(max((uint32_t)src[k], lo), hi);
    }
  }
}

}  // namespace nbc

using namespace nbc;

extern "C" size_t nbc_preprocess_workspace_bytes(int H, int W) {
  const int Ho = H / 4, Wo = W / 4;
  return pre_header_bytes(Ho > H ? Ho : H) + align_up((size_t)Ho * Wo * 3 * sizeof(int16_t), 256);
}

static int preprocess_4x_batch(const uint8_t* const* raw_spans, const int32_t* span_row0, const int32_t* span_rows, int n, int H,
                               int W, int64_t pitch, int flags, uint8_t* out, int64_t out_stride, int32_t* first_last,
                               void* workspace, size_t workspace_bytes, cudaStream_t stream, const char* who) {
  NBC_REQUIRE(raw_spans && out && first_last && workspace && n > 0, "%s: null pointer", who);
  NBC_REQUIRE(H > 0 && W > 0 && H % 4 == 0 && W % 4 == 0, "%s: H and W must be multiples of 4 (got %dx%d)", who, H, W);
  NBC_REQUIRE(pitch >= (int64_t)W * 3, "%s: pitch %lld < 3*W", who, (long long)pitch);
  const size_t ws_stride = nbc_preprocess_workspace_bytes(H, W);
  if (workspace_bytes < ws_stride * (size_t)n) {
    set_error("%s: workspace %zu < %zu", who, workspace_bytes, ws_stride * (size_t)n);
    return NBC_ERR_WORKSPACE;
  }
  const int Ho = H / 4, Wo = W / 4;
  // workspace: n headers (min / max + per-row non-dark counts) first -- one memset clears them all -- then the n saturated
  // u8 intermediates (Ho x Wo x 3 each)
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  const size_t hdr_stride = pre_header_bytes(H), r8_stride = ws_stride - hdr_stride;
  uint8_t* r8s = ws + (size_t)n * hdr_stride;
  NBC_CUDA(cudaMemsetAsync(ws, 0, (size_t)n * hdr_stride, stream));
  bool aligned = pitch % 16 == 0;
  for (int i = 0; i < n; ++i) {
    const int r0 = span_row0 ? span_row0[i] : 0, rows = span_rows ? span_rows[i] : H;
    NBC_REQUIRE((raw_spans[i] || rows == 0) && r0 >= 0 && rows >= 0 && r0 % 4 == 0 && rows % 4 == 0 && r0 + rows <= H,
                "%s: the span [%d, +%d) of scan %d must be made of whole groups of 4 rows inside the image", who, r0, rows, i);
    aligned = aligned && (reinterpret_cast<uintptr_t>(raw_spans[i]) % 16 == 0);
  }
  const int groups = (Wo + 3) / 4;
  const int64_t total16 = ceil_div64((int64_t)Ho * Wo * 3, 16);
  const int blocks2 = (int)(total16 < 256 ? 1 : (ceil_div64(total16, 256) < 4 * 148 ? ceil_div64(total16, 256) : 4 * 148));
  for (int i0 = 0; i0 < n; i0 += kPreBatch) {
    const int nb = n - i0 < kPreBatch ? n - i0 : kPreBatch;
    PreBatch b;
    for (int j = 0; j < kPreBatch; ++j) {
      const int i = i0 + (j < nb ? j : 0);
      const int r0 = span_row0 ? span_row0[i] : 0, rows = span_rows ? span_rows[i] : H;
      // the kernel addresses memory row r at raw + r * pitch and never touches a row outside the span
      b.raw[j] = raw_spans[i] ? raw_spans[i] - (int64_t)r0 * pitch : ws;
      b.lo[j] = r0, b.hi[j] = r0 + rows;
    }
    const dim3 grid(ceil_div(groups, 256), Ho, nb);
    if (aligned)
      resize4x_pass1<true><<<grid, 256, 0, stream>>>(b, H, W, pitch, flags, ws + i0 * hdr_stride, hdr_stride, r8s + i0 * r8_stride,
                                                     r8_stride);
    else
      resize4x_pass1<false><<<grid, 256, 0, stream>>>(b, H, W, pitch, flags, ws + i0 * hdr_stride, hdr_stride, r8s + i0 * r8_stride,
                                                      r8_stride);
    NBC_CHECK_LAUNCH();
  }
  trim_rows_kernel<<<n, 1024, 0, stream>>>(reinterpret_cast<const int*>(ws + sizeof(PreHeader)), reinterpret_cast<const PreHeader*>(ws),
                                          Ho, Wo, Ho == Wo ? 1 : 0, first_last, hdr_stride);
  NBC_CHECK_LAUNCH();
  resize4x_pass2<<<dim3(blocks2, n), 256, 0, stream>>>(ws, hdr_stride, r8s, r8_stride, Wo, first_last, out, out_stride);
  NBC_CHECK_LAUNCH();
  return 0;
}

extern "C" int nbc_preprocess_4x_u8(const uint8_t* raw, int H, int W, int64_t pitch, int flags, uint8_t* out,
                                    int32_t* first_last, void* workspace, size_t workspace_bytes, void* stream_) {
  NBC_REQUIRE(raw, "nbc_preprocess_4x_u8: null pointer");
  return preprocess_4x_batch(&raw, nullptr, nullptr, 1, H, W, pitch, flags, out, 0, first_last, workspace, workspace_bytes,
                             reinterpret_cast<cudaStream_t>(stream_), "nbc_preprocess_4x_u8");
}

extern "C" int nbc_preprocess_4x_span_u8(const uint8_t* raw_span, int H, int W, int64_t pitch, int flags, int span_row0,
                                         int span_rows, uint8_t* out, int32_t* first_last, void* workspace,
                                         size_t workspace_bytes, void* stream_) {
  const int32_t r0 = span_row0, rows = span_rows;
  return preprocess_4x_batch(&raw_span, &r0, &rows, 1, H, W, pitch, flags, out, 0, first_last, workspace, workspace_bytes,
                             reinterpret_cast<cudaStream_t>(stream_), "nbc_preprocess_4x_span_u8");
}

extern "C" int nbc_preprocess_4x_batch_u8(const uint8_t* const* raw_spans, const int32_t* span_row0, const int32_t* span_rows,
                                          int n, int H, int W, int64_t pitch, int flags, uint8_t* out, int64_t out_stride_bytes,
                                          int32_t* first_last, void* workspace, size_t workspace_bytes, void* stream_) {
  NBC_REQUIRE(n > 0 && n <= 4096, "nbc_preprocess_4x_batch_u8: bad scan count %d", n);
  NBC_REQUIRE(out_stride_bytes >= (int64_t)(H / 4) * (W / 4) * 3, "nbc_preprocess_4x_batch_u8: out stride smaller than one result");
  return preprocess_4x_batch(raw_spans, span_row0, span_rows, n, H, W, pitch, flags, out, out_stride_bytes, first_last, workspace,
                             workspace_bytes, reinterpret_cast<cudaStream_t>(stream_), "nbc_preprocess_4x_batch_u8");
}

extern "C" int nbc_trim_u8(const uint8_t* img, int H, int W, uint8_t* out, int32_t* first_last, void* workspace,
                           size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  NBC_REQUIRE(img && out && first_last && workspace, "nbc_trim_u8: null pointer");
  NBC_REQUIRE(H > 0 && W > 0, "nbc_trim_u8: bad shape");
  if (workspace_bytes < pre_header_bytes(H)) {
    set_error("nbc_trim_u8: workspace too small");
    return NBC_ERR_WORKSPACE;
  }
  char* ws = reinterpret_cast<char*>(workspace);
  int* rowcount = reinterpret_cast<int*>(ws + sizeof(PreHeader));
  NBC_CUDA(cudaMemsetAsync(ws, 0, sizeof(PreHeader) + (size_t)H * sizeof(int), stream));
  rowcount_u8<<<H, 256, 0, stream>>>(img, H, W, rowcount);
  NBC_CHECK_LAUNCH();
  trim_rows_kernel<<<1, 1024, 0, stream>>>(rowcount, nullptr, H, W, H == W ? 1 : 0, first_last);
  NBC_CHECK_LAUNCH();
  copy_rows_u8<<<4 * 148, 256, 0, stream>>>(img, W, first_last, out);
  NBC_CHECK_LAUNCH();
  return 0;
}

extern "C" size_t nbc_preprocess_general_workspace_bytes(int H, int W, int target) {
  (void)H, (void)W;
  if (target <= 0) return 0;
  return pre_header_bytes(target) + align_up((size_t)target * target * 3, 256);
}

extern "C" int nbc_preprocess_general_u8(const uint8_t* raw, int H, int W, int64_t pitch, int flags, int target, uint8_t* out,
                                         int32_t* first_last, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  NBC_REQUIRE(raw && out && first_last && workspace, "nbc_preprocess_general_u8: null pointer");
  NBC_REQUIRE(H > 0 && W > 0 && target > 0 && H < (1 << 20) && W < (1 << 20), "nbc_preprocess_general_u8: bad shape %dx%d -> %d", H, W,
              target);
  NBC_REQUIRE(pitch >= (int64_t)W * 3, "nbc_preprocess_general_u8: pitch %lld < 3*W", (long long)pitch);
  if (workspace_bytes < nbc_preprocess_general_workspace_bytes(H, W, target)) {
    set_error("nbc_preprocess_general_u8: workspace %zu < %zu", workspace_bytes, nbc_preprocess_general_workspace_bytes(H, W, target));
    return NBC_ERR_WORKSPACE;
  }
  const int Ho = target, Wo = target;
  char* ws = reinterpret_cast<char*>(workspace);
  PreHeader* hdr = reinterpret_cast<PreHeader*>(ws);
  int* rowcount = reinterpret_cast<int*>(ws + sizeof(PreHeader));
  uint8_t* r8 = reinterpret_cast<uint8_t*>(ws + pre_header_bytes(target));
  NBC_CUDA(cudaMemsetAsync(ws, 0, sizeof(PreHeader) + (size_t)Ho * sizeof(int), stream));
  minmax_u8<<<H < 4 * 148 ? H : 4 * 148, 256, 0, stream>>>(raw, H, W, pitch, hdr);
  NBC_CHECK_LAUNCH();
  resize_general_kernel<<<dim3(ceil_div(Wo, 256), Ho), 256, 0, stream>>>(raw, H, W, pitch, flags, Ho, Wo, hdr, r8, rowcount);
  NBC_CHECK_LAUNCH();
  // the resized image is target x target, i.e. square: trim_black always applies (models.py:200)
  trim_rows_kernel<<<1, 1024, 0, stream>>>(rowcount, hdr, Ho, Wo, 1, first_last);
  NBC_CHECK_LAUNCH();
  copy_rows_u8<<<4 * 148, 256, 0, stream>>>(r8, Wo, first_last, out);
  NBC_CHECK_LAUNCH();
  return 0;
}

// ---- mixed chunk ---------------------------------------------------------------------------------------------
static size_t mixed_table_bytes(int n) { return align_up((size_t)n * sizeof(MixedImage) + 4 * (size_t)n * sizeof(int), 256); }
static size_t mixed_hdr_stride(int target) { return pre_header_bytes(target); }
static size_t mixed_r8_stride(int target) { return align_up((size_t)target * target * 3, 256); }

extern "C" size_t nbc_preprocess_mixed_workspace_bytes(const nbc_mixed_desc* descs, int n, int target) {
  (void)descs;
  if (n <= 0 || target <= 0) return 0;
  return mixed_table_bytes(n) + (size_t)n * (mixed_hdr_stride(target) + mixed_r8_stride(target));
}

extern "C" int nbc_preprocess_mixed_batch_u8(const nbc_mixed_desc* descs, int n, int target, uint8_t* out, int64_t out_stride_bytes,
                                             int32_t* first_last, void* workspace, size_t workspace_bytes, void* stream_) {
  const char* who = "nbc_preprocess_mixed_batch_u8";
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  NBC_REQUIRE(descs && out && first_last && workspace, "%s: null pointer", who);
  NBC_REQUIRE(n > 0 && n <= 4096 && target > 0 && target < (1 << 14), "%s: bad image count %d or target %d", who, n, target);
  const size_t need = nbc_preprocess_mixed_workspace_bytes(descs, n, target);
  if (workspace_bytes < need) {
    set_error("%s: workspace %zu < %zu", who, workspace_bytes, need);
    return NBC_ERR_WORKSPACE;
  }
  // the table: images, then the four per-kind index lists; routed as Preprocessor.preprocess_array (models.py:194-201)
  std::vector<uint8_t> host(mixed_table_bytes(n), 0);
  MixedImage* img = reinterpret_cast<MixedImage*>(host.data());
  int* lists = reinterpret_cast<int*>(host.data() + (size_t)n * sizeof(MixedImage));
  int count[4] = {0, 0, 0, 0}, small_rows = 0, general_rows = 0;
  bool aligned = true;
  std::vector<int> order[4];
  for (int i = 0; i < n; ++i) {
    const nbc_mixed_desc& d = descs[i];
    NBC_REQUIRE(d.H > 0 && d.W > 0 && d.H < (1 << 20) && d.W < (1 << 20) && d.pitch >= (int64_t)d.W * 3 && d.flags >= 0 && d.flags <= 3,
                "%s: image %d: bad geometry %dx%d, pitch %lld, flags %d", who, i, d.H, d.W, (long long)d.pitch, d.flags);
    MixedImage& m = img[i];
    const bool resize = (d.H > d.W ? d.H : d.W) > target;
    m.kind = !resize ? (d.H == d.W ? kMixedTrim : kMixedCopy) : (d.H == 4 * target && d.W == 4 * target ? kMixed4x : kMixedGeneral);
    if (m.kind == kMixed4x) {
      NBC_REQUIRE((d.raw || d.span_rows == 0) && d.span_row0 >= 0 && d.span_rows >= 0 && d.span_row0 % 4 == 0 && d.span_rows % 4 == 0 &&
                      d.span_row0 + d.span_rows <= d.H,
                  "%s: image %d: the span [%d, +%d) must be made of whole groups of 4 rows inside the image", who, i, d.span_row0,
                  d.span_rows);
    } else {
      NBC_REQUIRE(d.raw && d.span_row0 == 0 && d.span_rows == d.H,
                  "%s: image %d (%dx%d): only a 4 * target square scan may hold a part of its rows", who, i, d.H, d.W);
    }
    // the kernels address memory row r at raw + r * pitch and never touch a row outside the span
    m.raw = d.raw ? d.raw - (int64_t)d.span_row0 * d.pitch : reinterpret_cast<const uint8_t*>(workspace);
    m.pitch = d.pitch, m.H = d.H, m.W = d.W, m.flags = d.flags;
    m.lo = d.span_row0, m.hi = d.span_row0 + d.span_rows;
    m.Ho = resize ? target : d.H, m.Wo = resize ? target : d.W;
    NBC_REQUIRE(out_stride_bytes >= (int64_t)m.Ho * m.Wo * 3, "%s: out stride %lld smaller than the %dx%d result of image %d", who,
                (long long)out_stride_bytes, m.Ho, m.Wo, i);
    if (m.kind == kMixed4x) aligned = aligned && d.pitch % 16 == 0 && reinterpret_cast<uintptr_t>(m.raw) % 16 == 0;
    if (m.kind == kMixedTrim || m.kind == kMixedCopy) small_rows = d.H > small_rows ? d.H : small_rows;
    if (m.kind == kMixedGeneral) general_rows = d.H > general_rows ? d.H : general_rows;
    order[m.kind].push_back(i);
  }
  uint8_t* ws = reinterpret_cast<uint8_t*>(workspace);
  MixedTable t;
  t.img = reinterpret_cast<const MixedImage*>(ws);
  for (int k = 0, off = 0; k < 4; ++k) {
    count[k] = (int)order[k].size();
    std::copy(order[k].begin(), order[k].end(), lists + off);
    t.list[k] = reinterpret_cast<const int*>(ws + (size_t)n * sizeof(MixedImage)) + off;
    off += count[k];
  }
  t.hdr_stride = mixed_hdr_stride(target), t.r8_stride = mixed_r8_stride(target);
  t.hdrs = ws + mixed_table_bytes(n);
  t.r8s = t.hdrs + (size_t)n * t.hdr_stride;
  // pageable source: the copy is staged before cudaMemcpyAsync returns, so `host` may go out of scope
  NBC_CUDA(cudaMemcpyAsync(ws, host.data(), host.size(), cudaMemcpyHostToDevice, stream));
  NBC_CUDA(cudaMemsetAsync(t.hdrs, 0, (size_t)n * t.hdr_stride, stream));
  if (count[kMixed4x]) {
    const dim3 grid(ceil_div((target + 3) / 4, 256), target, count[kMixed4x]);
    if (aligned)
      mixed_resize4x_pass1<true><<<grid, 256, 0, stream>>>(t, 4 * target, 4 * target);
    else
      mixed_resize4x_pass1<false><<<grid, 256, 0, stream>>>(t, 4 * target, 4 * target);
    NBC_CHECK_LAUNCH();
  }
  if (count[kMixedGeneral]) {
    mixed_minmax<<<dim3(general_rows < 4 * 148 ? general_rows : 4 * 148, 1, count[kMixedGeneral]), 256, 0, stream>>>(t);
    NBC_CHECK_LAUNCH();
    mixed_resize_general<<<dim3(ceil_div(target, 256), target, count[kMixedGeneral]), 256, 0, stream>>>(t);
    NBC_CHECK_LAUNCH();
  }
  for (int kind : {kMixedTrim, kMixedCopy}) {
    if (!count[kind]) continue;
    mixed_small_rows<<<dim3(small_rows, 1, count[kind]), 256, 0, stream>>>(t, kind);
    NBC_CHECK_LAUNCH();
  }
  mixed_trim_rows<<<n, 1024, 0, stream>>>(t, first_last);
  NBC_CHECK_LAUNCH();
  const int64_t total16 = ceil_div64((int64_t)target * target * 3, 16);
  const int blocks = (int)(ceil_div64(total16, 256) < 4 * 148 ? ceil_div64(total16, 256) : 4 * 148);
  mixed_store<<<dim3(blocks, n), 256, 0, stream>>>(t, first_last, out, out_stride_bytes);
  NBC_CHECK_LAUNCH();
  return 0;
}
