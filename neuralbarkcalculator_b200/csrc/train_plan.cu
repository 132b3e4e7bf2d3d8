// Native training step of FCN-ResNet50 (row a14; reference __main__.py:231-269 with the CustomWeightedCrossEntropy of
// utils.py:151-165 as the loss): train-mode forward (batch-statistics BatchNorm, Dropout), loss, full backward and
// Adam -- every FLOP in this library's kernels; the convolutions (forward and data gradient) run on conv_tc.cu.
//
// Parameters live in ONE flat f32 buffer (per unit: conv weight in [Cout][kh][kw][Cin] order, gamma, beta; then the
// classifier), gradients / Adam moments in buffers of the same layout, so the optimiser is one fused pass and the
// data-parallel gradient exchange is one NCCL all-reduce over the flat gradient buffer (done by the caller).
#include <vector>

#include "common.cuh"
#include "conv.h"
#include "train.h"

namespace nbc {

struct Unit {
  int Cin, Cout, k, stride, pad, dil, relu;
  int Hin, Win, Ho, Wo;
  size_t w_off, g_off, b_off;  // floats, in the flat parameter buffer
  size_t rs_off;               // floats, in the running-stats buffer: mean[C] then var[C]
  size_t x_off;                // bytes: input activation of this unit (workspace)
  size_t z_off, y_off;         // bytes: pre-BN / post-BN(+ReLU) output
  size_t st_off;               // bytes: save_mean, save_invstd, a, b (C floats each), sums (2C)
  size_t wf_off, wd_off;       // bytes: packed bf16 forward / dgrad weights
  int sd_index;                // index of the conv weight in the 326-tensor state_dict
  // backward schedule (bytes, workspace): where the data gradient goes and what is added to it
  size_t dgrad_out_off, dgrad_res_off;
  size_t cap_off;              // bytes, in the capture buffer: dy, then dz (each N*Ho*Wo*Cout bf16)
  bool dgrad_has_res = false, need_dgrad = true;
  bool frozen = false;         // nbc_train_set_frozen: eval-mode BN folded into the conv, no backward
  ConvTcPrepared fwd, dgrad;
};

struct TBlock {
  int c1, c2, c3, ds;     // unit indices, ds = -1 if none
  size_t gin_off, gout_off;  // gradient w.r.t. the block output / input
};

}  // namespace nbc

struct nbc_train_plan {
  int N, H, W;
  int H2, W2, H4, W4, H8, W8;
  std::vector<nbc::Unit> units;  // units[0] = stem, last = head conv
  std::vector<nbc::TBlock> blocks;
  int head_unit = -1;
  size_t cls_w_off = 0, cls_b_off = 0;  // floats
  size_t n_params = 0, n_stats = 0;
  size_t padded_off, pool_off, pidx_off, drop_off, low_off, full_off, dfull_off, dlow_off, upws_off, gA_off, gB_off, gskip_off, dz_off,
      d1_off, d2_off, up_off, partial_off, zeros_off, wce_off, ws_bytes;
  size_t big_bytes, small_bytes;
  size_t capture_bytes = 0;
  void* capture = nullptr;  // nbc_train_set_capture: per-unit copies of the BN backward's dy and dz (off when null)
  void* prepared_ws = nullptr;
  int wgrad_impl = 0;   // 0 = tcgen05 (wgrad_tc.cu), 1 = mma.sync / CUDA-core cross-check kernels
  int loss_kind = 0;    // 0 = weighted CE, 1 = Lovasz-Softmax, 2 = CE / 4 + Lovasz
  int accumulate = 0;   // 1: the step adds to `grads` (every gradient writer is an atomic / red add) instead of zeroing it
  // nbc_train_set_frozen: units [0, first_unit) and blocks [0, first_block) are frozen; both 0 = nothing frozen
  int frozen = 0, first_unit = 0, first_block = 0;
  size_t fold_off = 0;  // bytes, workspace: the frozen stem's folded f32 weights [64][7][7][3] before the w224 pack
  size_t lov_off = 0, dfull2_off = 0, loss2_off = 0;
  // scratch of the deterministic weight-gradient reductions: the split partials of one wgrad_tc launch (reused by
  // the next, which the stream orders behind its reduction) and the classifier's per-block partials
  size_t wgpart_off = 0, wgpart_bytes = 0, clspart_off = 0;
  // gradient-ready events, one per SEGMENT of the flat gradient buffer in the order the backward finishes them:
  // segment 0 = head conv + classifier, then the bottleneck blocks last to first, then the stem (created lazily)
  std::vector<cudaEvent_t> seg_events;
  ~nbc_train_plan() {
    for (cudaEvent_t e : seg_events) cudaEventDestroy(e);
  }
};

namespace nbc {

static size_t al(size_t x) { return align_up(x, 1024); }

static int add_unit(nbc_train_plan* p, int Cin, int Cout, int k, int stride, int pad, int dil, int relu, int Hin, int Win,
                    int sd_index) {
  Unit u;
  memset(&u.fwd, 0, sizeof(u.fwd));
  memset(&u.dgrad, 0, sizeof(u.dgrad));
  u.Cin = Cin, u.Cout = Cout, u.k = k, u.stride = stride, u.pad = pad, u.dil = dil, u.relu = relu;
  u.Hin = Hin, u.Win = Win;
  u.Ho = (Hin + 2 * pad - dil * (k - 1) - 1) / stride + 1;
  u.Wo = (Win + 2 * pad - dil * (k - 1) - 1) / stride + 1;
  u.w_off = p->n_params, p->n_params += (size_t)Cout * k * k * Cin;
  u.g_off = p->n_params, p->n_params += Cout;
  u.b_off = p->n_params, p->n_params += Cout;
  u.rs_off = p->n_stats, p->n_stats += 2 * (size_t)Cout;
  u.sd_index = sd_index;
  u.x_off = u.z_off = u.y_off = u.st_off = u.wf_off = u.wd_off = u.dgrad_out_off = u.dgrad_res_off = u.cap_off = 0;
  p->units.push_back(u);
  return (int)p->units.size() - 1;
}

}  // namespace nbc

using namespace nbc;

extern "C" nbc_train_plan* nbc_train_create(int N, int H, int W) {
  if (N <= 0 || H < 32 || W < 32) {
    set_error("nbc_train_create: bad shape");
    return nullptr;
  }
  nbc_train_plan* p = new nbc_train_plan();
  p->N = N, p->H = H, p->W = W;
  p->H2 = (H - 1) / 2 + 1, p->W2 = (W - 1) / 2 + 1;
  p->H4 = (p->H2 - 1) / 2 + 1, p->W4 = (p->W2 - 1) / 2 + 1;
  p->H8 = (p->H4 - 1) / 2 + 1, p->W8 = (p->W4 - 1) / 2 + 1;
  int sd = 0;
  add_unit(p, 3, 64, 7, 2, 3, 1, 1, H, W, sd);  // stem
  sd += 6;
  const int nblocks[4] = {3, 4, 6, 3}, planes[4] = {64, 128, 256, 512};
  int inpl = 64, dilation = 1, h = p->H4, w = p->W4;
  for (int li = 0; li < 4; ++li) {
    int stride = (li == 0) ? 1 : 2;
    const int prev_dil = dilation;
    if (li >= 2) dilation *= stride, stride = 1;
    for (int b = 0; b < nblocks[li]; ++b) {
      const int width = planes[li], outp = width * 4;
      const int s = (b == 0) ? stride : 1, dl = (b == 0) ? prev_dil : dilation;
      TBlock B;
      B.gin_off = B.gout_off = 0;
      B.c1 = add_unit(p, inpl, width, 1, 1, 0, 1, 1, h, w, sd);
      sd += 6;
      B.c2 = add_unit(p, width, width, 3, s, dl, dl, 1, h, w, sd);
      sd += 6;
      const int h2 = p->units[B.c2].Ho, w2 = p->units[B.c2].Wo;
      B.c3 = add_unit(p, width, outp, 1, 1, 0, 1, 1, h2, w2, sd);  // ReLU after the residual add
      sd += 6;
      B.ds = -1;
      if (b == 0) {
        B.ds = add_unit(p, inpl, outp, 1, s, 0, 1, 0, h, w, sd);
        sd += 6;
      }
      inpl = outp, h = h2, w = w2;
      p->blocks.push_back(B);
    }
  }
  p->head_unit = add_unit(p, 2048, 512, 3, 1, 1, 1, 1, h, w, sd);
  p->cls_w_off = p->n_params, p->n_params += 3 * 512;
  p->cls_b_off = p->n_params, p->n_params += 3;

  // ---- workspace layout -------------------------------------------------------------------------------------
  size_t off = 0, cap = 0;
  for (Unit& u : p->units) {
    const size_t bytes = al((size_t)N * u.Ho * u.Wo * u.Cout * 2);
    u.cap_off = cap, cap += 2 * bytes;
    u.z_off = off, off += bytes;
    u.y_off = off, off += bytes;
    u.st_off = off, off += al((size_t)u.Cout * 6 * 4);
    const size_t wbytes = u.Cin == 3 ? (size_t)64 * 224 * 2 : (size_t)u.Cout * u.k * u.k * u.Cin * 2;
    u.wf_off = off, off += al(wbytes);
    u.wd_off = off, off += al(wbytes);
  }
  const size_t p2 = (size_t)p->H2 * p->W2, p4 = (size_t)p->H4 * p->W4, p8 = (size_t)p->H8 * p->W8;
  size_t big = p2 * 64;
  if (p4 * 512 > big) big = p4 * 512;  // also the zero-inserted gradient of the stride-2 downsample (512 ch at H/4)
  if (p8 * 2048 > big) big = p8 * 2048;
  p->big_bytes = al(big * N * 2);
  size_t small = p4 * 128;
  if (p8 * 512 > small) small = p8 * 512;
  p->small_bytes = al(small * N * 2);
  p->padded_off = off, off += al(nbc_stem_tc_workspace_bytes(N, H, W));
  p->pool_off = off, off += al((size_t)N * p4 * 64 * 2);
  p->pidx_off = off, off += al((size_t)N * p4 * 64);
  p->drop_off = off, off += al((size_t)N * p8 * 512 * 2);
  p->low_off = off, off += al((size_t)N * 3 * p8 * 4);
  p->full_off = off, off += al((size_t)N * 3 * H * W * 4);
  p->dfull_off = off, off += al((size_t)N * 3 * H * W * 4);
  p->dlow_off = off, off += al((size_t)N * 3 * p8 * 4);
  p->upws_off = off, off += al(upsample_bwd_workspace_bytes(N, 3, p->H8, p->W8, H, W));
  p->gA_off = off, off += p->big_bytes;
  p->gB_off = off, off += p->big_bytes;
  p->gskip_off = off, off += p->big_bytes;
  p->dz_off = off, off += p->big_bytes;
  p->up_off = off, off += p->big_bytes;
  p->d1_off = off, off += p->small_bytes;
  p->d2_off = off, off += p->small_bytes;
  p->partial_off = off, off += al(bn_partial_bytes((int64_t)N * p2, 2048));
  p->zeros_off = off, off += al(2048 * 4);
  p->wce_off = off, off += al(nbc_wce_workspace_bytes(N, H, W));
  p->lov_off = off, off += al(nbc_lovasz_workspace_bytes(N, H, W));
  p->dfull2_off = off, off += al((size_t)N * 3 * H * W * 4);
  p->loss2_off = off, off += al(16);
  p->fold_off = off, off += al(64 * 147 * 4);
  for (const Unit& u : p->units) {
    const ConvGeom g{N, u.Hin, u.Win, u.Cin, u.Cout, u.k, u.k, u.stride, u.pad, u.dil, 0, 0};
    const size_t b = u.Cin == 3 ? stem_wgrad_tc_scratch_bytes(N, u.Ho, u.Wo) : wgrad_tc_scratch_bytes(g);
    if (b > p->wgpart_bytes) p->wgpart_bytes = b;
  }
  p->wgpart_off = off, off += al(p->wgpart_bytes);
  p->clspart_off = off, off += al(cls_partial_bytes(512));
  p->ws_bytes = off;
  p->capture_bytes = cap;

  // ---- static data flow: inputs of the units, gradient ping-pong of the blocks ----------------------------------
  size_t x = p->pool_off;
  for (TBlock& B : p->blocks) {
    p->units[B.c1].x_off = x;
    p->units[B.c2].x_off = p->units[B.c1].y_off;
    p->units[B.c3].x_off = p->units[B.c2].y_off;
    if (B.ds >= 0) p->units[B.ds].x_off = x;
    x = p->units[B.c3].y_off;
  }
  p->units[p->head_unit].x_off = x;
  // the head's data gradient (w.r.t. the layer4 output) lands in gA; blocks alternate from there, last block first
  size_t gin = p->gA_off, gout = p->gB_off;
  p->units[p->head_unit].dgrad_out_off = gin;
  for (int b = (int)p->blocks.size() - 1; b >= 0; --b) {
    TBlock& B = p->blocks[b];
    B.gin_off = gin, B.gout_off = gout;
    p->units[B.c3].dgrad_out_off = p->d2_off;
    p->units[B.c2].dgrad_out_off = p->d1_off;
    p->units[B.c1].dgrad_out_off = gout;
    p->units[B.c1].dgrad_has_res = true;
    p->units[B.c1].dgrad_res_off = p->gskip_off;
    if (B.ds >= 0) p->units[B.ds].dgrad_out_off = p->gskip_off;
    const size_t t = gin;
    gin = gout, gout = t;
  }
  p->units[0].need_dgrad = false;  // nothing upstream of the stem
  return p;
}

extern "C" void nbc_train_destroy(nbc_train_plan* p) { delete p; }

// ---- gradient segments (for overlapping the data-parallel all-reduce with the backward) ------------------------------
// segment i belongs to frozen units (nbc_train_set_frozen): the backward neither writes it nor records its event
static bool segment_frozen(const nbc_train_plan* p, int i) {
  const int nb = (int)p->blocks.size();
  if (i == 0) return false;
  if (i <= nb) return nb - i < p->first_block;
  return p->frozen > 0;
}

extern "C" int nbc_train_num_segments(const nbc_train_plan* p) { return p ? (int)p->blocks.size() + 2 : 0; }

extern "C" int nbc_train_segment(const nbc_train_plan* p, int i, int64_t* offset, int64_t* count) {
  NBC_REQUIRE(p && offset && count && i >= 0 && i < (int)p->blocks.size() + 2, "nbc_train_segment: bad argument");
  const int nb = (int)p->blocks.size();
  size_t lo, hi;
  if (i == 0) {
    lo = p->units[p->head_unit].w_off, hi = p->n_params;
  } else if (i <= nb) {
    const int b = nb - i;      // blocks last to first
    lo = p->units[p->blocks[b].c1].w_off;
    hi = (b + 1 < nb) ? p->units[p->blocks[b + 1].c1].w_off : p->units[p->head_unit].w_off;
  } else {
    lo = 0, hi = p->units[p->blocks[0].c1].w_off;      // the stem
  }
  if (segment_frozen(p, i)) hi = lo;
  *offset = (int64_t)lo, *count = (int64_t)(hi - lo);
  return 0;
}

static int record_segment(nbc_train_plan* p, int i, cudaStream_t stream) {
  if (p->seg_events.empty()) {
    p->seg_events.resize(p->blocks.size() + 2);
    for (cudaEvent_t& e : p->seg_events) NBC_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  }
  NBC_CUDA(cudaEventRecord(p->seg_events[i], stream));
  return 0;
}

extern "C" int nbc_train_wait_segment(nbc_train_plan* p, int i, void* stream) {
  NBC_REQUIRE(p && i >= 0 && i < (int)p->blocks.size() + 2, "nbc_train_wait_segment: bad argument");
  if (segment_frozen(p, i)) return 0;
  NBC_REQUIRE(!p->seg_events.empty(), "nbc_train_wait_segment: no backward has been enqueued yet");
  NBC_CUDA(cudaStreamWaitEvent(reinterpret_cast<cudaStream_t>(stream), p->seg_events[i], 0));
  return 0;
}
extern "C" int64_t nbc_train_param_count(const nbc_train_plan* p) { return p ? (int64_t)p->n_params : 0; }
extern "C" int64_t nbc_train_stats_count(const nbc_train_plan* p) { return p ? (int64_t)p->n_stats : 0; }
extern "C" size_t nbc_train_workspace_bytes(const nbc_train_plan* p) { return p ? p->ws_bytes : 0; }

// state_dict (326 device tensors, torchvision order) <-> flat buffers.  direction 0: load (tensors -> flat),
// 1: store (flat -> tensors; used for the updated weights and, with the gradient buffer, for per-layer gradients)
extern "C" int nbc_train_exchange(nbc_train_plan* p, void* const* tensors, int n_tensors, float* params, float* stats,
                                  int direction, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  NBC_REQUIRE(p && tensors && n_tensors == 326 && params, "nbc_train_exchange: bad arguments");
  for (const Unit& u : p->units) {
    float* w = reinterpret_cast<float*>(tensors[u.sd_index]);
    float* const* bn = reinterpret_cast<float* const*>(tensors + u.sd_index + 1);
    int rc = oihw_ohwi(direction == 0 ? w : params + u.w_off, u.Cout, u.Cin, u.k, u.k, direction == 0 ? params + u.w_off : w,
                       direction, stream);
    if (rc) return rc;
    const size_t cb = (size_t)u.Cout * 4;
    if (direction == 0) {
      NBC_CUDA(cudaMemcpyAsync(params + u.g_off, bn[0], cb, cudaMemcpyDeviceToDevice, stream));
      NBC_CUDA(cudaMemcpyAsync(params + u.b_off, bn[1], cb, cudaMemcpyDeviceToDevice, stream));
      if (stats) {
        NBC_CUDA(cudaMemcpyAsync(stats + u.rs_off, bn[2], cb, cudaMemcpyDeviceToDevice, stream));
        NBC_CUDA(cudaMemcpyAsync(stats + u.rs_off + u.Cout, bn[3], cb, cudaMemcpyDeviceToDevice, stream));
      }
    } else {
      NBC_CUDA(cudaMemcpyAsync(bn[0], params + u.g_off, cb, cudaMemcpyDeviceToDevice, stream));
      NBC_CUDA(cudaMemcpyAsync(bn[1], params + u.b_off, cb, cudaMemcpyDeviceToDevice, stream));
      if (stats) {
        NBC_CUDA(cudaMemcpyAsync(bn[2], stats + u.rs_off, cb, cudaMemcpyDeviceToDevice, stream));
        NBC_CUDA(cudaMemcpyAsync(bn[3], stats + u.rs_off + u.Cout, cb, cudaMemcpyDeviceToDevice, stream));
      }
    }
  }
  float* cw = reinterpret_cast<float*>(tensors[324]);
  float* cbias = reinterpret_cast<float*>(tensors[325]);
  if (direction == 0) {
    NBC_CUDA(cudaMemcpyAsync(params + p->cls_w_off, cw, 3 * 512 * 4, cudaMemcpyDeviceToDevice, stream));
    NBC_CUDA(cudaMemcpyAsync(params + p->cls_b_off, cbias, 3 * 4, cudaMemcpyDeviceToDevice, stream));
  } else {
    NBC_CUDA(cudaMemcpyAsync(cw, params + p->cls_w_off, 3 * 512 * 4, cudaMemcpyDeviceToDevice, stream));
    NBC_CUDA(cudaMemcpyAsync(cbias, params + p->cls_b_off, 3 * 4, cudaMemcpyDeviceToDevice, stream));
  }
  return 0;
}

namespace nbc {

// tensor maps depend on the workspace address: (re)build the conv launches when it changes
// the folded bias of a frozen unit lives in its (otherwise unused) BatchNorm scratch
static float* fold_bias(char* ws, const Unit& u) { return reinterpret_cast<float*>(ws + u.st_off); }

// frozen unit: y = act(conv(x, folded w) + folded bias (+ residual)) in one launch, straight into y
static int prepare_frozen(nbc_train_plan* p, char* ws, Unit& u, const void* residual) {
  ConvGeom g{p->N, u.Hin, u.Win, u.Cin, u.Cout, u.k, u.k, u.stride, u.pad, u.dil, u.relu, 0};
  return conv_tc_prepare(g, ws + u.x_off, ws + u.wf_off, fold_bias(ws, u), residual, ws + u.y_off, &u.fwd);
}

static int prepare(nbc_train_plan* p, char* ws) {
  if (p->prepared_ws == ws) return 0;
  const float* zeros = reinterpret_cast<const float*>(ws + p->zeros_off);
  const int N = p->N;
  Unit& s = p->units[0];
  int rc = s.frozen ? conv_tc_prepare_stem(N, s.Ho, s.Wo, 2 * s.Ho + 5, 2 * s.Wo + 6, ws + p->padded_off, ws + s.wf_off,
                                           fold_bias(ws, s), ws + s.y_off, &s.fwd, nullptr, 0, /*relu=*/1)
                    : conv_tc_prepare_stem(N, s.Ho, s.Wo, 2 * s.Ho + 5, 2 * s.Wo + 6, ws + p->padded_off, ws + s.wf_off, zeros,
                                           ws + s.z_off, &s.fwd, nullptr, 0, /*relu=*/0);   // BN sits between the conv and the ReLU
  if (rc) return rc;
  for (int b = 0; b < p->first_block; ++b) {
    const TBlock& B = p->blocks[b];
    const void* skip = ws + p->units[B.c1].x_off;
    if ((rc = prepare_frozen(p, ws, p->units[B.c1], nullptr))) return rc;
    if ((rc = prepare_frozen(p, ws, p->units[B.c2], nullptr))) return rc;
    if (B.ds >= 0) {
      if ((rc = prepare_frozen(p, ws, p->units[B.ds], nullptr))) return rc;
      skip = ws + p->units[B.ds].y_off;
    }
    if ((rc = prepare_frozen(p, ws, p->units[B.c3], skip))) return rc;
  }
  for (size_t i = 1; i < p->units.size(); ++i) {
    Unit& u = p->units[i];
    if (u.frozen) continue;
    ConvGeom g{N, u.Hin, u.Win, u.Cin, u.Cout, u.k, u.k, u.stride, u.pad, u.dil, 0, 0};
    rc = conv_tc_prepare(g, ws + u.x_off, ws + u.wf_off, zeros, nullptr, ws + u.z_off, &u.fwd);
    if (rc) return rc;
    if (!u.need_dgrad) continue;
    // data gradient = stride-1 conv of dz (zero-inserted for stride 2) with the flipped, transposed weights
    const bool s2 = u.stride == 2;
    ConvGeom d{N, s2 ? u.Hin : u.Ho, s2 ? u.Win : u.Wo, u.Cout, u.Cin, u.k, u.k, 1, u.pad, u.dil, 0, 0};
    if (d.Ho() != u.Hin || d.Wo() != u.Win) {
      set_error("train plan: dgrad geometry mismatch (unit %zu: %dx%d vs %dx%d)", i, d.Ho(), d.Wo(), u.Hin, u.Win);
      return NBC_ERR_INVALID;
    }
    const void* src = ws + (s2 ? p->up_off : p->dz_off);
    rc = conv_tc_prepare(d, src, ws + u.wd_off, zeros, u.dgrad_has_res ? ws + u.dgrad_res_off : nullptr,
                         ws + u.dgrad_out_off, &u.dgrad);
    if (rc) return rc;
  }
  p->prepared_ws = ws;
  return 0;
}

struct Ctx {
  nbc_train_plan* p;
  char* ws;
  float* params;
  float* stats;
  float* grads;
  cudaStream_t stream;
  float* st(const Unit& u, int which) const { return reinterpret_cast<float*>(ws + u.st_off) + (size_t)which * u.Cout; }
  float* partial() const { return reinterpret_cast<float*>(ws + p->partial_off); }
};

static int unit_forward(const Ctx& c, Unit& u, const void* residual, int relu) {
  int rc = conv_tc_run(&u.fwd, c.stream);
  if (rc || u.frozen) return rc;   // a frozen unit's launch already wrote y (bias, residual and ReLU in its epilogue)
  const int64_t M = (int64_t)c.p->N * u.Ho * u.Wo;
  return bn_forward_train(c.ws + u.z_off, M, u.Cout, c.params + u.g_off, c.params + u.b_off, 1e-5f, 0.1f,
                          c.stats ? c.stats + u.rs_off : nullptr, c.stats ? c.stats + u.rs_off + u.Cout : nullptr, c.st(u, 0),
                          c.st(u, 1), c.st(u, 2), c.st(u, 3), c.partial(), residual, relu, c.ws + u.y_off, c.stream);
}

// dy -> dz (in ws+dz_off), parameter gradients of the BN, weight gradient of the conv, data gradient
static int unit_backward(const Ctx& c, Unit& u, const void* dy, int relu, void* g_out) {
  nbc_train_plan* p = c.p;
  const int64_t M = (int64_t)p->N * u.Ho * u.Wo;
  void* dz = c.ws + p->dz_off;
  int rc = bn_backward(dy, c.ws + u.y_off, c.ws + u.z_off, M, u.Cout, c.params + u.g_off, c.st(u, 0), c.st(u, 1), relu,
                       c.partial(), c.st(u, 4), c.grads + u.g_off, c.grads + u.b_off, dz, g_out, c.stream);
  if (rc) return rc;
  if (p->capture != nullptr) {
    const size_t bytes = (size_t)M * u.Cout * 2;
    char* cap = reinterpret_cast<char*>(p->capture) + u.cap_off;
    NBC_CUDA(cudaMemcpyAsync(cap, dy, bytes, cudaMemcpyDeviceToDevice, c.stream));
    NBC_CUDA(cudaMemcpyAsync(cap + al(bytes), dz, bytes, cudaMemcpyDeviceToDevice, c.stream));
  }
  void* scratch = c.ws + p->wgpart_off;
  if (u.Cin == 3)
    return c.p->wgrad_impl == 1
               ? stem_wgrad(dz, c.ws + p->padded_off, p->N, u.Ho, u.Wo, c.grads + u.w_off, c.stream)
               : stem_wgrad_tc(dz, c.ws + p->padded_off, p->N, u.Ho, u.Wo, c.grads + u.w_off, scratch, p->wgpart_bytes, c.stream);
  ConvGeom g{p->N, u.Hin, u.Win, u.Cin, u.Cout, u.k, u.k, u.stride, u.pad, u.dil, 0, 0};
  rc = (c.p->wgrad_impl == 1 || !wgrad_tc_supported(g))
           ? wgrad_mma(g, dz, c.ws + u.x_off, c.grads + u.w_off, c.stream)
           : wgrad_tc(g, dz, c.ws + u.x_off, c.grads + u.w_off, scratch, p->wgpart_bytes, c.stream);
  if (rc) return rc;
  if (!u.need_dgrad) return 0;
  if (u.stride == 2) {
    rc = zero_insert(dz, p->N, u.Ho, u.Wo, u.Hin, u.Win, u.Cout, c.ws + p->up_off, c.stream);
    if (rc) return rc;
  }
  return conv_tc_run(&u.dgrad, c.stream);
}

}  // namespace nbc

extern "C" int nbc_train_forward_backward(nbc_train_plan* p, float* params, float* stats, float* grads, const void* input,
                                          int input_kind, const float* mean3_host, const float* std3_host,
                                          const uint8_t* target, const float* weights3, float dropout_p, uint64_t seed,
                                          float* loss, void* workspace, size_t workspace_bytes, void* stream_) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  NBC_REQUIRE(p && params && grads && input && target && weights3 && loss && workspace, "nbc_train_forward_backward: null pointer");
  NBC_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f, "nbc_train_forward_backward: dropout_p must be in [0,1)");
  NBC_REQUIRE(reinterpret_cast<uintptr_t>(workspace) % 1024 == 0, "nbc_train_forward_backward: workspace must be 1024-byte aligned");
  NBC_REQUIRE(stats || p->frozen == 0, "nbc_train_forward_backward: frozen stages need `stats` (their running statistics)");
  if (workspace_bytes < p->ws_bytes) {
    set_error("nbc_train_forward_backward: workspace %zu < %zu", workspace_bytes, p->ws_bytes);
    return NBC_ERR_WORKSPACE;
  }
  char* ws = reinterpret_cast<char*>(workspace);
  Ctx c{p, ws, params, stats, grads, stream};
  const int N = p->N, H = p->H, W = p->W;
  int rc = prepare(p, ws);
  if (rc) return rc;
  const size_t g0 = p->units[p->first_unit].w_off;   // the frozen prefix of `grads` is never written
  if (!p->accumulate) NBC_CUDA(cudaMemsetAsync(grads + g0, 0, (p->n_params - g0) * sizeof(float), stream));
  NBC_CUDA(cudaMemsetAsync(ws + p->zeros_off, 0, 2048 * 4, stream));

  // ---- weights of this step: bf16 copies for the forward and the data-gradient convolutions
  for (Unit& u : p->units) {
    if (u.frozen) {
      // eval-mode BatchNorm folded into the conv; the flat [Cout][kh][kw][Cin] row of each output channel is scaled
      // as a whole (fold_pack with Cin = kh = 1, kw = k*k*Cin), so the packed layout is the trainable forward's
      const float* rs = stats + u.rs_off;
      const int row = u.k * u.k * u.Cin;
      float* f32 = reinterpret_cast<float*>(ws + p->fold_off);
      rc = fold_pack(params + u.w_off, params + u.g_off, params + u.b_off, rs, rs + u.Cout, nullptr, 1e-5f, u.Cout, 1, 1, row, 1,
                     u.Cin == 3 ? nullptr : ws + u.wf_off, u.Cin == 3 ? f32 : nullptr, fold_bias(ws, u), stream);
      if (!rc && u.Cin == 3) rc = nbc_stem_pack_weights(f32, 0, ws + u.wf_off, stream);
    } else if (u.Cin == 3) {
      rc = nbc_stem_pack_weights(params + u.w_off, 0, ws + u.wf_off, stream);
    } else {
      rc = cast_pack(params + u.w_off, (int64_t)u.Cout * u.k * u.k * u.Cin, ws + u.wf_off, stream);
      if (!rc && u.need_dgrad) rc = dgrad_pack(params + u.w_off, u.Cout, u.Cin, u.k, u.k, ws + u.wd_off, stream);
    }
    if (rc) return rc;
  }

  // ---- forward ------------------------------------------------------------------------------------------------
  Unit& stem = p->units[0];
  rc = stem_tc_pad(input, input_kind, N, H, W, mean3_host, std3_host, ws + p->padded_off, stream, nullptr, 0);
  if (rc) return rc;
  rc = unit_forward(c, stem, nullptr, 1);
  if (rc) return rc;
  rc = stem.frozen ? maxpool_ragged(ws + stem.y_off, N, p->H2, p->W2, 64, ws + p->pool_off, nullptr, stream)
                   : maxpool_forward_idx(ws + stem.y_off, N, p->H2, p->W2, 64, ws + p->pool_off, ws + p->pidx_off, stream);
  if (rc) return rc;
  for (TBlock& B : p->blocks) {
    Unit &u1 = p->units[B.c1], &u2 = p->units[B.c2], &u3 = p->units[B.c3];
    if ((rc = unit_forward(c, u1, nullptr, 1))) return rc;
    if ((rc = unit_forward(c, u2, nullptr, 1))) return rc;
    const void* skip = ws + u1.x_off;
    if (B.ds >= 0) {
      Unit& ud = p->units[B.ds];
      if ((rc = unit_forward(c, ud, nullptr, 0))) return rc;
      skip = ws + ud.y_off;
    }
    if ((rc = unit_forward(c, u3, skip, 1))) return rc;
  }
  Unit& head = p->units[p->head_unit];
  if ((rc = unit_forward(c, head, nullptr, 1))) return rc;
  const int64_t P8 = (int64_t)p->H8 * p->W8;
  const void* cls_in = ws + head.y_off;
  if (dropout_p > 0.f) {
    if ((rc = dropout_apply(ws + head.y_off, (int64_t)N * P8 * 512, dropout_p, seed, ws + p->drop_off, stream))) return rc;
    cls_in = ws + p->drop_off;
  }
  float* low = reinterpret_cast<float*>(ws + p->low_off);
  float* full = reinterpret_cast<float*>(ws + p->full_off);
  float* dfull = reinterpret_cast<float*>(ws + p->dfull_off);
  float* dlow = reinterpret_cast<float*>(ws + p->dlow_off);
  if ((rc = head_1x1(cls_in, P8, N, 512, params + p->cls_w_off, params + p->cls_b_off, low, 0, stream))) return rc;
  if ((rc = nbc_upsample_bicubic(low, N, 3, p->H8, p->W8, H, W, full, stream))) return rc;
  if (p->loss_kind == 0) {
    if ((rc = nbc_wce_fwd_bwd(full, target, 0, weights3, N, H, W, loss, dfull, ws + p->wce_off, nbc_wce_workspace_bytes(N, H, W),
                              stream)))
      return rc;
  } else if (p->loss_kind == 1) {
    if ((rc = nbc_lovasz_softmax_fwd_bwd(full, target, 0, N, H, W, 1.f, loss, dfull, ws + p->lov_off,
                                         nbc_lovasz_workspace_bytes(N, H, W), stream)))
      return rc;
  } else {
    // MixedLoss (utils.py:185-192): CE / 4 + Lovasz, for the value and for the gradient
    float* dfull2 = reinterpret_cast<float*>(ws + p->dfull2_off);
    float* loss2 = reinterpret_cast<float*>(ws + p->loss2_off);
    if ((rc = nbc_wce_fwd_bwd(full, target, 0, weights3, N, H, W, loss2, dfull2, ws + p->wce_off, nbc_wce_workspace_bytes(N, H, W),
                              stream)))
      return rc;
    if ((rc = nbc_lovasz_softmax_fwd_bwd(full, target, 0, N, H, W, 1.f, loss2 + 1, dfull, ws + p->lov_off,
                                         nbc_lovasz_workspace_bytes(N, H, W), stream)))
      return rc;
    if ((rc = axpby(dfull2, 0.25f, dfull, 1.f, (int64_t)N * 3 * H * W, dfull, stream))) return rc;
    if ((rc = axpby(loss2, 0.25f, loss2 + 1, 1.f, 1, loss, stream))) return rc;
  }

  // ---- backward -----------------------------------------------------------------------------------------------
  if ((rc = upsample_backward(dfull, N, 3, p->H8, p->W8, H, W, dlow, ws + p->upws_off, stream))) return rc;
  // classifier: gradient w.r.t. the head activations (through the dropout mask) goes to d2
  if ((rc = cls_backward(dlow, cls_in, params + p->cls_w_off, N, P8, 512, dropout_p, seed, ws + p->d2_off,
                         grads + p->cls_w_off, grads + p->cls_b_off, ws + p->clspart_off, stream)))
    return rc;
  if ((rc = unit_backward(c, head, ws + p->d2_off, 1, nullptr))) return rc;
  if ((rc = record_segment(p, 0, stream))) return rc;
  const int nb = (int)p->blocks.size();
  for (int b = nb - 1; b >= p->first_block; --b) {   // the backward ends at the first trainable block
    TBlock& B = p->blocks[b];
    Unit &u1 = p->units[B.c1], &u2 = p->units[B.c2], &u3 = p->units[B.c3];
    // y3 = relu(bn3(z3) + skip): masked gradient g3 feeds both the main path and the skip path (kept in gskip)
    if ((rc = unit_backward(c, u3, ws + B.gin_off, 1, ws + p->gskip_off))) return rc;
    if ((rc = unit_backward(c, u2, ws + p->d2_off, 1, nullptr))) return rc;
    if (B.ds >= 0) {
      // downsample branch: BN (no ReLU) -> conv 1x1; its data gradient replaces g3 in gskip
      if ((rc = unit_backward(c, p->units[B.ds], ws + p->gskip_off, 0, nullptr))) return rc;
    }
    // conv1's data gradient + skip gradient = gradient w.r.t. the block input
    if ((rc = unit_backward(c, u1, ws + p->d1_off, 1, nullptr))) return rc;
    if ((rc = record_segment(p, nb - b, stream))) return rc;
  }
  if (p->frozen > 0) return 0;
  // maxpool and stem
  const size_t g_pool = p->blocks[0].gout_off;
  if ((rc = maxpool_backward(ws + g_pool, ws + p->pidx_off, N, p->H2, p->W2, 64, ws + p->gskip_off, stream))) return rc;
  if ((rc = unit_backward(c, stem, ws + p->gskip_off, 1, nullptr))) return rc;
  return record_segment(p, nb + 1, stream);
}

// debug / test accessor: byte offset into the workspace and geometry of an intermediate tensor.
// what: 0 = z (pre-BN, bf16 NHWC) of unit `index`, 1 = y (post BN/ReLU) of unit `index`, 2 = low-res logits (f32 planar),
// 3 = full-res logits (f32 planar), 4 = d loss / d full logits, 5 = d loss / d low-res logits;  6 = dy, 7 = dz of the BN
// backward of unit `index` (bf16 NHWC) -- offsets into the CAPTURE buffer (nbc_train_set_capture), not the workspace.
// dims_out[4] = N,H,W,C.
extern "C" int64_t nbc_train_debug_offset(const nbc_train_plan* p, int what, int index, int32_t* dims_out) {
  if (!p || !dims_out) return -1;
  if (what == 0 || what == 1 || what == 6 || what == 7) {
    if (index < 0 || index >= (int)p->units.size()) return -1;
    const Unit& u = p->units[index];
    if (u.frozen && what != 1) return -1;   // a frozen unit has only its y
    dims_out[0] = p->N, dims_out[1] = u.Ho, dims_out[2] = u.Wo, dims_out[3] = u.Cout;
    if (what >= 6) return (int64_t)(u.cap_off + (what == 7 ? al((size_t)p->N * u.Ho * u.Wo * u.Cout * 2) : 0));
    return (int64_t)(what == 0 ? u.z_off : u.y_off);
  }
  if (what == 2 || what == 5) {
    dims_out[0] = p->N, dims_out[1] = p->H8, dims_out[2] = p->W8, dims_out[3] = 3;
    return (int64_t)(what == 2 ? p->low_off : p->dlow_off);
  }
  if (what == 3 || what == 4) {
    dims_out[0] = p->N, dims_out[1] = p->H, dims_out[2] = p->W, dims_out[3] = 3;
    return (int64_t)(what == 3 ? p->full_off : p->dfull_off);
  }
  return -1;
}
extern "C" size_t nbc_train_capture_bytes(const nbc_train_plan* p) { return p ? p->capture_bytes : 0; }
extern "C" int nbc_train_set_capture(nbc_train_plan* p, void* buf, size_t bytes) {
  NBC_REQUIRE(p, "nbc_train_set_capture: null plan");
  if (buf != nullptr && bytes < p->capture_bytes) {
    set_error("nbc_train_set_capture: buffer %zu < %zu bytes", bytes, p->capture_bytes);
    return NBC_ERR_WORKSPACE;
  }
  p->capture = buf;
  return 0;
}
extern "C" int nbc_train_set_wgrad_impl(nbc_train_plan* p, int impl) {
  NBC_REQUIRE(p && (impl == 0 || impl == 1), "nbc_train_set_wgrad_impl: impl must be 0 (tcgen05) or 1 (mma.sync)");
  p->wgrad_impl = impl;
  return 0;
}
extern "C" int nbc_train_set_loss(nbc_train_plan* p, int kind) {
  NBC_REQUIRE(p && kind >= 0 && kind <= 2, "nbc_train_set_loss: kind must be 0 (weighted CE), 1 (Lovasz) or 2 (mixed)");
  p->loss_kind = kind;
  return 0;
}
extern "C" int nbc_train_set_accumulate(nbc_train_plan* p, int on) {
  NBC_REQUIRE(p && (on == 0 || on == 1), "nbc_train_set_accumulate: on must be 0 (overwrite) or 1 (add)");
  p->accumulate = on;
  return 0;
}
extern "C" int nbc_train_set_frozen(nbc_train_plan* p, int stages) {
  NBC_REQUIRE(p, "nbc_train_set_frozen: null plan");
  if (stages < 0 || stages > 5) {
    set_error("nbc_train_set_frozen: stages must be 0 (none), 1 (stem) or 2..5 (stem through layer1..layer4), got %d", stages);
    return NBC_ERR_INVALID;
  }
  const int first_block[6] = {0, 0, 3, 7, 13, 16};   // layers of 3, 4, 6 and 3 bottlenecks
  p->frozen = stages, p->first_block = first_block[stages];
  p->first_unit = stages == 0 ? 0 : (stages == 5 ? p->head_unit : p->blocks[p->first_block].c1);
  for (size_t i = 0; i < p->units.size(); ++i) {
    p->units[i].frozen = (int)i < p->first_unit;
    p->units[i].need_dgrad = i > 0 && (int)i >= p->first_unit;
  }
  // the first trainable unit(s) read a frozen activation: no data gradient is wanted there
  if (stages > 0 && stages < 5) {
    p->units[p->blocks[p->first_block].c1].need_dgrad = false;
    p->units[p->blocks[p->first_block].ds].need_dgrad = false;
  } else if (stages == 5) {
    p->units[p->head_unit].need_dgrad = false;
  }
  p->prepared_ws = nullptr;   // the launches change
  return 0;
}
extern "C" int nbc_train_trainable_offsets(const nbc_train_plan* p, int64_t* param_off, int64_t* stats_off) {
  NBC_REQUIRE(p && param_off && stats_off, "nbc_train_trainable_offsets: null pointer");
  *param_off = (int64_t)p->units[p->first_unit].w_off;
  *stats_off = (int64_t)p->units[p->first_unit].rs_off;
  return 0;
}
extern "C" int nbc_train_num_units(const nbc_train_plan* p) { return p ? (int)p->units.size() : 0; }

extern "C" int nbc_train_adam(float* params, const float* grads, float* m, float* v, int64_t n, float lr, float beta1,
                              float beta2, float eps, float weight_decay, int step, float grad_scale, void* stream) {
  NBC_REQUIRE(params && grads && m && v && n > 0 && step >= 1, "nbc_train_adam: bad arguments");
  return adam_step(params, grads, m, v, n, lr, beta1, beta2, eps, weight_decay, step, grad_scale,
                   reinterpret_cast<cudaStream_t>(stream));
}
