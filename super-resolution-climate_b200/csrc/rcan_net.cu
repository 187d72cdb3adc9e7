// Whole-network executor: enqueues the RCAN forward / backward kernel sequence on one stream from a
// single C call (no per-layer host round trips, capturable into a CUDA graph -- all buffers live in a
// caller-provided workspace at offsets computed from the network description only).
//
// Network (reference sres/model/rcan/network.py:9-27, blocks.py:58-76):
//   head conv Cin->64 | G x [ R x RCAB(conv,ReLU,conv,CA,+x) , conv, +x ] | conv, +head | Upsampler | conv 64->Cout
// Parameters cross the boundary as ONE flat fp32 buffer in state_dict order (the order of
// `model.state_dict()` of the reference RCAN, SURVEY.md 3.2), gradients likewise.
//
// Precision plan (SURVEY.md section 7 "hard parts"): bf16 only where the sole consumer is a
// tensor-core operand (conv inputs, weights, incoming gradients); the residual trunk, the gradient
// trunk, pooled statistics, parameter gradients and all accumulation are fp32.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <map>
#include <mutex>
#include <string>
#include <vector>
#include "internal.h"
#include "ptx.cuh"

namespace sres {

constexpr int kConvW = 64 * 64 * 9;  // floats of one 64->64 conv weight
// bf16 gradient buffers rotate through a ring: a deferred weight-gradient job keeps reading its buffer until its
// batch (8 jobs = 4 blocks by default, on the side stream) has been launched, so the ring holds one batch of blocks
// plus the block being written (WgQueue::before_write flushes / joins whenever a buffer would be overwritten early,
// so any ring length is correct -- a short one just cuts the batches short)
constexpr int kRing = 8;
static int ring_len() {   // buffers actually rotated through (<= kRing): fewer = better L2 locality, more = deeper batches
  static const int v = [] {
    const char* e = getenv("SRES_RING");
    int n = e ? atoi(e) : 5;
    return n < 3 ? 3 : (n > kRing ? kRing : n);
  }();
  return v;
}
static int wgrad_batch_jobs() {
  static const int v = [] {
    const char* e = getenv("SRES_WGRAD_BATCH");
    // Measured on B200 (tools/r2_ab3.sh, interleaved, medians): 4 jobs / ring 3 28.26 ms per step, 8 / 5 27.88, 12 / 7 27.93,
    // 16 / 9 27.74 (the 12- and 16-job runs needed > 4 KB of kernel parameters for the tensor maps, which ncu's launch
    // interception rejects, so the limit stays at 8): a launch costs ~13 us of prologue + accumulator drain + reduce whatever its job count (1 job 22.8 us,
    // 4 jobs 52.9 us), so eight jobs per launch halve that; deeper still is within noise (and the rings lose L2 locality).
    int n = e ? atoi(e) : 8;
    return n < 1 ? 1 : (n > SRES_WGRAD_MAX_JOBS ? SRES_WGRAD_MAX_JOBS : n);
  }();
  return v;
}

// ---------------------------------------------------------------------------------------------
// Optional in-situ profiler (SRES_PROFILE=1, eager mode only): CUDA events around every enqueued
// kernel group, aggregated per category by sres_profile_report().  Development aid; off by default.
// ---------------------------------------------------------------------------------------------
struct ProfRec { const char* cat; cudaEvent_t a, b; };
static std::vector<ProfRec>* t_prof = nullptr;  // process-wide (autograd runs backward on its own thread)
static std::mutex g_prof_mu;
static bool prof_on() {
  static const bool v = [] { const char* e = getenv("SRES_PROFILE"); return e && atoi(e) > 0; }();
  return v;
}
struct ProfScope {
  cudaStream_t st; ProfRec r; bool on;
  ProfScope(const char* cat, void* stream) : st((cudaStream_t)stream), on(prof_on()) {
    if (!on) return;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(st, &cs);
    if (cs != cudaStreamCaptureStatusNone) { on = false; return; }
    r.cat = cat;
    cudaEventCreate(&r.a); cudaEventCreate(&r.b);
    cudaEventRecord(r.a, st);
  }
  ~ProfScope() {
    if (!on) return;
    cudaEventRecord(r.b, st);
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (!t_prof) t_prof = new std::vector<ProfRec>();
    t_prof->push_back(r);
  }
};
#define PROF(cat) ProfScope prof_scope__(cat, st)

#define RC0(x)           \
  do {                   \
    int rc__ = (x);      \
    if (rc__) return rc__; \
  } while (0)

struct Net {
  sres_rcan_desc d;
  bool edsr;    // EDSR: one "group" of ResBlocks without channel attention, group-tail conv or group skip
  float rs;     // EDSR residual scaling (1 for RCAN)
  int per;      // 64->64 convs per group in the packed-weight tables: 2R (+1 group-tail conv for RCAN)
  int hid;
  // parameter offsets (floats)
  long long head_w, head_b, body0, rcab_sz, group_sz, bt_w, bt_b, up_w[4], up_b[4], tail_w, tail_b, n_params;
  int n_body_convs;
  // geometry per resolution level
  int lvH[5], lvW[5];
  long long lvRows[5];
  // workspace offsets (bytes)
  size_t o_wp_fwd, o_wp_dg, o_wp_up_fwd[4], o_wp_up_dg[4], o_wp_tail, o_bias_up[4], o_bias_tail;
  size_t o_xb, o_t1, o_t2, o_mean, o_s, o_ds, o_resb, o_u[4];
  size_t o_hf, o_gf[2], o_xf, o_pool_part, o_pool_sum;
  size_t o_sbias;  // EDSR: res_scale * bias of every ResBlock's second conv
  size_t o_pair_flags;   // ready / consumed counters of the fused convolution pairs, two sets (alternating RCABs)
  size_t o_ga, o_gb32, o_gb16, o_dt2[kRing], o_dt1[kRing], o_ds_part, o_wg_ws, o_sw_ws, o_ca_scr, o_du16[4], o_du32[4], o_dres32, o_dres16;
  size_t total;
  int n_xb, n_t;  // saved-buffer counts (1 in inference mode)
  long long cidx(int g, int r, int which) const { return (long long)g * per + 2 * r + which; }
  long long cidx_gt(int g) const { return (long long)g * per + 2 * d.n_blocks; }
  long long cidx_bt() const { return (long long)d.n_groups * per; }
  long long off_rcab(int g, int r) const { return body0 + g * group_sz + r * rcab_sz; }
  long long off_gt(int g) const { return body0 + g * group_sz + d.n_blocks * rcab_sz; }
};

static size_t align_up(size_t v, size_t a = 1024) { return (v + a - 1) / a * a; }

static int build_net(Net* n, const sres_rcan_desc* d, int training) {
  if (!d) return set_error(SRES_ERR_INVALID_ARG, "rcan: null description");
  if (d->B <= 0 || d->H <= 0 || d->W <= 0) return set_error(SRES_ERR_INVALID_ARG, "rcan: bad tile geometry");
  if (d->nfeatures != 64) return set_error(SRES_ERR_UNSUPPORTED, "rcan: kernels are specialised for nfeatures == 64");
  // 16: the narrow CUDA-core head / tail kernels (small_conv.cu) and the n_out = 16 tensor-core tail conv
  if (d->cin < 1 || d->cin > 16 || d->cout < 1 || d->cout > 16)
    return set_error(SRES_ERR_UNSUPPORTED, "rcan: 1..16 image channels supported");
  if (d->n_groups < 1 || d->n_blocks < 1) return set_error(SRES_ERR_INVALID_ARG, "rcan: need >= 1 group and block");
  if (d->arch != SRES_ARCH_RCAN && d->arch != SRES_ARCH_EDSR) return set_error(SRES_ERR_INVALID_ARG, "rcan: unknown arch");
  const bool edsr = d->arch == SRES_ARCH_EDSR;
  if (!edsr && (d->reduction < 1 || 64 % d->reduction)) return set_error(SRES_ERR_INVALID_ARG, "rcan: reduction must divide 64");
  if (edsr && d->n_groups != 1) return set_error(SRES_ERR_INVALID_ARG, "edsr: n_groups must be 1 (n_blocks = number of ResBlocks)");
  if (edsr && !(d->res_scale > 0.f)) return set_error(SRES_ERR_INVALID_ARG, "edsr: res_scale must be positive");
  if (d->n_up < 0 || d->n_up > 4) return set_error(SRES_ERR_UNSUPPORTED, "rcan: at most 4 upsampler stages");
  memset(n, 0, sizeof(*n));
  n->d = *d;
  n->edsr = edsr;
  n->rs = edsr ? d->res_scale : 1.f;
  n->hid = edsr ? 0 : 64 / d->reduction;
  n->per = 2 * d->n_blocks + (edsr ? 0 : 1);
  const int G = d->n_groups, R = d->n_blocks, hid = n->hid;
  long long o = 0;
  n->head_w = o; o += 64LL * d->cin * 9;
  n->head_b = o; o += 64;
  n->body0 = o;
  n->rcab_sz = 2LL * (kConvW + 64) + (edsr ? 0 : (hid * 64 + hid) + (64 * hid + 64));
  n->group_sz = R * n->rcab_sz + (edsr ? 0 : kConvW + 64);
  o += G * n->group_sz;
  n->bt_w = o; o += kConvW;
  n->bt_b = o; o += 64;
  n->lvH[0] = d->H; n->lvW[0] = d->W;
  for (int i = 0; i < d->n_up; ++i) {
    const int f = d->up_factor[i];
    if (f != 2 && f != 3) return set_error(SRES_ERR_UNSUPPORTED, "rcan: upsampler stage factor must be 2 or 3");
    n->up_w[i] = o; o += (long long)f * f * kConvW;
    n->up_b[i] = o; o += f * f * 64;
    n->lvH[i + 1] = n->lvH[i] * f; n->lvW[i + 1] = n->lvW[i] * f;
  }
  n->tail_w = o; o += (long long)d->cout * 64 * 9;
  n->tail_b = o; o += d->cout;
  n->n_params = o;
  n->n_body_convs = G * n->per + 1;
  for (int i = 0; i <= d->n_up; ++i) {
    n->lvRows[i] = (long long)d->B * (n->lvH[i] + 1) * (n->lvW[i] + 1);
    if (n->lvRows[i] > 0x7fffff00LL) return set_error(SRES_ERR_UNSUPPORTED, "rcan: batch too large");
  }
  const size_t r0 = (size_t)n->lvRows[0];
  const size_t bf = r0 * 128, f32 = r0 * 256;
  size_t w = 0;
  auto take = [&](size_t bytes) { size_t at = w; w = align_up(w + bytes); return at; };
  // packed weights
  n->o_wp_fwd = take((size_t)n->n_body_convs * kConvW * 2);
  n->o_wp_dg = take((size_t)n->n_body_convs * kConvW * 2);
  for (int i = 0; i < d->n_up; ++i) {
    const int f2 = d->up_factor[i] * d->up_factor[i];
    n->o_wp_up_fwd[i] = take((size_t)f2 * kConvW * 2);
    n->o_wp_up_dg[i] = take((size_t)f2 * kConvW * 2);
    n->o_bias_up[i] = take((size_t)f2 * 64 * 4);
  }
  n->o_wp_tail = take(9 * 16 * 64 * 2);
  n->o_bias_tail = take(16 * 4);
  // activations
  n->n_xb = training ? G * (R + 1) + 1 : 2;
  n->n_t = training ? G * R : 1;
  n->o_xb = take((size_t)n->n_xb * bf);
  n->o_t1 = take((size_t)n->n_t * bf);
  if (edsr) {
    n->o_sbias = take((size_t)R * 64 * 4);
  } else {
    n->o_t2 = take((size_t)n->n_t * bf);
    n->o_mean = take((size_t)n->n_t * d->B * 64 * 4);
    n->o_s = take((size_t)n->n_t * d->B * 64 * 4);
  }
  n->o_resb = take(bf);
  for (int i = 0; i < d->n_up; ++i) n->o_u[i] = take((size_t)n->lvRows[i + 1] * 128);
  n->o_hf = take(f32);
  n->o_gf[0] = take(f32);
  n->o_gf[1] = take(f32);
  n->o_xf = take(f32);
  n->o_pool_part = take((size_t)sres_conv_mtiles(d->B, d->H, d->W) * 2 * 4 * 64 * 4);
  n->o_pool_sum = take((size_t)d->B * 64 * 4);
  n->o_pair_flags = take(2 * sres_conv_pair_flag_bytes(d->B, d->H, d->W));
  if (training) {
    n->o_ga = take(f32);
    n->o_gb16 = take(bf);
    for (int k = 0; k < ring_len(); ++k) { n->o_dt2[k] = take(bf); n->o_dt1[k] = take(bf); }
    if (!edsr) {
      n->o_ds = take((size_t)n->n_t * d->B * 64 * 4);
      n->o_gb32 = take(f32);
      const int bpi = sres_ca_blocks_per_image(d->B, d->H, d->W);
      n->o_ds_part = take((size_t)d->B * (bpi > 0 ? bpi : 1) * 64 * 4);
      n->o_ca_scr = take(sres_ca_param_grads_scratch_bytes(R, d->B));
    }
    n->o_wg_ws = take(sres_conv_wgrad_workspace_bytes());
    n->o_sw_ws = take(sres_small_wgrad_workspace_bytes());
    for (int i = 0; i < d->n_up; ++i) {
      // gradient w.r.t. U[i] (level i+1), stored as f*f sub-grids of level-i rows (PixelUnshuffle layout)
      const int f2 = d->up_factor[i] * d->up_factor[i];
      n->o_du16[i] = take((size_t)f2 * n->lvRows[i] * 128);
      // the fp32 accumulator of stage i's OUTPUT gradient is only written by stage i+1's input-gradient convs
      if (i < d->n_up - 1) n->o_du32[i] = take((size_t)f2 * n->lvRows[i] * 256);
    }
    n->o_dres32 = take(f32);
    n->o_dres16 = take(bf);
  }
  n->total = w;
  return SRES_OK;
}

// ---------------------------------------------------------------------------------------------
// bulk weight packing (all 64->64 body convs in one launch; both operand forms)
// ---------------------------------------------------------------------------------------------
struct PackBody {
  const float* params;
  long long body0, rcab_sz, group_sz, bt_w;
  int G, R, per;
  float scale2;     // multiplier folded into every block's second conv (EDSR res_scale; 1 for RCAN)
  float* sbias;     // EDSR: scale2 * bias of the second convs, [R][64]
  uint16_t* fwd;
  uint16_t* dg;
};
__global__ void pack_body_kernel(PackBody pb) {
  const int conv = blockIdx.y;
  const int per = pb.per;
  long long off;
  float sc = 1.f;
  if (conv == pb.G * per) off = pb.bt_w;
  else {
    const int g = conv / per, k = conv % per;
    off = pb.body0 + g * pb.group_sz + (k < 2 * pb.R ? (k / 2) * pb.rcab_sz + (k & 1) * (kConvW + 64) : pb.R * pb.rcab_sz);
    if (k < 2 * pb.R && (k & 1)) {
      sc = pb.scale2;
      if (pb.sbias && blockIdx.x == 0 && threadIdx.x < 64)
        pb.sbias[(size_t)(g * pb.R + k / 2) * 64 + threadIdx.x] = sc * pb.params[off + kConvW + threadIdx.x];
    }
  }
  const float* w = pb.params + off;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < kConvW; idx += gridDim.x * blockDim.x) {
    const int k = idx & 63, n = (idx >> 6) & 63, t = idx >> 12;
    const int ky = t / 3, kx = t % 3;
    const float vf = sc * w[((n * 64 + k) * 3 + ky) * 3 + kx];
    const float vd = sc * w[((k * 64 + n) * 3 + (2 - ky)) * 3 + (2 - kx)];
    pb.fwd[(size_t)conv * kConvW + idx] = (uint16_t)(pack_bf16x2(vf, 0.f) & 0xFFFF);
    pb.dg[(size_t)conv * kConvW + idx] = (uint16_t)(pack_bf16x2(vd, 0.f) & 0xFFFF);
  }
}
__global__ void gather_bias_kernel(const float* __restrict__ b, float* __restrict__ out, int n_out, int stride, int offset,
                                   int n_src) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n_out) {
    const int s = i * stride + offset;
    out[i] = s < n_src ? b[s] : 0.f;
  }
}

static int pack_all(const Net& n, const float* params, uint8_t* ws, cudaStream_t st) {
  PackBody pb{params, n.body0, n.rcab_sz, n.group_sz, n.bt_w, n.d.n_groups, n.d.n_blocks, n.per, n.rs,
              n.edsr ? (float*)(ws + n.o_sbias) : nullptr, (uint16_t*)(ws + n.o_wp_fwd), (uint16_t*)(ws + n.o_wp_dg)};
  pack_body_kernel<<<dim3(8, n.n_body_convs), 256, 0, st>>>(pb);
  SRES_CHECK_LAUNCH("rcan: pack launch");
  for (int i = 0; i < n.d.n_up; ++i) {
    const int f = n.d.up_factor[i], f2 = f * f;
    for (int sub = 0; sub < f2; ++sub) {
      int rc = sres_pack_conv_weights(params + n.up_w[i], ws + n.o_wp_up_fwd[i] + (size_t)sub * kConvW * 2, 0, 64, 64,
                                      f2 * 64, f2, sub, st);
      if (rc) return rc;
      rc = sres_pack_conv_weights(params + n.up_w[i], ws + n.o_wp_up_dg[i] + (size_t)sub * kConvW * 2, 1, 64, 64,
                                  f2 * 64, f2, sub, st);
      if (rc) return rc;
      gather_bias_kernel<<<1, 64, 0, st>>>(params + n.up_b[i], (float*)(ws + n.o_bias_up[i]) + sub * 64, 64, f2, sub,
                                           f2 * 64);
      SRES_CHECK_LAUNCH("rcan: bias gather launch");
    }
  }
  int rc = sres_pack_conv_weights(params + n.tail_w, ws + n.o_wp_tail, 0, 16, 64, n.d.cout, 1, 0, st);
  if (rc) return rc;
  gather_bias_kernel<<<1, 64, 0, st>>>(params + n.tail_b, (float*)(ws + n.o_bias_tail), 16, 1, 0, n.d.cout);
  SRES_CHECK_LAUNCH("rcan: bias gather launch");
  return SRES_OK;
}

// ---------------------------------------------------------------------------------------------
// forward
// ---------------------------------------------------------------------------------------------
static sres_conv_args conv64_args(const void* in, const void* wp, const float* bias, int B, int H, int W, float* out_f32,
                                  void* out_bf16, unsigned flags = 0, float* pool = nullptr, const float* resid = nullptr,
                                  const float* resid2 = nullptr, const void* mask = nullptr, int map = SRES_MAP_IDENT,
                                  int si = 0, int sj = 0, int sf = 2) {
  sres_conv_args a;
  memset(&a, 0, sizeof(a));
  a.in_bf16 = in; a.wpack_bf16 = wp; a.bias = bias; a.resid_f32 = resid; a.resid2_f32 = resid2; a.mask_bf16 = mask;
  a.out_f32 = out_f32; a.out_bf16 = out_bf16; a.pool_part = pool;
  a.B = B; a.H = H; a.W = W; a.n_out = 64; a.epi_flags = flags; a.map_mode = map; a.sub_i = si; a.sub_j = sj;
  a.shuffle_factor = sf;
  return a;
}

static int conv64(const void* in, const void* wp, const float* bias, int B, int H, int W, void* st, float* out_f32,
                  void* out_bf16, unsigned flags = 0, float* pool = nullptr, const float* resid = nullptr,
                  const float* resid2 = nullptr, const void* mask = nullptr, int map = SRES_MAP_IDENT, int si = 0,
                  int sj = 0, int sf = 2) {
  PROF(map != SRES_MAP_IDENT ? "conv shuffle/unshuffle" : (flags & SRES_EPI_DOT) ? "conv dgrad +fp32 rmw +ds-dot" : mask ? "conv dgrad+relu-mask" : (resid && out_f32) ? "conv +fp32 addend (rmw)"
       : (flags & SRES_EPI_POOL) ? "conv fwd +pool" : (flags & SRES_EPI_RELU) ? "conv fwd +relu" : "conv other");
  const sres_conv_args a = conv64_args(in, wp, bias, B, H, W, out_f32, out_bf16, flags, pool, resid, resid2, mask, map, si, sj, sf);
  return sres_conv3x3_igemm(&a, st);
}

// two dependent convolutions: one fused launch when the pair kernel takes them, else one after the other
static int conv64_pair(const sres_conv_args& a1, const sres_conv_args& a2, void* flags, void* st, const char* cat) {
  if (sres_conv_pair_supported(&a1, &a2)) {
    PROF(cat);
    return sres_conv3x3_pair(&a1, &a2, flags, st);
  }
  { PROF((a1.epi_flags & SRES_EPI_RELU) ? "conv fwd +relu" : "conv dgrad+relu-mask"); RC0(sres_conv3x3_igemm(&a1, st)); }
  PROF((a2.epi_flags & SRES_EPI_DOT) ? "conv dgrad +fp32 rmw +ds-dot" : "conv fwd +pool");
  return sres_conv3x3_igemm(&a2, st);
}

#define RC(x)            \
  do {                   \
    int rc__ = (x);      \
    if (rc__) return rc__; \
  } while (0)

static int forward(const Net& n, const float* P, const float* x, float* out, uint8_t* ws, int training, void* st) {
  const sres_rcan_desc& d = n.d;
  const int B = d.B, H = d.H, W = d.W, G = d.n_groups, R = d.n_blocks;
  const size_t bf = (size_t)n.lvRows[0] * 128;
  const bool fused_pool = (H + 1) * (W + 1) >= 128;
  auto XB = [&](int i) { return ws + n.o_xb + (size_t)(training ? i : (i & 1)) * bf; };
  auto T1 = [&](int i) { return ws + n.o_t1 + (size_t)(training ? i : 0) * bf; };
  auto T2 = [&](int i) { return ws + n.o_t2 + (size_t)(training ? i : 0) * bf; };
  auto WF = [&](long long c) { return ws + n.o_wp_fwd + (size_t)c * kConvW * 2; };
  float* hf = (float*)(ws + n.o_hf);
  float* xf = (float*)(ws + n.o_xf);
  float* pool_part = (float*)(ws + n.o_pool_part);
  float* pool_sum = (float*)(ws + n.o_pool_sum);
  int xbi = 0;  // index of the bf16 copy of the current trunk value
  const bool l2hint = l2_hint_enabled();
  if (l2hint) RC(sres_l2_persist_window(xf, (size_t)n.lvRows[0] * 256, st));
  { PROF("head conv"); RC(sres_conv3x3_small_in(x, P + n.head_w, P + n.head_b, B, d.cin, H, W, 0, 0, hf, XB(0), st)); }
  const float* gin = hf;
  if (n.edsr) {
    // ResBlock r: t1 = relu(conv1(x)); x <- x + res_scale * conv2(t1)   (scale folded into the packed weights / bias)
    for (int r = 0; r < R; ++r) {
      const float* pr = P + n.off_rcab(0, r);
      RC(conv64(XB(xbi), WF(n.cidx(0, r, 0)), pr + kConvW, B, H, W, st, nullptr, T1(r), SRES_EPI_RELU));
      RC(conv64(T1(r), WF(n.cidx(0, r, 1)), (const float*)(ws + n.o_sbias) + (size_t)r * 64, B, H, W, st, xf, XB(xbi + 1), 0,
                nullptr, r == 0 ? hf : xf));
      ++xbi;
    }
  }
  for (int g = 0; g < (n.edsr ? 0 : G); ++g) {
    float* gout = (float*)(ws + n.o_gf[g & 1]);
    for (int r = 0; r < R; ++r) {
      const int ti = g * R + r;
      const float* pr = P + n.off_rcab(g, r);
      const float* c1b = pr + kConvW;
      const float* c2b = pr + 2 * kConvW + 64;
      const float* w1 = pr + 2 * (kConvW + 64);
      const float* b1 = w1 + n.hid * 64;
      const float* w2 = b1 + n.hid;
      const float* b2 = w2 + 64 * n.hid;
      RC(conv64_pair(conv64_args(XB(xbi), WF(n.cidx(g, r, 0)), c1b, B, H, W, nullptr, T1(ti), SRES_EPI_RELU),
                     conv64_args(T1(ti), WF(n.cidx(g, r, 1)), c2b, B, H, W, nullptr, T2(ti), fused_pool ? SRES_EPI_POOL : 0,
                                 fused_pool ? pool_part : nullptr),
                     ws + n.o_pair_flags + (size_t)(ti & 1) * sres_conv_pair_flag_bytes(B, H, W), st, "conv pair fwd (conv1 -> conv2 +pool)"));
      if (!fused_pool) RC(sres_ca_pool(T2(ti), pool_sum, B, H, W, st));
      float* mean = (float*)(ws + n.o_mean) + (size_t)(training ? ti : 0) * B * 64;
      float* sv = (float*)(ws + n.o_s) + (size_t)(training ? ti : 0) * B * 64;
      { PROF("ca_apply_fwd");
        RC(sres_ca_apply_fwd(T2(ti), fused_pool ? pool_part : nullptr, fused_pool ? nullptr : pool_sum, w1, b1, w2, b2,
                             n.hid, r == 0 ? gin : xf, xf, XB(xbi + 1), mean, sv, B, H, W, st)); }
      ++xbi;
    }
    const float* pg = P + n.off_gt(g);
    RC(conv64(XB(xbi), WF(n.cidx_gt(g)), pg + kConvW, B, H, W, st, gout, XB(xbi + 1), 0, nullptr, gin));
    ++xbi;
    gin = gout;
  }
  if (l2hint) RC(sres_l2_persist_window(nullptr, 0, st));
  void* resb = ws + n.o_resb;
  RC(conv64(XB(xbi), WF(n.cidx_bt()), P + n.bt_b, B, H, W, st, nullptr, resb, 0, nullptr, hf));
  const void* cur = resb;
  for (int i = 0; i < d.n_up; ++i) {
    const int f = d.up_factor[i];
    for (int sub = 0; sub < f * f; ++sub)
      RC(conv64(cur, ws + n.o_wp_up_fwd[i] + (size_t)sub * kConvW * 2, (const float*)(ws + n.o_bias_up[i]) + sub * 64, B,
                n.lvH[i], n.lvW[i], st, nullptr, ws + n.o_u[i], 0, nullptr, nullptr, nullptr, nullptr, SRES_MAP_SHUFFLE,
                sub / f, sub % f, f));
    cur = ws + n.o_u[i];
  }
  sres_conv_args a;
  memset(&a, 0, sizeof(a));
  a.in_bf16 = cur; a.wpack_bf16 = ws + n.o_wp_tail; a.bias = (const float*)(ws + n.o_bias_tail);
  a.out_nchw = out; a.c_real = d.cout; a.n_out = 16;
  a.B = B; a.H = n.lvH[d.n_up]; a.W = n.lvW[d.n_up];
  if (sres_conv_supported(a.H, a.W, 16)) {
    PROF("tail conv (N=16)");
    RC(sres_conv3x3_igemm(&a, st));
  } else {  // very wide images (x8 of 96x96): HBM-bound CUDA-core kernel, no halo window in shared memory
    PROF("tail conv (CUDA cores)");
    RC(sres_conv3x3_small_out(cur, P + n.tail_w, P + n.tail_b, B, d.cout, a.H, a.W, out, st));
  }
  return SRES_OK;
}

// ---------------------------------------------------------------------------------------------
// backward.  Segments: 0 = tail conv, upsampler, body-tail conv; 1..G = residual groups G-1..0;
// G+1 = head conv.  A caller overlapping the gradient all-reduce runs them one at a time.
// ---------------------------------------------------------------------------------------------
// Deferred weight-gradient jobs: up to SRES_WGRAD_BATCH (8) of the same geometry go out as one batched launch.  A job only
// reads saved activations and a bf16 output-gradient buffer; the queue is flushed before any kernel that
// overwrites such a buffer is enqueued, when it is full, and at the end of every backward segment.
// Optional second stream for the weight-gradient batches: they depend only on saved activations and on
// output-gradient buffers already produced, so they can run beside the input-gradient chain and fill the
// SM time that chain leaves idle (kernel tails, element-wise kernels that leave the tensor cores free).
struct AsyncCtx {
  static constexpr int kEvents = 8;
  cudaStream_t side = nullptr;
  cudaEvent_t fork[kEvents], done[kEvents];
  const void* bufs[kEvents][SRES_WGRAD_MAX_JOBS];  // dy buffers a side batch still reads
  bool live[kEvents];
  int next = 0;
};

struct WgQueue {
  sres_wgrad_job jobs[SRES_WGRAD_MAX_JOBS];
  int n = 0, B = 0, H = 0, W = 0;
  const Net* net = nullptr;
  uint8_t* ws = nullptr;
  void* st = nullptr;
  AsyncCtx* ax = nullptr;
  int wait_slot(int i) {  // main stream waits for side batch i
    if (ax && ax->live[i]) {
      cudaError_t e = cudaStreamWaitEvent((cudaStream_t)st, ax->done[i], 0);
      if (e != cudaSuccess) return set_cuda_error(e, "backward: join side stream");
      ax->live[i] = false;
    }
    return SRES_OK;
  }
  int join_all() {
    if (ax)
      for (int i = 0; i < AsyncCtx::kEvents; ++i) RC(wait_slot(i));
    return SRES_OK;
  }
  int flush() {
    if (n == 0) return SRES_OK;
    PROF("wgrad batch (+reduce)");
    int rc;
    if (ax) {
      const int i = ax->next;
      ax->next = (i + 1) % AsyncCtx::kEvents;
      RC(wait_slot(i));
      cudaError_t e = cudaEventRecord(ax->fork[i], (cudaStream_t)st);
      if (e == cudaSuccess) e = cudaStreamWaitEvent(ax->side, ax->fork[i], 0);
      if (e != cudaSuccess) return set_cuda_error(e, "backward: fork side stream");
      rc = sres_conv3x3_wgrad_batch(jobs, n, B, H, W, ws + net->o_wg_ws, sres_conv_wgrad_workspace_bytes(), ax->side);
      if (rc) return rc;
      e = cudaEventRecord(ax->done[i], ax->side);
      if (e != cudaSuccess) return set_cuda_error(e, "backward: side event");
      for (int k = 0; k < SRES_WGRAD_MAX_JOBS; ++k) ax->bufs[i][k] = k < n ? jobs[k].dy_bf16 : nullptr;
      ax->live[i] = true;
    } else {
      rc = sres_conv3x3_wgrad_batch(jobs, n, B, H, W, ws + net->o_wg_ws, sres_conv_wgrad_workspace_bytes(), st);
    }
    n = 0;
    return rc;
  }
  // Run one more piece of work that only depends on what the main stream has enqueued so far (the channel-attention
  // parameter gradients of a finished group) behind the weight-gradient batches on the side stream.
  template <class F>
  int run_side(F fn) {
    if (!ax) return fn(st);
    const int i = ax->next;
    ax->next = (i + 1) % AsyncCtx::kEvents;
    RC(wait_slot(i));
    cudaError_t e = cudaEventRecord(ax->fork[i], (cudaStream_t)st);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(ax->side, ax->fork[i], 0);
    if (e != cudaSuccess) return set_cuda_error(e, "backward: fork side stream");
    RC(fn((void*)ax->side));
    e = cudaEventRecord(ax->done[i], ax->side);
    if (e != cudaSuccess) return set_cuda_error(e, "backward: side event");
    for (int k = 0; k < SRES_WGRAD_MAX_JOBS; ++k) ax->bufs[i][k] = nullptr;
    ax->live[i] = true;
    return SRES_OK;
  }
  int push(const void* x, const void* dy, int B_, int H_, int W_, float* dw, float* db, int cout_total, int stride,
           int offset, int acc, float scale = 1.f) {
    if (n && (B_ != B || H_ != H || W_ != W)) RC(flush());
    B = B_; H = H_; W = W_;
    sres_wgrad_job& j = jobs[n++];
    j.x_bf16 = x; j.dy_bf16 = dy; j.dw_oihw = dw; j.dbias = db;
    j.cout_total = cout_total; j.oc_stride = stride; j.oc_offset = offset; j.accumulate = acc;
    j.scale = scale;
    if (n == wgrad_batch_jobs()) RC(flush());
    return SRES_OK;
  }
  // call before enqueuing a kernel that writes `buf`
  int before_write(const void* buf) {
    for (int i = 0; i < n; ++i)
      if (jobs[i].dy_bf16 == buf) { RC(flush()); break; }
    if (ax)
      for (int i = 0; i < AsyncCtx::kEvents; ++i)
        if (ax->live[i])
          for (int k = 0; k < SRES_WGRAD_MAX_JOBS; ++k)
            if (ax->bufs[i][k] == buf) { RC(wait_slot(i)); break; }
    return SRES_OK;
  }
};

static int backward(const Net& n, const float* P, const float* x, const float* dout, float* Gr, int accumulate,
                    uint8_t* ws, int seg_begin, int seg_end, AsyncCtx* ax, void* st) {
  const sres_rcan_desc& d = n.d;
  const int B = d.B, H = d.H, W = d.W, G = d.n_groups, R = d.n_blocks, L = d.n_up;
  const size_t bf = (size_t)n.lvRows[0] * 128;
  auto XB = [&](int i) { return ws + n.o_xb + (size_t)i * bf; };
  auto T1 = [&](int i) { return ws + n.o_t1 + (size_t)i * bf; };
  auto T2 = [&](int i) { return ws + n.o_t2 + (size_t)i * bf; };
  auto WD = [&](long long c) { return ws + n.o_wp_dg + (size_t)c * kConvW * 2; };
  float* ga = (float*)(ws + n.o_ga);
  float* gb32 = (float*)(ws + n.o_gb32);
  void* gb16 = ws + n.o_gb16;
  WgQueue wq;
  wq.net = &n; wq.ws = ws; wq.st = st; wq.ax = ax;
  if (ax) for (int i = 0; i < AsyncCtx::kEvents; ++i) ax->live[i] = false;
  float* dres32 = (float*)(ws + n.o_dres32);
  void* dres16 = ws + n.o_dres16;
  const int xb_last = n.edsr ? R : G * (R + 1);  // bf16 copy of the body's last output = body-tail conv input
  const bool fused_dot = (H + 1) * (W + 1) >= 128;  // per-tile two-segment partials need an image >= one M tile

  for (int seg = seg_begin; seg < seg_end; ++seg) {
    if (seg == 0) {
      const int Hh = n.lvH[L], Wh = n.lvW[L];
      const void* u_last = L > 0 ? (const void*)(ws + n.o_u[L - 1]) : (const void*)(ws + n.o_resb);
      { PROF("tail wgrad");
      RC(sres_small_out_wgrad(dout, u_last, B, d.cout, Hh, Wh, Gr + n.tail_w, Gr + n.tail_b, accumulate, ws + n.o_sw_ws,
                              sres_small_wgrad_workspace_bytes(), st)); }
      { PROF("tail dgrad");
      if (L == 0) {
        RC(sres_conv3x3_small_in(dout, P + n.tail_w, nullptr, B, d.cout, Hh, Wh, 1, 0, dres32, dres16, st));
      } else {
        RC(sres_conv3x3_small_in(dout, P + n.tail_w, nullptr, B, d.cout, Hh, Wh, 1, d.up_factor[L - 1], nullptr,
                                 ws + n.o_du16[L - 1], st));
      } }
      for (int i = L - 1; i >= 0; --i) {
        const int f = d.up_factor[i], f2 = f * f;
        const void* cur_in = i > 0 ? (const void*)(ws + n.o_u[i - 1]) : (const void*)(ws + n.o_resb);
        const size_t sub_bytes = (size_t)n.lvRows[i] * 128;
        // destination of the input gradient of this stage
        float* acc32 = i > 0 ? (float*)(ws + n.o_du32[i - 1]) : dres32;
        void* acc16 = i > 0 ? (void*)(ws + n.o_du16[i - 1]) : dres16;
        const int map = i > 0 ? SRES_MAP_UNSHUFFLE : SRES_MAP_IDENT;
        const int sf = i > 0 ? d.up_factor[i - 1] : 2;
        for (int sub = 0; sub < f2; ++sub) {
          const void* dy = ws + n.o_du16[i] + sub * sub_bytes;
          RC(wq.push(cur_in, dy, B, n.lvH[i], n.lvW[i], Gr + n.up_w[i], Gr + n.up_b[i], f2 * 64, f2, sub, accumulate));
          RC(conv64(dy, ws + n.o_wp_up_dg[i] + (size_t)sub * kConvW * 2, nullptr, B, n.lvH[i], n.lvW[i], st, acc32,
                    sub == f2 - 1 ? acc16 : nullptr, 0, nullptr, sub > 0 ? acc32 : nullptr, nullptr, nullptr, map, 0, 0,
                    sf));
        }
      }
      // body-tail conv
      RC(wq.push(XB(xb_last), dres16, B, H, W, Gr + n.bt_w, Gr + n.bt_b, 64, 1, 0, accumulate));
      RC(wq.before_write(gb16));
      RC(conv64(dres16, WD(n.cidx_bt()), nullptr, B, H, W, st, ga, gb16));
      RC(wq.flush());
    } else if (seg <= G && n.edsr) {
      // ResBlocks R-1..0.  ga = fp32 gradient trunk; its bf16 copy for block r lives in gb16 (r = R-1, written by
      // segment 0) or dt2[r % ring_len()] (written by block r+1's conv1 input-gradient).
      const bool l2hint = l2_hint_enabled();
      if (l2hint) RC(sres_l2_persist_window(ga, (size_t)n.lvRows[0] * 256, st));
      for (int r = R - 1; r >= 0; --r) {
        float* gr = Gr + n.off_rcab(0, r);
        const void* g16 = r == R - 1 ? gb16 : (const void*)(ws + n.o_dt2[r % ring_len()]);
        void* dt1 = ws + n.o_dt1[r % ring_len()];
        RC(wq.push(T1(r), g16, B, H, W, gr + kConvW + 64, gr + 2 * kConvW + 64, 64, 1, 0, accumulate, n.rs));
        RC(wq.before_write(dt1));
        RC(conv64(g16, WD(n.cidx(0, r, 1)), nullptr, B, H, W, st, nullptr, dt1, 0, nullptr, nullptr, nullptr, T1(r)));
        RC(wq.push(XB(r), dt1, B, H, W, gr, gr + kConvW, 64, 1, 0, accumulate));
        void* nxt = r > 0 ? (void*)(ws + n.o_dt2[(r - 1) % ring_len()]) : nullptr;
        if (nxt) RC(wq.before_write(nxt));
        RC(conv64(dt1, WD(n.cidx(0, r, 0)), nullptr, B, H, W, st, ga, nxt, 0, nullptr, ga));
      }
      RC(wq.flush());
      if (l2hint) RC(sres_l2_persist_window(nullptr, 0, st));
    } else if (seg <= G) {
      const int g = G - seg;
      const int xb0 = g * (R + 1);  // XB index of the group's input
      const bool l2hint = l2_hint_enabled();
      if (l2hint) RC(sres_l2_persist_window(gb32, (size_t)n.lvRows[0] * 256, st));
      float* Gg = Gr + n.off_gt(g);
      RC(wq.push(XB(xb0 + R), gb16, B, H, W, Gg, Gg + kConvW, 64, 1, 0, accumulate));
      // the convolution that produces the gradient of RCAB r's output also reduces ds = sum(g * t2_r) per tile
      float* dot_part = (float*)(ws + n.o_pool_part);
      RC(conv64(gb16, WD(n.cidx_gt(g)), nullptr, B, H, W, st, gb32, nullptr, fused_dot ? SRES_EPI_DOT : 0,
                fused_dot ? dot_part : nullptr, nullptr, nullptr, fused_dot ? T2(g * R + R - 1) : nullptr));
      for (int r = R - 1; r >= 0; --r) {
        const int ti = g * R + r;
        const float* pr = P + n.off_rcab(g, r);
        float* gr = Gr + n.off_rcab(g, r);
        const float* w1 = pr + 2 * (kConvW + 64);
        const float* b1 = w1 + n.hid * 64;
        const float* w2 = b1 + n.hid;
        const float* b2 = w2 + 64 * n.hid;
        const float* mean = (const float*)(ws + n.o_mean) + (size_t)ti * B * 64;
        float* dsv = (float*)(ws + n.o_ds) + (size_t)ti * B * 64;
        void* dt2 = ws + n.o_dt2[ti % ring_len()];
        void* dt1 = ws + n.o_dt1[ti % ring_len()];
        RC(wq.before_write(dt2));
        { PROF("ca_bwd");
        if (fused_dot) RC(sres_ca_bwd_apply(gb32, dot_part, w1, b1, w2, b2, n.hid, mean, dt2, dsv, B, H, W, st));
        else RC(sres_ca_bwd(gb32, T2(ti), w1, b1, w2, b2, n.hid, mean, (float*)(ws + n.o_ds_part), dt2, dsv, B, H, W, st)); }
        RC(wq.push(T1(ti), dt2, B, H, W, gr + kConvW + 64, gr + 2 * kConvW + 64, 64, 1, 0, accumulate));
        RC(wq.before_write(dt1));
        if (r > 0) {
          // dgrad of conv2 (ReLU mask) and dgrad of conv1 (fp32 read-modify-write of the gradient trunk + sum g*t2) as one launch
          RC(conv64_pair(conv64_args(dt2, WD(n.cidx(g, r, 1)), nullptr, B, H, W, nullptr, dt1, 0, nullptr, nullptr, nullptr, T1(ti)),
                         conv64_args(dt1, WD(n.cidx(g, r, 0)), nullptr, B, H, W, gb32, nullptr, fused_dot ? SRES_EPI_DOT : 0,
                                     fused_dot ? dot_part : nullptr, gb32, nullptr, fused_dot ? T2(ti - 1) : nullptr),
                         ws + n.o_pair_flags + (size_t)(ti & 1) * sres_conv_pair_flag_bytes(B, H, W), st,
                         "conv pair bwd (dgrad2 -> dgrad1 +rmw +dot)"));
          RC(wq.push(XB(xb0 + r), dt1, B, H, W, gr, gr + kConvW, 64, 1, 0, accumulate));
        } else {
          RC(conv64(dt2, WD(n.cidx(g, r, 1)), nullptr, B, H, W, st, nullptr, dt1, 0, nullptr, nullptr, nullptr, T1(ti)));
          RC(wq.push(XB(xb0 + r), dt1, B, H, W, gr, gr + kConvW, 64, 1, 0, accumulate));
          // grad wrt the group input = body path (gb32 + conv1 dgrad) + group skip (ga)
          RC(wq.before_write(gb16));
          RC(conv64(dt1, WD(n.cidx(g, r, 0)), nullptr, B, H, W, st, ga, gb16, 0, nullptr, gb32, ga));
        }
      }
      RC(wq.flush());
      if (l2hint) RC(sres_l2_persist_window(nullptr, 0, st));
      // The group's squeeze-excite parameter gradients (20 small latency-bound blocks, 66 us) only read what the
      // ca_bwd kernels above saved: they go behind the weight-gradient batches on the side stream instead of holding up
      // the next group's input-gradient chain.
      const long long first = n.off_rcab(g, 0) + 2 * (kConvW + 64);
      PROF("ca_param_grads");
      RC(wq.run_side([&](void* s) {
        return sres_ca_param_grads(P + first, Gr + first, n.rcab_sz, R, (const float*)(ws + n.o_mean) + (size_t)g * R * B * 64,
                                   (const float*)(ws + n.o_ds) + (size_t)g * R * B * 64, B, n.hid, accumulate,
                                   ws + n.o_ca_scr, sres_ca_param_grads_scratch_bytes(R, B), s);
      }));
    } else if (seg == G + 1) {
      PROF("head wgrad");
      RC(sres_small_in_wgrad(ga, dres32, x, B, d.cin, H, W, Gr + n.head_w, Gr + n.head_b, accumulate, ws + n.o_sw_ws,
                             sres_small_wgrad_workspace_bytes(), st));
    }
  }
  // One join per call, not per segment: the side stream's work only has to be complete when the caller may look at the
  // gradients (the data-parallel path calls segment by segment and so still joins before each all-reduce).
  RC(wq.join_all());
  return SRES_OK;
}

}  // namespace sres

using namespace sres;

extern "C" int64_t sres_rcan_param_count(const sres_rcan_desc* d) {
  Net n;
  if (build_net(&n, d, 0)) return -1;
  return n.n_params;
}

extern "C" int sres_rcan_workspace_bytes(const sres_rcan_desc* d, int training, size_t* bytes) {
  Net n;
  int rc = build_net(&n, d, training);
  if (rc) return rc;
  if (!bytes) return set_error(SRES_ERR_INVALID_ARG, "rcan: null output");
  *bytes = n.total;
  return SRES_OK;
}

extern "C" int sres_rcan_num_segments(const sres_rcan_desc* d) { return d ? d->n_groups + 2 : -1; }

extern "C" int sres_rcan_segment_params(const sres_rcan_desc* d, int seg, int64_t* offset, int64_t* count) {
  Net n;
  int rc = build_net(&n, d, 0);
  if (rc) return rc;
  if (!offset || !count || seg < 0 || seg > d->n_groups + 1) return set_error(SRES_ERR_INVALID_ARG, "rcan: bad segment");
  if (seg == 0) { *offset = n.bt_w; *count = n.n_params - n.bt_w; }
  else if (seg <= d->n_groups) { *offset = n.body0 + (long long)(d->n_groups - seg) * n.group_sz; *count = n.group_sz; }
  else { *offset = 0; *count = n.body0; }
  return SRES_OK;
}

extern "C" int sres_rcan_pack_weights(const sres_rcan_desc* d, const float* params, void* workspace, int training,
                                      void* stream) {
  Net n;
  int rc = build_net(&n, d, training);
  if (rc) return rc;
  if (!params || !workspace) return set_error(SRES_ERR_INVALID_ARG, "rcan: null pointer");
  return pack_all(n, params, (uint8_t*)workspace, (cudaStream_t)stream);
}

extern "C" int sres_rcan_forward(const sres_rcan_desc* d, const float* params, const float* x_nchw, float* out_nchw,
                                 void* workspace, int training, void* stream) {
  Net n;
  int rc = build_net(&n, d, training);
  if (rc) return rc;
  if (!params || !x_nchw || !out_nchw || !workspace) return set_error(SRES_ERR_INVALID_ARG, "rcan: null pointer");
  return forward(n, params, x_nchw, out_nchw, (uint8_t*)workspace, training, stream);
}

extern "C" int sres_async_create(void** out) {
  if (!out) return set_error(SRES_ERR_INVALID_ARG, "async_create: null output");
  AsyncCtx* a = new AsyncCtx();
  cudaError_t e = cudaStreamCreateWithFlags(&a->side, cudaStreamNonBlocking);
  for (int i = 0; i < AsyncCtx::kEvents && e == cudaSuccess; ++i) {
    e = cudaEventCreateWithFlags(&a->fork[i], cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&a->done[i], cudaEventDisableTiming);
    a->live[i] = false;
  }
  if (e != cudaSuccess) { delete a; return set_cuda_error(e, "async_create"); }
  *out = a;
  return SRES_OK;
}

extern "C" int sres_async_destroy(void* ctx) {
  AsyncCtx* a = (AsyncCtx*)ctx;
  if (!a) return SRES_OK;
  for (int i = 0; i < AsyncCtx::kEvents; ++i) { cudaEventDestroy(a->fork[i]); cudaEventDestroy(a->done[i]); }
  cudaStreamDestroy(a->side);
  delete a;
  return SRES_OK;
}

extern "C" int sres_rcan_backward(const sres_rcan_desc* d, const float* params, const float* x_nchw,
                                  const float* dout_nchw, float* grads, int accumulate, void* workspace, int seg_begin,
                                  int seg_end, void* async_ctx, void* stream) {
  Net n;
  int rc = build_net(&n, d, 1);
  if (rc) return rc;
  if (!params || !x_nchw || !dout_nchw || !grads || !workspace) return set_error(SRES_ERR_INVALID_ARG, "rcan: null pointer");
  if (seg_begin < 0 || seg_end > d->n_groups + 2 || seg_begin > seg_end)
    return set_error(SRES_ERR_INVALID_ARG, "rcan: bad segment range");
  return backward(n, params, x_nchw, dout_nchw, grads, accumulate, (uint8_t*)workspace, seg_begin, seg_end, (AsyncCtx*)async_ctx,
                  stream);
}

// Aggregate and clear the SRES_PROFILE records of the calling thread (synchronises the device).
extern "C" int sres_profile_report(char* buf, size_t nbuf) {
  using namespace sres;
  if (!buf || nbuf == 0) return set_error(SRES_ERR_INVALID_ARG, "profile_report: no buffer");
  buf[0] = 0;
  cudaDeviceSynchronize();
  std::lock_guard<std::mutex> lk(g_prof_mu);
  if (!t_prof || t_prof->empty()) return SRES_OK;
  std::map<std::string, std::pair<int, double>> agg;
  double total = 0;
  for (auto& r : *t_prof) {
    float ms = 0;
    cudaEventElapsedTime(&ms, r.a, r.b);
    agg[r.cat].first += 1; agg[r.cat].second += ms; total += ms;
    cudaEventDestroy(r.a); cudaEventDestroy(r.b);
  }
  t_prof->clear();
  size_t off = 0;
  off += snprintf(buf + off, nbuf - off, "total %.3f ms\n", total);
  for (auto& kv : agg)
    if (off < nbuf) off += snprintf(buf + off, nbuf - off, "%-40s n=%5d  %8.3f ms  %5.1f%%  avg %7.1f us\n", kv.first.c_str(),
                                    kv.second.first, kv.second.second, 100.0 * kv.second.second / total,
                                    1e3 * kv.second.second / kv.second.first);
  return SRES_OK;
}
