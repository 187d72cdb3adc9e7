// HBM-bound element-wise / reduction kernels around the network: bicubic resize, losses and their
// gradients, fused flat Adam.  All vectorised where alignment is guaranteed, reductions are
// two-stage with a fixed order (deterministic, no atomics).
#include "internal.h"
#include "ptx.cuh"

namespace sres {

static int ew_grid(long long n, int per_thread = 1) {
  int sms = device_sm_count();
  if (sms <= 0) sms = 148;
  long long blocks = (n + 256LL * per_thread - 1) / (256LL * per_thread);
  const long long cap = (long long)sms * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (int)blocks;
}

// ---------------------------------------------------------------------------------------------
// Bicubic resize, F.interpolate(mode='bicubic', align_corners=False, antialias=False) semantics
// (aten upsample_bicubic2d: A = -0.75, source index scale*(dst+0.5)-0.5, border clamp).
// Reference call sites: sres/base/util/array.py:72-76 (downsample), :84-87 (upsample).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float cc1(float x, float A) { return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; }
__device__ __forceinline__ float cc2(float x, float A) { return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; }
__device__ __forceinline__ void cubic_coeffs(float t, float (&c)[4]) {
  const float A = -0.75f;
  c[0] = cc2(t + 1.f, A);
  c[1] = cc1(t, A);
  c[2] = cc1(1.f - t, A);
  c[3] = cc2(2.f - t, A);
}

__global__ void bicubic_resize_kernel(const float* __restrict__ in, float* __restrict__ out, int planes, int Hi, int Wi,
                                      int Ho, int Wo, float scale_h, float scale_w) {
  const long long total = (long long)planes * Ho * Wo;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int ox = int(idx % Wo), oy = int((idx / Wo) % Ho);
    const int pl = int(idx / ((long long)Wo * Ho));
    const float ry = scale_h * (oy + 0.5f) - 0.5f, rx = scale_w * (ox + 0.5f) - 0.5f;
    const float fy = floorf(ry), fx = floorf(rx);
    const int iy = int(fy), ix = int(fx);
    float cy[4], cx[4];
    cubic_coeffs(ry - fy, cy);
    cubic_coeffs(rx - fx, cx);
    const float* ip = in + (size_t)pl * Hi * Wi;
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int yy = min(max(iy - 1 + i, 0), Hi - 1);
      float row = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int xx = min(max(ix - 1 + j, 0), Wi - 1);
        row += __ldg(ip + (size_t)yy * Wi + xx) * cx[j];
      }
      acc += row * cy[i];
    }
    out[idx] = acc;
  }
}

// ---------------------------------------------------------------------------------------------
// Nearest, nearest-exact, bilinear and area resize: F.interpolate(mode=..., align_corners=False,
// antialias=False) on 4-D input, the other settings of task.downsample_mode / upsample_mode
// (sres/base/util/array.py:37-41 passes them to F.interpolate unchanged).  Index arithmetic as in
// ATen (UpSample.h, AdaptiveAveragePooling), so nearest / nearest-exact pick the same source
// pixels as torch's CPU and CUDA kernels and area sums in the same order.
// ---------------------------------------------------------------------------------------------
// upsample_nearest2d on the CPU: a plain copy for equal sizes and a shift for exactly 2x, else
// floor(dst * scale) with the float scale 1/scale_factor.
__device__ __forceinline__ int nearest_src(int dst, int in, int out, float scale) {
  if (out == in) return dst;
  if (out == 2 * in) return dst >> 1;
  return min(int(floorf(__fmul_rn((float)dst, scale))), in - 1);
}
__device__ __forceinline__ int nearest_exact_src(int dst, int in, float scale) {
  return min(int(floorf(__fmul_rn(__fadd_rn((float)dst, 0.5f), scale))), in - 1);
}
// linear source index (area_pixel_compute_source_index, clamped at 0 unlike cubic) and lambdas
// (guard_index_and_lambda).  ATen's float build contracts scale * (dst + 0.5) - 0.5 into one FMA.
__device__ __forceinline__ void linear_src(int dst, int in, int out, float scale, int& i0, int& i1, float& l0, float& l1) {
  if (out == in) {
    i0 = i1 = dst;
    l0 = 1.f;
    l1 = 0.f;
    return;
  }
  const float r = fmaxf(__fmaf_rn(scale, __fadd_rn((float)dst, 0.5f), -0.5f), 0.f);
  i0 = min(int(floorf(r)), in - 1);
  l1 = fminf(fmaxf(r - (float)i0, 0.f), 1.f);
  l0 = 1.f - l1;
  i1 = i0 + (i0 < in - 1 ? 1 : 0);
}

__device__ __forceinline__ float add_in_order(float s, float q) { return s + q; }
__device__ __forceinline__ float add_in_order(float s, float4 q) { return (((s + q.x) + q.y) + q.z) + q.w; }
// Sum of rows [y0, y1) x columns [x0, x0 + kw) in fp32, row by row and left to right (ATen's order), read as pieces of
// sizeof(V) bytes (kw a multiple of the piece) four at a time, so that four loads are in flight before the adds.
template <typename V>
__device__ __forceinline__ float window_sum(const float* ip, int Wi, int y0, int y1, int x0, int kw) {
  constexpr int P = sizeof(V) / sizeof(float);
  const int per_row = kw / P, n = (y1 - y0) * per_row;
  float sum = 0.f;
  for (int p = 0; p < n; p += 4) {
    V q[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (p + k < n) {
        const int r = (p + k) / per_row, c = p + k - r * per_row;
        q[k] = __ldg(reinterpret_cast<const V*>(ip + (size_t)(y0 + r) * Wi + x0) + c);
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (p + k < n) sum = add_in_order(sum, q[k]);
  }
  return sum;
}

template <int MODE>
__global__ void __launch_bounds__(256)
resize_kernel(const float* __restrict__ in, float* __restrict__ out, int planes, int Hi, int Wi, int Ho, int Wo,
              float scale_h, float scale_w, int rows16) {
  const long long total = (long long)planes * Ho * Wo;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int ox = int(idx % Wo), oy = int((idx / Wo) % Ho);
    const int pl = int(idx / ((long long)Wo * Ho));
    const float* ip = in + (size_t)pl * Hi * Wi;
    float v;
    if (MODE == SRES_RESIZE_NEAREST) {
      v = __ldg(ip + (size_t)nearest_src(oy, Hi, Ho, scale_h) * Wi + nearest_src(ox, Wi, Wo, scale_w));
    } else if (MODE == SRES_RESIZE_NEAREST_EXACT) {
      v = __ldg(ip + (size_t)nearest_exact_src(oy, Hi, scale_h) * Wi + nearest_exact_src(ox, Wi, scale_w));
    } else if (MODE == SRES_RESIZE_BILINEAR) {
      int y0, y1, x0, x1;
      float a0, a1, b0, b1;
      linear_src(oy, Hi, Ho, scale_h, y0, y1, a0, a1);
      linear_src(ox, Wi, Wo, scale_w, x0, x1, b0, b1);
      const float* r0 = ip + (size_t)y0 * Wi;
      const float* r1 = ip + (size_t)y1 * Wi;
      v = a0 * (b0 * __ldg(r0 + x0) + b1 * __ldg(r0 + x1)) + a1 * (b0 * __ldg(r1 + x0) + b1 * __ldg(r1 + x1));
    } else {  // SRES_RESIZE_AREA: adaptive_avg_pool2d, rows [floor(o*in/out), ceil((o+1)*in/out))
      const int y0 = (int)(((long long)oy * Hi) / Ho), y1 = (int)(((long long)(oy + 1) * Hi + Ho - 1) / Ho);
      const int x0 = (int)(((long long)ox * Wi) / Wo), x1 = (int)(((long long)(ox + 1) * Wi + Wo - 1) / Wo);
      const int kw = x1 - x0;
      const float sum = (rows16 && ((x0 | kw) & 3) == 0)   // whole 16-byte row pieces (a x4 / x8 block mean)
                            ? window_sum<float4>(ip, Wi, y0, y1, x0, kw)
                            : window_sum<float>(ip, Wi, y0, y1, x0, kw);
      v = sum / (float)(y1 - y0) / (float)kw;
    }
    out[idx] = v;
  }
}

// ---------------------------------------------------------------------------------------------
// Losses.  kind 0 = l2 (RMSE, sres/controller/stats.py:5-8), 1 = charbonnier
// (sres/controller/dual_trainer.py:196-198), 2 = l1 (north_star variant, not in the reference).
// Forward stage 1: per-block sums of f(d); stage 2: one block sums the partials in order and
// writes  stat[0] = sum f(d),  stat[1] = loss.
// The target may be larger than the product (conform_to_product, dual_trainer.py:200-203): it is
// read with its own row pitch / plane size and cropped to the product's (H,W).
// ---------------------------------------------------------------------------------------------
struct LossGeom {
  long long n;       // product elements
  int H, W;          // product plane
  int tH, tW;        // target plane
};
__device__ __forceinline__ long long tgt_index(const LossGeom& g, long long i) {
  if (g.tH == g.H && g.tW == g.W) return i;
  const int x = int(i % g.W);
  const long long r = i / g.W;
  const int y = int(r % g.H);
  const long long pl = r / g.H;
  return (pl * g.tH + y) * g.tW + x;
}
__device__ __forceinline__ float loss_term(int kind, float d, float eps) {
  if (kind == 0) return d * d;
  if (kind == 1) return sqrtf(d * d + eps);
  return fabsf(d);
}

__global__ void __launch_bounds__(256)
loss_partial_kernel(const float* __restrict__ prd, const float* __restrict__ tgt, LossGeom g, int kind, float eps,
                    double* __restrict__ part) {
  __shared__ double sm[256];
  double a = 0.0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < g.n; i += (long long)gridDim.x * blockDim.x)
    a += (double)loss_term(kind, prd[i] - tgt[tgt_index(g, i)], eps);
  sm[threadIdx.x] = a;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) sm[threadIdx.x] += sm[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) part[blockIdx.x] = sm[0];
}

// stat (double[2]): [0] = sum over THIS rank, [1] = number of elements of THIS rank -- a data-parallel caller all-reduces
// both, so that ranks holding batches of different sizes (the short last batch of a timeslice) still agree on the
// global-batch loss.
__global__ void loss_final_kernel(const double* __restrict__ part, int nparts, double n_local, double* __restrict__ stat) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < nparts; ++i) s += part[i];
    stat[0] = s;
    stat[1] = n_local;
  }
}

// loss value from the (possibly all-reduced) sum:  l2: sqrt(sum/N),  others: sum/N.
__global__ void loss_value_kernel(const double* __restrict__ stat, double n_total, const double* __restrict__ n_total_dev,
                                  int kind, float* __restrict__ loss) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    if (n_total_dev) n_total = n_total_dev[0];
    const double m = n_total > 0.0 ? stat[0] / n_total : 0.0;   // (no elements anywhere: define the loss as 0)
    loss[0] = (float)(kind == 0 ? sqrt(m) : m);
  }
}

// d loss / d prd, times the upstream scalar `gscale`.
//   l2:  d / (N * L);  charbonnier: d / sqrt(d^2+eps) / N;  l1: sign(d) / N      (N = n_total)
__global__ void __launch_bounds__(256)
loss_grad_kernel(const float* __restrict__ prd, const float* __restrict__ tgt, LossGeom g, int kind, float eps,
                 const float* __restrict__ loss, double n_total, const double* __restrict__ n_total_dev, float gscale,
                 const float* __restrict__ gscale_dev, float* __restrict__ grad) {
  const float L = loss[0];
  if (gscale_dev) gscale *= gscale_dev[0];
  if (n_total_dev) n_total = n_total_dev[0];
  const float inv_n = n_total > 0.0 ? (float)(1.0 / n_total) : 0.f;
  const float k_l2 = (gscale != 0.f && L > 0.f) ? gscale * inv_n / L : 0.f;   // weight-0 participant / zero loss: no gradient
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < g.n; i += (long long)gridDim.x * blockDim.x) {
    const float d = prd[i] - tgt[tgt_index(g, i)];
    float r;
    if (kind == 0) r = d * k_l2;
    else if (kind == 1) r = gscale * inv_n * d / sqrtf(d * d + eps);
    else r = gscale * inv_n * (d > 0.f ? 1.f : (d < 0.f ? -1.f : 0.f));
    grad[i] = r;
  }
}

// ---------------------------------------------------------------------------------------------
// Fused flat Adam: torch.optim.Adam defaults semantics (sres/controller/dual_trainer.py:126,323):
//   g += wd*p;  m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;  p -= (lr/bc1) * m / (sqrt(v)/sqrt(bc2) + eps)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
adam_flat_kernel(float4* __restrict__ p, const float4* __restrict__ g, float4* __restrict__ m, float4* __restrict__ v,
                 long long n4, float lr_over_bc1, float inv_sqrt_bc2, float b1, float b2, float eps, float wd) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
    float4 pp = p[i], gg = g[i], mm = m[i], vv = v[i];
    float* P = &pp.x; float* G = &gg.x; float* M = &mm.x; float* V = &vv.x;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float gr = G[j];
      if (wd != 0.f) gr = fmaf(wd, P[j], gr);
      M[j] = fmaf(b1, M[j], (1.f - b1) * gr);
      V[j] = fmaf(b2, V[j], (1.f - b2) * gr * gr);
      const float denom = sqrtf(V[j]) * inv_sqrt_bc2 + eps;
      P[j] -= lr_over_bc1 * (M[j] / denom);
    }
    p[i] = pp; m[i] = mm; v[i] = vv;
  }
}

}  // namespace sres

using namespace sres;

extern "C" int sres_bicubic_resize(const float* in, float* out, int planes, int Hi, int Wi, int Ho, int Wo,
                                   double scale_h, double scale_w, void* stream) {
  if (!in || !out) return set_error(SRES_ERR_INVALID_ARG, "bicubic: null pointer");
  if (planes <= 0 || Hi <= 0 || Wi <= 0 || Ho <= 0 || Wo <= 0) return set_error(SRES_ERR_INVALID_ARG, "bicubic: bad shape");
  const long long total = (long long)planes * Ho * Wo;
  bicubic_resize_kernel<<<ew_grid(total), 256, 0, (cudaStream_t)stream>>>(in, out, planes, Hi, Wi, Ho, Wo,
                                                                          (float)scale_h, (float)scale_w);
  SRES_CHECK_LAUNCH("bicubic: launch");
  return SRES_OK;
}

extern "C" int sres_resize(const float* in, float* out, int planes, int Hi, int Wi, int Ho, int Wo, double scale_h,
                           double scale_w, int mode, void* stream) {
  if (!in || !out) return set_error(SRES_ERR_INVALID_ARG, "resize: null pointer");
  if (planes <= 0 || Hi <= 0 || Wi <= 0 || Ho <= 0 || Wo <= 0) return set_error(SRES_ERR_INVALID_ARG, "resize: bad shape");
  if (mode < SRES_RESIZE_NEAREST || mode > SRES_RESIZE_AREA)
    return set_error(SRES_ERR_INVALID_ARG, "resize: unknown mode (SRES_RESIZE_NEAREST .. SRES_RESIZE_AREA)");
  if (mode != SRES_RESIZE_AREA && !(scale_h > 0.0 && scale_w > 0.0 && scale_h < INFINITY && scale_w < INFINITY))
    return set_error(SRES_ERR_INVALID_ARG, "resize: scales must be positive and finite");
  if (mode == SRES_RESIZE_BICUBIC) return sres_bicubic_resize(in, out, planes, Hi, Wi, Ho, Wo, scale_h, scale_w, stream);
  const long long total = (long long)planes * Ho * Wo;
  const int grid = ew_grid(total);
  const float sh = (float)scale_h, sw = (float)scale_w;
  const cudaStream_t st = (cudaStream_t)stream;
  const int rows16 = (Wi % 4 == 0) && ((uintptr_t)in % 16 == 0);
  switch (mode) {
    case SRES_RESIZE_NEAREST:
      resize_kernel<SRES_RESIZE_NEAREST><<<grid, 256, 0, st>>>(in, out, planes, Hi, Wi, Ho, Wo, sh, sw, rows16);
      break;
    case SRES_RESIZE_NEAREST_EXACT:
      resize_kernel<SRES_RESIZE_NEAREST_EXACT><<<grid, 256, 0, st>>>(in, out, planes, Hi, Wi, Ho, Wo, sh, sw, rows16);
      break;
    case SRES_RESIZE_BILINEAR:
      resize_kernel<SRES_RESIZE_BILINEAR><<<grid, 256, 0, st>>>(in, out, planes, Hi, Wi, Ho, Wo, sh, sw, rows16);
      break;
    default:
      resize_kernel<SRES_RESIZE_AREA><<<grid, 256, 0, st>>>(in, out, planes, Hi, Wi, Ho, Wo, sh, sw, rows16);
      break;
  }
  SRES_CHECK_LAUNCH("resize: launch");
  return SRES_OK;
}

extern "C" size_t sres_loss_workspace_bytes(void) {
  int sms = device_sm_count();
  if (sms <= 0) sms = 148;
  return (size_t)sms * 8 * sizeof(double);
}

static int loss_geom(LossGeom* g, int planes, int H, int W, int tH, int tW) {
  if (planes <= 0 || H <= 0 || W <= 0 || tH < H || tW < W) return set_error(SRES_ERR_INVALID_ARG, "loss: bad shape");
  g->n = (long long)planes * H * W; g->H = H; g->W = W; g->tH = tH; g->tW = tW;
  return SRES_OK;
}

extern "C" int sres_loss_sum(const float* prd, const float* tgt, int planes, int H, int W, int tH, int tW, int kind,
                             double* stat, void* workspace, size_t workspace_bytes, void* stream) {
  LossGeom g;
  int rc = loss_geom(&g, planes, H, W, tH, tW);
  if (rc) return rc;
  if (!prd || !tgt || !stat || !workspace) return set_error(SRES_ERR_INVALID_ARG, "loss: null pointer");
  if (kind < 0 || kind > 2) return set_error(SRES_ERR_INVALID_ARG, "loss: kind must be 0 (l2), 1 (charbonnier), 2 (l1)");
  const int grid = ew_grid(g.n, 4);
  if (workspace_bytes < (size_t)grid * sizeof(double)) return set_error(SRES_ERR_INVALID_ARG, "loss: workspace too small");
  loss_partial_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(prd, tgt, g, kind, 1e-6f, (double*)workspace);
  SRES_CHECK_LAUNCH("loss: partial launch");
  loss_final_kernel<<<1, 32, 0, (cudaStream_t)stream>>>((const double*)workspace, grid, (double)g.n, stat);
  SRES_CHECK_LAUNCH("loss: final launch");
  return SRES_OK;
}

extern "C" int sres_loss_value(const double* stat, double n_total, const double* n_total_dev, int kind, float* loss,
                               void* stream) {
  if (!stat || !loss || (!n_total_dev && n_total <= 0)) return set_error(SRES_ERR_INVALID_ARG, "loss_value: bad argument");
  loss_value_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(stat, n_total, n_total_dev, kind, loss);
  SRES_CHECK_LAUNCH("loss_value: launch");
  return SRES_OK;
}

extern "C" int sres_loss_grad(const float* prd, const float* tgt, int planes, int H, int W, int tH, int tW, int kind,
                              const float* loss, double n_total, const double* n_total_dev, float gscale,
                              const float* gscale_dev, float* grad, void* stream) {
  LossGeom g;
  int rc = loss_geom(&g, planes, H, W, tH, tW);
  if (rc) return rc;
  if (!prd || !tgt || !loss || !grad || (!n_total_dev && n_total <= 0)) return set_error(SRES_ERR_INVALID_ARG, "loss_grad: bad argument");
  loss_grad_kernel<<<ew_grid(g.n, 4), 256, 0, (cudaStream_t)stream>>>(prd, tgt, g, kind, 1e-6f, loss, n_total, n_total_dev,
                                                                      gscale, gscale_dev, grad);
  SRES_CHECK_LAUNCH("loss_grad: launch");
  return SRES_OK;
}

extern "C" int sres_adam_step_flat(float* p, const float* g, float* m, float* v, int64_t n, int64_t step, double lr,
                                   double beta1, double beta2, double eps, double weight_decay, void* stream) {
  if (!p || !g || !m || !v || n <= 0 || step <= 0) return set_error(SRES_ERR_INVALID_ARG, "adam: bad argument");
  if (n % 4 || ((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) % 16)
    return set_error(SRES_ERR_INVALID_ARG, "adam: flat buffers must be 16-byte aligned with n % 4 == 0 (pad the tail)");
  const double bc1 = 1.0 - pow(beta1, (double)step), bc2 = 1.0 - pow(beta2, (double)step);
  adam_flat_kernel<<<ew_grid(n / 4), 256, 0, (cudaStream_t)stream>>>(
      (float4*)p, (const float4*)g, (float4*)m, (float4*)v, n / 4, (float)(lr / bc1), (float)(1.0 / sqrt(bc2)),
      (float)beta1, (float)beta2, (float)eps, (float)weight_decay);
  SRES_CHECK_LAUNCH("adam: launch");
  return SRES_OK;
}
