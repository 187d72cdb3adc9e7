/*
 * sres_b200 -- C ABI of the B200-native RCAN hot path for nasa-nccs-hpda/super-resolution-climate.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  The reference has no FFI of its own: its
 * hot path is stock torch.nn modules called from
 *     sres/model/rcan/network.py:22-27      RCAN.forward
 *     sres/controller/dual_trainer.py:557-571  ModelTrainer.apply_network  (bicubic down + model)
 *     sres/controller/dual_trainer.py:221-234  ModelTrainer.loss  -> sres/controller/stats.py:5-8
 *     sres/controller/dual_trainer.py:322-323  mloss.backward(); optimizer.step()
 *     sres/base/source/swot/raw.py:216-233   SWOTRawDataLoader.get_tiles
 *     sres/controller/dual_trainer.py:449-480  ModelTrainer.assemble_images
 * Each entry point below names the reference lines it replaces.  Signatures are plain C: raw
 * device pointers, explicit sizes, a cudaStream_t passed as void*.  Every function returns an
 * int status (SRES_OK == 0), never throws, never allocates device memory (the caller owns all
 * buffers, including workspaces), so calls on different streams are independent.  Process-wide state is limited to
 * read-once environment switches (DESIGN.md section 5), the L2 set-aside flag of sres_l2_set_aside and the optional
 * SRES_PROFILE event list; none of it is touched by the data path after the first call.  INTEGRATION.md shows the ctypes binding a maintainer would add.
 *
 * Activation layout ("padded tile layout", PTL).  A batch of B feature maps of H x W pixels with
 * 64 channels is stored as   rows = B*(H+1)*(W+1) positions,  64 channels per position,
 * position (b,y,x) at row  b*(H+1)*(W+1) + y*(W+1) + x.  Column x == W and row y == H of every
 * map are zero padding shared between neighbours, so the 3x3 tap (dy,dx) of position q is simply
 * row q + dy*(W+1) + dx -- a constant row shift.  Kernels keep the padding rows at exactly 0.
 * bf16 PTL rows are 128 bytes (one TMA/UMMA 128B-swizzle row); fp32 PTL rows are 256 bytes.
 */
#ifndef SRES_B200_H_
#define SRES_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* exported symbol (the library is built with -fvisibility=hidden) */
#define SRES_API __attribute__((visibility("default")))

#define SRES_OK 0
#define SRES_ERR_INVALID_ARG 1
#define SRES_ERR_UNSUPPORTED 2  /* geometry / channel count outside what the kernels cover */
#define SRES_ERR_CUDA 3         /* a CUDA runtime / driver call failed; see sres_last_error */
#define SRES_ERR_NO_DEVICE 4

#define SRES_NF 64 /* feature channels of the RCAN trunk (nfeatures, config/model/rcan-10-20-64.yaml:4) */

/* ------------------------------------------------------------------------------------------ */
/* library / device                                                                           */
/* ------------------------------------------------------------------------------------------ */
/* ABI version of this header (bumped on incompatible change). */
SRES_API int sres_abi_version(void);
/* Human readable text of the last failure on the calling thread. */
SRES_API const char* sres_last_error(void);
/* Number of SMs of the current device (grid sizing); <0 on error. */
SRES_API int sres_device_sm_count(void);
/* Kernels this library has enqueued so far in this process (eager launches and launches recorded into a stream capture
 * alike; graph replays do not pass through the library and are not counted).  Monotonic; read it before and after a call
 * to count that call's launches.  Not part of the reference's interface: accounting for bench.py's `gpu_launches`.  */
SRES_API long long sres_launch_count(void);
/* L2 residency hints (optional; plain CUDA access-policy windows).  sres_l2_set_aside reserves up to
 * `bytes` of L2 for persisting lines on the current device (process-wide CUDA limit);
 * sres_l2_persist_window marks [base, base+bytes) as persisting for kernels launched on `stream`
 * afterwards (bytes == 0 clears it).  After sres_l2_set_aside(bytes > 0) the network executor marks
 * the fp32 residual trunk (forward) and gradient trunk (backward) persisting by itself.        */
SRES_API int sres_l2_set_aside(size_t bytes);
SRES_API int sres_l2_persist_window(const void* base, size_t bytes, void* stream);
/* Development aid: with SRES_PROFILE=1 in the environment (eager launches only) the network executor brackets
 * every kernel group with CUDA events; this call aggregates them per category into `buf` and clears them. */
SRES_API int sres_profile_report(char* buf, size_t nbuf);
/* Rows of the padded tile layout for a (B,H,W) batch. */
SRES_API int64_t sres_ptl_rows(int B, int H, int W);

/* ------------------------------------------------------------------------------------------ */
/* 3x3 convolution, 64 input features, tensor cores (tcgen05 implicit GEMM)                   */
/* replaces nn.Conv2d(64, n, 3, padding=1) forward and its input-gradient:                    */
/*   sres/model/common/cnn.py:8-9 (default_conv) as used at sres/model/rcan/network.py:14-16, */
/*   55, 71 and sres/model/rcan/blocks.py:62-64 (Upsampler convs).                            */
/* ------------------------------------------------------------------------------------------ */
#define SRES_EPI_RELU 1u       /* v = max(v, 0)                       (network.py:57, nn.ReLU) */
#define SRES_EPI_POOL 2u       /* emit per-tile channel sums for the CA average pool (network.py:35,45) */
#define SRES_EPI_DOT 4u        /* mask_bf16 is not a ReLU mask but a second factor: emit per-tile channel sums of
                                  out * mask into pool_part (the ds = sum(g * t2) reduction of the CALayer backward) */

#define SRES_MAP_IDENT 0       /* output position == input position                              */
#define SRES_MAP_SHUFFLE 1     /* PixelShuffle(f) store: (b,y,x) -> (b,f*y+sub_i,f*x+sub_j) (blocks.py:65,70) */
#define SRES_MAP_UNSHUFFLE 2   /* inverse: (b,y,x) -> sub-grid (y%f,x%f), position (b,y/f,x/f)     */

typedef struct sres_conv_args {
  const void* in_bf16;     /* [rows_in][64] bf16 PTL, geometry (B,H,W)                          */
  const void* wpack_bf16;  /* [9][n_out][64] bf16, tap-major, from sres_pack_conv_weights        */
  const float* bias;       /* [n_out] fp32 or NULL                                              */
  const float* resid_f32;  /* fp32 PTL indexed like the OUTPUT, added before ReLU; may alias out_f32; or NULL */
  const float* resid2_f32; /* second fp32 PTL addend (group skip gradient), may alias out_f32; or NULL */
  const void* mask_bf16;   /* bf16 PTL indexed like the INPUT: v = mask > 0 ? v : 0 (ReLU backward) or NULL */
  float* out_f32;          /* fp32 PTL output or NULL                                           */
  void* out_bf16;          /* bf16 PTL output or NULL                                           */
  float* pool_part;        /* [n_mtiles][2][4][64] fp32 partial channel sums (SRES_EPI_POOL) or NULL */
  float* out_nchw;         /* [B][c_real][H][W] fp32 planar output (n_out == 16 path) or NULL   */
  int32_t B, H, W;         /* geometry of the input                                             */
  int32_t n_out;           /* 64, or 16 (narrow tail conv, c_real <= 16 real channels)          */
  int32_t c_real;          /* real output channels when out_nchw is used                        */
  uint32_t epi_flags;      /* SRES_EPI_*                                                        */
  int32_t map_mode;        /* SRES_MAP_*                                                        */
  int32_t sub_i, sub_j;    /* sub-pixel of SRES_MAP_SHUFFLE                                     */
  int32_t shuffle_factor;  /* PixelShuffle factor of SRES_MAP_(UN)SHUFFLE; 0 means 2             */
  int32_t debug_flags;     /* bring-up only: bit1 (2) forces the direct (non-TMA) epilogue, bit4 (16) the runtime-flag
                              instance, bit6 (64) the tap-per-MMA kernel for the n_out == 16 tail conv (bit1 does too)
                              instead of the three-taps-per-MMA one                                                     */
  void* debug_timeline;    /* bring-up only: int64 [grid][16] per-CTA clock stamps, or NULL          */
} sres_conv_args;

/* Output rows per M tile of the convolutions that emit per-tile partial sums for (H,W) images: 128 for every geometry.
 * pool_part is indexed [tile][segment][lane quarter][64] with tile = first output row / sres_conv_tile_rows.    */
SRES_API int sres_conv_tile_rows(int H, int W);
/* Number of M tiles of a (B,H,W) batch (size of pool_part's leading dim). */
SRES_API int sres_conv_mtiles(int B, int H, int W);
/* 1 when a (H,W) image fits the tensor-core kernel's shared-memory halo window for n_out outputs, else 0 */
SRES_API int sres_conv_supported(int H, int W, int n_out);
SRES_API int sres_conv3x3_igemm(const sres_conv_args* args, void* stream);

/* Two dependent identity-mapped 64 -> 64 convolutions in ONE persistent launch: the second reads the first's bf16 output
 * (a2->in_bf16 == a1->out_bf16), tile by tile behind per-tile ready counters, so one pipeline fill / drain and the wave
 * quantisation are paid once per pair.  Supported pairs (sres_conv_pair_supported): RCAB forward conv1 (bias, ReLU) ->
 * conv2 (bias, SRES_EPI_POOL), network.py:55-59; RCAB backward dgrad(conv2) (ReLU mask) -> dgrad(conv1) (fp32
 * read-modify-write, SRES_EPI_DOT).  flags: sres_conv_pair_flag_bytes() bytes of device memory, zero-filled ONCE (the
 * counters reset themselves); do not share one flag buffer between launches that may overlap.                          */
SRES_API size_t sres_conv_pair_flag_bytes(int B, int H, int W);
SRES_API int sres_conv_pair_supported(const sres_conv_args* first, const sres_conv_args* second);
SRES_API int sres_conv3x3_pair(const sres_conv_args* first, const sres_conv_args* second, void* flags, void* stream);

/* Repack fp32 OIHW 3x3 weights (the checkpoint layout, state_dict of nn.Conv2d) to the bf16
 * tap-major operand the tensor-core kernels read.
 *   mode 0 (forward):   out[t][n][k] = w[oc(n)][k][ky][kx],              t = ky*3+kx
 *   mode 1 (dgrad):     out[t][n][k] = w[oc(k)][n][2-ky][2-kx]           (transposed, flipped)
 *   oc(c) = c*oc_stride + oc_offset   (PixelShuffle sub-convs: oc_stride 4, oc_offset 2i+j)
 *   n_rows = rows of the packed operand (64, or 16 with zero rows beyond the real ones);
 *   cin = input channels of w (64);  cout_total = output channels of w.                      */
SRES_API int sres_pack_conv_weights(const float* w_oihw, void* out_bf16, int mode, int n_rows, int cin,
                           int cout_total, int oc_stride, int oc_offset, void* stream);

/* ------------------------------------------------------------------------------------------ */
/* 3x3 convolution weight + bias gradient (split-K tcgen05 GEMM + deterministic reduce)       */
/* replaces the grad_weight / grad_bias outputs of aten::convolution_backward for the same    */
/* nn.Conv2d modules, reached from mloss.backward() (sres/controller/dual_trainer.py:322).     */
/*   x_bf16  [rows][64] bf16 PTL, the conv input;  dy_bf16 [rows][64] bf16 PTL, grad of output */
/*   dw_oihw fp32 (cout_total, 64, 3, 3); channel n of dy maps to oc = n*oc_stride+oc_offset   */
/*   dbias   fp32 (cout_total) or NULL;  accumulate != 0 adds into dw/dbias instead of storing */
/*   workspace: at least sres_conv_wgrad_workspace_bytes() bytes of device memory              */
/* ------------------------------------------------------------------------------------------ */
SRES_API size_t sres_conv_wgrad_workspace_bytes(void);
/* Several independent weight gradients of the same geometry in ONE launch (split-K CTAs are divided
 * between the jobs; fewer partials per job, one prologue / accumulator drain per batch).            */
#define SRES_WGRAD_MAX_JOBS 8
typedef struct sres_wgrad_job {
  const void* x_bf16;      /* conv input, bf16 PTL                                               */
  const void* dy_bf16;     /* gradient of the conv output, bf16 PTL                              */
  float* dw_oihw;          /* fp32 (cout_total, 64, 3, 3)                                        */
  float* dbias;            /* fp32 (cout_total) or NULL                                          */
  int32_t cout_total, oc_stride, oc_offset, accumulate;   /* cout_total >= 1, oc_stride >= 1, 0 <= oc_offset < oc_stride */
  float scale;             /* result multiplier (1 for a plain conv; EDSR's res_scale for conv2) */
} sres_wgrad_job;
SRES_API int sres_conv3x3_wgrad_batch(const sres_wgrad_job* jobs, int njobs, int B, int H, int W, void* workspace,
                                      size_t workspace_bytes, void* stream);
SRES_API int sres_conv3x3_wgrad(const void* x_bf16, const void* dy_bf16, int B, int H, int W, float* dw_oihw,
                                float* dbias, int cout_total, int oc_stride, int oc_offset, int accumulate,
                                void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------------ */
/* Narrow 3x3 convolutions at the ends of the network (CUDA cores, HBM-bound)                 */
/* ------------------------------------------------------------------------------------------ */
/* Cs = 1..16 image channels in all five entry points below (SRES_ERR_UNSUPPORTED beyond).
 * planar fp32 (B,Cs,H,W)  ->  64-feature PTL rows (fp32 and/or bf16).
 *   transposed == 0: w (64,Cs,3,3) + bias: the head conv forward (sres/model/rcan/network.py:13,23)
 *   transposed == 1: w (Cs,64,3,3): input-gradient of the tail conv 64->Cs (network.py:16)
 *   unshuffle  > 1 : store with PixelUnshuffle(unshuffle) addressing (sub-grid-major PTL)          */
SRES_API int sres_conv3x3_small_in(const float* in_nchw, const float* w, const float* bias, int B, int Cs, int H,
                                   int W, int transposed, int unshuffle, float* out_f32, void* out_bf16,
                                   void* stream);
/* tail conv forward 64 -> Cs on CUDA cores (bf16 PTL in, planar fp32 out): the path for images too wide for the
 * tensor-core kernel's halo window; w (Cs,64,3,3)                                                       */
SRES_API int sres_conv3x3_small_out(const void* u_bf16, const float* w, const float* bias, int B, int Cs, int H, int W,
                                    float* out_nchw, void* stream);
/* workspace of the two weight gradients below, for any Cs (channel chunks run in stream order and reuse it) */
SRES_API size_t sres_small_wgrad_workspace_bytes(void);
/* head conv weight/bias gradient; the output gradient is g1 (+ g2 when not NULL), fp32 PTL      */
SRES_API int sres_small_in_wgrad(const float* g1_f32, const float* g2_f32, const float* in_nchw, int B, int Cs,
                                 int H, int W, float* dw, float* db, int accumulate, void* workspace,
                                 size_t workspace_bytes, void* stream);
/* tail conv weight/bias gradient from the planar output gradient and the bf16 PTL conv input    */
SRES_API int sres_small_out_wgrad(const float* dout_nchw, const void* u_bf16, int B, int Cs, int H, int W,
                                  float* dw, float* db, int accumulate, void* workspace, size_t workspace_bytes,
                                  void* stream);

/* ------------------------------------------------------------------------------------------ */
/* Channel attention + RCAB residual  (sres/model/rcan/network.py:31-47 CALayer, :61-64 RCAB)  */
/*   w1 (hidden,64) b1 (hidden) = conv_du.0 ; w2 (64,hidden) b2 (64) = conv_du.2               */
/* ------------------------------------------------------------------------------------------ */
SRES_API int sres_ca_blocks_per_image(int B, int H, int W);
/* per-image channel sums of a bf16 PTL tensor -> pool_sum [B][64] (small images only)          */
SRES_API int sres_ca_pool(const void* t2_bf16, float* pool_sum, int B, int H, int W, void* stream);
/* x_out = x_in + t2 * sigmoid(MLP(mean(t2)));  xb_out = bf16(x_out);  saves mean and scale [B][64].
 * The pooled sums come either from the conv epilogue partials (pool_part) or from pool_sum.      */
SRES_API int sres_ca_apply_fwd(const void* t2_bf16, const float* pool_part, const float* pool_sum, const float* w1,
                               const float* b1, const float* w2, const float* b2, int hidden, const float* x_in,
                               float* x_out, void* xb_out_bf16, float* save_mean, float* save_s, int B, int H, int W,
                               void* stream);
/* backward of the above w.r.t. t2: dt2 (bf16 PTL) from the fp32 trunk gradient; saves ds [B][64];
 * ds_part: scratch [B][sres_ca_blocks_per_image][64] floats                                       */
SRES_API int sres_ca_bwd(const float* grad_f32, const void* t2_bf16, const float* w1, const float* b1,
                         const float* w2, const float* b2, int hidden, const float* save_mean, float* ds_part,
                         void* dt2_bf16, float* save_ds, int B, int H, int W, void* stream);
/* same, when ds = sum(g * t2) was already reduced per M tile by the convolution that produced g
 * (SRES_EPI_DOT): tile_part has the layout of pool_part                                             */
SRES_API int sres_ca_bwd_apply(const float* grad_f32, const float* tile_part, const float* w1, const float* b1,
                               const float* w2, const float* b2, int hidden, const float* save_mean, void* dt2_bf16,
                               float* save_ds, int B, int H, int W, void* stream);
/* parameter gradients of `nlayers` CALayers whose parameters sit layer_stride floats apart;
 * scratch: sres_ca_param_grads_scratch_bytes(nlayers, B) bytes of device memory                   */
SRES_API size_t sres_ca_param_grads_scratch_bytes(int nlayers, int B);
SRES_API int sres_ca_param_grads(const float* params_first, float* grads_first, int64_t layer_stride, int nlayers,
                                 const float* save_mean, const float* save_ds, int B, int hidden, int accumulate,
                                 void* scratch, size_t scratch_bytes, void* stream);

/* ------------------------------------------------------------------------------------------ */
/* Bicubic resize = F.interpolate(mode="bicubic", align_corners=False)                         */
/*   sres/base/util/array.py:72-76 (downsample, scale = s) and :84-87 (upsample, scale = 1/s)  */
/* ------------------------------------------------------------------------------------------ */
SRES_API int sres_bicubic_resize(const float* in, float* out, int planes, int Hi, int Wi, int Ho, int Wo,
                                 double scale_h, double scale_w, void* stream);

/* ------------------------------------------------------------------------------------------ */
/* Resize in any mode the reference's task.downsample_mode / upsample_mode can name            */
/*   sres/base/util/array.py:37-41 (torch_interp_mode: linear -> bilinear, cubic -> bicubic,    */
/*   every other name passed through), :72-76 (downsample) and :84-87 (upsample):              */
/*   F.interpolate(t, scale_factor=..., mode=...) on 4-D fp32 NCHW, align_corners=False, no     */
/*   antialias.  planes = N*C; (Ho,Wo) = floor((Hi,Wi) * scale_factor) as F.interpolate sizes   */
/*   it; scale_h / scale_w = 1 / scale_factor (positive, finite; SRES_RESIZE_AREA ignores them:  */
/*   adaptive_avg_pool2d to (Ho,Wo), output o averages input [floor(o*in/out), ceil((o+1)*in/out))). */
/*   SRES_RESIZE_BICUBIC runs the sres_bicubic_resize kernel.  Null pointers, sizes <= 0, an    */
/*   unknown mode or a bad scale return SRES_ERR_INVALID_ARG before anything is enqueued.       */
/* ------------------------------------------------------------------------------------------ */
#define SRES_RESIZE_NEAREST 0        /* "nearest":       src = min(floor(dst*scale), in-1) (1:1 copy, 2x shift) */
#define SRES_RESIZE_NEAREST_EXACT 1  /* "nearest-exact": src = min(floor((dst+0.5)*scale), in-1)              */
#define SRES_RESIZE_BILINEAR 2       /* "bilinear" ("linear"): src = max(scale*(dst+0.5)-0.5, 0), two taps    */
#define SRES_RESIZE_BICUBIC 3        /* "bicubic" ("cubic"): the kernel above                                 */
#define SRES_RESIZE_AREA 4           /* "area": block mean (adaptive average pool)                            */
SRES_API int sres_resize(const float* in, float* out, int planes, int Hi, int Wi, int Ho, int Wo, double scale_h,
                         double scale_w, int mode, void* stream);

/* ------------------------------------------------------------------------------------------ */
/* Losses: kind 0 = l2 / RMSE (sres/controller/stats.py:5-8), 1 = charbonnier                  */
/* (sres/controller/dual_trainer.py:196-198), 2 = l1 (BASELINE north_star variant).            */
/* The target plane (tH,tW) may exceed the product's (H,W): conform_to_product,                */
/* dual_trainer.py:200-203.  stat: device double[2]; stat[0] = sum_i f(d_i) and stat[1] = number */
/* of elements of THIS rank -- a data-parallel caller all-reduces both (sum) and passes          */
/* n_total_dev = stat + 1, so ranks with batches of different sizes agree on the global-batch    */
/* loss (SURVEY.md 8e).  n_total_dev == NULL: the element count is the host value n_total.       */
/* ------------------------------------------------------------------------------------------ */
SRES_API size_t sres_loss_workspace_bytes(void);
SRES_API int sres_loss_sum(const float* prd, const float* tgt, int planes, int H, int W, int tH, int tW, int kind,
                           double* stat, void* workspace, size_t workspace_bytes, void* stream);
SRES_API int sres_loss_value(const double* stat, double n_total, const double* n_total_dev, int kind, float* loss,
                             void* stream);
SRES_API int sres_loss_grad(const float* prd, const float* tgt, int planes, int H, int W, int tH, int tW, int kind,
                            const float* loss, double n_total, const double* n_total_dev, float gscale,
                            const float* gscale_dev, float* grad,
                            void* stream); /* upstream factor = gscale * (gscale_dev ? *gscale_dev : 1) */

/* ------------------------------------------------------------------------------------------ */
/* Fused Adam over flat fp32 buffers = torch.optim.Adam(lr, betas, eps, weight_decay).step()   */
/*   sres/controller/dual_trainer.py:126, :323.  n % 4 == 0, 16-byte aligned.                  */
/* ------------------------------------------------------------------------------------------ */
SRES_API int sres_adam_step_flat(float* p, const float* g, float* m, float* v, int64_t n, int64_t step, double lr,
                                 double beta1, double beta2, double eps, double weight_decay, void* stream);

/* ------------------------------------------------------------------------------------------ */
/* Whole network: RCAN forward / backward  (sres/model/rcan/network.py:9-27)                   */
/*   and EDSR through the same entry points (sres/model/edsr/network.py:9-32: head conv,       */
/*   n_blocks x ResBlock(conv, ReLU, conv, *res_scale, +x) common/residual.py:30-54, conv,      */
/*   +head, SPUpsample common/upsample.py:34-66, conv)                                          */
/* ------------------------------------------------------------------------------------------ */
#define SRES_ARCH_RCAN 0
#define SRES_ARCH_EDSR 1
typedef struct sres_rcan_desc {
  int32_t B, H, W;         /* low-resolution tile batch                                         */
  int32_t cin, cout;       /* image channels, 1..16 each (nchannels_in / nchannels_out, manager.py:52) */
  int32_t nfeatures;       /* 64                                                                 */
  int32_t n_groups;        /* nlayers  (residual groups)                                         */
  int32_t n_blocks;        /* nblocks  (RCABs per group)                                         */
  int32_t reduction;       /* cbottleneck                                                        */
  int32_t n_up;            /* upsampler stages                                                   */
  int32_t up_factor[4];    /* PixelShuffle factor of each stage: 2,2 for x4; 3 for x3            */
  int32_t arch;            /* SRES_ARCH_RCAN (0) or SRES_ARCH_EDSR: n_groups = 1, n_blocks = nlayers, */
                           /* reduction ignored                                                  */
  float res_scale;         /* EDSR only: ResBlock residual scaling (edsr.yaml res_scale)         */
} sres_rcan_desc;

/* Parameters / gradients are ONE flat fp32 buffer in the reference's state_dict order.        */
SRES_API int64_t sres_rcan_param_count(const sres_rcan_desc* d);
/* Workspace size.  The workspace must be zero-filled once before first use (padding rows of the
 * PixelUnshuffle-layout gradient buffers are never written) and must persist from forward to
 * backward in training mode.                                                                   */
SRES_API int sres_rcan_workspace_bytes(const sres_rcan_desc* d, int training, size_t* bytes);
/* Re-derive the bf16 tensor-core operands from the fp32 parameters (after every update).       */
SRES_API int sres_rcan_pack_weights(const sres_rcan_desc* d, const float* params, void* workspace, int training,
                                    void* stream);
/* x (B,cin,H,W) fp32 -> out (B,cout,H*s,W*s) fp32.  training != 0 keeps activations for backward. */
SRES_API int sres_rcan_forward(const sres_rcan_desc* d, const float* params, const float* x_nchw, float* out_nchw,
                               void* workspace, int training, void* stream);
/* Backward in segments [seg_begin, seg_end): 0 = tail + upsampler + body-tail conv,
 * 1..G = residual groups G-1..0 (EDSR: 1 = all ResBlocks), G+1 = head conv.  Each segment completes the gradients of the
 * parameter range reported by sres_rcan_segment_params, so a data-parallel caller can start
 * the all-reduce of that range while the next segment runs.                                     */
SRES_API int sres_rcan_num_segments(const sres_rcan_desc* d);
SRES_API int sres_rcan_segment_params(const sres_rcan_desc* d, int seg, int64_t* offset, int64_t* count);
/* async_ctx (optional, from sres_async_create; NULL = everything on `stream`): a side stream + events owned by the
 * caller on which the weight-gradient batches run beside the input-gradient chain; every segment joins it back
 * into `stream` before returning, so stream order (and CUDA-graph capture of `stream`) still covers all work.   */
SRES_API int sres_async_create(void** ctx);
SRES_API int sres_async_destroy(void* ctx);
SRES_API int sres_rcan_backward(const sres_rcan_desc* d, const float* params, const float* x_nchw,
                                const float* dout_nchw, float* grads, int accumulate, void* workspace, int seg_begin,
                                int seg_end, void* async_ctx, void* stream);

/* ------------------------------------------------------------------------------------------ */
/* Tile extraction / normalisation / stitching (index-exact data movement around the model)   */
/*   region (C,Y,X) fp32; tile grid gy x gx of T x T tiles starting at (y0,x0)                 */
/*   (sres/data/tiles.py:110-127).  A "candidate" tile index is c*gy*gx + ty*gx + tx.          */
/* ------------------------------------------------------------------------------------------ */
/* flags[cand] = 1 when every element of the candidate tile is finite -- the survivors of the
 * reference's NaN-tile drop, isfinite(tile.mean(-1).mean(-1)) (sres/base/source/swot/raw.py:226) */
SRES_API int sres_tiles_finite_flags(const float* region, int C, int Y, int X, int y0, int x0, int T, int gy, int gx,
                                     int32_t* flags, void* stream);
/* out[slot] (T x T) = candidate tile src_tile[slot]; slot = n*C + c of the (N,C,T,T) result
 * (raw.py:216-233; the table encodes the reference's channel-major order or the corrected one)  */
SRES_API int sres_tiles_gather(const float* region, int C, int Y, int X, int y0, int x0, int T, int gy, int gx,
                               const int32_t* src_tile, int nslots, float* out, void* stream);
/* per plane (x-mean)/std, NaN-skipping, population std (raw.py:176-183), with the xyflip
 * orientation flip_index = 0..7 (bit0 flip x, bit1 flip y, bit2 transpose; source/batch.py:37-49)
 * fused into the store; mean/std [nplanes] are returned for denorm                               */
SRES_API int sres_tiles_lnorm(const float* in, int nplanes, int T, int flip_index, float* out, float* mean,
                              float* std_, void* stream);
/* image (gy*t, gx*t) of variable ivar: tile cell_to_tile[cy*gx+cx] (or NaN when < 0), optionally
 * de-normalised x*std+mean (sres/controller/dual_trainer.py:449-480 assemble_images, :67-77 denorm) */
SRES_API int sres_tiles_stitch(const float* tiles, int C, int ivar, int t, int gy, int gx, const int32_t* cell_to_tile,
                               const float* mean, const float* std_, float* out, void* stream);

/* Rectangular tiles (task.tile_size {x, y} with x != y; sres/data/tiles.py:110-127 and raw.py:216-233 treat the two
 * axes separately).  Same contracts as the square entry points above, which are these with Th = Tw = T.        */
/* candidate tile (c, ty, tx) starts at (y0 + ty*Th, x0 + tx*Tw); the grid must fit the region on each axis      */
SRES_API int sres_tiles_finite_flags_hw(const float* region, int C, int Y, int X, int y0, int x0, int Th, int Tw, int gy,
                                        int gx, int32_t* flags, void* stream);
/* out[slot] (Th x Tw) = candidate tile src_tile[slot]; slot = n*C + c of the (N,C,Th,Tw) result                */
SRES_API int sres_tiles_gather_hw(const float* region, int C, int Y, int X, int y0, int x0, int Th, int Tw, int gy, int gx,
                                  const int32_t* src_tile, int nslots, float* out, void* stream);
/* in: nplanes Th x Tw planes.  Flips 0-3 write Th x Tw planes, out[r][c] = in[fy(r)][fx(c)]; flips 4-7 write
 * Tw x Th planes, out[r][c] = in[fy(c)][fx(r)] (the reference flips x, then y, then swapaxes(-1,-2);
 * source/batch.py:37-49), with fy(j) = (flip & 2) ? Th-1-j : j and fx(i) = (flip & 1) ? Tw-1-i : i.
 * Statistics as sres_tiles_lnorm.  In-place only with flip_index 0.                                           */
SRES_API int sres_tiles_lnorm_hw(const float* in, int nplanes, int Th, int Tw, int flip_index, float* out, float* mean,
                                 float* std_, void* stream);
/* tiles (N,C,th,tw) -> image (gy*th, gx*tw) of variable ivar; tile cell_to_tile[cy*gx+cx] lands at rows
 * [cy*th, (cy+1)*th) and columns [cx*tw, (cx+1)*tw) (dual_trainer.py:449-480), NaN when < 0                   */
SRES_API int sres_tiles_stitch_hw(const float* tiles, int C, int ivar, int th, int tw, int gy, int gx,
                                  const int32_t* cell_to_tile, const float* mean, const float* std_, float* out,
                                  void* stream);

/* ------------------------------------------------------------------------------------------ */
/* Raw LLC4320 fields -> region of interest (the reference's file reader, SURVEY.md 8f rank 4)  */
/*   sres/base/source/swot/raw.py:133-145 load_file: big-endian f4 ocean-only ("shrunk") file,  */
/*   scattered through the template's land mask (template != 0), land = NaN, LLC faces unfolded */
/*   by mds2d (sres/base/source/swot/util.py:3-55) into (3 nx, 4 nx), cropped by subset_roi      */
/*   (raw.py:38-45).  The template is digested once into a gather index of the region; a file   */
/*   then costs one host->device copy of its bytes and one gather kernel.                       */
/* ------------------------------------------------------------------------------------------ */
SRES_API size_t sres_llc_index_workspace_bytes(int nx);
/* template_be: the 13 nx^2 big-endian floats of the template file, on the device (raw bytes).
 * roi_index [ys*xs] int32: position of the pixel's value in a shrunk file, -1 for land.
 * n_ocean_dev: device int64, number of ocean points = number of floats a shrunk file holds.     */
SRES_API int sres_llc_build_roi_index(const void* template_be, int nx, int y0, int ys, int x0, int xs, void* workspace,
                                      size_t workspace_bytes, int32_t* roi_index, int64_t* n_ocean_dev, void* stream);
/* data_be: the n_data big-endian floats of one shrunk file, on the device (raw bytes); out [npix] fp32. */
SRES_API int sres_llc_gather_roi(const void* data_be, int64_t n_data, const int32_t* roi_index, int64_t npix, float* out,
                                 void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SRES_B200_H_ */
