/*
 * dust3r_b200 — C ABI of the B200-native DUSt3R hot paths (sm_100a).
 *
 * The reference (naver/dust3r) has no FFI/plugin registry; its only native entry point is the
 * pybind function `curope.rope_2d` (croco/models/curope/curope.cpp:49-69).  Everything else on
 * the two hot paths is Python calling torch.  This header is therefore the boundary a
 * maintainer binds with ctypes (see INTEGRATION.md): plain pointers + sizes + a cudaStream_t,
 * int return codes, no torch / ATen / Python types.
 *
 * Conventions
 *   - every pointer marked `dev` is a CUDA device pointer owned by the caller (PyTorch owns all
 *     memory; the library never allocates caller-visible memory);
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - return value 0 = success, negative = error; d3r_last_error() gives the message of the
 *     last failure on the calling thread;
 *   - calls are asynchronous w.r.t. the host unless stated; thread-safe for distinct streams.
 */
#ifndef DUST3R_B200_H_
#define DUST3R_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define D3R_OK 0
#define D3R_ERR_INVALID (-1)   /* bad argument / unsupported shape   */
#define D3R_ERR_CUDA (-2)      /* CUDA runtime / driver error        */
#define D3R_ERR_UNSUPPORTED_DEVICE (-3)

const char* d3r_last_error(void);
/* ABI version of this header; bumped on any signature change. */
int d3r_abi_version(void);
/* 0 when the current device is sm_100 (B200); D3R_ERR_UNSUPPORTED_DEVICE otherwise. */
int d3r_check_device(void);

/* Launch accounting / profiling aid: number of kernels this library launched since the last reset;
 * with d3r_prof_enable(1) every launch is bracketed by CUDA events on its stream and
 * d3r_prof_report() returns a JSON object {tag: {count, ms, flops, bytes}} (returns length, -1 if
 * the buffer is too small). */
long long d3r_launch_count(void);
void d3r_launch_count_reset(void);
void d3r_prof_enable(int on);
int d3r_prof_report(char* buf, int cap);
/* every recorded launch in order: JSON list [{tag, detail, ms, flops, bytes}] (length, or -1 if it does not fit) */
int d3r_prof_dump(char* buf, int cap);

/* ------------------------------------------------------------------------------------------
 * Path 2 — global alignment (replaces the body of global_alignment_iter(),
 * dust3r/cloud_opt/base_opt.py:352-366: zero_grad + PointCloudOptimizer.forward
 * (optimizer.py:188-201) or BasePCOptimizer.forward (base_opt.py:246-273) + loss.backward() +
 * torch.optim.Adam.step(), for every iteration of global_alignment_loop, base_opt.py:326-349).
 *
 * One launch per iteration: unproject depth -> 3D, confidence-weighted pairwise distance,
 * analytic backward, Adam on the per-pixel log-depths; the last CTA folds the per-edge /
 * per-image partial sums into pose / focal / principal-point / pairwise-pose gradients, applies
 * Adam to them and refreshes the transforms for the next launch.
 * ------------------------------------------------------------------------------------------ */

/* Small parameters live in ONE float buffer `small` (and two more of the same layout for Adam's
 * exp_avg / exp_avg_sq, plus a uint8 buffer of trainable flags):
 *   [ im_poses n*7 | im_focals n*2 | im_pp n*2 | pw_poses E*8 | pw_adaptors E*2 ]
 * im_poses / pw_poses rows are [qx,qy,qz,qw, tx,ty,tz(, log_scale)] exactly as
 * optimizer.py:30 / base_opt.py:90 store them; im_focals holds focal_break*log(f) twice when the
 * model has a single focal (fx == fy, tied). */
typedef struct d3r_align_desc {
  int32_t n_imgs;          /* n                                                             */
  int32_t n_edges;         /* E (directed edges, base_opt.py:61)                            */
  int32_t n_entries;       /* 2*E : one entry per (edge, side)                              */
  int32_t n_chunks;        /* total CTAs = sum_i ceil(P_i / chunk_px)                       */
  int32_t max_deg;         /* max entries incident to one image                             */
  int32_t max_chunks;      /* max CTAs of one image                                         */
  int32_t chunk_px;        /* pixels per CTA, 1..d3r_align_chunk_pixels() (host picks it so
                              the grid is a whole number of waves)                          */
  int32_t dist_l2;         /* 0: l1_dist, 1: l2_dist (commons.py:62-70)                     */
  int32_t norm_pw_scale;   /* base_opt.py:86,178-184                                        */
  int32_t tied_focal;      /* 1: one focal per image (fx==fy), 0: fx_and_fy                 */
  int32_t eval_only;       /* 1: only write the loss (net.forward()), no parameter update   */
  float base_scale;        /* base_opt.py:49                                                */
  float pw_break;          /* base_opt.py:51                                                */
  float focal_break;       /* optimizer.py:22 / modular_optimizer.py:24 (focal_brake)       */
  float adam_eps;          /* 1e-8                                                          */
  float beta1, beta2;      /* (0.9, 0.9) base_opt.py:337                                    */

  /* per image (dev) */
  const int32_t* img_hw;        /* [n][2] = H, W                                            */
  const int64_t* img_pix_off;   /* [n+1] offset of image i's pixels in logd / adam buffers  */
  const int32_t* img_ent_ptr;   /* [n+1] CSR into the entry arrays                          */
  const int32_t* img_chunk_ptr; /* [n+1] first CTA index of image i                         */
  /* per CTA (dev) */
  const int32_t* chunk_img;     /* [n_chunks] image handled by CTA c                        */
  /* per entry, CSR order (dev) */
  const int32_t* ent_edge;      /* [2E] edge id                                             */
  const int64_t* ent_obs_off;   /* [2E] offset (in float4) of the entry's observations      */
  const float*   ent_coef;      /* [2E] loss coefficient: 1/total_area (stacked) or 1/(P*E) */
  const int32_t* edge_ent;      /* [E][2] entry index of (edge, side i) and (edge, side j)  */
  /* observations (dev): float4 = (pred.x, pred.y, pred.z, weight) per pixel per entry.
   * 32*E*P bytes in total = the read-once traffic of SURVEY §8d.                          */
  const void* obs;

  /* trainable state (dev) */
  float* logd;                  /* [sum P_i] log-depth, optimizer.py:29                     */
  float* logd_m;                /* Adam exp_avg                                             */
  float* logd_v;                /* Adam exp_avg_sq                                          */
  float* small;                 /* layout above                                             */
  float* small_m;
  float* small_v;
  const uint8_t* small_trainable; /* same layout, 1 = requires_grad                         */

  /* derived per-iteration state + scratch (dev), sizes from d3r_align_workspace_floats()  */
  float* workspace;
  /* [niter_total][4] = lr, lr/bias_correction1, sqrt(bias_correction2), 0 for every step   */
  const float* sched;
  float* loss_out;              /* [niter_total] loss of every iteration                    */
  int32_t* counters;            /* [n + 2] zero-initialised by the caller once              */
  /* `workspace` must be zero-initialised by the caller once as well (accumulators live there).  */

  /* ---- streaming kernel (csrc/align_stream.cu), used when every image has P % 4 == 0 and a pixel stride
   * that is a multiple of 4 (always true for DUSt3R inputs: H, W are multiples of the 16-pixel patch).
   * stream_kernel = 1 selects it; obs then holds the slot-interleaved layout written by
   * d3r_align_pack_obs_stream (same 16 bytes per observation):
   *   per entry: slots of 64 pixels = [32 x (xA,xB,yA,yB)] [32 x (zA,zB,wA,wB)] for the 32 pixel pairs
   *   (A,B) = (2j, 2j+1) of the slot, the loss coefficient folded into w; every image's slab is padded to
   *   whole slots with w = 0.
   * The pixel range of every image is cut into work items of <= ppt slots; persistent warp w owns items
   * [warp_item_ptr[w], warp_item_ptr[w+1]).                                                           */
  int32_t stream_kernel;
  int32_t stream_grid;          /* CTAs of the persistent grid                                       */
  int32_t stream_ppt;           /* slots (64 pixels) per work item, 2..4                              */
  int32_t stream_window;        /* entries whose partial sums a warp keeps in shared memory            */
  int32_t n_items;
  int32_t reserved0;
  const void* items;            /* [n_items] d3r_align_item                                            */
  const int32_t* warp_item_ptr; /* [stream_grid * 8 + 1]                                               */
  /* Optional second traversal of the same items in REVERSE global order (items_rev[k] = items[n_items-1-k],
   * with its own warp split).  When set, odd iterations walk it: what an iteration streamed last is what
   * the next one streams first, so the tail of every pass is still resident in the 126 MB L2 (observations
   * are constants of the problem).  NULL = every iteration walks `items`.                              */
  const void* items_rev;
  const int32_t* warp_item_ptr_rev;
} d3r_align_desc;

/* One work item of the streaming kernel: `nslots` consecutive 64-pixel slots of image `img`. */
typedef struct d3r_align_item {
  int32_t img, slot0, nslots, npx;     /* npx: valid pixels of the item (multiple of 4)               */
  int32_t e0, deg, W, u0;              /* first entry / number of entries of the image; width; column of the first pixel */
  int32_t v0;                          /* row of the first pixel                                      */
  float inv_w;                         /* 1 / W                                                       */
  int64_t pix0;                        /* img_pix_off[img] + 64 * slot0: index into logd / adam moments */
  int64_t obs0;                        /* 16-byte units: first entry's slab of the image + 64 * slot0   */
  int32_t slab_units;                  /* 16-byte units per entry slab of this image (64 * slots)      */
  int32_t reserved;
} d3r_align_item;

/* sizeof(d3r_align_desc) / sizeof(d3r_align_item) as compiled into the library (binding self-check). */
int d3r_sizeof_align_desc(void);
int d3r_sizeof_align_item(void);
/* Maximum pixels one CTA of the alignment kernel can take (compile-time constant of the library). */
int d3r_align_chunk_pixels(void);
/* Number of floats of `workspace` needed for a problem of this size. */
int64_t d3r_align_workspace_floats(int32_t n_imgs, int32_t n_edges, int32_t n_chunks, int32_t max_chunks);
/* Computes the transforms used by the first iteration from `small` (call once after the
 * parameters are (re)initialised or modified from the host). */
int d3r_align_prepare(const d3r_align_desc* desc, void* stream);
/* Runs iterations [it_begin, it_end) (indices into sched / loss_out).  Asynchronous. */
int d3r_align_run(const d3r_align_desc* desc, int32_t it_begin, int32_t it_end, void* stream);
/* Cross-CTA sums use order-independent 2^40 fixed-point integer atomics (bit-reproducible).  *host_out = 1 when a
 * partial sum (|x| >= 2^18) or a total (|x| >= 2^22) left the supported range (unreasonably scaled scene, NaN / Inf input)
 * since iteration 0 of the current d3r_align_run batch. */
int d3r_align_overflow_flag(const d3r_align_desc* desc, int32_t* host_out, void* stream);
/* World-frame pointmaps X[i] = R_i * unproject(depth_i) + T_i for every image
 * (PointCloudOptimizer.depth_to_pts3d, optimizer.py:170-180).  out: [sum P_i][3] float. */
int d3r_align_pts3d(const d3r_align_desc* desc, float* out_dev, void* stream);
/* Debug aid: when dev_buf != NULL every CTA of the next alignment launches writes 4 uint64 %globaltimer stamps
 * (start, end of pixel phase, end/exit, end of small-parameter step) at dev_buf[4*cta]. */
int d3r_align_set_debug(void* dev_buf);
/* Packs pred (P,3) + weight (P) rows into the float4 observation layout. */
int d3r_align_pack_obs(const float* pts_dev, const float* weight_dev, void* obs_dev, int64_t obs_off,
                       int64_t n_pix, void* stream);

/* Packs EVERY entry's observations in one launch, straight from the (device-resident) output of the forward:
 * replaces the ParameterStack copies + conf_trf of optimizer.py:50-57 / base_opt.py:72-75.  `table` (dev) has one
 * row per entry; the confidence transform (commons.py:73-80: D3R_CONF_ID / LOG / SQRT / M1) is applied on the fly.
 * stream_layout = 0: plain float4 (x, y, z, w) rows; 1: the slot-interleaved layout of the streaming kernel, the
 * loss coefficient folded into w and slabs padded to whole 64-pixel slots with zeros. */
#define D3R_CONF_ID 0
#define D3R_CONF_LOG 1
#define D3R_CONF_SQRT 2
#define D3R_CONF_M1 3
typedef struct d3r_pack_entry {
  const float* pts;        /* dev: (area, 3) pointmap of the entry                                       */
  const float* conf;       /* dev: (area) raw confidence                                                  */
  int64_t obs_off;         /* float4 units: where the entry's slab starts in obs                          */
  int32_t area;            /* pixels of the entry                                                         */
  float coef;              /* loss coefficient of the entry (folded into w when stream_layout = 1)        */
} d3r_pack_entry;
int d3r_sizeof_pack_entry(void);
/* Compile-time constants of the streaming kernel the host needs to build the work-item table: slots (64 pixels) per
 * item, persistent warps per CTA, and the largest entry window for which two CTAs still fit one SM. */
int d3r_align_stream_slots_per_item(void);
int d3r_align_stream_warps_per_cta(void);
int d3r_align_stream_max_window(void);
int d3r_align_pack_entries(const d3r_pack_entry* table_dev, int32_t n_entries, int32_t max_area, int32_t conf_mode,
                           int32_t stream_layout, void* obs_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Path 1 building blocks — exported so the parity tests can exercise each kernel in isolation.
 * Integrators use d3r_forward_* below; these are the ops it is composed of.
 * ------------------------------------------------------------------------------------------ */

/* epilogue flags of d3r_gemm_bf16 / d3r_conv3x3_bf16 */
#define D3R_F_BIAS          (1u << 0)
#define D3R_F_GELU          (1u << 1)   /* exact erf GELU (croco/models/blocks.py Mlp act_layer=nn.GELU) */
#define D3R_F_RELU          (1u << 2)
#define D3R_F_OUT_F32       (1u << 3)
#define D3R_F_RESID_INPLACE (1u << 4)   /* out(f32) += result : residual stream update                   */
#define D3R_F_ADD0          (1u << 5)
#define D3R_F_ADD1          (1u << 6)
#define D3R_F_OUT2_RELU     (1u << 7)
#define D3R_F_ROPE          (1u << 8)   /* 2D RoPE on columns < rope_cols; replaces curope.rope_2d        */
#define D3R_F_OUT2_BF16     (1u << 11)

/* out[M,N] = epilogue(A[M,K] * B[N,K]^T); A, B bf16 row-major (nn.Linear weight layout), tcgen05.
 * N % 32 == 0, K % 8 == 0.  With D3R_F_ROPE: rope_cos/sin are [max_pos][16] fp32 tables
 * (angle = pos * base^(-k/16), croco/models/curope/kernels.cu:41-52), rows are tokens of images of
 * `tokens_per_img` tokens laid out row-major on a grid `grid_w` wide. */
int d3r_gemm_bf16(const void* A_dev, const void* B_dev, void* out_dev, const float* bias_dev, const void* add0_dev,
                  void* out2_dev, int32_t M, int32_t N, int32_t K, int64_t ldo, uint32_t flags,
                  const float* rope_cos_dev, const float* rope_sin_dev, int32_t rope_cols, int32_t tokens_per_img,
                  int32_t grid_w, void* stream);

/* 3x3 stride-1 pad-1 convolution as implicit GEMM on tcgen05.  x: (B,H,W,Cin) bf16 NHWC;
 * w_packed: [Cout][ky*3+kx][Cin] bf16; out/add0/add1/out2: (B,H,W,Cout) bf16 NHWC.
 * (croco/models/dpt_block.py ResidualConvUnit_custom / layer_rn / head convs) */
int d3r_conv3x3_bf16(const void* x_nhwc_dev, const void* w_packed_dev, void* out_dev, const float* bias_dev,
                     const void* add0_dev, const void* add1_dev, void* out2_dev, int32_t B, int32_t H, int32_t W,
                     int32_t Cin, int32_t Cout, uint32_t flags, void* stream);

/* softmax(q k^T * scale) v, head dim 64, bf16 in/out, fp32 softmax (croco/models/blocks.py:94-112,
 * 146-169).  q rows at (b*Nq+i)*ldq + h*64, k/v rows at (b*Nk+j)*ld{k,v} + h*64, out like q.
 * Range: the exponent reference of a row moves lazily (DESIGN.md section 4); a key whose scaled logit leads the keys before
 * it by 86 or more (natural-log units) overflows fp32 and the row's output is NaN (measured on a B200; finite up to 84). */
int d3r_attention_hd64(const void* q_dev, int64_t ldq, const void* k_dev, int64_t ldk, const void* v_dev, int64_t ldv,
                       void* out_dev, int64_t ldo, int32_t B, int32_t heads, int32_t Nq, int32_t Nk, float scale,
                       void* stream);

/* ConvTranspose2d with kernel == stride == k (act_postprocess 0 / 1, dpt_head.py via croco/models/dpt_block.py) as a
 * GEMM whose epilogue scatters every (ky,kx,co) column to its output pixel.  x: (B,h,w,Cin) bf16 NHWC;
 * w_packed: [(ky*k+kx)*Cout + co][Cin] bf16; bias [Cout] fp32 or NULL; out: (B,h*k,w*k,Cout) bf16 NHWC.
 * Cin % 8 == 0, Cout % 32 == 0 (a 32-column chunk of the epilogue must stay inside one (ky,kx) tap). */
int d3r_convT_bf16(const void* x_nhwc_dev, const void* w_packed_dev, const float* bias_dev, void* out_dev, int32_t B, int32_t h,
                   int32_t w, int32_t Cin, int32_t Cout, int32_t k, void* stream);

/* Last DPT conv with the head tail fused into its epilogue: 3x3 conv 128 -> 128 (+ bias) -> ReLU -> 1x1 conv to 4
 * channels (w4 fp32 [4][128], b4 fp32 [4]; always four rows, row 3 is the confidence logit) -> postprocess
 * (heads/postprocess.py: depth_mode 0 linear, 1 square, 2 exp; conf_mode 0 none, 1 exp, 2 sigmoid, range
 * [conf_min, conf_max]).  x: (B,H,W,128) bf16 NHWC; w_packed: [128][9][128] bf16; pts3d: (B,H,W,3) fp32;
 * conf: (B,H,W) fp32, or NULL for no confidence output (conf_mode is then ignored). */
int d3r_conv3x3_head_tail(const void* x_nhwc_dev, const void* w_packed_dev, const float* bias_dev, const float* w4_dev,
                          const float* b4_dev, float* pts3d_dev, float* conf_dev, int32_t B, int32_t H, int32_t W,
                          int32_t depth_mode, int32_t conf_mode, float conf_min, float conf_max, void* stream);

/* LayerNorm over the last dimension, fp32 in, bf16 out: out[m] = (x[m] - mean) / sqrt(var + eps) * g + b (biased
 * variance, like nn.LayerNorm).  x: [M][C] fp32, g, b: [C] fp32.  C % 4 == 0, C <= 2048. */
int d3r_layernorm_bf16(const float* x_dev, const float* g_dev, const float* b_dev, void* out_dev, int32_t M, int32_t C, float eps,
                       void* stream);

/* Bilinear x2 upsampling with align_corners=True of x (B,H,W,C) bf16 NHWC onto the (2H, 2W) grid, of which the first
 * Ho x Wo pixels are written to out (B,Ho,Wo,C) (Ho <= 2H, Wo <= 2W: the crop of refinenet4, dpt_head.py:57).
 * C % 8 == 0 and C / 8 a power of two. */
int d3r_upsample2x_bf16(const void* x_dev, void* out_dev, int32_t B, int32_t H, int32_t W, int32_t C, int32_t Ho, int32_t Wo,
                        void* stream);

/* im2col of a 3x3 stride-2 pad-1 convolution: x (B,H,W,C) bf16 NHWC -> out [B*Ho*Wo][9][C] bf16 (tap = ky*3+kx, zeros
 * outside the image), Ho = (H-1)/2+1, Wo = (W-1)/2+1.  C % 8 == 0. */
int d3r_im2col_3x3_s2_bf16(const void* x_dev, void* out_dev, int32_t B, int32_t H, int32_t W, int32_t C, void* stream);

/* Patch-embedding im2col, 16 x 16 patches: img (B,3,H,W) fp32 -> out [B*(H/16)*(W/16)][3*16*16] bf16 with column
 * c*256 + py*16 + px (the flattening of the Conv2d weight).  H % 16 == 0, W % 16 == 0. */
int d3r_patch_im2col16(const float* img_dev, void* out_dev, int32_t B, int32_t H, int32_t W, void* stream);

/* Row gather by image: out[i*rows_per_img + r] = in[map[i]*rows_per_img + r] for i < n_out, rows of C bf16.
 * map_dev: int32 [n_out] (device).  C % 8 == 0. */
int d3r_gather_images_bf16(const void* in_dev, void* out_dev, const int32_t* map_dev, int32_t n_out, int32_t rows_per_img,
                           int32_t C, void* stream);

/* fp32 -> bf16, round to nearest even, n elements, n % 4 == 0. */
int d3r_cast_f32_bf16(const float* x_dev, void* out_dev, int64_t n, void* stream);

/* Linear head tail (heads/linear_head.py + postprocess.py): feat [B*gh*gw][nch*256] fp32 (channel-major, then
 * py*16 + px) -> pixel shuffle -> pts3d (B,gh*16,gw*16,3) and, when nch == 4, conf (B,gh*16,gw*16) fp32.  Modes as for
 * d3r_conv3x3_head_tail. */
int d3r_linear_head_postprocess(const float* feat_dev, float* pts3d_dev, float* conf_dev, int32_t B, int32_t gh, int32_t gw,
                                int32_t nch, int32_t depth_mode, int32_t conf_mode, float conf_min, float conf_max, void* stream);

/* Selects the GEMM / conv kernel family: 0 = 1-CTA tcgen05 kernels, 1 = CTA-pair (cta_group::2) kernels,
 * 2 (default) = CTA-pair kernels from 4 k-blocks of 64 on (K >= 256), 1-CTA for shorter reductions. */
void d3r_set_gemm_impl(int32_t impl);
/* Tuning aid for impl 2: minimum number of 64-wide k-blocks for which the CTA-pair kernel is used (default 4). */
void d3r_set_gemm_pair_min_kblocks(int32_t kblocks);

/* Debug aid: per-image timeline stamps (64 x uint64 %globaltimer per traced CTA) of the tcgen05 attention. */
int d3r_attention_set_debug(void* dev_buf);

/* Selects the attention kernel: 3 (default) = tcgen05/TMEM split-row kernel (two warps per 32 query rows, 128-key blocks) with P
 * kept in tensor memory (A-from-TMEM tcgen05.mma); 2 = the same dataflow with P through shared memory (A/B reference). */
void d3r_set_attention_impl(int32_t impl);

/* ------------------------------------------------------------------------------------------
 * Scene-level operators either side of the alignment loop (SURVEY section 8f).  Device pointers, fp32.
 * ------------------------------------------------------------------------------------------ */
/* clean_pointcloud (dust3r/cloud_opt/base_opt.py:369-405): conf[i][p] is cut to bad_conf when image i's world point p lands
 * in image j in front of j's surface ((1 - tol) * depth_j) where j is more confident; (i, j) visited in the reference's order
 * (later tests see earlier cuts).  Images are packed back to back: image i = rows [off[i], off[i] + hw[2i] * hw[2i+1]) of
 * pts3d [.][3] (world frame), conf (updated in place) and depth.  K: [n][3][3], cams: [n][4][4] world-to-camera, row-major. */
int d3r_clean_pointcloud(int32_t n_imgs, const int32_t* hw_dev, const int64_t* off_dev, int32_t max_area, const float* pts3d_dev,
                         float* conf_dev, const float* depth_dev, const float* K_dev, const float* cams_dev, float tol,
                         float bad_conf, void* stream);
/* Moments of the weighted Umeyama / Kabsch problems roma.rigid_points_registration solves for
 * dust3r/cloud_opt/init_im_poses.py:66-110, 253-262: per problem b, out[b][17] (fp64) =
 * { sum w | sum w x (3) | sum w y (3) | sum w y x^T (9, row-major) | sum w |x|^2 } over the n_points rows of x, y [B][P][3], w [B][P]. */
int d3r_procrustes_moments(int32_t n_problems, int32_t n_points, const float* x_dev, const float* y_dev, const float* w_dev,
                           double* out_dev, void* stream);
/* estimate_focal_knowing_depth(..., focal_mode='weiszfeld') (dust3r/post_process.py:12-60) without its final clipping:
 * pts3d [B][H][W][3] in the camera frame, pp [B][2] -> focal [B] after `steps` re-weighted iterations. */
int d3r_weiszfeld_focal(int32_t n_maps, int32_t H, int32_t W, const float* pts3d_dev, const float* pp_dev, int32_t steps,
                        float* focal_dev, void* stream);
/* Index of the nearest of `points` [M][3] for every row of `queries` [N][3] (squared Euclidean distance, lowest index on a
 * tie): the two tree queries of find_reciprocal_matches (dust3r/utils/geometry.py:345-361), brute force on the GPU. */
int d3r_nearest_neighbours(int32_t n_queries, int32_t n_points, const float* queries_dev, const float* points_dev, int32_t* nn_dev,
                           void* stream);
/* Per-image pixel work of load_images (dust3r/utils/image.py:62-71 `_resize_pil_image`, :101-124 crop + ImgNorm): Pillow's 8-bit
 * Image.resize (src/libImaging/Resample.c: horizontal then vertical pass, 22-bit fixed-point coefficients, each pass rounded and
 * clipped to uint8), the centre crop, and torchvision's ToTensor + Normalize(0.5, 0.5), bit-exact.
 *   src [H0][W0][3] uint8 RGB (decoded image)            ->  out [3][H2][W2] fp32 in [-1, 1]
 *   x/ybounds [W1 | H1][2] = (first source index, taps <= kx | ky), x/ycoefs [kx | ky][W1 | H1] (tap-major) int32 with 22
 *   fractional bits: the tables of Resample.c precompute_coeffs + normalize_coeffs_8bpc for W0 -> W1 and H0 -> H1 (a dimension
 *   that does not change gets the identity table: bounds (i, 1), coefficient 1 << 22); the output is the window [crop_y0, crop_y0 + H2) x [crop_x0, crop_x0 + W2)
 *   of the resized image; [row0, row0 + rows) = the source rows those output rows read (union of their ybounds);
 *   lut [256] = the fp32 value of every byte after ImgNorm; tmp = workspace of rows * W2 * 3 bytes. */
int d3r_image_resize_crop_normalize(const uint8_t* src_dev, int32_t H0, int32_t W0, int32_t H1, int32_t W1,
                                    const int32_t* xbounds_dev, const int32_t* xcoefs_dev, int32_t kx,
                                    const int32_t* ybounds_dev, const int32_t* ycoefs_dev, int32_t ky, int32_t row0, int32_t rows,
                                    int32_t crop_x0, int32_t crop_y0, int32_t H2, int32_t W2, const float* lut_dev, uint8_t* tmp_dev,
                                    float* out_dev, void* stream);

/* ------------------------------------------------------------------------------------------
 * Path 1 — pairwise forward: replaces AsymmetricCroCo3DStereo.forward (dust3r/model.py:199-211 =
 * _encode_symmetrized :153-170, _decoder :172-191, downstream heads :193-208) for one batch of
 * same-sized pairs.  Weights are caller-owned device buffers, repacked once by the host side
 * (dust3r_b200/model.py: bf16 GEMM operands, fp32 biases / LayerNorm parameters).
 * ------------------------------------------------------------------------------------------ */
typedef struct d3r_linear { const void* w; const float* b; } d3r_linear;  /* w: bf16 [out][in]; b may be NULL */
typedef struct d3r_norm { const float* g; const float* b; } d3r_norm;     /* LayerNorm weight / bias (fp32)   */

typedef struct d3r_enc_block {      /* croco/models/blocks.py:114-130 */
  d3r_norm norm1, norm2;
  d3r_linear qkv, proj, fc1, fc2;
} d3r_enc_block;

typedef struct d3r_dec_block {      /* croco/models/blocks.py:171-191 */
  d3r_norm norm1, norm2, norm3, norm_y;
  d3r_linear qkv, proj;             /* self attention                                             */
  d3r_linear projq, projkv, cproj;  /* cross attention; projkv = rows of projk then projv          */
  d3r_linear fc1, fc2;
} d3r_dec_block;

typedef struct d3r_fusion {         /* FeatureFusionBlock_custom, croco/models/dpt_block.py:130-212 */
  d3r_linear rcu1_conv1, rcu1_conv2, rcu2_conv1, rcu2_conv2; /* 3x3, packed [Cout][9][Cin]           */
  d3r_linear out_conv;                                     /* 1x1 [256][256]                        */
} d3r_fusion;

typedef struct d3r_dpt_head {       /* DPTOutputAdapter_fix, dust3r/heads/dpt_head.py:20-65         */
  d3r_linear act_conv[4];           /* 1x1 convs on the 4 hooked token maps                        */
  d3r_linear act0_up;               /* ConvTranspose k4 s4 as GEMM  [(ky*4+kx)*96+co][ci]           */
  d3r_linear act1_up;               /* ConvTranspose k2 s2 as GEMM  [(ky*2+kx)*192+co][ci]          */
  d3r_linear act3_down;             /* 3x3 s2 p1 as GEMM over im2col [768][9*768]                   */
  d3r_linear layer_rn[4];           /* 3x3, no bias, packed                                        */
  d3r_fusion refine[4];             /* refinenet1..4                                               */
  d3r_linear head0;                 /* 3x3 256->128 packed                                         */
  d3r_linear head2;                 /* 3x3 128->128 packed                                         */
  const float* head4_w;             /* fp32 [4][128], always 4 rows: row 3 zero when nch == 3      */
  const float* head4_b;             /* fp32 [4], entry 3 zero when nch == 3                        */
} d3r_dpt_head;

typedef struct d3r_model {
  int32_t enc_dim, enc_depth, enc_heads, dec_dim, dec_depth, dec_heads, mlp_ratio, patch;
  int32_t head_type;                /* 0 = linear (LinearPts3d), 1 = dpt                            */
  int32_t nch;                      /* 3 + has_conf                                                */
  int32_t depth_mode;               /* 0 linear, 1 square, 2 exp  (postprocess.py:23-44)            */
  int32_t conf_mode;                /* 0 none, 1 exp, 2 sigmoid   (postprocess.py:47-58)            */
  float conf_min, conf_max, ln_eps;
  int32_t hooks[4];                 /* DPT hooks into [enc_out, dec_1..dec_L] (dpt_head.py:110)     */
  int32_t rope_max_pos;
  const float* rope_cos;            /* [rope_max_pos][16]                                          */
  const float* rope_sin;
  d3r_linear patch_embed;           /* [enc_dim][3*patch*patch]                                    */
  const d3r_enc_block* enc;         /* host array [enc_depth]                                      */
  d3r_norm enc_norm;
  d3r_linear decoder_embed;
  const d3r_dec_block* dec1;        /* dec_blocks   (host array [dec_depth])                       */
  const d3r_dec_block* dec2;        /* dec_blocks2                                                 */
  d3r_norm dec_norm;
  const d3r_dpt_head* dpt[2];       /* downstream_head1/2 when head_type == 1                      */
  d3r_linear lin_head[2];           /* downstream_head{1,2}.proj when head_type == 0               */
} d3r_model;

/* sizeof(d3r_model) as compiled into the library (binding self-check). */
int d3r_sizeof_model(void);

/* Bytes of device workspace d3r_forward_pairs needs for (n_enc images to encode, B pairs, HxW). */
int64_t d3r_forward_workspace_bytes(const d3r_model* m, int32_t n_enc, int32_t B, int32_t H, int32_t W);

/* imgs: (n_enc,3,H,W) fp32 in [-1,1] — the images the encoder runs on (model.py:142-170 decides which:
 * cat(img1,img2), or only the even halves for a symmetrised batch).  idx1/idx2: HOST int32[B], the
 * encoded image acting as view1 / view2 of pair b.  Outputs (fp32, device):
 * pts3d_1 (B,H,W,3), conf_1 (B,H,W) in view1's frame for view1; pts3d_2 / conf_2 for view2
 * ('pts3d_in_other_view').  conf pointers may be NULL when the model has no confidence channel. */
int d3r_forward_pairs(const d3r_model* m, const float* imgs_dev, int32_t n_enc, const int32_t* idx1_host,
                      const int32_t* idx2_host, int32_t B, int32_t H, int32_t W, float* pts3d_1, float* conf_1,
                      float* pts3d_2, float* conf_2, void* workspace_dev, int64_t workspace_bytes, void* stream);

/* Pairs whose two images differ in size (the reference encodes them separately, dust3r/model.py:147-151, and
 * inference() then runs one pair per call, dust3r/inference.py:60-64): imgs1 (B,3,H1,W1) are the first views,
 * imgs2 (B,3,H2,W2) the second views; outputs pts3d_1 (B,H1,W1,3), conf_1 (B,H1,W1), pts3d_2 (B,H2,W2,3),
 * conf_2 (B,H2,W2).  No symmetrisation shortcut on this path. */
int64_t d3r_forward_mixed_workspace_bytes(const d3r_model* m, int32_t B, int32_t H1, int32_t W1, int32_t H2, int32_t W2);
int d3r_forward_pairs_mixed(const d3r_model* m, const float* imgs1_dev, int32_t H1, int32_t W1, const float* imgs2_dev,
                            int32_t H2, int32_t W2, int32_t B, float* pts3d_1, float* conf_1, float* pts3d_2,
                            float* conf_2, void* workspace_dev, int64_t workspace_bytes, void* stream);

/* Optional taps for the parity tests: when non-NULL, fp32 copies of intermediate stages are written.
 * (set with d3r_forward_set_debug before a call; cleared after it).  stage ids in DESIGN.md. */
int d3r_forward_set_debug(int32_t stage_id, float* out_dev, int64_t capacity_floats);

#ifdef __cplusplus
}
#endif
#endif /* DUST3R_B200_H_ */
