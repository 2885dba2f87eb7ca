// Bandwidth-bound glue kernels of the forward path (everything that is not a GEMM / attention):
// LayerNorm (fp32 residual stream -> bf16 GEMM operand), patch im2col, casts, row gathers,
// bilinear x2 upsampling (align_corners=True), strided 3x3 im2col, linear-head pixel shuffle +
// postprocess.  All coalesced, 16-byte vectorised where the layout allows.
#include "d3r_common.cuh"
#include "elementwise.h"
#include "prof.h"
#include "pdl.cuh"
#include <cuda_bf16.h>

namespace d3r {
namespace ew {

__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// ---- LayerNorm: one warp per row, row kept in registers (C <= 2048, C % 4 == 0) -----------------
template <int MAXV>  // float4 per lane
__global__ void __launch_bounds__(256) layernorm_kernel(const float* __restrict__ x, const float* __restrict__ g,
                                                        const float* __restrict__ b, __nv_bfloat16* __restrict__ out,
                                                        const int* __restrict__ row_map, int M, int C, float eps) {
  pdl::sync_with_predecessor();   // PDL: nothing above touches memory produced by other kernels
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const int nv = C >> 2;
  const float4* xr = reinterpret_cast<const float4*>(x + (size_t)row * C);
  float4 v[MAXV];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int c = lane + i * 32;
    if (c < nv) {
      v[i] = xr[c];
      s += v[i].x + v[i].y + v[i].z + v[i].w;
    }
  }
  s = warp_sum(s);
  const float mean = s / float(C);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int c = lane + i * 32;
    if (c < nv) {
      const float a = v[i].x - mean, bb = v[i].y - mean, cc = v[i].z - mean, d = v[i].w - mean;
      q += a * a + bb * bb + cc * cc + d * d;
    }
  }
  q = warp_sum(q);
  const float rstd = rsqrtf(q / float(C) + eps);
  const int orow = row_map ? row_map[row] : row;
  uint2* o = reinterpret_cast<uint2*>(out + (size_t)orow * C);
  const float4* g4 = reinterpret_cast<const float4*>(g);
  const float4* b4 = reinterpret_cast<const float4*>(b);
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int c = lane + i * 32;
    if (c < nv) {
      const float4 gg = __ldg(g4 + c), bb = __ldg(b4 + c);
      const float y0 = (v[i].x - mean) * rstd * gg.x + bb.x, y1 = (v[i].y - mean) * rstd * gg.y + bb.y;
      const float y2 = (v[i].z - mean) * rstd * gg.z + bb.z, y3 = (v[i].w - mean) * rstd * gg.w + bb.w;
      o[c] = make_uint2(pack2(y0, y1), pack2(y2, y3));
    }
  }
}

int layernorm(const float* x, const float* g, const float* b, void* out_bf16, const int* row_map, int M, int C, float eps,
              cudaStream_t st) {
  D3R_CHECK_ARG(C % 4 == 0 && C <= 2048, "layernorm: C=%d unsupported", C);
  const int warps = 8;
  const int blocks = (M + warps - 1) / warps;
  prof::Scope scope("layernorm", st, 0.0, double(M) * C * 6.0);
  if (C <= 1024)
    D3R_CUDA(pdl::launch(layernorm_kernel<8>, dim3(blocks), dim3(warps * 32), 0, st, x, g, b, (__nv_bfloat16*)out_bf16, row_map, M, C, eps));
  else
    D3R_CUDA(pdl::launch(layernorm_kernel<16>, dim3(blocks), dim3(warps * 32), 0, st, x, g, b, (__nv_bfloat16*)out_bf16, row_map, M, C, eps));
  D3R_LAUNCH_CHECK();
  return D3R_OK;
}

// ---- fp32 -> bf16 cast ----------------------------------------------------------------------------
__global__ void cast_kernel(const float4* __restrict__ x, uint2* __restrict__ o, size_t n4) {
  pdl::sync_with_predecessor();   // PDL: nothing above touches memory produced by other kernels
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n4) {
    const float4 v = x[i];
    o[i] = make_uint2(pack2(v.x, v.y), pack2(v.z, v.w));
  }
}
int cast_f32_bf16(const float* x, void* out, size_t n, cudaStream_t st) {
  D3R_CHECK_ARG(n % 4 == 0, "cast: n must be a multiple of 4");
  const size_t n4 = n / 4;
  if (n4 == 0) return D3R_OK;
  prof::Scope scope("cast_f32_bf16", st, 0.0, double(n) * 6.0);
  D3R_CUDA(pdl::launch(cast_kernel, dim3((unsigned)((n4 + 255) / 256)), dim3(256), 0, st, (const float4*)x, (uint2*)out, n4));
  D3R_LAUNCH_CHECK();
  return D3R_OK;
}

// ---- gather rows of a bf16 matrix: out[r] = in[map[r / rows_per] * rows_per + r % rows_per] -------
__global__ void gather_rows_kernel(const uint4* __restrict__ in, uint4* __restrict__ out, const int* __restrict__ img_map,
                                   int rows_per_img, int vec_per_row, size_t total) {
  pdl::sync_with_predecessor();   // PDL: nothing above touches memory produced by other kernels
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const size_t row = i / vec_per_row;
  const int v = (int)(i - row * vec_per_row);
  const int img = (int)(row / rows_per_img);
  const int r = (int)(row - (size_t)img * rows_per_img);
  out[i] = in[((size_t)img_map[img] * rows_per_img + r) * vec_per_row + v];
}
int gather_images_bf16(const void* in, void* out, const int* img_map_dev, int n_out_imgs, int rows_per_img, int C, cudaStream_t st) {
  D3R_CHECK_ARG(C % 8 == 0, "gather: C must be a multiple of 8");
  const int vpr = C / 8;
  const size_t total = (size_t)n_out_imgs * rows_per_img * vpr;
  if (!total) return D3R_OK;
  prof::Scope scope("gather_images", st, 0.0, double(total) * 32.0);
  D3R_CUDA(pdl::launch(gather_rows_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, (const uint4*)in, (uint4*)out, img_map_dev, rows_per_img, vpr, total));
  D3R_LAUNCH_CHECK();
  return D3R_OK;
}

// ---- patch im2col: (B,3,H,W) fp32 -> [B*gh*gw][3*P*P] bf16, k = c*P*P + py*P + px (Conv2d weight flatten)
__global__ void patch_im2col_kernel(const float* __restrict__ img, __nv_bfloat16* __restrict__ out, int B, int H, int W,
                                    int gh, int gw) {
  pdl::sync_with_predecessor();   // PDL: nothing above touches memory produced by other kernels
  // one thread per (token, c, py): 16 contiguous pixels
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)B * gh * gw * 48;
  if (idx >= total) return;
  const int cpy = (int)(idx % 48);
  const size_t tok = idx / 48;
  const int c = cpy / 16, py = cpy % 16;
  const int b = (int)(tok / (gh * gw));
  const int t = (int)(tok - (size_t)b * gh * gw);
  const int ty = t / gw, tx = t % gw;
  const float4* src = reinterpret_cast<const float4*>(img + (((size_t)b * 3 + c) * H + ty * 16 + py) * W + tx * 16);
  uint4* dst = reinterpret_cast<uint4*>(out + tok * 768 + c * 256 + py * 16);
  const float4 a = src[0], bb = src[1], cc = src[2], d = src[3];
  dst[0] = make_uint4(pack2(a.x, a.y), pack2(a.z, a.w), pack2(bb.x, bb.y), pack2(bb.z, bb.w));
  dst[1] = make_uint4(pack2(cc.x, cc.y), pack2(cc.z, cc.w), pack2(d.x, d.y), pack2(d.z, d.w));
}
int patch_im2col16(const float* img, void* out, int B, int H, int W, cudaStream_t st) {
  D3R_CHECK_ARG(H % 16 == 0 && W % 16 == 0, "patch_im2col: image %dx%d is not a multiple of the 16-pixel patch", H, W);
  const size_t total = (size_t)B * (H / 16) * (W / 16) * 48;
  prof::Scope scope("patch_im2col", st, 0.0, double(total) * 96.0);
  D3R_CUDA(pdl::launch(patch_im2col_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, img, (__nv_bfloat16*)out, B, H, W, H / 16, W / 16));
  D3R_LAUNCH_CHECK();
  return D3R_OK;
}

// ---- bilinear x2 upsample, align_corners=True, NHWC bf16 (F.interpolate in dpt_block.py:226,247) ----
// One thread = one 16-byte channel vector of one output column, walking kRowsPerBlock consecutive output rows.  An input row
// feeds two to three output rows: the thread keeps the two source rows of the current output row (2 x 2 vectors) in registers
// and fetches a new pair only when the source row advances, so a vector of output costs ~1.3 instead of 4 loads -- the
// one-output-per-thread version was bound by L2 -> L1 traffic (64 B read per 16 B written, 2.3 TB/s of output).
constexpr int kUpRows = 8;
__device__ __forceinline__ uint4 lerp4(const uint4& a, const uint4& b, const uint4& c, const uint4& d, float w00, float w01, float w10,
                                       float w11) {
  const uint32_t av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w}, cv[4] = {c.x, c.y, c.z, c.w}, dv[4] = {d.x, d.y, d.z, d.w};
  uint32_t r[4];
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const __nv_bfloat162 ha = *reinterpret_cast<const __nv_bfloat162*>(&av[t]);
    const __nv_bfloat162 hb = *reinterpret_cast<const __nv_bfloat162*>(&bv[t]);
    const __nv_bfloat162 hc = *reinterpret_cast<const __nv_bfloat162*>(&cv[t]);
    const __nv_bfloat162 hd = *reinterpret_cast<const __nv_bfloat162*>(&dv[t]);
    const float lo = w00 * __low2float(ha) + w01 * __low2float(hb) + w10 * __low2float(hc) + w11 * __low2float(hd);
    const float hi = w00 * __high2float(ha) + w01 * __high2float(hb) + w10 * __high2float(hc) + w11 * __high2float(hd);
    r[t] = pack2(lo, hi);
  }
  return make_uint4(r[0], r[1], r[2], r[3]);
}
__global__ void __launch_bounds__(256) upsample2x_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                                          int H, int W, int C, int Ho, int Wo, int vpc_shift) {
  pdl::sync_with_predecessor();   // PDL: nothing above touches memory produced by other kernels
  // grid = (x tiles, row groups, B)
  const int b = blockIdx.z;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int vpc = 1 << vpc_shift;
  const int ox = idx >> vpc_shift, v = idx & (vpc - 1);
  if (ox >= Wo) return;
  // source coordinate for an output grid of (2H, 2W) (cropping keeps the scale of the full map)
  const float sx = (W > 1) ? ox * (float(W - 1) / float(2 * W - 1)) : 0.f;
  const int x0 = (int)sx;
  const int x1 = min(x0 + 1, W - 1);
  const float fx = sx - x0;
  const __nv_bfloat16* base = x + (size_t)b * H * W * C + v * 8;
  const int oy_begin = blockIdx.y * kUpRows, oy_end = min(oy_begin + kUpRows, Ho);
  const float ystep = (H > 1) ? (float(H - 1) / float(2 * H - 1)) : 0.f;
  int cy0 = -1, cy1 = -1;
  uint4 a0, a1, c0, c1;            // rows cy0 / cy1 at columns x0 / x1
  for (int oy = oy_begin; oy < oy_end; ++oy) {
    const float sy = oy * ystep;
    const int y0 = (int)sy;
    const int y1 = min(y0 + 1, H - 1);
    const float fy = sy - y0;
    if (y0 != cy0) {
      if (y0 == cy1) { a0 = c0; a1 = c1; }          // the old lower row becomes the upper one
      else {
        const __nv_bfloat16* r0 = base + (size_t)y0 * W * C;
        a0 = __ldg(reinterpret_cast<const uint4*>(r0 + (size_t)x0 * C));
        a1 = __ldg(reinterpret_cast<const uint4*>(r0 + (size_t)x1 * C));
      }
      cy0 = y0;
    }
    if (y1 != cy1) {
      if (y1 == y0) { c0 = a0; c1 = a1; }           // clamped at the last row
      else {
        const __nv_bfloat16* r1 = base + (size_t)y1 * W * C;
        c0 = __ldg(reinterpret_cast<const uint4*>(r1 + (size_t)x0 * C));
        c1 = __ldg(reinterpret_cast<const uint4*>(r1 + (size_t)x1 * C));
      }
      cy1 = y1;
    }
    const float w00 = (1.f - fy) * (1.f - fx), w01 = (1.f - fy) * fx, w10 = fy * (1.f - fx), w11 = fy * fx;
    __stcs(reinterpret_cast<uint4*>(out + (((size_t)b * Ho + oy) * Wo + ox) * C + v * 8), lerp4(a0, a1, c0, c1, w00, w01, w10, w11));
  }
}
int upsample2x_bf16(const void* x, void* out, int B, int H, int W, int C, int Ho, int Wo, cudaStream_t st) {
  D3R_CHECK_ARG(C % 8 == 0 && Ho <= 2 * H && Wo <= 2 * W, "upsample2x: bad shape");
  const int vpc = C / 8;
  D3R_CHECK_ARG((vpc & (vpc - 1)) == 0, "upsample2x: C/8 must be a power of two (C=%d)", C);
  int shift = 0;
  while ((1 << shift) < vpc) ++shift;
  const size_t total = (size_t)B * Ho * Wo * vpc;
  prof::Scope scope("upsample2x", st, 0.0, double(total) * 20.0);
  dim3 grid((unsigned)(((size_t)Wo * vpc + 255) / 256), (unsigned)((Ho + kUpRows - 1) / kUpRows), (unsigned)B);
  D3R_CUDA(pdl::launch(upsample2x_kernel, dim3(grid), dim3(256), 0, st, (const __nv_bfloat16*)x, (__nv_bfloat16*)out, H, W, C, Ho, Wo, shift));
  D3R_LAUNCH_CHECK();
  return D3R_OK;
}

// ---- im2col for the one strided conv (3x3, stride 2, pad 1): (B,H,W,C) -> [B*Ho*Wo][9*C] ------------
__global__ void im2col_s2_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ out, int B, int H, int W,
                                 int C, int Ho, int Wo) {
  pdl::sync_with_predecessor();   // PDL: nothing above touches memory produced by other kernels
  const int vpc = C / 8;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)B * Ho * Wo * 9 * vpc;
  if (idx >= total) return;
  const int v = (int)(idx % vpc);
  size_t r = idx / vpc;
  const int tap = (int)(r % 9);
  r /= 9;
  const int ox = (int)(r % Wo);
  r /= Wo;
  const int oy = (int)(r % Ho);
  const int b = (int)(r / Ho);
  const int iy = oy * 2 + tap / 3 - 1, ix = ox * 2 + tap % 3 - 1;
  uint4 val = make_uint4(0, 0, 0, 0);
  if (iy >= 0 && iy < H && ix >= 0 && ix < W) val = *reinterpret_cast<const uint4*>(x + (((size_t)b * H + iy) * W + ix) * C + v * 8);
  *reinterpret_cast<uint4*>(out + ((((size_t)b * Ho + oy) * Wo + ox) * 9 + tap) * C + v * 8) = val;
}
int im2col_3x3_s2_bf16(const void* x, void* out, int B, int H, int W, int C, cudaStream_t st) {
  D3R_CHECK_ARG(C % 8 == 0, "im2col_s2: C must be a multiple of 8");
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  const size_t total = (size_t)B * Ho * Wo * 9 * (C / 8);
  prof::Scope scope("im2col_s2", st, 0.0, double(total) * 32.0);
  D3R_CUDA(pdl::launch(im2col_s2_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, (const __nv_bfloat16*)x, (__nv_bfloat16*)out, B, H, W, C, Ho, Wo));
  D3R_LAUNCH_CHECK();
  return D3R_OK;
}

// ---- postprocess (dust3r/heads/postprocess.py:10-58) ---------------------------------------------
__device__ __forceinline__ void post_one(float x, float y, float z, float c, float* pts, float* conf, int depth_mode,
                                         int conf_mode, float cmin, float cmax) {
  float ox = x, oy = y, oz = z;
  if (depth_mode != 0) {
    const float d = sqrtf(x * x + y * y + z * z);
    const float dc = fmaxf(d, 1e-8f);
    const float s = (depth_mode == 2) ? expm1f(d) : d * d;
    ox = x / dc * s; oy = y / dc * s; oz = z / dc * s;
  }
  pts[0] = ox; pts[1] = oy; pts[2] = oz;
  if (conf_mode == 1) *conf = cmin + fminf(expf(c), cmax - cmin);
  else if (conf_mode == 2) *conf = (cmax - cmin) * (1.f / (1.f + expf(-c))) + cmin;
}

// linear head: feat [B*gh*gw][nch*256] fp32, channel-major then (py,px)  -> pixel shuffle -> postprocess
__global__ void linear_head_post_kernel(const float* __restrict__ feat, float* __restrict__ pts3d, float* __restrict__ conf,
                                        int B, int gh, int gw, int nch, int depth_mode, int conf_mode, float cmin, float cmax) {
  pdl::sync_with_predecessor();   // PDL: nothing above touches memory produced by other kernels
  const int H = gh * 16, W = gw * 16;
  const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (size_t)B * H * W) return;
  const int x = (int)(idx % W);
  const int y = (int)((idx / W) % H);
  const int b = (int)(idx / ((size_t)W * H));
  const size_t tok = ((size_t)b * gh + y / 16) * gw + x / 16;
  const int sub = (y % 16) * 16 + (x % 16);
  const float* f = feat + tok * (size_t)(nch * 256) + sub;
  float c = nch > 3 ? f[3 * 256] : 0.f;
  float dummy;
  post_one(f[0], f[256], f[512], c, pts3d + idx * 3, nch > 3 ? conf + idx : &dummy, depth_mode, nch > 3 ? conf_mode : 0, cmin, cmax);
}
int linear_head_postprocess(const float* feat, float* pts3d, float* conf, int B, int gh, int gw, int nch, int depth_mode,
                            int conf_mode, float cmin, float cmax, cudaStream_t st) {
  const size_t total = (size_t)B * gh * gw * 256;
  prof::Scope scope("linear_head_post", st, 0.0, double(total) * 32.0);
  D3R_CUDA(pdl::launch(linear_head_post_kernel, dim3((unsigned)((total + 255) / 256)), dim3(256), 0, st, feat, pts3d, conf, B, gh, gw, nch, depth_mode, conf_mode, cmin, cmax));
  D3R_LAUNCH_CHECK();
  return D3R_OK;
}

}  // namespace ew
}  // namespace d3r

// ---- building blocks exported through the C ABI (unit tests; forward.cu calls the ew:: functions) ----
using namespace d3r;

extern "C" int d3r_layernorm_bf16(const float* x, const float* g, const float* b, void* out, int32_t M, int32_t C, float eps, void* stream) {
  return ew::layernorm(x, g, b, out, nullptr, M, C, eps, (cudaStream_t)stream);
}
extern "C" int d3r_upsample2x_bf16(const void* x, void* out, int32_t B, int32_t H, int32_t W, int32_t C, int32_t Ho, int32_t Wo, void* stream) {
  return ew::upsample2x_bf16(x, out, B, H, W, C, Ho, Wo, (cudaStream_t)stream);
}
extern "C" int d3r_im2col_3x3_s2_bf16(const void* x, void* out, int32_t B, int32_t H, int32_t W, int32_t C, void* stream) {
  return ew::im2col_3x3_s2_bf16(x, out, B, H, W, C, (cudaStream_t)stream);
}
extern "C" int d3r_patch_im2col16(const float* img, void* out, int32_t B, int32_t H, int32_t W, void* stream) {
  return ew::patch_im2col16(img, out, B, H, W, (cudaStream_t)stream);
}
extern "C" int d3r_gather_images_bf16(const void* in, void* out, const int32_t* map_dev, int32_t n_out, int32_t rows_per_img, int32_t C,
                                      void* stream) {
  return ew::gather_images_bf16(in, out, map_dev, n_out, rows_per_img, C, (cudaStream_t)stream);
}
extern "C" int d3r_cast_f32_bf16(const float* x, void* out, int64_t n, void* stream) {
  D3R_CHECK_ARG(n >= 0, "cast: negative length");
  return ew::cast_f32_bf16(x, out, (size_t)n, (cudaStream_t)stream);
}
extern "C" int d3r_linear_head_postprocess(const float* feat, float* pts3d, float* conf, int32_t B, int32_t gh, int32_t gw, int32_t nch,
                                           int32_t depth_mode, int32_t conf_mode, float cmin, float cmax, void* stream) {
  D3R_CHECK_ARG(feat && pts3d && (nch == 3 || nch == 4), "linear head: null buffer or nch=%d not 3 / 4", nch);
  D3R_CHECK_ARG(nch == 3 || conf_mode == 0 || conf, "linear head: conf_mode %d without a conf buffer", conf_mode);
  return ew::linear_head_postprocess(feat, pts3d, conf, B, gh, gw, nch, depth_mode, conf_mode, cmin, cmax, (cudaStream_t)stream);
}
