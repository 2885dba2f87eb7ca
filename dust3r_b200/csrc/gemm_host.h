// Internal host API of the tcgen05 GEMM (C++ side; the C ABI wrappers live in gemm_host.cu).
#pragma once
#include "gemm_tcgen05.cuh"

namespace d3r {
namespace gemm {
int pick_block_n(int N, uint32_t flags);
void set_impl(int impl);
void set_pair_min_kb(int kb);
// A: [M][lda] bf16 row-major (K valid columns), B: [N][K] bf16.  p.{M,N,K,flags,out,...} filled by the caller.
int gemm_bf16(const void* A, long long lda, const void* B, Params p, cudaStream_t st);
// x: (B,H,W,Cin) bf16 NHWC, w_packed: [Cout][9][Cin] bf16, output (B,H,W,Cout).
int conv3x3_bf16(const void* x_nhwc, const void* w_packed, int B, int H, int W, int Cin, int Cout, Params p, cudaStream_t st);
// k == stride transposed conv as GEMM + scatter: x (B,h,w,Cin), w_packed [(ky*k+kx)*Cout + co][Cin], out (B,h*k,w*k,Cout).
int convT_bf16(const void* x_nhwc, const void* w_packed, const float* bias, void* out, int B, int h, int w, int Cin, int Cout, int k,
               cudaStream_t st);
// last DPT conv (3x3, 128 -> 128) + ReLU + 1x1 conv to 4 channels (w4 [4][128], b4 [4]) + pts3d / conf postprocess.
// conf == nullptr: no confidence output (conf_mode ignored).
int conv3x3_head_tail(const void* x_nhwc, const void* w_packed, const float* bias, const float* w4, const float* b4, float* pts3d,
                      float* conf, int B, int H, int W, int depth_mode, int conf_mode, float conf_min, float conf_max, cudaStream_t st);
}  // namespace gemm
}  // namespace d3r
