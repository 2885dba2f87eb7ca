// Host side of the tcgen05 GEMM / conv kernels: tensor-map construction, tile-shape selection, launch.
#include "gemm_tcgen05.cuh"
#include "gemm2_tcgen05.cuh"
#include "gemm_host.h"
#include "prof.h"
#include <mutex>

namespace d3r {
namespace gemm {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

static int encode(CUtensorMap* m, const void* ptr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes,
                  const cuuint32_t* box, CUtensorMapDataType dtype = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16) {
  EncodeTiledFn fn = get_encode();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled is not available from the CUDA driver");
    return D3R_ERR_CUDA;
  }
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = fn(m, dtype, (cuuint32_t)rank, const_cast<void*>(ptr), dims, strides_bytes, box,
                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rank %d, dims %llu,%llu)", (int)r, rank,
              (unsigned long long)dims[0], (unsigned long long)dims[1]);
    return D3R_ERR_CUDA;
  }
  return D3R_OK;
}

bool use_pair(int bn, int num_kb);

int pick_block_n(int N, uint32_t flags) {
  if (flags & F_HEAD_FINAL) return 128;
  if (N % 256 == 0) return 256;
  if (N % 128 == 0) return 128;
  if (N % 64 == 0) return (N >= 512) ? 256 : 64;
  return (N > 128) ? 256 : 128;
}

template <int BN, int EPI>
static int launch(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& to, const Params& p, int total_tiles, cudaStream_t st) {
  static unsigned long long attr_devices = 0;
  if (first_launch_on_this_device(attr_devices))
    D3R_CUDA(cudaFuncSetAttribute(gemm_kernel<BN, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<BN, EPI>::kSmemBytes));
  int grid = total_tiles < num_sms() ? total_tiles : num_sms();
  const char* tag = (p.mode == 1) ? ((p.flags & F_HEAD_FINAL) ? "conv3x3_head_tail" : "conv3x3_tcgen05")
                                  : (BN == 256 ? "gemm_tcgen05_bn256" : (BN == 128 ? "gemm_tcgen05_bn128" : "gemm_tcgen05_bn64"));
  char detail[96];
  snprintf(detail, sizeof(detail), "M=%d N=%d K=%d flags=0x%x mode=%d epi=%d", p.M, p.N, p.K, (unsigned)p.flags, p.mode, EPI);
  prof::Scope scope(tag, st, 2.0 * double(p.M) * double(p.N) * double(p.K), 0.0, 1, detail);
  D3R_CUDA(pdl::launch(gemm_kernel<BN, EPI>, dim3(grid), dim3(kNumThreads), size_t(Cfg<BN, EPI>::kSmemBytes), st, ta, tb, to, p));
  D3R_LAUNCH_CHECK();
  return D3R_OK;
}

// 0: 1-CTA kernels, 1: CTA-pair (cta_group::2) kernels whenever BLOCK_N >= 128, 2 (default): pair kernels from
// g_pair_min_kb k-blocks of 64 on, 1-CTA kernels for the shortest reductions (K = 96 / 192 of the DPT re-assembly).
// Round 1 drew the line at 16 k-blocks from isolated-GEMM timings; interleaved A/B runs of the WHOLE forward step
// (scripts/gemm_policy_ab.py, round 2) put >= 4 ahead by 1 %: 67.5-67.7 ms against 68.3 ms at >= 16.
static int g_impl = 2;
static int g_pair_min_kb = 4;
void set_impl(int impl) { g_impl = impl; }
void set_pair_min_kb(int kb) { g_pair_min_kb = kb; }
bool use_pair(int bn, int num_kb) { return bn >= 128 && (g_impl == 1 || (g_impl == 2 && num_kb >= g_pair_min_kb)); }

template <int BN, int EPI>
static int launch2(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& to, const Params& p, int m_tiles, int n_tiles,
                   cudaStream_t st) {
  static unsigned long long attr_devices = 0;
  if (first_launch_on_this_device(attr_devices))
    D3R_CUDA(cudaFuncSetAttribute(gemm2_kernel<BN, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg2<BN, EPI>::kSmemBytes));
  const int cluster_tiles = ((m_tiles + 1) / 2) * n_tiles;
  const int max_clusters = num_sms() / 2;
  const int clusters = cluster_tiles < max_clusters ? cluster_tiles : max_clusters;
  const char* tag = (p.mode == 1) ? ((p.flags & F_HEAD_FINAL) ? "conv3x3_head_tail_2cta" : "conv3x3_tcgen05_2cta")
                                  : (BN == 256 ? (p.K >= 1024 ? "gemm_tcgen05_2cta_bn256" : "gemm_tcgen05_2cta_bn256_shortk")
                                               : "gemm_tcgen05_2cta_bn128");   // short-K projections (decoder K = 768, DPT K = 256)
                                                                               // are epilogue-bound: a class of their own in the breakdown
  char detail[96];
  snprintf(detail, sizeof(detail), "M=%d N=%d K=%d flags=0x%x mode=%d epi=%d", p.M, p.N, p.K, (unsigned)p.flags, p.mode, EPI);
  prof::Scope scope(tag, st, 2.0 * double(p.M) * double(p.N) * double(p.K), 0.0, 1, detail);
  D3R_CUDA(pdl::launch(gemm2_kernel<BN, EPI>, dim3(2 * clusters), dim3(kNumThreads), size_t(Cfg2<BN, EPI>::kSmemBytes), st, ta, tb, to, p));
  D3R_LAUNCH_CHECK();
  return D3R_OK;
}

static int dispatch(int bn, const CUtensorMap& ta, const CUtensorMap& tb, const Params& p, int total_tiles, cudaStream_t st) {
  // epilogue specialisation (BLOCK_N = 256 only: every hot projection of the two ViTs has N % 256 == 0)
  int epi = (bn == 256) ? pick_epi(p.mode, p.flags) : EPI_GENERIC;
  CUtensorMap to = ta;   // placeholder unless the epilogue stores through TMA
  if (epi == EPI_RESID) {
    if ((reinterpret_cast<uintptr_t>(p.out) & 15) != 0 || p.ldo % 4 != 0) {
      epi = EPI_GENERIC;   // TMA needs 16-byte aligned rows; the register epilogue has no such requirement
    } else {
      cuuint64_t dims[2] = {(cuuint64_t)p.N, (cuuint64_t)p.M};
      cuuint64_t str[1] = {(cuuint64_t)p.ldo * 4};
      cuuint32_t box[2] = {32, 32};
      int rc = encode(&to, p.out, 2, dims, str, box, CU_TENSOR_MAP_DATA_TYPE_FLOAT32);
      if (rc) return rc;
    }
  }
  if (use_pair(bn, p.num_kb)) {
    const int n_tiles = (p.N + bn - 1) / bn;
    const int m_tiles = total_tiles / n_tiles;
    if (bn == 256) {
      switch (epi) {
        case EPI_RESID: return launch2<256, EPI_RESID>(ta, tb, to, p, m_tiles, n_tiles, st);
        case EPI_ACT: return launch2<256, EPI_ACT>(ta, tb, to, p, m_tiles, n_tiles, st);
        case EPI_ROPE: return launch2<256, EPI_ROPE>(ta, tb, to, p, m_tiles, n_tiles, st);
        default: return launch2<256, EPI_GENERIC>(ta, tb, to, p, m_tiles, n_tiles, st);
      }
    }
    return launch2<128, EPI_GENERIC>(ta, tb, to, p, m_tiles, n_tiles, st);
  }
  switch (bn) {
    case 256:
      switch (epi) {
        case EPI_RESID: return launch<256, EPI_RESID>(ta, tb, to, p, total_tiles, st);
        case EPI_ACT: return launch<256, EPI_ACT>(ta, tb, to, p, total_tiles, st);
        case EPI_ROPE: return launch<256, EPI_ROPE>(ta, tb, to, p, total_tiles, st);
        default: return launch<256, EPI_GENERIC>(ta, tb, to, p, total_tiles, st);
      }
    case 128: return launch<128, EPI_GENERIC>(ta, tb, to, p, total_tiles, st);
    case 64: return launch<64, EPI_GENERIC>(ta, tb, to, p, total_tiles, st);
  }
  set_error("unsupported BLOCK_N %d", bn);
  return D3R_ERR_INVALID;
}

// B operand: [N][taps][Kc] bf16, K-major
static int make_tmap_b(CUtensorMap* m, const void* B, int N, int taps, int Kc, int bn, int num_kb) {
  cuuint64_t dims[3] = {(cuuint64_t)Kc, (cuuint64_t)taps, (cuuint64_t)N};
  cuuint64_t str[2] = {(cuuint64_t)Kc * 2, (cuuint64_t)taps * Kc * 2};
  cuuint32_t box[3] = {(cuuint32_t)BLOCK_K, 1, (cuuint32_t)(use_pair(bn, num_kb) ? bn / 2 : bn)};   // each CTA of a pair stages half of B
  return encode(m, B, 3, dims, str, box);
}

int gemm_bf16(const void* A, long long lda, const void* B, Params p, cudaStream_t st) {
  D3R_CHECK_ARG(A && B, "gemm: null operand");
  D3R_CHECK_ARG(p.M > 0 && p.N > 0 && p.K > 0, "gemm: bad shape %d %d %d", p.M, p.N, p.K);
  D3R_CHECK_ARG(p.N % 32 == 0, "gemm: N=%d must be a multiple of 32", p.N);
  D3R_CHECK_ARG(p.K % 8 == 0 && lda % 8 == 0, "gemm: K=%d / lda=%lld must be multiples of 8 (16-byte TMA strides)", p.K, lda);
  D3R_CHECK_ARG((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(B) & 15) == 0, "gemm: operands must be 16-byte aligned");
  p.mode = 0;
  p.num_kb = (p.K + BLOCK_K - 1) / BLOCK_K;
  const int bn = pick_block_n(p.N, p.flags);
  CUtensorMap ta, tb;
  {
    cuuint64_t dims[2] = {(cuuint64_t)p.K, (cuuint64_t)p.M};
    cuuint64_t str[1] = {(cuuint64_t)lda * 2};
    cuuint32_t box[2] = {(cuuint32_t)BLOCK_K, (cuuint32_t)BLOCK_M};
    int rc = encode(&ta, A, 2, dims, str, box);
    if (rc) return rc;
  }
  int rc = make_tmap_b(&tb, B, p.N, 1, p.K, bn, p.num_kb);
  if (rc) return rc;
  const int total = ((p.M + BLOCK_M - 1) / BLOCK_M) * ((p.N + bn - 1) / bn);
  return dispatch(bn, ta, tb, p, total, st);
}

int conv3x3_bf16(const void* x_nhwc, const void* w_packed, int B, int H, int W, int Cin, int Cout, Params p, cudaStream_t st) {
  D3R_CHECK_ARG(x_nhwc && w_packed, "conv3x3: null operand");
  D3R_CHECK_ARG(Cin % 8 == 0 && Cout % 32 == 0, "conv3x3: Cin=%d must be a multiple of 8 and Cout=%d of 32", Cin, Cout);
  p.mode = 1;
  p.M = B * H * W;
  p.N = Cout;
  p.cin_blocks = (Cin + BLOCK_K - 1) / BLOCK_K;
  p.K = 9 * Cin;
  p.num_kb = 9 * p.cin_blocks;
  p.cB = B; p.cH = H; p.cW = W;
  int tw = 16;
  while (tw < W && tw < 128) tw *= 2;
  p.tile_w = tw;
  p.tile_h = BLOCK_M / tw;
  p.tiles_x = (W + p.tile_w - 1) / p.tile_w;
  p.tiles_y = (H + p.tile_h - 1) / p.tile_h;
  p.ldo = Cout;
  const int bn = pick_block_n(p.N, p.flags);
  CUtensorMap ta, tb;
  {
    cuuint64_t dims[4] = {(cuuint64_t)Cin, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
    cuuint64_t str[3] = {(cuuint64_t)Cin * 2, (cuuint64_t)W * Cin * 2, (cuuint64_t)H * W * Cin * 2};
    cuuint32_t box[4] = {(cuuint32_t)BLOCK_K, (cuuint32_t)p.tile_w, (cuuint32_t)p.tile_h, 1};
    int rc = encode(&ta, x_nhwc, 4, dims, str, box);
    if (rc) return rc;
  }
  int rc = make_tmap_b(&tb, w_packed, Cout, 9, Cin, bn, p.num_kb);
  if (rc) return rc;
  const int total = B * p.tiles_x * p.tiles_y * ((p.N + bn - 1) / bn);
  return dispatch(bn, ta, tb, p, total, st);
}

int convT_bf16(const void* x_nhwc, const void* w_packed, const float* bias, void* out, int B, int h, int w, int Cin, int Cout, int k,
               cudaStream_t st) {
  D3R_CHECK_ARG(x_nhwc && w_packed && out, "convT: null buffer");
  D3R_CHECK_ARG(B > 0 && h > 0 && w > 0 && k > 0, "convT: bad shape");
  // the epilogue scatters 32-column chunks: each must lie inside one (ky, kx) tap
  D3R_CHECK_ARG(Cout % 32 == 0, "convT: Cout=%d must be a multiple of 32", Cout);
  Params p{};
  p.M = B * h * w; p.N = k * k * Cout; p.K = Cin;
  p.flags = F_CONVT | (bias ? F_BIAS : 0);
  p.out = out; p.bias = bias; p.ldo = 0;
  p.tk = k; p.th_in = h; p.tw_in = w; p.tCout = Cout;
  return gemm_bf16(x_nhwc, Cin, w_packed, p, st);
}

int conv3x3_head_tail(const void* x_nhwc, const void* w_packed, const float* bias, const float* w4, const float* b4, float* pts3d,
                      float* conf, int B, int H, int W, int depth_mode, int conf_mode, float conf_min, float conf_max, cudaStream_t st) {
  D3R_CHECK_ARG(w4 && b4 && pts3d, "head tail: null buffer");
  D3R_CHECK_ARG(depth_mode >= 0 && depth_mode <= 2 && conf_mode >= 0 && conf_mode <= 2, "head tail: bad postprocess mode");
  Params p{};
  p.flags = F_HEAD_FINAL | (bias ? F_BIAS : 0);
  p.bias = bias;
  p.w4 = w4; p.b4 = b4;
  p.pts3d = pts3d; p.conf = conf;
  p.depth_mode = depth_mode; p.conf_mode = conf ? conf_mode : 0;
  p.conf_min = conf_min; p.conf_max = conf_max;
  return conv3x3_bf16(x_nhwc, w_packed, B, H, W, 128, 128, p, st);
}

}  // namespace gemm
}  // namespace d3r

// ---- building blocks exported through the C ABI (used by the unit tests and by forward.cu) ----
using namespace d3r;

extern "C" void d3r_set_gemm_impl(int32_t impl) { gemm::set_impl(impl); }
extern "C" void d3r_set_gemm_pair_min_kblocks(int32_t kb) { gemm::set_pair_min_kb(kb); }

extern "C" int d3r_gemm_bf16(const void* A, const void* B, void* out, const float* bias, const void* add0, void* out2,
                             int32_t M, int32_t N, int32_t K, int64_t ldo, uint32_t flags, const float* rope_cos,
                             const float* rope_sin, int32_t rope_cols, int32_t tokens_per_img, int32_t grid_w, void* stream) {
  gemm::Params p{};
  p.M = M; p.N = N; p.K = K;
  p.flags = flags;
  p.out = out; p.out2 = out2; p.add0 = add0; p.bias = bias; p.ldo = ldo;
  p.rope_cos = rope_cos; p.rope_sin = rope_sin; p.rope_cols = rope_cols; p.tokens_per_img = tokens_per_img; p.grid_w = grid_w;
  D3R_CHECK_ARG(!(flags & gemm::F_BIAS) || bias, "gemm: F_BIAS without bias");
  D3R_CHECK_ARG(!(flags & gemm::F_ROPE) || (rope_cos && rope_sin && tokens_per_img > 0 && grid_w > 0), "gemm: F_ROPE without tables");
  D3R_CHECK_ARG(!(flags & (gemm::F_CONVT | gemm::F_HEAD_FINAL)), "gemm: use the dedicated entry points for convT / head tail");
  return gemm::gemm_bf16(A, K, B, p, (cudaStream_t)stream);
}

extern "C" int d3r_conv3x3_bf16(const void* x_nhwc, const void* w_packed, void* out, const float* bias, const void* add0,
                                const void* add1, void* out2, int32_t B, int32_t H, int32_t W, int32_t Cin, int32_t Cout,
                                uint32_t flags, void* stream) {
  gemm::Params p{};
  p.flags = flags;
  p.out = out; p.out2 = out2; p.add0 = add0; p.add1 = add1; p.bias = bias;
  D3R_CHECK_ARG(!(flags & (gemm::F_CONVT | gemm::F_HEAD_FINAL | gemm::F_ROPE)), "conv3x3: unsupported flag");
  return gemm::conv3x3_bf16(x_nhwc, w_packed, B, H, W, Cin, Cout, p, (cudaStream_t)stream);
}

extern "C" int d3r_convT_bf16(const void* x_nhwc, const void* w_packed, const float* bias, void* out, int32_t B, int32_t h, int32_t w,
                              int32_t Cin, int32_t Cout, int32_t k, void* stream) {
  return gemm::convT_bf16(x_nhwc, w_packed, bias, out, B, h, w, Cin, Cout, k, (cudaStream_t)stream);
}

extern "C" int d3r_conv3x3_head_tail(const void* x_nhwc, const void* w_packed, const float* bias, const float* w4, const float* b4,
                                     float* pts3d, float* conf, int32_t B, int32_t H, int32_t W, int32_t depth_mode, int32_t conf_mode,
                                     float conf_min, float conf_max, void* stream) {
  return gemm::conv3x3_head_tail(x_nhwc, w_packed, bias, w4, b4, pts3d, conf, B, H, W, depth_mode, conf_mode, conf_min, conf_max,
                                 (cudaStream_t)stream);
}
