// Pairwise forward orchestration (host side, C++): replaces AsymmetricCroCo3DStereo.forward
// (dust3r/model.py:199-211) for one batch of same-sized pairs with a fixed launch sequence on ONE stream:
//
//   encoder   patch im2col -> GEMM(+bias)->x(f32) ; 24 x { LN -> GEMM(qkv,+bias,+RoPE) -> attention ->
//             GEMM(proj,+bias,+=x) -> LN -> GEMM(fc1,+bias,GELU) -> GEMM(fc2,+bias,+=x) } ; LN(enc_norm)
//   decoder   GEMM(decoder_embed) ; 12 x two branches { LN ; norm_y of the other branch ; self-attn ;
//             cross-attn (q from x, fused k|v projection of norm_y(other)) ; MLP }, hooks kept in bf16
//   heads     DPT: 1x1 GEMMs, transposed convs as GEMM+scatter, 3x3 convs as implicit GEMM (TMA im2col),
//             bilinear x2 kernels, final 1x1 conv + postprocess fused in the last conv's epilogue;
//             or linear head GEMM + pixel-shuffle/postprocess kernel.
//
// The residual stream stays fp32 (as in the reference), GEMM operands are bf16, accumulation fp32.
#include "gemm_host.h"
#include "elementwise.h"
#include <vector>
#include <cstring>

namespace d3r {
namespace fwd {

using gemm::Params;

struct Arena {
  uint8_t* base;
  size_t cap, off;
  bool dry;  // size-only pass
  void* take(size_t bytes) {
    off = (off + 255) & ~size_t(255);
    void* p = dry ? nullptr : base + off;
    off += bytes;
    return p;
  }
  template <class T>
  T* arr(size_t n) { return reinterpret_cast<T*>(take(n * sizeof(T))); }
};

struct DebugTap { int stage; float* out; long long cap; };
static thread_local DebugTap g_tap = {-1, nullptr, 0};

__global__ void bf16_to_f32_kernel(const __nv_bfloat16* x, float* o, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) o[i] = __bfloat162float(x[i]);
}
static void tap_f32(int stage, const float* x, size_t n, cudaStream_t st) {
  if (g_tap.stage == stage && g_tap.out && (long long)n <= g_tap.cap)
    cudaMemcpyAsync(g_tap.out, x, n * sizeof(float), cudaMemcpyDeviceToDevice, st);
}
static void tap_bf16(int stage, const void* x, size_t n, cudaStream_t st) {
  if (g_tap.stage == stage && g_tap.out && (long long)n <= g_tap.cap)
    bf16_to_f32_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const __nv_bfloat16*)x, g_tap.out, n);
}

#define RC(x)            \
  do {                   \
    int _rc = (x);       \
    if (_rc) return _rc; \
  } while (0)

struct Ctx {
  const d3r_model* m;
  cudaStream_t st;
  int gh, gw, N;  // token grid
};

static int linear(const Ctx& c, const void* A, long long lda, const d3r_linear& w, int M, int N, int K, void* out, uint32_t flags,
                  void* out2 = nullptr, const void* add0 = nullptr, int rope_cols = 0) {
  Params p{};
  p.M = M; p.N = N; p.K = K;
  p.flags = flags | (w.b ? gemm::F_BIAS : 0);
  p.out = out; p.out2 = out2; p.add0 = add0; p.bias = w.b; p.ldo = N;
  if (flags & gemm::F_ROPE) {
    p.rope_cos = c.m->rope_cos; p.rope_sin = c.m->rope_sin; p.rope_cols = rope_cols; p.tokens_per_img = c.N; p.grid_w = c.gw;
  }
  return gemm::gemm_bf16(A, lda, w.w, p, c.st);
}

static int conv3(const Ctx& c, const void* x, const d3r_linear& w, int B, int H, int W, int Cin, int Cout, void* out, uint32_t flags,
                 const void* add0 = nullptr, const void* add1 = nullptr, void* out2 = nullptr) {
  Params p{};
  p.flags = flags | (w.b ? gemm::F_BIAS : 0) | (add0 ? gemm::F_ADD0 : 0) | (add1 ? gemm::F_ADD1 : 0) | (out2 ? gemm::F_OUT2_RELU : 0);
  p.out = out; p.out2 = out2; p.add0 = add0; p.add1 = add1; p.bias = w.b;
  return gemm::conv3x3_bf16(x, w.w, B, H, W, Cin, Cout, p, c.st);
}

// k == stride transposed convolution: rows = input pixels, columns = (ky,kx,co)
static int convT(const Ctx& c, const void* x, const d3r_linear& w, int B, int h, int wd, int Cin, int Cout, int k, void* out) {
  return gemm::convT_bf16(x, w.w, w.b, out, B, h, wd, Cin, Cout, k, c.st);
}

// ---- encoder ---------------------------------------------------------------------------------
static int run_encoder(const Ctx& c, Arena& ar, const float* imgs, int n_enc, int H, int W, void** enc_out_bf16) {
  const d3r_model& m = *c.m;
  const int E = m.enc_dim, M = n_enc * c.N, hid = E * m.mlp_ratio;
  float* x = ar.arr<float>((size_t)M * E);
  __nv_bfloat16* ln = ar.arr<__nv_bfloat16>((size_t)M * E);
  __nv_bfloat16* qkv = ar.arr<__nv_bfloat16>((size_t)M * 3 * E);
  __nv_bfloat16* att = ar.arr<__nv_bfloat16>((size_t)M * E);
  __nv_bfloat16* hidb = ar.arr<__nv_bfloat16>((size_t)M * hid);
  __nv_bfloat16* eout = ar.arr<__nv_bfloat16>((size_t)M * E);
  *enc_out_bf16 = eout;
  if (ar.dry) return D3R_OK;
  const int pk = 3 * m.patch * m.patch;
  RC(ew::patch_im2col16(imgs, hidb, n_enc, H, W, c.st));
  RC(linear(c, hidb, pk, m.patch_embed, M, E, pk, x, gemm::F_OUT_F32));
  tap_f32(1, x, (size_t)M * E, c.st);
  const float scale = 1.0f / sqrtf(float(E / m.enc_heads));
  for (int l = 0; l < m.enc_depth; ++l) {
    const d3r_enc_block& b = m.enc[l];
    RC(ew::layernorm(x, b.norm1.g, b.norm1.b, ln, nullptr, M, E, m.ln_eps, c.st));
    RC(linear(c, ln, E, b.qkv, M, 3 * E, E, qkv, gemm::F_ROPE, nullptr, nullptr, 2 * E));
    RC(attn::attention_hd64(qkv, 3 * E, qkv + E, 3 * E, qkv + 2 * E, 3 * E, att, E, n_enc, m.enc_heads, c.N, c.N, scale, c.st));
    RC(linear(c, att, E, b.proj, M, E, E, x, gemm::F_RESID_INPLACE));
    RC(ew::layernorm(x, b.norm2.g, b.norm2.b, ln, nullptr, M, E, m.ln_eps, c.st));
    RC(linear(c, ln, E, b.fc1, M, hid, E, hidb, gemm::F_GELU));
    RC(linear(c, hidb, hid, b.fc2, M, E, hid, x, gemm::F_RESID_INPLACE));
    if (l == 0) tap_f32(2, x, (size_t)M * E, c.st);
  }
  tap_f32(3, x, (size_t)M * E, c.st);
  RC(ew::layernorm(x, m.enc_norm.g, m.enc_norm.b, eout, nullptr, M, E, m.ln_eps, c.st));
  tap_bf16(4, eout, (size_t)M * E, c.st);
  return D3R_OK;
}

// one decoder block applied to branch `x` (fp32, updated in place) attending to ynorm (bf16, already norm_y'ed)
struct DecBufs {
  __nv_bfloat16 *ln, *qkv, *att, *q, *kv, *hid;
};
static int dec_block(const Ctx& c, const Ctx& cy, const d3r_dec_block& b, float* x, const __nv_bfloat16* ynorm, const DecBufs& w,
                     int B) {
  // c: token grid of this branch (queries), cy: token grid of the other view (memory) -- they differ for pairs whose
  // two images have different sizes (model.py:147-151 encodes such images separately)
  const d3r_model& m = *c.m;
  const int D = m.dec_dim, M = B * c.N, My = B * cy.N, hid = D * m.mlp_ratio;
  const float scale = 1.0f / sqrtf(float(D / m.dec_heads));
  RC(ew::layernorm(x, b.norm1.g, b.norm1.b, w.ln, nullptr, M, D, m.ln_eps, c.st));
  RC(linear(c, w.ln, D, b.qkv, M, 3 * D, D, w.qkv, gemm::F_ROPE, nullptr, nullptr, 2 * D));
  RC(attn::attention_hd64(w.qkv, 3 * D, w.qkv + D, 3 * D, w.qkv + 2 * D, 3 * D, w.att, D, B, m.dec_heads, c.N, c.N, scale, c.st));
  RC(linear(c, w.att, D, b.proj, M, D, D, x, gemm::F_RESID_INPLACE));
  RC(ew::layernorm(x, b.norm2.g, b.norm2.b, w.ln, nullptr, M, D, m.ln_eps, c.st));
  RC(linear(c, w.ln, D, b.projq, M, D, D, w.q, gemm::F_ROPE, nullptr, nullptr, D));
  RC(linear(cy, ynorm, D, b.projkv, My, 2 * D, D, w.kv, gemm::F_ROPE, nullptr, nullptr, D));  // k rotated (memory positions), v not
  RC(attn::attention_hd64(w.q, D, w.kv, 2 * D, w.kv + D, 2 * D, w.att, D, B, m.dec_heads, c.N, cy.N, scale, c.st));
  RC(linear(c, w.att, D, b.cproj, M, D, D, x, gemm::F_RESID_INPLACE));
  RC(ew::layernorm(x, b.norm3.g, b.norm3.b, w.ln, nullptr, M, D, m.ln_eps, c.st));
  RC(linear(c, w.ln, D, b.fc1, M, hid, D, w.hid, gemm::F_GELU));
  RC(linear(c, w.hid, hid, b.fc2, M, D, hid, x, gemm::F_RESID_INPLACE));
  return D3R_OK;
}

// ---- DPT head for one branch ---------------------------------------------------------------------
static int run_dpt(const Ctx& c, Arena& ar, const d3r_dpt_head& hd, const void* const tok[4], int B, float* pts3d, float* conf) {
  const d3r_model& m = *c.m;
  const int gh = c.gh, gw = c.gw, F = 256;
  const int dims[4] = {m.enc_dim, m.dec_dim, m.dec_dim, m.dec_dim};
  const int ld[4] = {96, 192, 384, 768};
  const int Mt = B * c.N;
  // resolutions of the four pyramid levels
  const int h3 = (gh - 1) / 2 + 1, w3 = (gw - 1) / 2 + 1;
  const int Hs[4] = {gh * 4, gh * 2, gh, h3}, Ws[4] = {gw * 4, gw * 2, gw, w3};
  typedef __nv_bfloat16 bf;
  bf* a0 = ar.arr<bf>((size_t)Mt * 96);
  bf* a1 = ar.arr<bf>((size_t)Mt * 192);
  bf* a3 = ar.arr<bf>((size_t)Mt * 768);
  bf* l[4];
  l[0] = ar.arr<bf>((size_t)B * Hs[0] * Ws[0] * 96);
  l[1] = ar.arr<bf>((size_t)B * Hs[1] * Ws[1] * 192);
  l[2] = ar.arr<bf>((size_t)Mt * 384);
  l[3] = ar.arr<bf>((size_t)B * h3 * w3 * 768);
  bf* col = ar.arr<bf>((size_t)B * h3 * w3 * 9 * 768);
  bf *r[4], *rr[4];  // layer_rn outputs: raw + relu copy
  for (int k = 0; k < 4; ++k) {
    r[k] = ar.arr<bf>((size_t)B * Hs[k] * Ws[k] * F);
    rr[k] = ar.arr<bf>((size_t)B * Hs[k] * Ws[k] * F);
  }
  const size_t big = (size_t)B * Hs[0] * Ws[0] * F;  // largest 256-channel map
  bf* t = ar.arr<bf>(big);      // conv1 output (relu'ed)
  bf* s = ar.arr<bf>(big);      // fused sum (raw)
  bf* sr = ar.arr<bf>(big);     // relu(sum)
  bf* y = ar.arr<bf>(big);      // RCU2 output
  bf* z = ar.arr<bf>(big);      // out_conv output (low res)
  bf* path = ar.arr<bf>(big * 4);  // upsampled path (level 0 output is 2x the level-0 resolution)
  const int Hf = gh * 16, Wf = gw * 16;
  bf* h0 = ar.arr<bf>((size_t)B * (Hf / 2) * (Wf / 2) * 128);
  bf* h1 = ar.arr<bf>((size_t)B * Hf * Wf * 128);
  if (ar.dry) return D3R_OK;

  // act_postprocess (dpt_block.py:341-398)
  RC(linear(c, tok[0], dims[0], hd.act_conv[0], Mt, ld[0], dims[0], a0, 0));
  RC(convT(c, a0, hd.act0_up, B, gh, gw, 96, 96, 4, l[0]));
  RC(linear(c, tok[1], dims[1], hd.act_conv[1], Mt, ld[1], dims[1], a1, 0));
  RC(convT(c, a1, hd.act1_up, B, gh, gw, 192, 192, 2, l[1]));
  RC(linear(c, tok[2], dims[2], hd.act_conv[2], Mt, ld[2], dims[2], l[2], 0));
  RC(linear(c, tok[3], dims[3], hd.act_conv[3], Mt, ld[3], dims[3], a3, 0));
  RC(ew::im2col_3x3_s2_bf16(a3, col, B, gh, gw, 768, c.st));
  RC(linear(c, col, 9 * 768, hd.act3_down, B * h3 * w3, 768, 9 * 768, l[3], 0));
  // layer_rn (no bias): raw + relu copies
  for (int k = 0; k < 4; ++k) RC(conv3(c, l[k], hd.layer_rn[k], B, Hs[k], Ws[k], ld[k], F, r[k], 0, nullptr, nullptr, rr[k]));
  tap_bf16(20, r[0], (size_t)B * Hs[0] * Ws[0] * F, c.st);
  tap_bf16(23, r[3], (size_t)B * Hs[3] * Ws[3] * F, c.st);

  // refinenet4 (single input): RCU2 -> out_conv -> x2 (cropped to level-2 size)
  const bf* prev_path = nullptr;
  for (int lvl = 3; lvl >= 0; --lvl) {
    const d3r_fusion& f = hd.refine[lvl];
    const int Hc = Hs[lvl], Wc = Ws[lvl];
    const bf *sum_raw, *sum_relu;
    if (lvl == 3) {
      sum_raw = r[3];
      sum_relu = rr[3];
    } else {
      // output = path + RCU1(r[lvl]) ; RCU1(x) = conv2(relu(conv1(relu(x)))) + x
      RC(conv3(c, rr[lvl], f.rcu1_conv1, B, Hc, Wc, F, F, t, gemm::F_RELU));
      RC(conv3(c, t, f.rcu1_conv2, B, Hc, Wc, F, F, s, 0, r[lvl], prev_path, sr));
      sum_raw = s;
      sum_relu = sr;
    }
    RC(conv3(c, sum_relu, f.rcu2_conv1, B, Hc, Wc, F, F, t, gemm::F_RELU));
    RC(conv3(c, t, f.rcu2_conv2, B, Hc, Wc, F, F, y, 0, sum_raw));
    // out_conv (1x1) commutes with the bilinear interpolation (both linear, weights sum to 1): run it on
    // the low-res map (4x fewer FLOPs), then upsample.  Same function as dpt_block.py:207-211.
    RC(linear(c, y, F, f.out_conv, B * Hc * Wc, F, F, z, 0));
    const int Ho = (lvl == 3) ? Hs[2] : 2 * Hc, Wo = (lvl == 3) ? Ws[2] : 2 * Wc;
    RC(ew::upsample2x_bf16(z, path, B, Hc, Wc, F, Ho, Wo, c.st));
    prev_path = path;
    if (lvl == 3) tap_bf16(24, path, (size_t)B * Ho * Wo * F, c.st);
    if (lvl == 0) tap_bf16(21, path, (size_t)B * Ho * Wo * F, c.st);
    // `path` is consumed by the next level's rcu1_conv2 epilogue before being overwritten (stream order)
  }
  // head: conv3x3 256->128, x2, conv3x3 128->128 + ReLU + 1x1 conv + postprocess (fused tail)
  const int Hp = Hs[0] * 2, Wp = Ws[0] * 2;
  RC(conv3(c, path, hd.head0, B, Hp, Wp, F, 128, h0, 0));
  RC(ew::upsample2x_bf16(h0, h1, B, Hp, Wp, 128, Hf, Wf, c.st));
  RC(gemm::conv3x3_head_tail(h1, hd.head2.w, hd.head2.b, hd.head4_w, hd.head4_b, pts3d, m.nch > 3 ? conf : nullptr, B, Hf, Wf,
                             m.depth_mode, m.conf_mode, m.conf_min, m.conf_max, c.st));
  return D3R_OK;
}

// decoder + heads.  cv[br]: token grid of view br; enc[br]: encoder output holding view br's images; maps_host[br]: image
// index of each pair inside enc[br] (nullptr = identity, pair b uses image b).
static int decode_heads(const d3r_model* mp, const Ctx cv[2], const void* const enc[2], const int32_t* const maps_host[2], int B,
                        float* pts1, float* conf1, float* pts2, float* conf2, Arena& ar, cudaStream_t st) {
  const d3r_model& m = *mp;
  const int E = m.enc_dim, D = m.dec_dim, hid = D * m.mlp_ratio;
  const int Md[2] = {B * cv[0].N, B * cv[1].N};
  const int Mx = Md[0] > Md[1] ? Md[0] : Md[1];
  typedef __nv_bfloat16 bf;

  // per-pair encoder features (bf16): f[br] = enc[br][maps[br]]
  bf* f[2];
  f[0] = ar.arr<bf>((size_t)Md[0] * E);
  f[1] = ar.arr<bf>((size_t)Md[1] * E);
  int* maps = ar.arr<int>((size_t)2 * B);
  float* x[2] = {ar.arr<float>((size_t)Md[0] * D), ar.arr<float>((size_t)Md[1] * D)};
  bf* yn[2] = {ar.arr<bf>((size_t)Md[1] * D), ar.arr<bf>((size_t)Md[0] * D)};   // yn[br]: the OTHER view, normalised for branch br
  DecBufs w;
  w.ln = ar.arr<bf>((size_t)Mx * D);
  w.qkv = ar.arr<bf>((size_t)Mx * 3 * D);
  w.att = ar.arr<bf>((size_t)Mx * D);
  w.q = ar.arr<bf>((size_t)Mx * D);
  w.kv = ar.arr<bf>((size_t)Mx * 2 * D);
  w.hid = ar.arr<bf>((size_t)Mx * hid);
  // hooked decoder outputs (bf16): hooks[1], hooks[2] raw; hooks[3] (= last) after dec_norm
  bf* hook[2][3];
  for (int br = 0; br < 2; ++br)
    for (int k = 0; k < 3; ++k) hook[br][k] = ar.arr<bf>((size_t)Md[br] * D);
  float* lin_feat = nullptr;
  if (m.head_type == 0) lin_feat = ar.arr<float>((size_t)Mx * m.nch * m.patch * m.patch);

  const size_t mark_head = ar.off;
  if (m.head_type == 1) {
    // both heads reuse the same scratch region (sized for the larger view)
    size_t top = ar.off;
    for (int br = 0; br < 2; ++br) {
      Arena probe = ar;
      const void* none[4] = {nullptr, nullptr, nullptr, nullptr};
      probe.dry = true;
      RC(run_dpt(cv[br], probe, *m.dpt[br], none, B, nullptr, nullptr));
      if (probe.off > top) top = probe.off;
    }
    if (ar.dry) ar.off = top;
  }
  if (ar.dry) return D3R_OK;

  if (ar.off > ar.cap && m.head_type != 1) {
    set_error("forward: workspace too small (%zu > %zu bytes)", ar.off, ar.cap);
    return D3R_ERR_INVALID;
  }

  for (int br = 0; br < 2; ++br) {
    if (maps_host[br]) {
      D3R_CUDA(cudaMemcpyAsync(maps + br * B, maps_host[br], sizeof(int) * B, cudaMemcpyHostToDevice, st));
      RC(ew::gather_images_bf16(enc[br], f[br], maps + br * B, B, cv[br].N, E, st));
    } else {
      D3R_CUDA(cudaMemcpyAsync(f[br], enc[br], sizeof(bf) * (size_t)Md[br] * E, cudaMemcpyDeviceToDevice, st));
    }
  }

  // decoder (model.py:172-191)
  RC(linear(cv[0], f[0], E, m.decoder_embed, Md[0], D, E, x[0], gemm::F_OUT_F32));
  RC(linear(cv[1], f[1], E, m.decoder_embed, Md[1], D, E, x[1], gemm::F_OUT_F32));
  tap_f32(5, x[0], (size_t)Md[0] * D, st);
  for (int l = 0; l < m.dec_depth; ++l) {
    // memory normalisation of the *previous* outputs, each with the consuming block's norm_y
    RC(ew::layernorm(x[1], m.dec1[l].norm_y.g, m.dec1[l].norm_y.b, yn[0], nullptr, Md[1], D, m.ln_eps, st));  // for branch 1
    RC(ew::layernorm(x[0], m.dec2[l].norm_y.g, m.dec2[l].norm_y.b, yn[1], nullptr, Md[0], D, m.ln_eps, st));  // for branch 2
    RC(dec_block(cv[0], cv[1], m.dec1[l], x[0], yn[0], w, B));
    RC(dec_block(cv[1], cv[0], m.dec2[l], x[1], yn[1], w, B));
    if (l == 0) { tap_f32(6, x[0], (size_t)Md[0] * D, st); tap_f32(7, x[1], (size_t)Md[1] * D, st); }
    for (int k = 1; k <= 2; ++k) {
      if (m.head_type == 1 && l + 1 == m.hooks[k]) {
        RC(ew::cast_f32_bf16(x[0], hook[0][k - 1], (size_t)Md[0] * D, st));
        RC(ew::cast_f32_bf16(x[1], hook[1][k - 1], (size_t)Md[1] * D, st));
      }
    }
  }
  tap_f32(8, x[0], (size_t)Md[0] * D, st);
  tap_f32(9, x[1], (size_t)Md[1] * D, st);
  RC(ew::layernorm(x[0], m.dec_norm.g, m.dec_norm.b, hook[0][2], nullptr, Md[0], D, m.ln_eps, st));
  RC(ew::layernorm(x[1], m.dec_norm.g, m.dec_norm.b, hook[1][2], nullptr, Md[1], D, m.ln_eps, st));

  float* outs[2][2] = {{pts1, conf1}, {pts2, conf2}};
  if (m.head_type == 0) {
    const int nf = m.nch * m.patch * m.patch;
    for (int br = 0; br < 2; ++br) {
      RC(linear(cv[br], hook[br][2], D, m.lin_head[br], Md[br], nf, D, lin_feat, gemm::F_OUT_F32));
      RC(ew::linear_head_postprocess(lin_feat, outs[br][0], outs[br][1], B, cv[br].gh, cv[br].gw, m.nch, m.depth_mode, m.conf_mode,
                                     m.conf_min, m.conf_max, st));
    }
  } else {
    for (int br = 0; br < 2; ++br) {
      Arena head = ar;
      head.off = mark_head;
      const void* tok[4] = {f[br], hook[br][0], hook[br][1], hook[br][2]};
      RC(run_dpt(cv[br], head, *m.dpt[br], tok, B, outs[br][0], outs[br][1]));
      if (head.off > head.cap) {
        set_error("forward: workspace too small (%zu > %zu bytes)", head.off, head.cap);
        return D3R_ERR_INVALID;
      }
    }
  }
  return D3R_OK;
}

// all images share one size: one encoder pass over the n_enc distinct images, pairs address them through idx1 / idx2
static int forward(const d3r_model* mp, const float* imgs, int n_enc, const int32_t* idx1, const int32_t* idx2, int B, int H, int W,
                   float* pts1, float* conf1, float* pts2, float* conf2, Arena& ar, cudaStream_t st) {
  const d3r_model& m = *mp;
  Ctx c{mp, st, H / m.patch, W / m.patch, (H / m.patch) * (W / m.patch)};
  void* enc_out = nullptr;
  RC(run_encoder(c, ar, imgs, n_enc, H, W, &enc_out));
  const Ctx cv[2] = {c, c};
  const void* enc[2] = {enc_out, enc_out};
  const int32_t* maps[2] = {idx1, idx2};
  // a dry (size-only) pass has no index lists; the gather path is what the real call takes
  static const int32_t kDummy = 0;
  if (ar.dry) maps[0] = maps[1] = &kDummy;
  return decode_heads(mp, cv, enc, maps, B, pts1, conf1, pts2, conf2, ar, st);
}

// the two views of every pair have different sizes (all first views H1 x W1, all second views H2 x W2): the reference
// encodes them separately (model.py:147-151) and the decoder cross-attends between the two token grids
static int forward_mixed(const d3r_model* mp, const float* imgs1, int H1, int W1, const float* imgs2, int H2, int W2, int B, float* pts1,
                         float* conf1, float* pts2, float* conf2, Arena& ar, cudaStream_t st) {
  const d3r_model& m = *mp;
  const Ctx cv[2] = {Ctx{mp, st, H1 / m.patch, W1 / m.patch, (H1 / m.patch) * (W1 / m.patch)},
                     Ctx{mp, st, H2 / m.patch, W2 / m.patch, (H2 / m.patch) * (W2 / m.patch)}};
  void* e[2] = {nullptr, nullptr};
  RC(run_encoder(cv[0], ar, imgs1, B, H1, W1, &e[0]));
  RC(run_encoder(cv[1], ar, imgs2, B, H2, W2, &e[1]));
  const void* enc[2] = {e[0], e[1]};
  const int32_t* maps[2] = {nullptr, nullptr};
  return decode_heads(mp, cv, enc, maps, B, pts1, conf1, pts2, conf2, ar, st);
}

}  // namespace fwd
}  // namespace d3r

using namespace d3r;

static int check_model(const d3r_model* m, int H, int W) {
  D3R_CHECK_ARG(m != nullptr, "forward: null model");
  D3R_CHECK_ARG(m->patch == 16, "forward: patch size %d unsupported (16 only)", m->patch);
  D3R_CHECK_ARG(m->enc_dim % 64 == 0 && m->enc_dim / m->enc_heads == 64, "forward: encoder head dim must be 64");
  D3R_CHECK_ARG(m->dec_dim % 64 == 0 && m->dec_dim / m->dec_heads == 64, "forward: decoder head dim must be 64");
  D3R_CHECK_ARG(H > 0 && W > 0 && H % 16 == 0 && W % 16 == 0, "forward: image %dx%d is not a multiple of the patch size", H, W);
  D3R_CHECK_ARG(m->rope_cos && m->rope_sin && m->rope_max_pos >= (H > W ? H : W) / 16, "forward: RoPE tables too small");
  D3R_CHECK_ARG(m->head_type == 0 || m->head_type == 1, "forward: bad head type");
  D3R_CHECK_ARG(m->head_type == 0 || (m->enc_dim % 32 == 0 && m->dpt[0] && m->dpt[1]), "forward: missing DPT weights");
  return D3R_OK;
}

extern "C" int64_t d3r_forward_workspace_bytes(const d3r_model* m, int32_t n_enc, int32_t B, int32_t H, int32_t W) {
  if (check_model(m, H, W)) return -1;
  fwd::Arena ar{nullptr, 0, 0, true};
  if (fwd::forward(m, nullptr, n_enc, nullptr, nullptr, B, H, W, nullptr, nullptr, nullptr, nullptr, ar, 0)) return -1;
  return (int64_t)ar.off + 4096;
}

extern "C" int d3r_forward_pairs(const d3r_model* m, const float* imgs_dev, int32_t n_enc, const int32_t* idx1_host,
                                 const int32_t* idx2_host, int32_t B, int32_t H, int32_t W, float* pts3d_1, float* conf_1,
                                 float* pts3d_2, float* conf_2, void* workspace_dev, int64_t workspace_bytes, void* stream) {
  int rc = check_model(m, H, W);
  if (rc) return rc;
  D3R_CHECK_ARG(imgs_dev && idx1_host && idx2_host && pts3d_1 && pts3d_2 && workspace_dev, "forward: null buffer");
  D3R_CHECK_ARG(n_enc > 0 && B > 0, "forward: empty batch");
  for (int b = 0; b < B; ++b)
    D3R_CHECK_ARG(idx1_host[b] >= 0 && idx1_host[b] < n_enc && idx2_host[b] >= 0 && idx2_host[b] < n_enc, "forward: pair index out of range");
  const int64_t need = d3r_forward_workspace_bytes(m, n_enc, B, H, W);
  D3R_CHECK_ARG(need > 0 && workspace_bytes >= need, "forward: workspace of %lld bytes needed, %lld given", (long long)need, (long long)workspace_bytes);
  fwd::Arena ar{reinterpret_cast<uint8_t*>(workspace_dev), (size_t)workspace_bytes, 0, false};
  rc = fwd::forward(m, imgs_dev, n_enc, idx1_host, idx2_host, B, H, W, pts3d_1, conf_1, pts3d_2, conf_2, ar, (cudaStream_t)stream);
  fwd::g_tap = {-1, nullptr, 0};
  return rc;
}

extern "C" int64_t d3r_forward_mixed_workspace_bytes(const d3r_model* m, int32_t B, int32_t H1, int32_t W1, int32_t H2, int32_t W2) {
  if (check_model(m, H1, W1) || check_model(m, H2, W2)) return -1;
  fwd::Arena ar{nullptr, 0, 0, true};
  if (fwd::forward_mixed(m, nullptr, H1, W1, nullptr, H2, W2, B, nullptr, nullptr, nullptr, nullptr, ar, 0)) return -1;
  return (int64_t)ar.off + 4096;
}

extern "C" int d3r_forward_pairs_mixed(const d3r_model* m, const float* imgs1_dev, int32_t H1, int32_t W1, const float* imgs2_dev,
                                       int32_t H2, int32_t W2, int32_t B, float* pts3d_1, float* conf_1, float* pts3d_2,
                                       float* conf_2, void* workspace_dev, int64_t workspace_bytes, void* stream) {
  int rc = check_model(m, H1, W1);
  if (rc) return rc;
  if ((rc = check_model(m, H2, W2))) return rc;
  D3R_CHECK_ARG(imgs1_dev && imgs2_dev && pts3d_1 && pts3d_2 && workspace_dev, "forward: null buffer");
  D3R_CHECK_ARG(B > 0, "forward: empty batch");
  const int64_t need = d3r_forward_mixed_workspace_bytes(m, B, H1, W1, H2, W2);
  D3R_CHECK_ARG(need > 0 && workspace_bytes >= need, "forward: workspace of %lld bytes needed, %lld given", (long long)need, (long long)workspace_bytes);
  fwd::Arena ar{reinterpret_cast<uint8_t*>(workspace_dev), (size_t)workspace_bytes, 0, false};
  rc = fwd::forward_mixed(m, imgs1_dev, H1, W1, imgs2_dev, H2, W2, B, pts3d_1, conf_1, pts3d_2, conf_2, ar, (cudaStream_t)stream);
  fwd::g_tap = {-1, nullptr, 0};
  return rc;
}

extern "C" int d3r_sizeof_model(void) { return (int)sizeof(d3r_model); }

extern "C" int d3r_forward_set_debug(int32_t stage_id, float* out_dev, int64_t capacity_floats) {
  fwd::g_tap = {stage_id, out_dev, capacity_floats};
  return D3R_OK;
}
