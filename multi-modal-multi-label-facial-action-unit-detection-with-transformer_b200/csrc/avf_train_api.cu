// Training half of the C ABI (include/avformer_b200.h, section "training"): the encoder stack with an activation
// tape, its backward, the AU_former front end with batch statistics, and the small backward / optimiser entry points.
// Host-side orchestration only — kernels live in avf_train.cu, avf_gemm_umma.cu, avf_simt.cu, avf_rowops.cu.
#include <algorithm>
#include <cstring>

#include "avf_common.cuh"
#include "avf_internal.h"

namespace avf {

static inline size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }
static inline size_t elt(int mode) { return mode == AVF_BF16 ? 2 : 4; }

// Per-layer activation tape (what the backward pass re-reads).  e = 2 bytes (bf16 mode) or 4 (fp32 mode).
struct LayerTape {
  float* x_in;    // [R, D]  fp32 residual stream entering the attention sub-layer
  void* xn1;      // [R, D]  e    LN1(x_in)
  void* qkv;      // [R, 3I] e
  void* o;        // [R, I]  e    merged heads
  float* x_mid;   // [R, D]  fp32 residual stream entering the MLP sub-layer
  void* xn2;      // [R, D]  e    LN2(x_mid)
  void* hpre;     // [R, M]  e    W1 xn2 + b1
  void* g;        // [R, M]  e    gelu(hpre)
};

static size_t layer_tape_bytes(const avf_stack_shape* s, int mode) {
  const size_t R = size_t(s->n_seq) * s->n_tok, D = s->dim, I = size_t(s->heads) * s->dim_head, M = s->mlp_dim, e = elt(mode);
  return 2 * align_up(R * D * 4) + 2 * align_up(R * D * e) + align_up(R * 3 * I * e) + align_up(R * I * e) + 2 * align_up(R * M * e);
}

static LayerTape carve_tape(const avf_stack_shape* s, int mode, void* base, int layer) {
  const size_t R = size_t(s->n_seq) * s->n_tok, D = s->dim, I = size_t(s->heads) * s->dim_head, M = s->mlp_dim, e = elt(mode);
  uint8_t* p = static_cast<uint8_t*>(base) + size_t(layer) * layer_tape_bytes(s, mode);
  LayerTape t;
  t.x_in = reinterpret_cast<float*>(p);  p += align_up(R * D * 4);
  t.xn1 = p;                             p += align_up(R * D * e);
  t.qkv = p;                             p += align_up(R * 3 * I * e);
  t.o = p;                               p += align_up(R * I * e);
  t.x_mid = reinterpret_cast<float*>(p); p += align_up(R * D * 4);
  t.xn2 = p;                             p += align_up(R * D * e);
  t.hpre = p;                            p += align_up(R * M * e);
  t.g = p;
  return t;
}

static int check_train_shape(const avf_stack_shape* s) {
  AVF_REQUIRE(s != nullptr, AVF_EINVAL, "null stack shape");
  AVF_REQUIRE(s->n_seq > 0 && s->n_tok > 0 && s->depth > 0, AVF_EINVAL, "empty stack: n_seq=%d n_tok=%d depth=%d", s->n_seq, s->n_tok, s->depth);
  AVF_REQUIRE(s->dim % 128 == 0 && s->dim <= 512, AVF_EUNSUPPORTED, "training: dim=%d must be a multiple of 128 (<= 512)", s->dim);
  AVF_REQUIRE(s->dim_head == 32 || s->dim_head == 64, AVF_EUNSUPPORTED, "dim_head=%d (supported: 32, 64)", s->dim_head);
  AVF_REQUIRE((s->heads * s->dim_head) % 64 == 0 && s->mlp_dim % 64 == 0, AVF_EUNSUPPORTED, "inner=%d / mlp=%d must be multiples of 64",
              s->heads * s->dim_head, s->mlp_dim);
  AVF_REQUIRE(s->n_tok <= 64 || s->dim_head == 64, AVF_EUNSUPPORTED,
              "n_tok=%d: sequences longer than 64 tokens are not part of this path for dim_head=%d", s->n_tok, s->dim_head);
  AVF_REQUIRE(s->n_tok <= 256, AVF_EUNSUPPORTED, "n_tok=%d: sequences longer than 256 tokens are not part of this path", s->n_tok);
  return 0;
}

// C = epi(op(A) op(B)) in either arithmetic mode (see gemm_umma for the operand conventions).
int gemm(int mode, int ta, int tb, const void* a, int lda, const void* b, int ldb, const float* bias, const float* res, int ld_res,
         void* aux, int ld_aux, void* c, int ldc, int c_mode, int m, int n, int k, int flags, void* ws, size_t ws_bytes, cudaStream_t st,
         DropSpec drop = DropSpec{}) {
  if (drop.thresh != 0) flags |= AVF_EPI_DROPOUT;
  if (mode == AVF_BF16)
    return gemm_umma(ta, tb, a, lda, b, ldb, bias, res, ld_res, aux, ld_aux, c, ldc, c_mode, m, n, k, flags, ws, ws_bytes, st, drop);
  return gemm_f32(ta, tb, static_cast<const float*>(a), lda, static_cast<const float*>(b), ldb, bias, res, ld_res, static_cast<float*>(aux),
                  ld_aux, c, ldc, c_mode, m, n, k, flags, st, drop);
}

// Dropout site (layer, 0 = after to_out, 1 = after GELU, 2 = after net.3): models/heads.py:216,194,197
static DropSpec drop_site(float p, uint64_t seed, const uint32_t* salt, int layer, int site) {
  DropSpec d;
  if (!(p > 0.f)) return d;
  d.salt = salt;
  d.seed = mix32(uint32_t(seed) ^ mix32(uint32_t(seed >> 32) + 0x9E3779B9u * uint32_t(layer * 3 + site + 1)));
  const double t = double(p) * 4294967296.0;
  d.thresh = t >= 4294967295.0 ? 4294967295u : uint32_t(t);
  d.scale = 1.f / (1.f - p);
  return d;
}

static int copy_rows(float* dst, int ld_dst, const float* src, int ld_src, int rows, int dim, cudaStream_t st) {
  AVF_CUDA(cudaMemcpy2DAsync(dst, size_t(ld_dst) * 4, src, size_t(ld_src) * 4, size_t(dim) * 4, rows, cudaMemcpyDeviceToDevice, st));
  return 0;
}

// ---------------------------------------------------------------------------------------------
// forward with tape:  the residual stream walks x_in(0) -> x_mid(0) -> x_in(1) -> ... -> out
// keep (optional, [n_seq, n_tok] uint8): attention mask of every layer; the backward needs the same one
// ---------------------------------------------------------------------------------------------
static int encoder_fwd_train(int mode, const avf_stack_shape* s, const avf_layer_weights* L, const float* x, int ld_x, float* out, int ld_out,
                             void* tape, size_t tape_bytes, float p_drop, uint64_t seed, const uint32_t* salt, cudaStream_t st,
                             const uint8_t* keep = nullptr) {
  int e = check_train_shape(s);
  if (e) return e;
  AVF_REQUIRE(p_drop >= 0.f && p_drop < 1.f, AVF_EINVAL, "dropout p=%f", p_drop);
  AVF_REQUIRE(mode == AVF_BF16 || mode == AVF_FP32, AVF_EINVAL, "mode=%d", mode);
  AVF_REQUIRE(L && x && out && tape, AVF_EINVAL, "encoder_stack_fwd_train: null pointer");
  const size_t need = layer_tape_bytes(s, mode) * s->depth;
  AVF_REQUIRE(tape_bytes >= need, AVF_EWORKSPACE, "tape too small: %zu < %zu bytes", tape_bytes, need);
  const int R = s->n_seq * s->n_tok, D = s->dim, I = s->heads * s->dim_head, M = s->mlp_dim;
  LayerTape t = carve_tape(s, mode, tape, 0);
  if ((e = copy_rows(t.x_in, D, x, ld_x, R, D, st))) return e;
  for (int l = 0; l < s->depth; ++l) {
    const avf_layer_weights& W = L[l];
    t = carve_tape(s, mode, tape, l);
    const bool last = l == s->depth - 1;
    float* next = last ? out : carve_tape(s, mode, tape, l + 1).x_in;
    const int ld_next = last ? ld_out : D;
    if ((e = layernorm(mode, t.x_in, D, W.ln1_gamma, W.ln1_beta, t.xn1, R, D, st))) return e;
    if ((e = gemm(mode, 0, 0, t.xn1, D, W.w_qkv, D, nullptr, nullptr, 0, nullptr, 0, t.qkv, 3 * I, mode, R, 3 * I, D, 0, nullptr, 0, st))) return e;
    if ((e = attention_small(mode, t.qkv, t.o, s->n_seq, s->n_tok, s->heads, s->dim_head, st, keep))) return e;
    if ((e = gemm(mode, 0, 0, t.o, I, W.w_out, I, W.b_out, t.x_in, D, nullptr, 0, t.x_mid, D, AVF_FP32, R, D, I, AVF_EPI_BIAS | AVF_EPI_RESIDUAL,
                  nullptr, 0, st, drop_site(p_drop, seed, salt, l, 0))))
      return e;
    if ((e = layernorm(mode, t.x_mid, D, W.ln2_gamma, W.ln2_beta, t.xn2, R, D, st))) return e;
    if ((e = gemm(mode, 0, 0, t.xn2, D, W.w_ff1, D, W.b_ff1, nullptr, 0, t.hpre, M, t.g, M, mode, R, M, D,
                  AVF_EPI_BIAS | AVF_EPI_SAVE_PRE | AVF_EPI_GELU, nullptr, 0, st, drop_site(p_drop, seed, salt, l, 1))))
      return e;
    if ((e = gemm(mode, 0, 0, t.g, M, W.w_ff2, M, W.b_ff2, t.x_mid, D, nullptr, 0, next, ld_next, AVF_FP32, R, D, M,
                  AVF_EPI_BIAS | AVF_EPI_RESIDUAL, nullptr, 0, st, drop_site(p_drop, seed, salt, l, 2))))
      return e;
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------
// backward
// ---------------------------------------------------------------------------------------------
struct BwdWs {
  void* dyb;     // [R, D]            e: GEMM-operand copy of the gradient stream (masked by the consumer's dropout); fp32 mode
                 //                      without dropout reads the stream itself
  float* dxn;    // [R, D]            fp32 gradient wrt a LayerNorm output
  void* big;     // [R, max(M, 3I)]   e: dh, then dqkv
  void* dob;     // [R, I]            e
  void* red;     // reductions: split-K partial tiles / LayerNorm and column-sum partials
  size_t red_bytes, total;
};

static BwdWs carve_bwd_ws(const avf_stack_shape* s, int mode, void* base) {
  const size_t R = size_t(s->n_seq) * s->n_tok, D = s->dim, I = size_t(s->heads) * s->dim_head, M = s->mlp_dim, e = elt(mode);
  uint8_t* p = static_cast<uint8_t*>(base);
  BwdWs w;
  size_t off = 0;
  w.dyb = p + off;                             off += align_up(R * D * e);
  w.dxn = reinterpret_cast<float*>(p + off);   off += align_up(R * D * 4);
  w.big = p + off;                             off += align_up(R * std::max(M, 3 * I) * e);
  w.dob = p + off;                             off += align_up(R * I * e);
  size_t red = std::max(layernorm_bwd_workspace_bytes(int(R), int(D)), colsum_workspace_bytes(int(R), int(M)));
  if (mode == AVF_BF16) {
    red = std::max(red, gemm_umma_workspace_bytes(int(D), int(M), int(R)));
    red = std::max(red, gemm_umma_workspace_bytes(int(M), int(D), int(R)));
    red = std::max(red, gemm_umma_workspace_bytes(int(D), int(I), int(R)));
    red = std::max(red, gemm_umma_workspace_bytes(int(3 * I), int(D), int(R)));
  }
  w.red = p + off;
  w.red_bytes = align_up(red);
  off += w.red_bytes;
  w.total = off;
  return w;
}

// gmaps (optional): layer l's gradient map G = P o dP goes to gmaps + l * n_seq*heads*n_tok*n_tok (fp32 [depth, n_seq, heads, n_tok, n_tok]),
// written by that layer's attention backward launch.
static int encoder_bwd(int mode, const avf_stack_shape* s, const avf_layer_weights* L, const void* tape, size_t tape_bytes, float* dx, int ld_dx,
                       const avf_layer_grads* G, int accumulate, void* ws, size_t ws_bytes, float p_drop, uint64_t seed, const uint32_t* salt,
                       cudaStream_t st, const uint8_t* keep = nullptr, float* gmaps = nullptr) {
  int e = check_train_shape(s);
  if (e) return e;
  AVF_REQUIRE(p_drop >= 0.f && p_drop < 1.f, AVF_EINVAL, "dropout p=%f", p_drop);
  const bool dropping = p_drop > 0.f;
  const int wg = accumulate ? AVF_EPI_ACCUMULATE : 0;       // wgrad epilogue
  const float beta = accumulate ? 1.f : 0.f;
  AVF_REQUIRE(mode == AVF_BF16 || mode == AVF_FP32, AVF_EINVAL, "mode=%d", mode);
  AVF_REQUIRE(L && tape && dx && ws, AVF_EINVAL, "encoder_stack_bwd: null pointer");
  AVF_REQUIRE(tape_bytes >= layer_tape_bytes(s, mode) * s->depth, AVF_EWORKSPACE, "tape too small");
  const BwdWs w = carve_bwd_ws(s, mode, ws);
  AVF_REQUIRE(ws_bytes >= w.total, AVF_EWORKSPACE, "workspace too small: %zu < %zu bytes", ws_bytes, w.total);
  AVF_REQUIRE(ld_dx == s->dim, AVF_EINVAL, "encoder_stack_bwd: the gradient stream must be dense (ld_dx=%d, dim=%d)", ld_dx, s->dim);
  const int R = s->n_seq * s->n_tok, D = s->dim, I = s->heads * s->dim_head, M = s->mlp_dim;
  static const avf_layer_grads none = {};
  // GEMM-operand copy of the incoming gradient: bf16 and / or masked by the dropout on the top layer's output
  // (fp32 mode without dropout: the GEMMs read the stream directly)
  const void* dyb = dx;
  int ld_dyb = ld_dx;
  if (mode == AVF_BF16 || dropping) {
    if ((e = masked_copy(dx, w.dyb, mode, R, D, drop_site(p_drop, seed, salt, s->depth - 1, 2), st))) return e;
    dyb = w.dyb;
    ld_dyb = D;
  }
  void* dxb_out = (mode == AVF_BF16 || dropping) ? w.dyb : nullptr;
  for (int l = s->depth - 1; l >= 0; --l) {
    const avf_layer_weights& W = L[l];
    const avf_layer_grads& g = G ? G[l] : none;
    const LayerTape t = carve_tape(s, mode, const_cast<void*>(tape), l);
    // ---- MLP sub-layer:  y = x_mid + W2 gelu(W1 LN2(x_mid) + b1) + b2 ---------------------------------------
    if (g.w_ff2 && (e = gemm(mode, 1, 1, dyb, ld_dyb, t.g, M, nullptr, nullptr, 0, nullptr, 0, g.w_ff2, M, AVF_FP32, D, M, R, wg, w.red, w.red_bytes, st))) return e;
    if ((e = gemm(mode, 0, 1, dyb, ld_dyb, W.w_ff2, M, nullptr, nullptr, 0, t.hpre, M, w.big, M, mode, R, M, D, AVF_EPI_DGELU, nullptr, 0, st,
                  drop_site(p_drop, seed, salt, l, 1))))
      return e;
    if (g.w_ff1 && (e = gemm(mode, 1, 1, w.big, M, t.xn2, D, nullptr, nullptr, 0, nullptr, 0, g.w_ff1, D, AVF_FP32, M, D, R, wg, w.red, w.red_bytes, st))) return e;
    if (g.b_ff1 && (e = colsum(mode, w.big, M, R, M, g.b_ff1, beta, w.red, w.red_bytes, st))) return e;
    if ((e = gemm(mode, 0, 1, w.big, M, W.w_ff1, D, nullptr, nullptr, 0, nullptr, 0, w.dxn, D, AVF_FP32, R, D, M, 0, nullptr, 0, st))) return e;
    if ((e = layernorm_bwd(t.x_mid, D, W.ln2_gamma, w.dxn, dx, ld_dx, dxb_out, mode, g.ln2_gamma, g.ln2_beta, g.b_ff2, beta, R, D, w.red, w.red_bytes, st,
                           drop_site(p_drop, seed, salt, l, 2), drop_site(p_drop, seed, salt, l, 0))))
      return e;
    // ---- attention sub-layer:  x_mid = x_in + Wo attn(Wqkv LN1(x_in)) + bo -----------------------------------
    if (g.w_out && (e = gemm(mode, 1, 1, dyb, ld_dyb, t.o, I, nullptr, nullptr, 0, nullptr, 0, g.w_out, I, AVF_FP32, D, I, R, wg, w.red, w.red_bytes, st))) return e;
    if ((e = gemm(mode, 0, 1, dyb, ld_dyb, W.w_out, I, nullptr, nullptr, 0, nullptr, 0, w.dob, I, mode, R, I, D, 0, nullptr, 0, st))) return e;
    float* gmap = gmaps ? gmaps + size_t(l) * s->n_seq * s->heads * s->n_tok * s->n_tok : nullptr;
    if ((e = attention_bwd(mode, t.qkv, w.dob, w.big, s->n_seq, s->n_tok, s->heads, s->dim_head, st, keep, gmap))) return e;
    if (g.w_qkv && (e = gemm(mode, 1, 1, w.big, 3 * I, t.xn1, D, nullptr, nullptr, 0, nullptr, 0, g.w_qkv, D, AVF_FP32, 3 * I, D, R, wg, w.red, w.red_bytes, st))) return e;
    if ((e = gemm(mode, 0, 1, w.big, 3 * I, W.w_qkv, D, nullptr, nullptr, 0, nullptr, 0, w.dxn, D, AVF_FP32, R, D, 3 * I, 0, nullptr, 0, st))) return e;
    if ((e = layernorm_bwd(t.x_in, D, W.ln1_gamma, w.dxn, dx, ld_dx, dxb_out, mode, g.ln1_gamma, g.ln1_beta, g.b_out, beta, R, D, w.red, w.red_bytes, st,
                           drop_site(p_drop, seed, salt, l, 0), l > 0 ? drop_site(p_drop, seed, salt, l - 1, 2) : DropSpec{})))
      return e;
  }
  return 0;
}

static int require_device_train() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    cudaGetLastError();
    set_error("no CUDA device: the AVFormer B200 path has no CPU fallback");
    return AVF_ENODEVICE;
  }
  return 0;
}

}  // namespace avf

using namespace avf;

extern "C" {

size_t avf_encoder_tape_bytes(const avf_stack_shape* s, int mode) {
  if (s == nullptr || s->n_seq <= 0 || s->n_tok <= 0 || s->depth <= 0) return 0;
  return layer_tape_bytes(s, mode) * s->depth;
}

size_t avf_encoder_bwd_workspace_bytes(const avf_stack_shape* s, int mode) {
  if (s == nullptr || s->n_seq <= 0 || s->n_tok <= 0) return 0;
  return carve_bwd_ws(s, mode, nullptr).total;
}

int avf_encoder_stack_fwd_train(int mode, const avf_stack_shape* s, const avf_layer_weights* layers, const float* x, int32_t ld_x, float* out,
                                int32_t ld_out, void* tape, size_t tape_bytes, float dropout_p, uint64_t dropout_seed, const uint32_t* dropout_salt,
                                void* stream) {
  int e = require_device_train();
  if (e) return e;
  return encoder_fwd_train(mode, s, layers, x, ld_x, out, ld_out, tape, tape_bytes, dropout_p, dropout_seed, dropout_salt, static_cast<cudaStream_t>(stream));
}

int avf_encoder_stack_bwd(int mode, const avf_stack_shape* s, const avf_layer_weights* layers, const void* tape, size_t tape_bytes, float* dx,
                          int32_t ld_dx, const avf_layer_grads* grads, int accumulate, void* workspace, size_t workspace_bytes, float dropout_p,
                          uint64_t dropout_seed, const uint32_t* dropout_salt, void* stream) {
  int e = require_device_train();
  if (e) return e;
  return encoder_bwd(mode, s, layers, tape, tape_bytes, dx, ld_dx, grads, accumulate, workspace, workspace_bytes, dropout_p, dropout_seed, dropout_salt,
                     static_cast<cudaStream_t>(stream));
}

int avf_encoder_stack_fwd_train_masked(int mode, const avf_stack_shape* s, const avf_layer_weights* layers, const uint8_t* keep, const float* x,
                                       int32_t ld_x, float* out, int32_t ld_out, void* tape, size_t tape_bytes, float dropout_p, uint64_t dropout_seed,
                                       const uint32_t* dropout_salt, void* stream) {
  int e = require_device_train();
  if (e) return e;
  return encoder_fwd_train(mode, s, layers, x, ld_x, out, ld_out, tape, tape_bytes, dropout_p, dropout_seed, dropout_salt, static_cast<cudaStream_t>(stream),
                           keep);
}

int avf_encoder_stack_bwd_masked(int mode, const avf_stack_shape* s, const avf_layer_weights* layers, const uint8_t* keep, const void* tape,
                                 size_t tape_bytes, float* dx, int32_t ld_dx, const avf_layer_grads* grads, int accumulate, void* workspace,
                                 size_t workspace_bytes, float dropout_p, uint64_t dropout_seed, const uint32_t* dropout_salt, void* stream) {
  int e = require_device_train();
  if (e) return e;
  return encoder_bwd(mode, s, layers, tape, tape_bytes, dx, ld_dx, grads, accumulate, workspace, workspace_bytes, dropout_p, dropout_seed, dropout_salt,
                     static_cast<cudaStream_t>(stream), keep);
}

int avf_dropout_mask(float dropout_p, uint64_t dropout_seed, const uint32_t* dropout_salt, int32_t layer, int32_t site, int32_t rows,
                     int32_t cols, float* out, void* stream) {
  int e = require_device_train();
  if (e) return e;
  AVF_REQUIRE(dropout_p >= 0.f && dropout_p < 1.f && site >= 0 && site < 3 && layer >= 0, AVF_EINVAL, "dropout_mask: p=%f layer=%d site=%d", dropout_p, layer, site);
  return dropout_mask(out, rows, cols, drop_site(dropout_p, dropout_seed, dropout_salt, layer, site), static_cast<cudaStream_t>(stream));
}

size_t avf_gemm_workspace_bytes(int mode, int trans_a, int trans_b, int32_t m, int32_t n, int32_t k) {
  return (mode == AVF_BF16 && trans_a && trans_b) ? gemm_umma_workspace_bytes(m, n, k) : 0;
}

int avf_gemm(int mode, int trans_a, int trans_b, const void* a, int32_t lda, const void* b, int32_t ldb, const float* bias, const float* residual,
             int32_t ld_res, void* aux, int32_t ld_aux, void* c, int32_t ldc, int c_mode, int32_t m, int32_t n, int32_t k, int epilogue_flags,
             void* workspace, size_t workspace_bytes, void* stream) {
  int e = require_device_train();
  if (e) return e;
  AVF_REQUIRE(a && b && c, AVF_EINVAL, "gemm: null pointer");
  AVF_REQUIRE(!(epilogue_flags & AVF_EPI_BIAS) || bias, AVF_EINVAL, "gemm: bias flag without bias");
  AVF_REQUIRE(!(epilogue_flags & AVF_EPI_RESIDUAL) || residual, AVF_EINVAL, "gemm: residual flag without residual");
  return gemm(mode, trans_a, trans_b, a, lda, b, ldb, bias, residual, ld_res, aux, ld_aux, c, ldc, c_mode, m, n, k, epilogue_flags, workspace,
              workspace_bytes, static_cast<cudaStream_t>(stream));
}

size_t avf_tformer_embed_indexed_bwd_workspace_bytes(int32_t n_clips, int32_t n_frames, int32_t n_bank) {
  return n_clips > 0 && n_frames > 0 && n_bank >= 0 ? tformer_embed_indexed_bwd_workspace_bytes(n_clips, n_frames, n_bank) : 0;
}

int avf_tformer_embed_indexed_bwd(int out_mode, const float* dtok, const int32_t* index, int32_t n_clips, int32_t n_frames, int32_t dim, int32_t n_bank,
                                  void* dbank, void* workspace, size_t workspace_bytes, void* stream) {
  int e = require_device_train();
  if (e) return e;
  AVF_REQUIRE(dtok && index && dbank, AVF_EINVAL, "tformer_embed_indexed_bwd: null pointer");
  return tformer_embed_indexed_bwd(out_mode, dtok, index, n_clips, n_frames, dim, n_bank, dbank, workspace, workspace_bytes,
                                   static_cast<cudaStream_t>(stream));
}

size_t avf_colsum_workspace_bytes(int32_t rows, int32_t cols) { return rows > 0 && cols > 0 ? colsum_workspace_bytes(rows, cols) : 0; }

int avf_colsum(int in_mode, const void* x, size_t ld, int32_t rows, int32_t cols, float* out, void* workspace, size_t workspace_bytes, void* stream) {
  int e = require_device_train();
  if (e) return e;
  return colsum(in_mode, x, ld, rows, cols, out, 0.f, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

size_t avf_layernorm_bwd_workspace_bytes(int32_t rows, int32_t dim) { return rows > 0 && dim > 0 ? layernorm_bwd_workspace_bytes(rows, dim) : 0; }

int avf_layernorm_bwd(const float* x, int32_t ld_x, const float* gamma, const float* dy_norm, float* dres, int32_t ld_d, void* dx_bf16,
                      float* dgamma, float* dbeta, float* dbias, int32_t rows, int32_t dim, void* workspace, size_t workspace_bytes, void* stream) {
  int e = require_device_train();
  if (e) return e;
  return layernorm_bwd(x, ld_x, gamma, dy_norm, dres, ld_d, dx_bf16, AVF_BF16, dgamma, dbeta, dbias, 0.f, rows, dim, workspace, workspace_bytes,
                       static_cast<cudaStream_t>(stream));
}

int avf_attention_bwd(int io_mode, const void* qkv, const void* dout, void* dqkv, int32_t n_seq, int32_t n_tok, int32_t heads, int32_t dim_head,
                      void* stream) {
  int e = require_device_train();
  if (e) return e;
  AVF_REQUIRE(qkv && dout && dqkv, AVF_EINVAL, "attention_bwd: null pointer");
  return attention_bwd(io_mode, qkv, dout, dqkv, n_seq, n_tok, heads, dim_head, static_cast<cudaStream_t>(stream));
}

int avf_attention_bwd_masked(int io_mode, const void* qkv, const void* dout, void* dqkv, int32_t n_seq, int32_t n_tok, int32_t heads, int32_t dim_head,
                             const uint8_t* keep, void* stream) {
  int e = require_device_train();
  if (e) return e;
  AVF_REQUIRE(qkv && dout && dqkv, AVF_EINVAL, "attention_bwd: null pointer");
  return attention_bwd(io_mode, qkv, dout, dqkv, n_seq, n_tok, heads, dim_head, static_cast<cudaStream_t>(stream), keep);
}

int avf_attention_bwd_gradmaps(int io_mode, const void* qkv, const void* dout, void* dqkv, int32_t n_seq, int32_t n_tok, int32_t heads,
                               int32_t dim_head, const uint8_t* keep, float* gmap, void* stream) {
  int e = require_device_train();
  if (e) return e;
  AVF_REQUIRE(qkv && dout && dqkv && gmap, AVF_EINVAL, "attention_bwd_gradmaps: null pointer");
  return attention_bwd(io_mode, qkv, dout, dqkv, n_seq, n_tok, heads, dim_head, static_cast<cudaStream_t>(stream), keep, gmap);
}

int avf_encoder_stack_bwd_gradmaps(int mode, const avf_stack_shape* s, const avf_layer_weights* layers, const uint8_t* keep, const void* tape,
                                   size_t tape_bytes, float* dx, int32_t ld_dx, const avf_layer_grads* grads, int accumulate, void* workspace,
                                   size_t workspace_bytes, float dropout_p, uint64_t dropout_seed, const uint32_t* dropout_salt, float* gmaps,
                                   void* stream) {
  int e = require_device_train();
  if (e) return e;
  AVF_REQUIRE(gmaps, AVF_EINVAL, "encoder_stack_bwd_gradmaps: null pointer");
  return encoder_bwd(mode, s, layers, tape, tape_bytes, dx, ld_dx, grads, accumulate, workspace, workspace_bytes, dropout_p, dropout_seed, dropout_salt,
                     static_cast<cudaStream_t>(stream), keep, gmaps);
}

int avf_attention_rollout(const float* gmaps, int32_t depth, int32_t n_seq, int32_t heads, int32_t n_tok, float* R, void* stream) {
  int e = require_device_train();
  if (e) return e;
  return attention_rollout(gmaps, depth, n_seq, heads, n_tok, R, static_cast<cudaStream_t>(stream));
}

/* ---- AU_former front end with tape ------------------------------------------------------------------------- */
size_t avf_au_former_front_tape_bytes(int mode, int32_t n_clips, int32_t in_dim) {
  return n_clips > 0 && in_dim > 0 ? align_up(size_t(n_clips) * in_dim * elt(mode)) + 2 * align_up(size_t(in_dim) * 4) : 0;
}

int avf_au_former_front_fwd_train(int mode, const float* emb, int32_t ld_emb, const float* bn_gamma, const float* bn_beta, float* bn_mean,
                                  float* bn_var, int batch_stats, float momentum, const void* w_cat, const float* b_cat, const float* pos,
                                  float* x, int32_t n_clips, int32_t in_dim, int32_t emb_dim, void* tape, size_t tape_bytes, void* stream) {
  int e = require_device_train();
  if (e) return e;
  AVF_REQUIRE(emb && bn_gamma && bn_beta && bn_mean && bn_var && w_cat && b_cat && pos && x && tape, AVF_EINVAL, "au_former_front: null pointer");
  AVF_REQUIRE(n_clips > 0 && in_dim > 0 && emb_dim > 0, AVF_EINVAL, "au_former_front: n_clips=%d", n_clips);
  AVF_REQUIRE(tape_bytes >= avf_au_former_front_tape_bytes(mode, n_clips, in_dim), AVF_EWORKSPACE, "au_former_front: tape too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  uint8_t* p = static_cast<uint8_t*>(tape);
  void* xb = p;
  float* save_mean = reinterpret_cast<float*>(p + align_up(size_t(n_clips) * in_dim * elt(mode)));
  float* save_rstd = save_mean + align_up(size_t(in_dim) * 4) / 4;
  if (batch_stats) {
    if ((e = bn_train_fwd(mode, emb, ld_emb, bn_gamma, bn_beta, bn_mean, bn_var, momentum, xb, save_mean, save_rstd, n_clips, in_dim, st))) return e;
  } else {
    if ((e = bn_rows(mode, emb, ld_emb, bn_gamma, bn_beta, bn_mean, bn_var, xb, n_clips, in_dim, st))) return e;
  }
  if ((e = gemm(mode, 0, 0, xb, in_dim, w_cat, in_dim, b_cat, nullptr, 0, nullptr, 0, x, 12 * emb_dim, AVF_FP32, n_clips, 12 * emb_dim, in_dim,
                AVF_EPI_BIAS, nullptr, 0, st)))
    return e;
  return add_row_periodic(x, emb_dim, pos, n_clips * 12, emb_dim, 12, st);
}

size_t avf_au_former_front_bwd_workspace_bytes(int mode, int32_t n_clips, int32_t in_dim, int32_t emb_dim) {
  if (n_clips <= 0 || in_dim <= 0 || emb_dim <= 0) return 0;
  const size_t n_out = size_t(12) * emb_dim;
  size_t red = colsum_workspace_bytes(n_clips, int(n_out));
  if (mode == AVF_BF16) red = std::max(red, gemm_umma_workspace_bytes(int(n_out), in_dim, n_clips));
  return (mode == AVF_BF16 ? align_up(size_t(n_clips) * n_out * 2) : 0) + align_up(size_t(n_clips) * in_dim * 4) + align_up(red);
}

int avf_au_former_front_bwd(int mode, const float* emb, int32_t ld_emb, const float* bn_gamma, const float* bn_mean, const float* bn_var,
                            int batch_stats, const void* w_cat, const void* tape, size_t tape_bytes, const float* dx, float* demb,
                            int32_t ld_demb, float* dbn_gamma, float* dbn_beta, float* dw_cat, float* db_cat, int32_t n_clips, int32_t in_dim,
                            int32_t emb_dim, void* workspace, size_t workspace_bytes, void* stream) {
  int e = require_device_train();
  if (e) return e;
  AVF_REQUIRE(emb && bn_gamma && bn_mean && bn_var && w_cat && tape && dx && workspace, AVF_EINVAL, "au_former_front_bwd: null pointer");
  AVF_REQUIRE(tape_bytes >= avf_au_former_front_tape_bytes(mode, n_clips, in_dim), AVF_EWORKSPACE, "au_former_front_bwd: tape too small");
  AVF_REQUIRE(workspace_bytes >= avf_au_former_front_bwd_workspace_bytes(mode, n_clips, in_dim, emb_dim), AVF_EWORKSPACE,
              "au_former_front_bwd: workspace too small");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int n_out = 12 * emb_dim;
  const uint8_t* tp = static_cast<const uint8_t*>(tape);
  const void* xb = tp;
  const float* save_mean = reinterpret_cast<const float*>(tp + align_up(size_t(n_clips) * in_dim * elt(mode)));
  const float* save_rstd = save_mean + align_up(size_t(in_dim) * 4) / 4;
  uint8_t* wp = static_cast<uint8_t*>(workspace);
  const void* dxo = dx;                      // GEMM operand view of dx: [n_clips, 12*emb_dim]
  if (mode == AVF_BF16) {
    if ((e = cast_f32_bf16(dx, wp, size_t(n_clips) * n_out, st))) return e;
    dxo = wp;
    wp += align_up(size_t(n_clips) * n_out * 2);
  }
  float* dxb = reinterpret_cast<float*>(wp);
  wp += align_up(size_t(n_clips) * in_dim * 4);
  const size_t red_bytes = workspace_bytes - size_t(wp - static_cast<uint8_t*>(workspace));
  // bias and positional embedding both add to every clip's [12*emb_dim] vector: one column sum serves both
  if (db_cat && (e = colsum(AVF_FP32, dx, n_out, n_clips, n_out, db_cat, 0.f, wp, red_bytes, st))) return e;
  if (dw_cat && (e = gemm(mode, 1, 1, dxo, n_out, xb, in_dim, nullptr, nullptr, 0, nullptr, 0, dw_cat, in_dim, AVF_FP32, n_out, in_dim, n_clips, 0,
                          wp, red_bytes, st)))
    return e;
  if (demb == nullptr && dbn_gamma == nullptr && dbn_beta == nullptr) return 0;
  if ((e = gemm(mode, 0, 1, dxo, n_out, w_cat, in_dim, nullptr, nullptr, 0, nullptr, 0, dxb, in_dim, AVF_FP32, n_clips, in_dim, n_out, 0, nullptr, 0, st)))
    return e;
  return bn_bwd(emb, ld_emb, dxb, bn_gamma, batch_stats ? save_mean : bn_mean, batch_stats ? save_rstd : bn_var, batch_stats, demb, ld_demb,
                dbn_gamma, dbn_beta, n_clips, in_dim, st);
}

int avf_au_logits_bwd(const float* dlogits, int32_t ld_dlogits, const float* x, int32_t ld_x, const float* w_last, float* dx, int32_t ld_dx,
                      float* dw_last, int32_t n_clips, int32_t dim, void* stream) {
  int e = require_device_train();
  if (e) return e;
  return au_logits_bwd(dlogits, ld_dlogits, x, ld_x, w_last, dx, ld_dx, dw_last, n_clips, dim, static_cast<cudaStream_t>(stream));
}

int avf_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, void* bf16_shadow, size_t n, float lr, float beta1,
                  float beta2, float eps, float weight_decay, int32_t step, int decoupled, float grad_scale, void* stream) {
  int e = require_device_train();
  if (e) return e;
  return adam_step(params, grads, exp_avg, exp_avg_sq, bf16_shadow, n, lr, beta1, beta2, eps, weight_decay, step, decoupled, grad_scale,
                   static_cast<cudaStream_t>(stream));
}

}  // extern "C"
