// extern "C" surface of libavformer_b200.so (include/avformer_b200.h) and the host-side
// orchestration of one encoder stack.  No torch types, no CPU compute path.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "avf_common.cuh"
#include "avf_internal.h"

namespace avf {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};
static std::atomic<int> g_pdl{1};        // avf_set_pdl_enabled
bool pdl_enabled() { return g_pdl.load() != 0; }
static std::atomic<int> g_sm_cap{0};     // avf_set_sm_cap
int sm_cap() { return g_sm_cap.load(); }
static std::atomic<int> g_fused{1};      // avf_set_fused_enabled: 0 forces the kernel-per-op path (A/B tests)

void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return 0;
  set_error("CUDA error %d (%s) at %s", int(e), cudaGetErrorString(e), what);
  return int(e);
}

static int require_device() {
  static int state = 0;   // 0 unknown, 1 ok, -1 none
  if (state == 0) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
      cudaGetLastError();
      state = -1;
    } else {
      state = 1;
    }
  }
  if (state < 0) {
    set_error("no CUDA device: the AVFormer B200 path has no CPU fallback");
    return AVF_ENODEVICE;
  }
  return 0;
}

static bool tcgen05_ok() {
  static int state = 0;
  if (state == 0) {
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) == cudaSuccess)
      state = (major == 10) ? 1 : -1;
    else
      state = -1;
  }
  return state > 0;
}

static inline size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }
static inline size_t elt(int mode) { return mode == AVF_BF16 ? 2 : 4; }

struct EncoderWs {
  void* ln;      // [R, D]
  void* qkv;     // [R, 3I]
  void* attn;    // [R, I]
  void* hid;     // [R, M]
  size_t total;
};

static EncoderWs carve_encoder_ws(const avf_stack_shape* s, int mode, void* base) {
  const size_t R = size_t(s->n_seq) * s->n_tok, I = size_t(s->heads) * s->dim_head, e = elt(mode);
  uint8_t* p = static_cast<uint8_t*>(base);
  EncoderWs w;
  size_t off = 0;
  w.ln = p + off;   off += align_up(R * s->dim * e);
  w.qkv = p + off;  off += align_up(R * 3 * I * e);
  w.attn = p + off; off += align_up(R * I * e);
  w.hid = p + off;  off += align_up(R * s->mlp_dim * e);
  w.total = off;
  return w;
}

static int check_shape(const avf_stack_shape* s) {
  AVF_REQUIRE(s != nullptr, AVF_EINVAL, "null stack shape");
  AVF_REQUIRE(s->n_seq > 0 && s->n_tok > 0 && s->depth > 0, AVF_EINVAL, "empty stack: n_seq=%d n_tok=%d depth=%d", s->n_seq, s->n_tok, s->depth);
  AVF_REQUIRE(s->dim % 128 == 0 && s->dim <= 1536, AVF_EUNSUPPORTED, "dim=%d must be a multiple of 128 (<= 1536)", s->dim);
  AVF_REQUIRE(s->dim_head == 32 || s->dim_head == 64, AVF_EUNSUPPORTED, "dim_head=%d (supported: 32, 64)", s->dim_head);
  AVF_REQUIRE((s->heads * s->dim_head) % 64 == 0 && s->mlp_dim % 64 == 0, AVF_EUNSUPPORTED, "inner=%d / mlp=%d must be multiples of 64", s->heads * s->dim_head, s->mlp_dim);
  AVF_REQUIRE(s->n_tok <= 64 || s->dim_head == 64, AVF_EUNSUPPORTED,
              "n_tok=%d: sequences longer than 64 tokens are not part of this path for dim_head=%d", s->n_tok, s->dim_head);
  AVF_REQUIRE(s->n_tok <= 256, AVF_EUNSUPPORTED, "n_tok=%d: sequences longer than 256 tokens are not part of this path", s->n_tok);
  return 0;
}

int linear(int mode, const void* a, int lda, const void* w, const float* bias, const float* res, int ld_res, void* c, int ldc,
           int c_mode, int m, int n, int k, int flags, cudaStream_t st) {
  if (mode == AVF_BF16) {
    AVF_REQUIRE(tcgen05_ok(), AVF_EUNSUPPORTED, "bf16 mode needs an sm_100 device (tcgen05)");
    return linear_umma(a, lda, w, bias, res, ld_res, c, ldc, c_mode, m, n, k, flags, st);
  }
  return linear_f32(static_cast<const float*>(a), lda, static_cast<const float*>(w), bias, res, ld_res, c, ldc, c_mode, m, n, k, flags, st);
}

// Does a stack of fp32 token rows run as one fused kernel?
static bool fused_rows(int mode, const avf_stack_shape* s, int ld_x, const float* out, int ld_out) {
  return mode == AVF_BF16 && g_fused.load() && tcgen05_ok() && encoder_fused_supported(s) &&
         ld_x % 4 == 0 && (out == nullptr || ld_out % 4 == 0);
}

// keep (optional, [n_seq, n_tok] uint8): attention mask of every layer; the fused kernel has none, so a masked stack runs kernel by kernel.
// probs (optional): layer l's attention probabilities go to probs + l * n_seq*heads*n_tok*n_tok (fp32 [depth, n_seq, heads, n_tok, n_tok]),
// written by the attention launch itself; the fused kernel keeps them on chip, so such a stack runs kernel by kernel too.
static size_t probs_per_layer(const avf_stack_shape* s) { return size_t(s->n_seq) * s->heads * s->n_tok * s->n_tok; }

static int encoder_stack(int mode, const avf_stack_shape* s, const avf_layer_weights* L, float* x, int ld_x, float* out, int ld_out,
                         void* ws, size_t ws_bytes, cudaStream_t st, const uint8_t* keep = nullptr, float* probs = nullptr) {
  int e = check_shape(s);
  if (e) return e;
  AVF_REQUIRE(mode == AVF_BF16 || mode == AVF_FP32, AVF_EINVAL, "mode=%d", mode);
  AVF_REQUIRE(L != nullptr && x != nullptr && ws != nullptr, AVF_EINVAL, "null pointer argument");
  if (keep == nullptr && probs == nullptr && fused_rows(mode, s, ld_x, out, ld_out))     // whole stack, one persistent kernel
    return encoder_fused(1, s, L, x, ld_x, out ? out : x, out ? ld_out : ld_x, nullptr, nullptr, nullptr, nullptr, nullptr, st);
  const EncoderWs w = carve_encoder_ws(s, mode, ws);
  AVF_REQUIRE(ws_bytes >= w.total, AVF_EWORKSPACE, "workspace too small: %zu < %zu bytes", ws_bytes, w.total);
  const int R = s->n_seq * s->n_tok, D = s->dim, I = s->heads * s->dim_head, M = s->mlp_dim;
  for (int l = 0; l < s->depth; ++l) {
    const avf_layer_weights& W = L[l];
    // x + to_out(attn(to_qkv(LN(x))))                                     models/heads.py:175,185,219-239
    if ((e = layernorm(mode, x, ld_x, W.ln1_gamma, W.ln1_beta, w.ln, R, D, st))) return e;
    if ((e = linear(mode, w.ln, D, W.w_qkv, nullptr, nullptr, 0, w.qkv, 3 * I, mode, R, 3 * I, D, 0, st))) return e;
    if ((e = attention_small(mode, w.qkv, w.attn, s->n_seq, s->n_tok, s->heads, s->dim_head, st, keep, probs ? probs + l * probs_per_layer(s) : nullptr)))
      return e;
    if ((e = linear(mode, w.attn, I, W.w_out, W.b_out, x, ld_x, x, ld_x, AVF_FP32, R, D, I, AVF_EPI_BIAS | AVF_EPI_RESIDUAL, st))) return e;
    // x + W2 gelu(W1 LN(x) + b1) + b2                                     models/heads.py:188-200
    if ((e = layernorm(mode, x, ld_x, W.ln2_gamma, W.ln2_beta, w.ln, R, D, st))) return e;
    if ((e = linear(mode, w.ln, D, W.w_ff1, W.b_ff1, nullptr, 0, w.hid, M, mode, R, M, D, AVF_EPI_BIAS | AVF_EPI_GELU, st))) return e;
    const bool last = (l == s->depth - 1) && out != nullptr;
    if ((e = linear(mode, w.hid, M, W.w_ff2, W.b_ff2, x, ld_x, last ? out : x, last ? ld_out : ld_x, AVF_FP32, R, D, M,
                    AVF_EPI_BIAS | AVF_EPI_RESIDUAL, st)))
      return e;
  }
  return 0;
}

// Checks shared by the TFormer entry points; `in` is the frames or the frame bank, `need` the workspace the entry point carves.
static int tformer_check(const avf_stack_shape* s, const avf_layer_weights* layers, const void* in, const float* cls_token, const float* pos,
                         const float* cls_out, const void* workspace, size_t workspace_bytes, size_t need) {
  int e = check_shape(s);
  if (e) return e;
  AVF_REQUIRE(layers && in && cls_token && pos && cls_out && workspace, AVF_EINVAL, "tformer_fwd: null pointer");
  AVF_REQUIRE(s->n_tok >= 2, AVF_EINVAL, "tformer_fwd: n_tok=%d (cls + at least one frame)", s->n_tok);
  AVF_REQUIRE(workspace_bytes >= need, AVF_EWORKSPACE, "workspace too small: %zu < %zu bytes", workspace_bytes, need);
  return 0;
}

// The layers of the TFormer on the embedded tokens x [n_seq*n_tok, dim] fp32 that start the workspace -> cls_out.
// probs (optional): the maps of every layer (encoder_stack); the last layer's attention then runs every query row (full map) while
// everything after the softmax stays on the cls rows.
static int tformer_layers(int mode, const avf_stack_shape* s, const avf_layer_weights* layers, void* workspace, float* cls_out, const uint8_t* keep,
                          cudaStream_t st, float* probs = nullptr) {
  int e = 0;
  const int B = s->n_seq, N = s->n_tok, R = B * N, D = s->dim, I = s->heads * s->dim_head, M = s->mlp_dim;
  uint8_t* p = static_cast<uint8_t*>(workspace);
  float* x = reinterpret_cast<float*>(p);   p += align_up(size_t(R) * D * 4);
  void* enc_ws = p;
  const EncoderWs w = carve_encoder_ws(s, mode, enc_ws);
  p += w.total;
  float* xc = reinterpret_cast<float*>(p);  p += align_up(size_t(B) * D * 4);
  void* lnc = p;                            p += align_up(size_t(B) * D * elt(mode));
  void* oc = p;                             p += align_up(size_t(B) * I * elt(mode));
  void* hc = p;
  if (s->depth > 1) {
    avf_stack_shape head = *s;
    head.depth = s->depth - 1;
    if ((e = encoder_stack(mode, &head, layers, x, D, nullptr, 0, enc_ws, w.total, st, keep, probs))) return e;
  }
  float* last_probs = probs ? probs + size_t(s->depth - 1) * probs_per_layer(s) : nullptr;
  // Last layer (models/vformer.py:288-290 returns x[:, 0] only): keys / values need every row, everything after the softmax only
  // the cls row of each clip — out-projection, LayerNorm, MLP run on [n_clips, dim] instead of [n_clips * (T+1), dim].
  const avf_layer_weights& W = layers[s->depth - 1];
  if ((e = layernorm(mode, x, D, W.ln1_gamma, W.ln1_beta, w.ln, R, D, st))) return e;
  if ((e = linear(mode, w.ln, D, W.w_qkv, nullptr, nullptr, 0, w.qkv, 3 * I, mode, R, 3 * I, D, 0, st))) return e;
  if (mode == AVF_BF16) {
    if ((e = attention_mma_bf16(w.qkv, oc, B, N, s->heads, s->dim_head, st, 1, keep, last_probs))) return e;
  } else {
    if ((e = attention_small(mode, w.qkv, w.attn, B, N, s->heads, s->dim_head, st, keep, last_probs))) return e;
    AVF_CUDA(cudaMemcpy2DAsync(oc, size_t(I) * 4, w.attn, size_t(N) * I * 4, size_t(I) * 4, B, cudaMemcpyDeviceToDevice, st));
  }
  if ((e = rows_gather(x, size_t(N) * D, xc, B, D, st))) return e;
  if ((e = linear(mode, oc, I, W.w_out, W.b_out, xc, D, xc, D, AVF_FP32, B, D, I, AVF_EPI_BIAS | AVF_EPI_RESIDUAL, st))) return e;
  if ((e = layernorm(mode, xc, D, W.ln2_gamma, W.ln2_beta, lnc, B, D, st))) return e;
  if ((e = linear(mode, lnc, D, W.w_ff1, W.b_ff1, nullptr, 0, hc, M, mode, B, M, D, AVF_EPI_BIAS | AVF_EPI_GELU, st))) return e;
  return linear(mode, hc, M, W.w_ff2, W.b_ff2, xc, D, cls_out, D, AVF_FP32, B, D, M, AVF_EPI_BIAS | AVF_EPI_RESIDUAL, st);
}

static int tformer_fwd(int mode, int io_mode, const avf_stack_shape* s, const avf_layer_weights* layers, const void* frames, const float* cls_token,
                       const float* pos, float* cls_out, void* workspace, size_t workspace_bytes, const uint8_t* keep, cudaStream_t st,
                       float* probs = nullptr) {
  int e = tformer_check(s, layers, frames, cls_token, pos, cls_out, workspace, workspace_bytes, avf_tformer_workspace_bytes(s, mode));
  if (e) return e;
  if ((e = tformer_embed(io_mode, frames, cls_token, pos, static_cast<float*>(workspace), s->n_seq, s->n_tok - 1, s->dim, st))) return e;
  return tformer_layers(mode, s, layers, workspace, cls_out, keep, st, probs);
}

// Clips described by frame indices into a bank: gather, keep rows and embed in one launch, then the masked layers.  The keep rows
// follow the workspace of avf_tformer_fwd.
static int tformer_fwd_indexed(int mode, int io_mode, const avf_stack_shape* s, const avf_layer_weights* layers, const void* bank, int n_bank,
                               const int32_t* index, const float* cls_token, const float* pos, float* cls_out, void* workspace, size_t workspace_bytes,
                               cudaStream_t st, float* probs = nullptr) {
  int e = tformer_check(s, layers, index, cls_token, pos, cls_out, workspace, workspace_bytes, avf_tformer_indexed_workspace_bytes(s, mode));
  if (e) return e;
  AVF_REQUIRE(n_bank >= 0 && (bank != nullptr || n_bank == 0), AVF_EINVAL, "tformer_fwd_indexed: bank of %d frames at %p", n_bank, bank);
  uint8_t* keep = static_cast<uint8_t*>(workspace) + avf_tformer_workspace_bytes(s, mode);
  if ((e = tformer_embed_indexed(io_mode, bank, n_bank, index, cls_token, pos, static_cast<float*>(workspace), keep, s->n_seq, s->n_tok - 1, s->dim, st)))
    return e;
  return tformer_layers(mode, s, layers, workspace, cls_out, keep, st, probs);
}

}  // namespace avf

using namespace avf;

extern "C" {

int avf_abi_version(void) { return AVF_ABI_VERSION; }

const char* avf_last_error(void) { return g_err; }

uint64_t avf_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int avf_set_fused_enabled(int enabled) {
  const int old = g_fused.exchange(enabled ? 1 : 0);
  return old;
}

int avf_set_pdl_enabled(int enabled) { return g_pdl.exchange(enabled ? 1 : 0); }

int avf_set_sm_cap(int cap) { return g_sm_cap.exchange(cap > 0 ? cap : 0); }

int avf_encoder_fused_supported(const avf_stack_shape* s, int mode) {
  return (s != nullptr && mode == AVF_BF16 && s->n_seq > 0 && encoder_fused_supported(s)) ? 1 : 0;
}

/* Debug: per-phase cycle counters of the fused encoder kernel (library built with -DAVF_FUSED_PROF); else AVF_EUNSUPPORTED. */
int avf_debug_fused_prof(uint64_t* out64, int reset) { return fused_prof_read(reinterpret_cast<unsigned long long*>(out64), reset); }

int avf_debug_tmap_cache(uint64_t* hits, uint64_t* misses) {
  if (hits == nullptr || misses == nullptr) return AVF_EINVAL;
  tmap_cache_stats(hits, misses);
  return 0;
}

int avf_debug_gemm_prof(uint64_t* out16) { return gemm_prof_read(reinterpret_cast<unsigned long long*>(out16)); }

int avf_debug_set_trap_buffer(void* host_mapped_words) { return fused_set_trap_buffer(host_mapped_words); }

int avf_device_info(int32_t* sm_count, int32_t* cc, int32_t* has_tcgen05) {
  int e = require_device();
  if (e) return e;
  int dev = 0, sms = 0, major = 0, minor = 0;
  AVF_CUDA(cudaGetDevice(&dev));
  AVF_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  AVF_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  AVF_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  if (sm_count) *sm_count = sms;
  if (cc) *cc = major * 10 + minor;
  if (has_tcgen05) *has_tcgen05 = major == 10 ? 1 : 0;
  return 0;
}

size_t avf_encoder_workspace_bytes(const avf_stack_shape* s, int mode) {
  if (s == nullptr || s->n_seq <= 0 || s->n_tok <= 0) return 0;
  return carve_encoder_ws(s, mode, nullptr).total;
}

int avf_encoder_stack_fwd(int mode, const avf_stack_shape* s, const avf_layer_weights* layers, float* x, int32_t ld_x, float* out,
                          int32_t ld_out, void* workspace, size_t workspace_bytes, void* stream) {
  int e = require_device();
  if (e) return e;
  return encoder_stack(mode, s, layers, x, ld_x, out, ld_out, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
}

int avf_encoder_stack_fwd_masked(int mode, const avf_stack_shape* s, const avf_layer_weights* layers, const uint8_t* keep, float* x, int32_t ld_x,
                                 float* out, int32_t ld_out, void* workspace, size_t workspace_bytes, void* stream) {
  int e = require_device();
  if (e) return e;
  return encoder_stack(mode, s, layers, x, ld_x, out, ld_out, workspace, workspace_bytes, static_cast<cudaStream_t>(stream), keep);
}

int avf_token_stack_fwd(int mode, const avf_stack_shape* s, const avf_layer_weights* layers, float* x, int32_t ld_x, const float* pos, float* out,
                        int32_t ld_out, const float* w_last, float* out21, int32_t* decisions, void* workspace, size_t workspace_bytes, void* stream) {
  int e = require_device();
  if (e) return e;
  if ((e = check_shape(s))) return e;
  AVF_REQUIRE(layers && x && workspace, AVF_EINVAL, "token_stack: null pointer");
  AVF_REQUIRE(w_last == nullptr || (s->n_tok == 12 && out21 != nullptr), AVF_EINVAL, "token_stack: AU logits need 12 tokens per clip and out21 (n_tok=%d)",
              s->n_tok);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (fused_rows(mode, s, ld_x, out, ld_out))      // positional add, stack and AU logits in one launch
    return encoder_fused(1, s, layers, x, ld_x, (out || w_last) ? out : x, out ? ld_out : ld_x, pos, nullptr, w_last, out21, decisions, st);
  if (pos != nullptr && (e = add_row_periodic(x, ld_x, pos, s->n_seq * s->n_tok, s->dim, s->n_tok, st))) return e;
  if ((e = encoder_stack(mode, s, layers, x, ld_x, out, ld_out, workspace, workspace_bytes, st))) return e;
  return w_last == nullptr ? 0 : au_logits(out ? out : x, out ? ld_out : ld_x, w_last, out21, decisions, s->n_seq, s->dim, st);
}

int avf_layernorm_fwd(int out_mode, const float* x, int32_t ld_x, const float* gamma, const float* beta, void* y, int32_t rows,
                      int32_t dim, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(x && gamma && beta && y, AVF_EINVAL, "layernorm: null pointer");
  return layernorm(out_mode, x, ld_x, gamma, beta, y, rows, dim, static_cast<cudaStream_t>(stream));
}

int avf_linear_fwd(int mode, const void* a, int32_t lda, const void* w, const float* bias, const float* residual, int32_t ld_res,
                   void* c, int32_t ldc, int c_mode, int32_t m, int32_t n, int32_t k, int epilogue_flags, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(a && w && c, AVF_EINVAL, "linear: null pointer");
  AVF_REQUIRE(!(epilogue_flags & AVF_EPI_BIAS) || bias, AVF_EINVAL, "linear: bias flag without bias");
  AVF_REQUIRE(!(epilogue_flags & AVF_EPI_RESIDUAL) || residual, AVF_EINVAL, "linear: residual flag without residual");
  return linear(mode, a, lda, w, bias, residual, ld_res, c, ldc, c_mode, m, n, k, epilogue_flags, static_cast<cudaStream_t>(stream));
}

int avf_attention_fwd(int io_mode, const void* qkv, void* out, int32_t n_seq, int32_t n_tok, int32_t heads, int32_t dim_head, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(qkv && out, AVF_EINVAL, "attention: null pointer");
  return attention_small(io_mode, qkv, out, n_seq, n_tok, heads, dim_head, static_cast<cudaStream_t>(stream));
}

int avf_attention_fwd_masked(int io_mode, const void* qkv, void* out, int32_t n_seq, int32_t n_tok, int32_t heads, int32_t dim_head, const uint8_t* keep,
                             void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(qkv && out, AVF_EINVAL, "attention: null pointer");
  return attention_small(io_mode, qkv, out, n_seq, n_tok, heads, dim_head, static_cast<cudaStream_t>(stream), keep);
}

int avf_attention_fwd_probs(int io_mode, const void* qkv, void* out, int32_t n_seq, int32_t n_tok, int32_t heads, int32_t dim_head, const uint8_t* keep,
                            float* probs, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(qkv && out && probs, AVF_EINVAL, "attention_probs: null pointer");
  return attention_small(io_mode, qkv, out, n_seq, n_tok, heads, dim_head, static_cast<cudaStream_t>(stream), keep, probs);
}

int avf_encoder_stack_fwd_probs(int mode, const avf_stack_shape* s, const avf_layer_weights* layers, const uint8_t* keep, float* x, int32_t ld_x,
                                const float* pos, float* out, int32_t ld_out, float* probs, void* workspace, size_t workspace_bytes, void* stream) {
  int e = require_device();
  if (e) return e;
  if ((e = check_shape(s))) return e;
  AVF_REQUIRE(layers && x && probs && workspace, AVF_EINVAL, "encoder_stack_probs: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (pos != nullptr && (e = add_row_periodic(x, ld_x, pos, s->n_seq * s->n_tok, s->dim, s->n_tok, st))) return e;
  return encoder_stack(mode, s, layers, x, ld_x, out, ld_out, workspace, workspace_bytes, st, keep, probs);
}

int avf_sformer_tokens_pack(int io_mode, const void* fmap, const float* pos, float* x, int32_t n_frames, int32_t dim, int32_t hw, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(fmap && x, AVF_EINVAL, "sformer_tokens_pack: null pointer");      // pos == NULL: plain transpose (backward of unpack)
  return sformer_pack(io_mode, fmap, pos, x, n_frames, dim, hw, static_cast<cudaStream_t>(stream));
}

int avf_sformer_tokens_unpack(int io_mode, const float* x, void* fmap, int32_t n_frames, int32_t dim, int32_t hw, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(fmap && x, AVF_EINVAL, "sformer_tokens_unpack: null pointer");
  return sformer_unpack(io_mode, x, fmap, n_frames, dim, hw, static_cast<cudaStream_t>(stream));
}

size_t avf_sformer_workspace_bytes(const avf_stack_shape* s, int mode) {
  if (s == nullptr || s->n_seq <= 0 || s->n_tok <= 0) return 0;
  return align_up(size_t(s->n_seq) * s->n_tok * s->dim * 4) + carve_encoder_ws(s, mode, nullptr).total + align_up(encoder_fused_scratch_bytes());
}

int avf_sformer_fwd(int mode, int io_mode, const avf_stack_shape* s, const avf_layer_weights* layers, const float* pos,
                    const void* fmap_in, void* fmap_out, void* workspace, size_t workspace_bytes, void* stream) {
  int e = require_device();
  if (e) return e;
  if ((e = check_shape(s))) return e;
  AVF_REQUIRE(layers && pos && fmap_in && fmap_out && workspace, AVF_EINVAL, "sformer_fwd: null pointer");
  const size_t need = avf_sformer_workspace_bytes(s, mode);
  AVF_REQUIRE(workspace_bytes >= need, AVF_EWORKSPACE, "workspace too small: %zu < %zu bytes", workspace_bytes, need);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (mode == AVF_BF16 && io_mode == AVF_BF16 && g_fused.load() && tcgen05_ok() && encoder_fused_supported(s) && s->dim == 256)
    return encoder_fused(0, s, layers, fmap_in, 0, fmap_out, 0, pos, workspace, nullptr, nullptr, nullptr, st);   // frames in, frames out: nothing else touches HBM
  float* x = static_cast<float*>(workspace);
  const size_t xbytes = align_up(size_t(s->n_seq) * s->n_tok * s->dim * 4);
  if ((e = sformer_pack(io_mode, fmap_in, pos, x, s->n_seq, s->dim, s->n_tok, st))) return e;
  if ((e = encoder_stack(mode, s, layers, x, s->dim, nullptr, 0, static_cast<uint8_t*>(workspace) + xbytes, workspace_bytes - xbytes, st))) return e;
  return sformer_unpack(io_mode, x, fmap_out, s->n_seq, s->dim, s->n_tok, st);
}

int avf_tformer_embed(int io_mode, const void* frames, const float* cls_token, const float* pos, float* x, int32_t n_clips,
                      int32_t n_frames, int32_t dim, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(frames && cls_token && pos && x, AVF_EINVAL, "tformer_embed: null pointer");
  return tformer_embed(io_mode, frames, cls_token, pos, x, n_clips, n_frames, dim, static_cast<cudaStream_t>(stream));
}

size_t avf_tformer_workspace_bytes(const avf_stack_shape* s, int mode) {
  if (s == nullptr || s->n_seq <= 0 || s->n_tok <= 0) return 0;
  const size_t B = s->n_seq, D = s->dim, I = size_t(s->heads) * s->dim_head, M = s->mlp_dim, e = elt(mode);
  return align_up(B * s->n_tok * D * 4) + carve_encoder_ws(s, mode, nullptr).total + align_up(B * D * 4) + align_up(B * D * e) + align_up(B * I * e) +
         align_up(B * M * e);
}

int avf_tformer_fwd(int mode, int io_mode, const avf_stack_shape* s, const avf_layer_weights* layers, const void* frames,
                    const float* cls_token, const float* pos, float* cls_out, void* workspace, size_t workspace_bytes, void* stream) {
  int e = require_device();
  if (e) return e;
  return tformer_fwd(mode, io_mode, s, layers, frames, cls_token, pos, cls_out, workspace, workspace_bytes, nullptr, static_cast<cudaStream_t>(stream));
}

int avf_tformer_fwd_masked(int mode, int io_mode, const avf_stack_shape* s, const avf_layer_weights* layers, const uint8_t* keep, const void* frames,
                           const float* cls_token, const float* pos, float* cls_out, void* workspace, size_t workspace_bytes, void* stream) {
  int e = require_device();
  if (e) return e;
  return tformer_fwd(mode, io_mode, s, layers, frames, cls_token, pos, cls_out, workspace, workspace_bytes, keep, static_cast<cudaStream_t>(stream));
}

int avf_tformer_fwd_probs(int mode, int io_mode, const avf_stack_shape* s, const avf_layer_weights* layers, const uint8_t* keep, const void* frames,
                          const float* cls_token, const float* pos, float* cls_out, float* probs, void* workspace, size_t workspace_bytes, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(probs, AVF_EINVAL, "tformer_fwd_probs: null pointer");
  return tformer_fwd(mode, io_mode, s, layers, frames, cls_token, pos, cls_out, workspace, workspace_bytes, keep, static_cast<cudaStream_t>(stream), probs);
}

size_t avf_tformer_indexed_workspace_bytes(const avf_stack_shape* s, int mode) {
  if (s == nullptr || s->n_seq <= 0 || s->n_tok <= 0) return 0;
  return avf_tformer_workspace_bytes(s, mode) + align_up(size_t(s->n_seq) * s->n_tok);
}

int avf_tformer_fwd_indexed(int mode, int io_mode, const avf_stack_shape* s, const avf_layer_weights* layers, const void* bank, int32_t n_bank,
                            const int32_t* index, const float* cls_token, const float* pos, float* cls_out, void* workspace, size_t workspace_bytes,
                            void* stream) {
  int e = require_device();
  if (e) return e;
  return tformer_fwd_indexed(mode, io_mode, s, layers, bank, n_bank, index, cls_token, pos, cls_out, workspace, workspace_bytes,
                             static_cast<cudaStream_t>(stream));
}

int avf_tformer_fwd_indexed_probs(int mode, int io_mode, const avf_stack_shape* s, const avf_layer_weights* layers, const void* bank, int32_t n_bank,
                                  const int32_t* index, const float* cls_token, const float* pos, float* cls_out, float* probs, void* workspace,
                                  size_t workspace_bytes, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(probs, AVF_EINVAL, "tformer_fwd_indexed_probs: null pointer");
  return tformer_fwd_indexed(mode, io_mode, s, layers, bank, n_bank, index, cls_token, pos, cls_out, workspace, workspace_bytes,
                             static_cast<cudaStream_t>(stream), probs);
}

int avf_tformer_embed_indexed(int io_mode, const void* bank, int32_t n_bank, const int32_t* index, const float* cls_token, const float* pos, float* x,
                              uint8_t* keep, int32_t n_clips, int32_t n_frames, int32_t dim, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(index && cls_token && pos && x && keep, AVF_EINVAL, "tformer_embed_indexed: null pointer");
  AVF_REQUIRE(bank != nullptr || n_bank == 0, AVF_EINVAL, "tformer_embed_indexed: bank of %d frames at %p", n_bank, bank);
  return tformer_embed_indexed(io_mode, bank, n_bank, index, cls_token, pos, x, keep, n_clips, n_frames, dim, static_cast<cudaStream_t>(stream));
}

int avf_tformer_cls_extract(const float* x, float* cls, int32_t n_clips, int32_t n_tok, int32_t dim, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(x && cls, AVF_EINVAL, "tformer_cls_extract: null pointer");
  return rows_gather(x, size_t(n_tok) * dim, cls, n_clips, dim, static_cast<cudaStream_t>(stream));
}

int avf_token_front_fwd(int mode, const float* emb, int32_t ld_emb, const float* bn_gamma, const float* bn_beta, const float* bn_mean,
                        const float* bn_var, const void* w_cat, const float* b_cat, const float* pos, float* x, int32_t n_clips,
                        int32_t in_dim, int32_t emb_dim, int32_t n_tok, void* workspace, size_t workspace_bytes, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(emb && bn_gamma && bn_beta && bn_mean && bn_var && w_cat && b_cat && x && workspace, AVF_EINVAL, "token_front: null pointer");
  AVF_REQUIRE(n_clips > 0 && in_dim > 0 && emb_dim > 0 && n_tok > 0, AVF_EINVAL, "token_front: n_clips=%d n_tok=%d", n_clips, n_tok);
  const size_t need = align_up(size_t(n_clips) * in_dim * elt(mode));
  AVF_REQUIRE(workspace_bytes >= need, AVF_EWORKSPACE, "workspace too small: %zu < %zu bytes", workspace_bytes, need);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if ((e = bn_rows(mode, emb, ld_emb, bn_gamma, bn_beta, bn_mean, bn_var, workspace, n_clips, in_dim, st))) return e;
  // [n_clips, n_tok*emb_dim] row-major IS [n_clips*n_tok, emb_dim]: token i = the i-th stacked projection  (models/heads.py:294-319, 356-364)
  if ((e = linear(mode, workspace, in_dim, w_cat, b_cat, nullptr, 0, x, n_tok * emb_dim, AVF_FP32, n_clips, n_tok * emb_dim, in_dim, AVF_EPI_BIAS, st))) return e;
  return pos == nullptr ? 0 : add_row_periodic(x, emb_dim, pos, n_clips * n_tok, emb_dim, n_tok, st);     // NULL: added by avf_token_stack_fwd
}

int avf_au_former_front_fwd(int mode, const float* emb, int32_t ld_emb, const float* bn_gamma, const float* bn_beta, const float* bn_mean,
                            const float* bn_var, const void* w_cat, const float* b_cat, const float* pos, float* x, int32_t n_clips,
                            int32_t in_dim, int32_t emb_dim, void* workspace, size_t workspace_bytes, void* stream) {
  return avf_token_front_fwd(mode, emb, ld_emb, bn_gamma, bn_beta, bn_mean, bn_var, w_cat, b_cat, pos, x, n_clips, in_dim, emb_dim, 12, workspace,
                             workspace_bytes, stream);
}

int avf_au_logits_fwd(const float* x, int32_t ld_x, const float* w_last, float* out21, int32_t* decisions, int32_t n_clips, int32_t dim, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(x && w_last, AVF_EINVAL, "au_logits: null pointer");
  return au_logits(x, ld_x, w_last, out21, decisions, n_clips, dim, static_cast<cudaStream_t>(stream));
}

int avf_au_bce_loss(const float* logits, int32_t ld_logits, const float* labels, const float* pos_weight, float* loss_out, float* dlogits,
                    int32_t n_clips, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(logits && labels && pos_weight && loss_out, AVF_EINVAL, "au_bce_loss: null pointer");
  return au_bce(logits, ld_logits, labels, pos_weight, loss_out, dlogits, n_clips, static_cast<cudaStream_t>(stream));
}

size_t avf_peer_gather_bytes(int32_t world, size_t n_floats) { return (world > 0 && world <= 1024) ? peer_gather_bytes(world, n_floats) : 0; }

int avf_logits_push(const float* logits, size_t n_floats, const uint64_t* peer_base, int32_t world, int32_t rank, const uint32_t* state, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(logits && peer_base && state, AVF_EINVAL, "logits_push: null pointer");
  AVF_REQUIRE(world > 0 && world <= 1024 && rank >= 0 && rank < world && n_floats > 0, AVF_EINVAL, "logits_push: world %d rank %d n %zu", world, rank, n_floats);
  return logits_push(logits, n_floats, reinterpret_cast<const unsigned long long*>(peer_base), world, rank, state, static_cast<cudaStream_t>(stream));
}

int avf_logits_wait(const void* my_base, size_t n_floats, int32_t world, uint32_t* state, uint64_t timeout_ns, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(my_base && state, AVF_EINVAL, "logits_wait: null pointer");
  AVF_REQUIRE(world > 0 && world <= 1024 && n_floats > 0, AVF_EINVAL, "logits_wait: world %d n %zu", world, n_floats);
  return logits_wait(my_base, n_floats, world, state, timeout_ns, static_cast<cudaStream_t>(stream));
}

size_t avf_peer_allreduce_bytes(int32_t world, size_t n_floats) { return (world > 0 && world <= 16) ? peer_allreduce_bytes(world, n_floats) : 0; }

int avf_grad_allreduce(const uint64_t* peer_base, size_t n_floats, int32_t world, int32_t rank, uint32_t* state, uint64_t timeout_ns, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(peer_base && state, AVF_EINVAL, "grad_allreduce: null pointer");
  AVF_REQUIRE(world > 0 && world <= 16 && rank >= 0 && rank < world && n_floats > 0, AVF_EINVAL, "grad_allreduce: world %d (1..16) rank %d n %zu", world, rank, n_floats);
  return grad_allreduce(reinterpret_cast<const unsigned long long*>(peer_base), n_floats, world, rank, state, timeout_ns, static_cast<cudaStream_t>(stream));
}

int avf_adam_allreduce_step(const uint64_t* peer_base, size_t n_floats, int32_t world, int32_t rank, uint32_t* state, uint64_t timeout_ns, float* params,
                            float* exp_avg, float* exp_avg_sq, void* bf16_shadow, float lr, float beta1, float beta2, float eps, float weight_decay, int32_t step,
                            int decoupled, float grad_scale, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(peer_base && state, AVF_EINVAL, "adam_allreduce_step: null pointer");
  AVF_REQUIRE(world > 0 && world <= 16 && rank >= 0 && rank < world && n_floats > 0, AVF_EINVAL, "adam_allreduce_step: world %d (1..16) rank %d n %zu", world, rank, n_floats);
  return adam_allreduce_step(reinterpret_cast<const unsigned long long*>(peer_base), n_floats, world, rank, state, timeout_ns, params, exp_avg, exp_avg_sq, bf16_shadow,
                             lr, beta1, beta2, eps, weight_decay, step, decoupled, grad_scale, static_cast<cudaStream_t>(stream));
}

int avf_au_confusion_update(const float* pred, int32_t ld_pred, float threshold, const float* labels, int32_t ld_labels, float ignore,
                            uint64_t* counts48, int32_t n_rows, void* stream) {
  int e = require_device();
  if (e) return e;
  return au_confusion(pred, ld_pred, threshold, labels, ld_labels, ignore, reinterpret_cast<unsigned long long*>(counts48), n_rows,
                      static_cast<cudaStream_t>(stream));
}

int avf_cast_f32_to_bf16(const float* src, void* dst, size_t n, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE((src && dst) || n == 0, AVF_EINVAL, "cast: null pointer");
  return cast_f32_bf16(src, dst, n, static_cast<cudaStream_t>(stream));
}

int avf_cast_bf16_to_f32(const void* src, float* dst, size_t n, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE((src && dst) || n == 0, AVF_EINVAL, "cast: null pointer");
  return cast_bf16_f32(src, dst, n, static_cast<cudaStream_t>(stream));
}

int avf_add_row_periodic(float* x, int32_t ld_x, const float* pos, int32_t rows, int32_t dim, int32_t period, void* stream) {
  int e = require_device();
  if (e) return e;
  AVF_REQUIRE(x && pos, AVF_EINVAL, "add_row_periodic: null pointer");
  return add_row_periodic(x, ld_x, pos, rows, dim, period, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
