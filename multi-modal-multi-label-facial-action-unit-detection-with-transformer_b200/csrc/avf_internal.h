// Internal C++ launchers shared between the translation units of libavformer_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

#include "../../include/avformer_b200.h"
#include "avf_common.cuh"

namespace avf {

// avf_rowops.cu
int layernorm(int out_mode, const float* x, int ld_x, const float* g, const float* b, void* y, int rows, int dim, cudaStream_t st);
int bn_rows(int out_mode, const float* x, int ld_x, const float* g, const float* b, const float* mean, const float* var, void* y,
            int rows, int dim, cudaStream_t st);
int sformer_pack(int io_mode, const void* fmap, const float* pos, float* x, int n_frames, int dim, int hw, cudaStream_t st);
int sformer_unpack(int io_mode, const float* x, void* fmap, int n_frames, int dim, int hw, cudaStream_t st);
int tformer_embed(int io_mode, const void* frames, const float* cls, const float* pos, float* x, int n_clips, int T, int dim, cudaStream_t st);
int tformer_embed_indexed(int io_mode, const void* bank, int n_bank, const int* index, const float* cls, const float* pos, float* x, uint8_t* keep,
                          int n_clips, int T, int dim, cudaStream_t st);
int rows_gather(const float* x, size_t src_row_stride, float* y, int rows, int dim, cudaStream_t st);
int add_row_periodic(float* x, int ld_x, const float* pos, int rows, int dim, int period, cudaStream_t st);
int cast_f32_bf16(const float* s, void* d, size_t n, cudaStream_t st);
int cast_bf16_f32(const void* s, float* d, size_t n, cudaStream_t st);
int au_logits(const float* x, int ld_x, const float* w_last, float* out21, int* decisions, int n_clips, int dim, cudaStream_t st);
int au_bce(const float* logits, int ld, const float* labels, const float* pw, float* loss_out, float* dlogits, int n_clips, cudaStream_t st);
// avf_peer.cu: logit gather as pushes over NVLink peer memory
size_t peer_gather_bytes(int world, size_t n);
int logits_push(const float* logits, size_t n, const unsigned long long* peer_base, int world, int rank, const uint32_t* state, cudaStream_t st);
size_t peer_allreduce_bytes(int world, size_t n);
int grad_allreduce(const unsigned long long* peer_base, size_t n, int world, int rank, uint32_t* state, unsigned long long timeout_ns, cudaStream_t st);
int adam_allreduce_step(const unsigned long long* peer_base, size_t n, int world, int rank, uint32_t* state, unsigned long long timeout_ns, float* p, float* m,
                        float* v, void* shadow, float lr, float b1, float b2, float eps, float wd, int step, int decoupled, float grad_scale, cudaStream_t st);
int logits_wait(const void* my_base, size_t n, int world, uint32_t* state, unsigned long long timeout_ns, cudaStream_t st);
int au_confusion(const float* pred, int ld_pred, float thresh, const float* labels, int ld_lab, float ignore, unsigned long long* counts, int n_rows,
                 cudaStream_t st);

// avf_simt.cu
int linear_f32(const float* a, int lda, const float* w, const float* bias, const float* res, int ld_res, void* c, int ldc,
               int c_mode, int m, int n, int k, int flags, cudaStream_t st);
// keep (optional): [n_seq, n_tok] uint8, 1 = keep; score (i, j) survives only when tokens i and j are both kept (include/avformer_b200.h).
int attention_small(int io_mode, const void* qkv, void* out, int n_seq, int n_tok, int heads, int dim_head, cudaStream_t st,
                    const uint8_t* keep = nullptr);

int gemm_f32(int trans_a, int trans_b, const float* a, int lda, const float* w, int ldw, const float* bias, const float* res, int ld_res,
             float* aux, int ld_aux, void* c, int ldc, int c_mode, int m, int n, int k, int flags, cudaStream_t st, DropSpec drop = DropSpec{});

// avf_train.cu
size_t colsum_workspace_bytes(int rows, int cols);
int colsum(int in_mode, const void* x, size_t ld, int rows, int cols, float* out, float beta, void* ws, size_t ws_bytes, cudaStream_t st);
size_t layernorm_bwd_workspace_bytes(int rows, int dim);
// drop_in masks the incoming dres for the dbias sums (dropout on the output of the sub-layer being differentiated);
// drop_out masks the copy written to dxb (dropout on the output of the sub-layer BELOW, whose GEMMs consume dxb).
// dxb is bf16 (dxb_mode AVF_BF16) or fp32.
int layernorm_bwd(const float* x, int ld_x, const float* gamma, const float* dyn, float* dres, int ld_d, void* dxb, int dxb_mode, float* dgamma,
                  float* dbeta, float* dbias, float beta_acc, int rows, int dim, void* ws, size_t ws_bytes, cudaStream_t st,
                  DropSpec drop_in = DropSpec{}, DropSpec drop_out = DropSpec{});
// y = x * mask(drop) as bf16 / fp32 (dense [rows, dim]); without dropout a plain cast / copy
int masked_copy(const float* x, void* y, int y_mode, int rows, int dim, DropSpec drop, cudaStream_t st);
int dropout_mask(float* out, int rows, int cols, DropSpec drop, cudaStream_t st);
int attention_bwd(int io_mode, const void* qkv, const void* dout, void* dqkv, int n_seq, int n_tok, int heads, int dim_head, cudaStream_t st,
                  const uint8_t* keep = nullptr);
int au_logits_bwd(const float* dl, int ld_dl, const float* x, int ld_x, const float* w_last, float* dx, int ld_dx, float* dw, int n_clips,
                  int dim, cudaStream_t st);
int bn_train_fwd(int out_mode, const float* x, int ld_x, const float* g, const float* b, float* run_mean, float* run_var, float momentum,
                 void* y, float* save_mean, float* save_rstd, int rows, int dim, cudaStream_t st);
int bn_bwd(const float* x, int ld_x, const float* dy, const float* g, const float* mean, const float* rstd_or_var, int batch_stats, float* dx,
           int ld_dx, float* dgamma, float* dbeta, int rows, int dim, cudaStream_t st);
int adam_step(float* p, const float* g, float* m, float* v, void* shadow, size_t n, float lr, float b1, float b2, float eps, float wd, int step,
              int decoupled, float grad_scale, cudaStream_t st);

// avf_attention_mma.cu
int attention_mma_bf16(const void* qkv, void* out, int n_seq, int n_tok, int heads, int dim_head, cudaStream_t st, int q_rows = 0,
                       const uint8_t* keep = nullptr);
int attention_bwd_mma_bf16(const void* qkv, const void* dout, void* dqkv, int n_seq, int n_tok, int heads, int dim_head, cudaStream_t st,
                           const uint8_t* keep = nullptr);

// avf_layer_fused.cu: whole encoder stack in one persistent tcgen05 kernel (dim 256 or 128, 8 heads x 32)
bool encoder_fused_supported(const avf_stack_shape* s);
int fused_prof_read(unsigned long long* out64, int reset);   // phase counters, only with -DAVF_FUSED_PROF
int fused_set_trap_buffer(void* host_mapped_words);          // 4 host-mapped words a timed-out wait fills in before trapping
size_t encoder_fused_scratch_bytes();                        // scratch of the NCHW form (channel-major positional table)
int encoder_fused(int io_kind, const avf_stack_shape* s, const avf_layer_weights* L, const void* in, int ld_in, void* out, int ld_out,
                  const float* pos, void* scratch, const float* w_last, float* out21, int* decisions, cudaStream_t st);

// avf_gemm_umma.cu
int gemm_umma(int trans_a, int trans_b, const void* a, int lda, const void* w, int ldw, const float* bias, const float* res, int ld_res,
              const void* aux, int ld_aux, void* c, int ldc, int c_mode, int m, int n, int k, int flags, void* ws, size_t ws_bytes,
              cudaStream_t stream, DropSpec drop = DropSpec{});
size_t gemm_umma_workspace_bytes(int m, int n, int k);
void tmap_cache_stats(uint64_t* hits, uint64_t* misses);     // CUtensorMap cache (keyed by pointer / shape / pitch / box)
int gemm_prof_read(unsigned long long* out16);               // milestone timestamps of CTA 0, only with -DAVF_GEMM_PROF
int linear_umma(const void* a, int lda, const void* w, const float* bias, const float* res, int ld_res, void* c, int ldc,
                int c_mode, int m, int n, int k, int flags, cudaStream_t st);

}  // namespace avf
