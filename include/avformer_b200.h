/*
 * avformer_b200.h — C ABI of the B200-native AVFormer transformer hot path.
 *
 * Drop-in boundary for the transformer-encoder stack of the reference
 * (paths relative to the reference repo root):
 *   models/heads.py:164-256   GELU / Residual / PreNorm / FeedForward / Attention / Transformer
 *   models/vformer.py:245-259 SFormer token region of ResFormer.forward
 *   models/vformer.py:270-293 TFormer
 *   models/heads.py:258-339   AU_former
 *   models/tformer.py:362-403 fusion head (former_AU_head)
 *   models/loss.py:63-103     AULoss;   train.py:155  decision rule
 *
 * The reference has no FFI (it is pure Python/PyTorch); these are the entry points a
 * ctypes/cffi binding of that path binds (INTEGRATION.md shows the stub).  Conventions:
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream);
 *   - every function returns 0 on success, a negative AVF_E* code on a usage error, or a
 *     positive cudaError_t; avf_last_error() returns a human readable message for the
 *     calling thread.  Nothing is ever computed on the CPU: without a CUDA device every
 *     compute entry point fails with AVF_ENODEVICE.
 *   - activations are row-major; "tokens" are rows of a [n_seq * n_tok, dim] matrix;
 *   - mode AVF_BF16: GEMM operands bf16 (tcgen05 / TMEM accumulators in fp32), residual stream,
 *     LayerNorm statistics, softmax and all accumulators fp32.  mode AVF_FP32: everything fp32 on
 *     the CUDA cores (parity mode, 1e-4 relative to the reference).
 */
#ifndef AVFORMER_B200_H_
#define AVFORMER_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AVF_ABI_VERSION 1

enum { AVF_FP32 = 0, AVF_BF16 = 1 };                 /* compute mode / storage dtype selector */
enum { AVF_EINVAL = -1, AVF_ENODEVICE = -2, AVF_EWORKSPACE = -3, AVF_EUNSUPPORTED = -4 };

/* epilogue flags of avf_linear_fwd */
enum { AVF_EPI_BIAS = 1, AVF_EPI_GELU = 2, AVF_EPI_RESIDUAL = 4, AVF_EPI_DGELU = 8 /* x gelu'(aux), training */,
       AVF_EPI_SAVE_PRE = 16 /* store the pre-GELU value (after bias) to aux, training */,
       AVF_EPI_DROPOUT = 32 /* dropout mask after bias/GELU, before the residual add (internal: needs a seed) */,
       AVF_EPI_ACCUMULATE = 64 /* C += result (wgrad form: gradient accumulation straight into p.grad) */ };

/* One pre-LN encoder layer (models/heads.py:246-250).  Weight matrices are [out, in] row-major
 * exactly as nn.Linear stores them; `w_dtype` says whether they are fp32 or bf16 copies
 * (avf_cast_f32_to_bf16 makes the latter).  Vectors are always fp32. */
typedef struct avf_layer_weights {
  const float* ln1_gamma;   /* [dim]            layers.L.0.fn.norm.weight          */
  const float* ln1_beta;    /* [dim]            layers.L.0.fn.norm.bias            */
  const void*  w_qkv;       /* [3*inner, dim]   layers.L.0.fn.fn.to_qkv.weight  (rows q|k|v, head-major) */
  const void*  w_out;       /* [dim, inner]     layers.L.0.fn.fn.to_out.0.weight   */
  const float* b_out;       /* [dim]            layers.L.0.fn.fn.to_out.0.bias     */
  const float* ln2_gamma;   /* [dim]            layers.L.1.fn.norm.weight          */
  const float* ln2_beta;    /* [dim]            layers.L.1.fn.norm.bias            */
  const void*  w_ff1;       /* [mlp, dim]       layers.L.1.fn.fn.net.0.weight      */
  const float* b_ff1;       /* [mlp]            layers.L.1.fn.fn.net.0.bias        */
  const void*  w_ff2;       /* [dim, mlp]       layers.L.1.fn.fn.net.3.weight      */
  const float* b_ff2;       /* [dim]            layers.L.1.fn.fn.net.3.bias        */
} avf_layer_weights;

/* Geometry of an encoder stack (SURVEY.md appendix B). */
typedef struct avf_stack_shape {
  int32_t n_seq;      /* sequences (frames for SFormer, clips otherwise) */
  int32_t n_tok;      /* tokens per sequence: 49 / T+1 / 12; <= 64 with 32-wide heads, <= 256 with 64-wide heads */
  int32_t dim;        /* model dim D: 256 / 512 / 128 / 256               */
  int32_t heads;      /* 8                                                */
  int32_t dim_head;   /* 32 or 64                                         */
  int32_t mlp_dim;    /* 512 / 1024 / 256 / 256                           */
  int32_t depth;      /* layers                                           */
} avf_stack_shape;

/* ---- library / device ------------------------------------------------------------------- */
int         avf_abi_version(void);
const char* avf_last_error(void);
/* Number of kernels this library has launched in this process (bench.py's gpu_launches evidence). */
uint64_t    avf_launch_count(void);
/* SM count, compute capability major*10+minor, and whether the tcgen05 path is usable. */
int         avf_device_info(int32_t* sm_count, int32_t* cc, int32_t* has_tcgen05);

/* The encoder stacks with dim 256 or 128 / 8 heads x 32 (SFormer, fusion head, AU_formers, VA_former) run as ONE persistent
 * tcgen05 kernel per stack in mode AVF_BF16 (residual stream in TMEM, see csrc/avf_layer_fused.cu).  avf_set_fused_enabled(0) forces
 * the kernel-per-operation path instead (used by the A/B parity tests); returns the previous setting. */
int         avf_set_fused_enabled(int enabled);
int         avf_encoder_fused_supported(const avf_stack_shape* s, int mode);
/* Upper bound on the grid of the persistent kernels (fused encoder, tcgen05 GEMM) launched AFTER the call; 0 = all SMs.
 * Returns the previous value.  Lets a caller run two kernel chains side by side on disjoint SM sets (each persistent CTA
 * owns a whole SM): e.g. cap 116 around the SFormer launch, cap 32 around the TFormer / head chain on another stream. */
int         avf_set_sm_cap(int cap);
/* Programmatic dependent launch of every kernel of the library (default on): a kernel is scheduled while its predecessor in
 * the stream still runs and waits (griddepcontrol.wait) for it to complete before it touches memory.  0 = plain launches
 * (A/B tests).  Returns the previous setting. */
int         avf_set_pdl_enabled(int enabled);
/* Developer aid: 64 per-phase cycle counters of the fused kernel when the library is built with -DAVF_FUSED_PROF
 * (tools/fused_phases.py); AVF_EUNSUPPORTED otherwise. */
int         avf_debug_fused_prof(uint64_t* out64, int reset);
/* Developer aid: `host_mapped_words` = 4 uint32 in pinned (device-visible) host memory, or NULL.  A wait inside the fused
 * kernel that times out (a protocol bug) writes {block, thread, barrier index, parity} there before it traps. */
int         avf_debug_set_trap_buffer(void* host_mapped_words);
/* Developer aid: hits / misses of the CUtensorMap cache (maps are keyed by pointer, shape, pitch and box, so the steady state of
 * an eagerly launched step encodes none). */
int         avf_debug_tmap_cache(uint64_t* hits, uint64_t* misses);
/* Developer aid: 16 %globaltimer stamps (ns) of CTA 0 of the last tcgen05 GEMM launch when the library is built with
 * -DAVF_GEMM_PROF (tools/gemm_phases.py); AVF_EUNSUPPORTED otherwise. */
int         avf_debug_gemm_prof(uint64_t* out16);

/* ---- workspace ---------------------------------------------------------------------------- */
/* Bytes of scratch avf_encoder_stack_fwd needs for this shape/mode (replaces the implicit ATen
 * temporaries of models/heads.py:219-239). */
size_t avf_encoder_workspace_bytes(const avf_stack_shape* s, int mode);

/* ---- a1..a5: the encoder ------------------------------------------------------------------- */
/* x [n_seq*n_tok, ld_x] fp32 residual stream, updated IN PLACE through `depth` layers (n_tok <= 64 with dim_head 32, <= 256 with
 * dim_head 64; longer sequences return AVF_EUNSUPPORTED)
 * (models/heads.py:252-256).  If out != NULL the LAST layer's result is written to
 * out [.., ld_out] instead of x (used to write the two AU_former outputs side by side into the
 * [B,12,256] fusion input, models/avformer.py:100). */
int avf_encoder_stack_fwd(int mode, const avf_stack_shape* s, const avf_layer_weights* layers,
                          float* x, int32_t ld_x, float* out, int32_t ld_out,
                          void* workspace, size_t workspace_bytes, void* stream);
/* The encoder stack of a token head (AU_former, VA_former, fusion head): x [n_seq*n_tok, ld_x] fp32 (+ pos[n_tok, dim] when
 * pos != NULL) -> `depth` layers -> out (or x in place when out == NULL), like avf_encoder_stack_fwd.  With w_last [12, dim]
 * (n_tok = 12) the AU logits of the result follow as in avf_au_logits_fwd: out21 [n_seq, 21] (required) and decisions [n_seq, 12]
 * (may be NULL); the token rows are then only stored when out != NULL.  x is scratch whenever out != NULL or w_last != NULL.
 * Same workspace as avf_encoder_stack_fwd.  In mode AVF_BF16 a stack the fused kernel supports (dim 256 or 128) is ONE launch,
 * positional add and logits included; otherwise the sequence avf_add_row_periodic -> avf_encoder_stack_fwd -> avf_au_logits_fwd. */
int avf_token_stack_fwd(int mode, const avf_stack_shape* s, const avf_layer_weights* layers, float* x, int32_t ld_x, const float* pos,
                        float* out, int32_t ld_out, const float* w_last, float* out21, int32_t* decisions,
                        void* workspace, size_t workspace_bytes, void* stream);


/* Building blocks (exposed for tests and for callers that fuse differently). */
/* y[r,:] = LayerNorm(x[r,:]) * gamma + beta, eps 1e-5; y is bf16 (mode BF16) or fp32. */
int avf_layernorm_fwd(int out_mode, const float* x, int32_t ld_x, const float* gamma, const float* beta,
                      void* y, int32_t rows, int32_t dim, void* stream);
/* C[M,N] = epi(A[M,K] * W[N,K]^T): bias[N], tanh-GELU, + residual[M,ld_res] (fp32), in that order.
 * mode BF16: A, W bf16, tcgen05; mode FP32: A, W fp32.  C is bf16 or fp32 per c_mode. */
int avf_linear_fwd(int mode, const void* a, int32_t lda, const void* w, const float* bias,
                   const float* residual, int32_t ld_res, void* c, int32_t ldc, int c_mode,
                   int32_t m, int32_t n, int32_t k, int epilogue_flags, void* stream);
/* softmax(q k^T * dh^-0.5) v per (sequence, head); qkv [rows, 3*heads*dh] with columns q|k|v
 * head-major (models/heads.py:221-237); out [rows, heads*dh].  io_mode = dtype of qkv and out.  n_tok 65..256 needs dh = 64
 * (bf16: any n_tok; fp32 unmasked: n_tok with K|V of one head in shared memory). */
int avf_attention_fwd(int io_mode, const void* qkv, void* out, int32_t n_seq, int32_t n_tok,
                      int32_t heads, int32_t dim_head, void* stream);

/* ---- a6: SFormer token (un)packing, models/vformer.py:247-253 and :257-259 ---------------- */
/* fmap [n_frames, dim, hw] (NCHW, fp32 or bf16 per io_mode) -> x [n_frames*hw, dim] fp32 + pos[hw, dim]
 * (pos == NULL: plain transpose — the backward of avf_sformer_tokens_unpack) */
int avf_sformer_tokens_pack(int io_mode, const void* fmap, const float* pos, float* x,
                            int32_t n_frames, int32_t dim, int32_t hw, void* stream);
int avf_sformer_tokens_unpack(int io_mode, const float* x, void* fmap,
                              int32_t n_frames, int32_t dim, int32_t hw, void* stream);
/* Whole SFormer region: pack, `depth` layers, unpack (fmap_out may alias fmap_in). */
int avf_sformer_fwd(int mode, int io_mode, const avf_stack_shape* s, const avf_layer_weights* layers,
                    const float* pos, const void* fmap_in, void* fmap_out,
                    void* workspace, size_t workspace_bytes, void* stream);
size_t avf_sformer_workspace_bytes(const avf_stack_shape* s, int mode);

/* ---- a7: TFormer glue, models/vformer.py:280-290 ------------------------------------------- */
/* frames [n_clips*T, dim] (fp32/bf16 per io_mode) -> x [n_clips*(T+1), dim] fp32 =
 * cat(cls, frames) + pos[T+1, dim] */
int avf_tformer_embed(int io_mode, const void* frames, const float* cls_token, const float* pos, float* x,
                      int32_t n_clips, int32_t n_frames, int32_t dim, void* stream);
/* Whole TFormer (models/vformer.py:279-290) for inference: embed, `depth` layers, cls rows -> cls_out [n_clips, dim] fp32.  s->n_seq
 * = clips, s->n_tok = T+1.  Only x[:, 0] leaves the module, so the LAST layer computes keys / values for every row but the attention
 * output, out-projection, LayerNorm and MLP for the cls row of each clip only (1/(T+1) of that work).  T <= 255 (n_tok <= 256) with
 * 64-wide heads, T <= 63 with 32-wide heads. */
size_t avf_tformer_workspace_bytes(const avf_stack_shape* s, int mode);
int avf_tformer_fwd(int mode, int io_mode, const avf_stack_shape* s, const avf_layer_weights* layers, const void* frames,
                    const float* cls_token, const float* pos, float* cls_out, void* workspace, size_t workspace_bytes, void* stream);
/* cls[c,:] = x[c*(T+1), :] */
int avf_tformer_cls_extract(const float* x, float* cls, int32_t n_clips, int32_t n_tok, int32_t dim, void* stream);

/* ---- a8: AU_former front end, models/heads.py:293-323 --------------------------------------- */
/* emb [n_clips, 512] fp32 (row stride ld_emb, so the cls rows of a TFormer output can be read in
 * place) -> BatchNorm1d with running statistics (eval) -> 12 Linear(512,128)+b stacked as
 * w_cat [12*128, 512], b_cat [12*128] -> + pos[12,128] -> x [n_clips*12, 128] fp32.  pos == NULL: no positional add
 * (avf_token_stack_fwd adds it inside the stack launch). */
int avf_au_former_front_fwd(int mode, const float* emb, int32_t ld_emb,
                            const float* bn_gamma, const float* bn_beta, const float* bn_mean, const float* bn_var,
                            const void* w_cat, const float* b_cat, const float* pos, float* x,
                            int32_t n_clips, int32_t in_dim, int32_t emb_dim,
                            void* workspace, size_t workspace_bytes, void* stream);
/* The same front for any number of tokens per clip: BatchNorm1d (running statistics) -> n_tok stacked Linear(in_dim, emb_dim) ->
 * view [n_clips*n_tok, emb_dim] -> + pos[n_tok, emb_dim] (if pos != NULL).  n_tok = 12 is the AU_former above; n_tok = 2 is VA_former
 * (models/heads.py:341-372: VA_BN1, VA_linear_p1..2). */
int avf_token_front_fwd(int mode, const float* emb, int32_t ld_emb,
                        const float* bn_gamma, const float* bn_beta, const float* bn_mean, const float* bn_var,
                        const void* w_cat, const float* b_cat, const float* pos, float* x,
                        int32_t n_clips, int32_t in_dim, int32_t emb_dim, int32_t n_tok,
                        void* workspace, size_t workspace_bytes, void* stream);

/* ---- a9 tail + a11 + a12 -------------------------------------------------------------------- */
/* logits[c,i] = <x[c*12+i, :], w_last[i, :]>  written to out21 [n_clips, 21] (cols 12..20 zeroed,
 * models/avformer.py:102-105) and decisions [n_clips,12] int32 = (logit > 0) (train.py:155).
 * Either output may be NULL. */
int avf_au_logits_fwd(const float* x, int32_t ld_x, const float* w_last, float* out21, int32_t* decisions,
                      int32_t n_clips, int32_t dim, void* stream);
/* AULoss (models/loss.py:75-103): rows with labels[c,0] == -1 are dropped; pos_weight [12];
 * loss_out[0] = mean BCE, loss_out[1] = number of valid rows.  If dlogits != NULL it receives
 * d loss / d logits [n_clips,12] (zero on dropped rows). logits has row stride ld_logits (21). */
int avf_au_bce_loss(const float* logits, int32_t ld_logits, const float* labels, const float* pos_weight,
                    float* loss_out, float* dlogits, int32_t n_clips, void* stream);

/* MultiLabelAccF1 (metrics/accf1.py:45-77) without leaving the device: counts48 [12][4] (uint64, ACCUMULATED) += {TP, FP, FN, TN} per AU
 * over the entries whose label != ignore; pred > threshold is the positive decision (logits: 0, i.e. round(sigmoid), train.py:155;
 * 0/1 predictions: 0.5).  acc = sum(TP+TN) / sum(all), f1 = mean_i 2 TP_i / (2 TP_i + FP_i + FN_i); across ranks the 48 counters add. */
int avf_au_confusion_update(const float* pred, int32_t ld_pred, float threshold, const float* labels, int32_t ld_labels, float ignore,
                            uint64_t* counts48, int32_t n_rows, void* stream);

/* ---- evaluation-time logit gather over NVLink peer memory (SURVEY.md section 8(e); replaces the host-side concatenation of the
 * per-batch predictions in train.py:150-170 and the NCCL all-gather of a data-parallel evaluation) ------------------------------
 * Every rank owns one PEER-MAPPED block of avf_peer_gather_bytes(world, n_floats) bytes, zeroed once, laid out as
 * table[2][world][n_floats] fp32 followed (128-byte aligned) by flags[2][world] u32.  peer_base = DEVICE array of the `world` base
 * pointers as mapped into this process (own block included).  state = two DEVICE words, zeroed once: [0] step counter, [1] error.
 * avf_logits_push: store my n_floats logits into slot (step & 1), row block `rank`, of every peer's table and release the flag.
 * avf_logits_wait: spin (bounded by timeout_ns; on expiry state[1] = 1 + the missing rank) until all `world` blocks of the step
 * are in MY table, then step += 1.  The complete table of step i is table[i & 1]; it is overwritten by the pushes of step i + 2,
 * which no rank issues before every rank has pushed step i + 1 — so read it before this rank's push of step i + 1 (stream order).
 * Both are asynchronous on `stream`, graph-capturable, and must be issued the same number of times on every rank. */
size_t avf_peer_gather_bytes(int32_t world, size_t n_floats);
int avf_logits_push(const float* logits, size_t n_floats, const uint64_t* peer_base, int32_t world, int32_t rank, const uint32_t* state, void* stream);
int avf_logits_wait(const void* my_base, size_t n_floats, int32_t world, uint32_t* state, uint64_t timeout_ns, void* stream);

/* ---- data-parallel gradient all-reduce over NVLink peer memory (the reference trains on one GPU, train.py:206-236; this is the
 * exchange step of the clip-sharded training of SURVEY.md section 8(e), in place of torch DDP / an NCCL all-reduce) -----------------
 * Every rank keeps its flat fp32 gradient bucket of n_floats at the start of a PEER-MAPPED block of avf_peer_allreduce_bytes(world,
 * n_floats) bytes (zeroed once: padding and two flag rows follow the bucket).  peer_base = DEVICE array of the `world` base pointers
 * as mapped here; state = three DEVICE words zeroed once ([0] completed reductions, [1] error: 1 + r / 101 + r = rank r missing at
 * entry / exit, [2] scratch).  avf_grad_allreduce sums the buckets of all ranks IN PLACE (every rank ends with the same bits: slice r
 * is added up by rank r in rank order 0..W-1 and stored into all buckets); asynchronous on `stream`, graph-capturable, to be issued
 * once per step on every rank; bounded spins: after timeout_ns the kernel records the missing rank in state[1], prints it and traps
 * (unsummed gradients never reach the optimiser silently).  world <= 16, one node. */
size_t avf_peer_allreduce_bytes(int32_t world, size_t n_floats);
int avf_grad_allreduce(const uint64_t* peer_base, size_t n_floats, int32_t world, int32_t rank, uint32_t* state, uint64_t timeout_ns, void* stream);

/* `adam_allreduce_step` of SURVEY.md section 8(b): the reduction above and the optimiser step of train.py:235-236 (torch.optim.Adam with
 * coupled L2, train.py:334; decoupled != 0 = AdamW) as ONE kernel — as soon as the sums of all slices are in this rank's bucket every CTA
 * updates its share of the replicated parameters (params / exp_avg / exp_avg_sq: flat fp32 buckets of n_floats, a multiple of 4, 16-byte
 * aligned; bf16_shadow: optional bf16 image of the updated parameters).  grad_scale is applied to the summed gradient (1 / world for the
 * mean over shards); step is 1-based (bias correction).  Bit-identical to avf_grad_allreduce followed by avf_adam_step. */
int avf_adam_allreduce_step(const uint64_t* peer_base, size_t n_floats, int32_t world, int32_t rank, uint32_t* state, uint64_t timeout_ns,
                            float* params, float* exp_avg, float* exp_avg_sq, void* bf16_shadow, float lr, float beta1, float beta2, float eps,
                            float weight_decay, int32_t step, int decoupled, float grad_scale, void* stream);

/* ---- parameter preparation ------------------------------------------------------------------ */
int avf_cast_f32_to_bf16(const float* src, void* dst, size_t n, void* stream);
int avf_cast_bf16_to_f32(const void* src, float* dst, size_t n, void* stream);
/* x[r,:] += pos[r % period, :] */
int avf_add_row_periodic(float* x, int32_t ld_x, const float* pos, int32_t rows, int32_t dim, int32_t period, void* stream);

/* ============================================================================================
 * Training (train.py:206-236 restricted to the transformer stack): loss.backward() through the
 * drop-in modules lands here.  bf16 mode keeps GEMM operands (activations on the tape, gradient
 * operands, weights) in bf16 and everything else — residual / gradient streams, statistics,
 * reductions, weight gradients, optimiser state — in fp32.  All reductions have a fixed order.
 * ============================================================================================ */

/* Gradient destinations of one layer, same field order as avf_layer_weights; every buffer is fp32 with the shape
 * of its parameter and is OVERWRITTEN.  A NULL field skips that gradient (frozen parameter). */
typedef struct avf_layer_grads {
  float* ln1_gamma; float* ln1_beta; float* w_qkv; float* w_out; float* b_out;
  float* ln2_gamma; float* ln2_beta; float* w_ff1; float* b_ff1; float* w_ff2; float* b_ff2;
} avf_layer_grads;

/* General GEMM behind every linear of the forward and backward pass:  C[M,N] = epi(op(A) op(B)).
 *   trans_a = 0: A is [M,K] row-major (lda);   1: A is stored [K,M] row-major.
 *   trans_b = 0: B is [N,K] row-major (nn.Linear layout: C = A B^T);   1: B is stored [K,N] row-major.
 * so  forward  Y = X W^T (0,0);  dgrad  dX = dY W (0,1, B = W itself);  wgrad  dW = dY^T X (1,1, K = token rows).
 * mode BF16: operands bf16 on tcgen05 (operands with the reduction index as row index are fed as MN-major tiles, no
 * transposed copy); the (1,1) form splits K over the SMs and needs avf_gemm_workspace_bytes() of scratch, writes plain
 * fp32.  mode FP32: CUDA cores.  `aux` [M, ld_aux] (bf16 / fp32 per mode): AVF_EPI_SAVE_PRE stores the pre-GELU value
 * there, AVF_EPI_DGELU multiplies the accumulator by gelu'(aux) before anything else. */
size_t avf_gemm_workspace_bytes(int mode, int trans_a, int trans_b, int32_t m, int32_t n, int32_t k);
int avf_gemm(int mode, int trans_a, int trans_b, const void* a, int32_t lda, const void* b, int32_t ldb,
             const float* bias, const float* residual, int32_t ld_res, void* aux, int32_t ld_aux,
             void* c, int32_t ldc, int c_mode, int32_t m, int32_t n, int32_t k, int epilogue_flags,
             void* workspace, size_t workspace_bytes, void* stream);

/* Encoder stack, forward with an activation tape (x is NOT modified; the result goes to out, row stride ld_out)
 * and backward.  dx [n_seq*n_tok, dim] dense fp32 holds the gradient wrt the stack output on entry and the gradient
 * wrt its input on return; grads[depth] receives the parameter gradients (NULL: none wanted); with accumulate != 0 they are
 * ADDED to the buffers (which then are the optimiser's gradient bucket itself) instead of overwriting them.
 * dropout_p > 0 applies nn.Dropout at the reference's three sites per layer (after to_out, after GELU, after net.3;
 * models/heads.py:216,194,197) with a stateless counter-based mask derived from dropout_seed: the backward call must be given
 * the same (p, seed, salt) and regenerates the masks instead of storing them.  dropout_salt (optional) points to one DEVICE
 * uint32 that is hashed into the seed when the kernels start: a captured CUDA graph gets fresh masks on every replay by
 * changing that word between replays.  avf_dropout_mask writes the scaled mask
 * (0 or 1/(1-p)) of one site (0 = to_out [rows, dim], 1 = GELU [rows, mlp_dim], 2 = net.3 [rows, dim]) for tests.
 * n_tok <= 64 with dim_head 32, <= 256 with dim_head 64, as in avf_encoder_stack_fwd. */
size_t avf_encoder_tape_bytes(const avf_stack_shape* s, int mode);
size_t avf_encoder_bwd_workspace_bytes(const avf_stack_shape* s, int mode);
int avf_encoder_stack_fwd_train(int mode, const avf_stack_shape* s, const avf_layer_weights* layers,
                                const float* x, int32_t ld_x, float* out, int32_t ld_out,
                                void* tape, size_t tape_bytes, float dropout_p, uint64_t dropout_seed,
                                const uint32_t* dropout_salt, void* stream);
int avf_encoder_stack_bwd(int mode, const avf_stack_shape* s, const avf_layer_weights* layers,
                          const void* tape, size_t tape_bytes, float* dx, int32_t ld_dx,
                          const avf_layer_grads* grads, int accumulate, void* workspace, size_t workspace_bytes,
                          float dropout_p, uint64_t dropout_seed, const uint32_t* dropout_salt, void* stream);
int avf_dropout_mask(float dropout_p, uint64_t dropout_seed, const uint32_t* dropout_salt, int32_t layer, int32_t site,
                     int32_t rows, int32_t cols, float* out, void* stream);

/* Building blocks of the backward pass (exposed for tests). */
/* out[c] = sum_r x[r, c]; x is fp32 or bf16 per in_mode with row stride ld (elements). */
size_t avf_colsum_workspace_bytes(int32_t rows, int32_t cols);
int avf_colsum(int in_mode, const void* x, size_t ld, int32_t rows, int32_t cols, float* out,
               void* workspace, size_t workspace_bytes, void* stream);
/* Backward of y = x + f(LN(x)): dres (in: dL/dy, out: dL/dx) += LN'(dy_norm); optional bf16 copy of the result;
 * dgamma / dbeta of the LayerNorm and dbias = column sums of the incoming dres (bias gradient of f's last linear). */
size_t avf_layernorm_bwd_workspace_bytes(int32_t rows, int32_t dim);
int avf_layernorm_bwd(const float* x, int32_t ld_x, const float* gamma, const float* dy_norm, float* dres, int32_t ld_d,
                      void* dx_bf16, float* dgamma, float* dbeta, float* dbias, int32_t rows, int32_t dim,
                      void* workspace, size_t workspace_bytes, void* stream);
/* dqkv [rows, 3*heads*dh] from qkv and dout [rows, heads*dh] (softmax recomputed).  n_tok <= 64, or <= 256 with dh = 64. */
int avf_attention_bwd(int io_mode, const void* qkv, const void* dout, void* dqkv, int32_t n_seq, int32_t n_tok,
                      int32_t heads, int32_t dim_head, void* stream);

/* AU_former front end for training.  batch_stats = 1: BatchNorm1d uses batch statistics and updates the running
 * ones in place with `momentum` (nn.BatchNorm1d in train()); 0: running statistics (eval(), or a frozen model). */
size_t avf_au_former_front_tape_bytes(int mode, int32_t n_clips, int32_t in_dim);
int avf_au_former_front_fwd_train(int mode, const float* emb, int32_t ld_emb,
                                  const float* bn_gamma, const float* bn_beta, float* bn_mean, float* bn_var,
                                  int batch_stats, float momentum, const void* w_cat, const float* b_cat, const float* pos,
                                  float* x, int32_t n_clips, int32_t in_dim, int32_t emb_dim,
                                  void* tape, size_t tape_bytes, void* stream);
size_t avf_au_former_front_bwd_workspace_bytes(int mode, int32_t n_clips, int32_t in_dim, int32_t emb_dim);
/* dx [n_clips*12, emb_dim] fp32 dense -> demb [n_clips, in_dim] (row stride ld_demb), dbn_gamma, dbn_beta [in_dim],
 * dw_cat [12*emb_dim, in_dim], db_cat [12*emb_dim] (== the gradient of pos_embedding).  Any output may be NULL. */
int avf_au_former_front_bwd(int mode, const float* emb, int32_t ld_emb, const float* bn_gamma,
                            const float* bn_mean, const float* bn_var, int batch_stats, const void* w_cat,
                            const void* tape, size_t tape_bytes, const float* dx,
                            float* demb, int32_t ld_demb, float* dbn_gamma, float* dbn_beta, float* dw_cat, float* db_cat,
                            int32_t n_clips, int32_t in_dim, int32_t emb_dim,
                            void* workspace, size_t workspace_bytes, void* stream);

/* Backward of avf_au_logits_fwd: dx[c*12+i,:] = dlogits[c,i] w_last[i,:]; dw_last[i,:] = sum_c dlogits[c,i] x[c*12+i,:]. */
int avf_au_logits_bwd(const float* dlogits, int32_t ld_dlogits, const float* x, int32_t ld_x, const float* w_last,
                      float* dx, int32_t ld_dx, float* dw_last, int32_t n_clips, int32_t dim, void* stream);

/* One Adam step on a flat fp32 bucket (train.py:334: torch.optim.Adam, weight decay coupled into the gradient;
 * decoupled = 1 gives AdamW).  grads are multiplied by grad_scale first (1/world_size after a sum all-reduce).
 * bf16_shadow (optional) receives the updated parameters as bf16.  step counts from 1. */
int avf_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, void* bf16_shadow, size_t n,
                  float lr, float beta1, float beta2, float eps, float weight_decay, int32_t step, int decoupled,
                  float grad_scale, void* stream);

/* ---- attention masks (the `mask` of Transformer.forward, models/heads.py:225-232) ---------------
 * keep [n_seq, n_tok] DEVICE uint8, 1 = keep.  Score (i, j) of every head of sequence b survives iff keep[b, i] and keep[b, j]; the
 * other scores are filled with the same very negative value before the softmax.  So a kept query attends only to kept keys (dropped
 * keys get probability exactly 0), and a dropped query attends uniformly to all n_tok tokens (its output is the mean of V, never NaN).
 * The mask is generic: a caller that wants a token kept always (the cls slot) sets its byte.  n_tok <= 64, or <= 256 with 64-wide
 * heads.  keep == NULL is exactly
 * the unmasked call.  A masked stack never takes the fused kernel (it runs kernel by kernel); the backward must be given the keep
 * array of its forward.  Same workspace / tape sizes as the unmasked calls. */
int avf_attention_fwd_masked(int io_mode, const void* qkv, void* out, int32_t n_seq, int32_t n_tok,
                             int32_t heads, int32_t dim_head, const uint8_t* keep, void* stream);
int avf_attention_bwd_masked(int io_mode, const void* qkv, const void* dout, void* dqkv, int32_t n_seq, int32_t n_tok,
                             int32_t heads, int32_t dim_head, const uint8_t* keep, void* stream);
int avf_encoder_stack_fwd_masked(int mode, const avf_stack_shape* s, const avf_layer_weights* layers, const uint8_t* keep,
                                 float* x, int32_t ld_x, float* out, int32_t ld_out,
                                 void* workspace, size_t workspace_bytes, void* stream);
int avf_encoder_stack_fwd_train_masked(int mode, const avf_stack_shape* s, const avf_layer_weights* layers, const uint8_t* keep,
                                       const float* x, int32_t ld_x, float* out, int32_t ld_out,
                                       void* tape, size_t tape_bytes, float dropout_p, uint64_t dropout_seed,
                                       const uint32_t* dropout_salt, void* stream);
int avf_encoder_stack_bwd_masked(int mode, const avf_stack_shape* s, const avf_layer_weights* layers, const uint8_t* keep,
                                 const void* tape, size_t tape_bytes, float* dx, int32_t ld_dx,
                                 const avf_layer_grads* grads, int accumulate, void* workspace, size_t workspace_bytes,
                                 float dropout_p, uint64_t dropout_seed, const uint32_t* dropout_salt, void* stream);
/* avf_tformer_fwd with keep [n_clips, T+1] (row 0 of each clip is its cls token); the cls-only last layer honours it too. */
int avf_tformer_fwd_masked(int mode, int io_mode, const avf_stack_shape* s, const avf_layer_weights* layers, const uint8_t* keep,
                           const void* frames, const float* cls_token, const float* pos, float* cls_out,
                           void* workspace, size_t workspace_bytes, void* stream);

/* ---- whole-video inference: TFormer clips gathered from a per-video frame bank (models/vformer.py:280-290) --------------------
 * bank [n_bank, dim] DEVICE, contiguous, fp32 or bf16 per io_mode (16- / 8-byte aligned): the frame features of one video, each
 * frame computed once.  index [n_clips, T] DEVICE int32: clip c's slot t is frame index[c*T + t].  s->n_seq = n_clips,
 * s->n_tok = T+1.  An entry outside [0, n_bank) is a MISSING frame: its token is pos[1+t] alone and it is masked out of every layer
 * (keep of avf_tformer_fwd_masked, with the cls slot kept); the bank is never read outside [0, n_bank), whatever the index holds.
 * The gather, the keep rows and the embed are one launch; the layers always run masked, so the result equals avf_tformer_fwd_masked
 * on the gathered frames (any value in the missing slots) with keep = (0 <= index < n_bank).  Inference only; the workspace is
 * avf_tformer_workspace_bytes plus the keep rows. */
size_t avf_tformer_indexed_workspace_bytes(const avf_stack_shape* s, int mode);
int avf_tformer_fwd_indexed(int mode, int io_mode, const avf_stack_shape* s, const avf_layer_weights* layers,
                            const void* bank, int32_t n_bank, const int32_t* index,
                            const float* cls_token, const float* pos, float* cls_out,
                            void* workspace, size_t workspace_bytes, void* stream);

/* ---- training over a frame bank: the indexed embed and its backward (models/vformer.py:280-290) ------------------------------
 * avf_tformer_embed_indexed: the gather + embed step of avf_tformer_fwd_indexed alone.  bank / index as there; writes the fp32 token
 * matrix x [n_clips*(T+1), dim] (T = n_frames) and keep [n_clips, T+1] uint8 (1 = kept, the cls slot always), the input and the
 * mask of the tape-keeping avf_encoder_stack_fwd_train_masked.
 * avf_tformer_embed_indexed_bwd: dbank [n_bank, dim] (fp32, or bf16 for a bf16 bank: out_mode) =
 *   dbank[i] = sum of dtok[c*(T+1) + 1 + t] over every slot s = c*T + t with index[s] == i,
 * each column one fp32 chain over the slots in ascending s starting from +0.0 (bf16: that sum rounded once), so the result is
 * bit-reproducible and independent of the grid.  No float atomics.  Every row is written (+0.0 where no slot points); an entry
 * outside [0, n_bank) contributes nowhere, and nothing outside dbank is written.  dtok 16-byte aligned, dbank 16- (fp32) or 8-byte
 * (bf16) aligned.  The gradients of cls_token and pos are avf_colsum over dtok, as for avf_tformer_embed.  Three launches. */
int avf_tformer_embed_indexed(int io_mode, const void* bank, int32_t n_bank, const int32_t* index, const float* cls_token,
                              const float* pos, float* x, uint8_t* keep, int32_t n_clips, int32_t n_frames, int32_t dim, void* stream);
size_t avf_tformer_embed_indexed_bwd_workspace_bytes(int32_t n_clips, int32_t n_frames, int32_t n_bank);
int avf_tformer_embed_indexed_bwd(int out_mode, const float* dtok, const int32_t* index, int32_t n_clips, int32_t n_frames,
                                  int32_t dim, int32_t n_bank, void* dbank, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* AVFORMER_B200_H_ */
