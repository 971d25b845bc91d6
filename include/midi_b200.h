/* midi_b200.h -- C ABI of libmidi_b200.so: the sm_100a kernels behind the drop-in MIDIModel.
 *
 * The reference (SkyTNT/midi-model) has no FFI: its hot path is the Python class
 * `MIDIModel` (midi_model.py:99-250) whose arithmetic is delegated to HF transformers /
 * ATen.  This header is therefore the *new* boundary a maintainer binds with ctypes (see
 * INTEGRATION.md): plain pointers and sizes, no torch types, no allocation inside, the caller's
 * cudaStream_t last.  Each entry cites the reference call it replaces.
 *
 * Conventions
 *   - every function returns 0 (B200_OK) or a negative code; b200_last_error() gives the message
 *     (thread-local).  Nothing is allocated or synchronised inside; workspaces are caller-owned and
 *     sized by the *_workspace_bytes / *_parts queries.
 *   - all device pointers: bf16 activations/weights unless typed otherwise; token ids are int64
 *     (torch.long, the MIDITokenizerV2 tensor layout (batch, events, 8)); row-major.
 *   - kernels are re-entrant per stream (no global mutable state).
 */
#ifndef MIDI_B200_H
#define MIDI_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __DRIVER_TYPES_H__
typedef struct CUstream_st* cudaStream_t;
#endif

#define B200_OK 0
#define B200_ERR_ARG (-1)
#define B200_ERR_CUDA (-2)
#define B200_ERR_UNSUPPORTED (-3)

/* ---- runtime ------------------------------------------------------------------------------ */
const char* b200_last_error(void);
int b200_abi_version(void);
long long b200_launch_count(void);   /* kernels launched by this library so far (all threads) */
int b200_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- embeddings (midi_model.py:145-146 `embed_tokens(x).sum(-2)`; :126-131 cat([hidden, embed(x)])) */
int b200_embed_sum_fwd(const long long* ids, const void* table, void* out, int M, int T, int H, int V, cudaStream_t s);
int b200_inner_input_fwd(const void* hidden /*may be NULL*/, const long long* ids, const void* table, void* out,
                         int n_events, int n_ids, int H, int V, cudaStream_t s);
int b200_inner_input_bwd_hidden(const void* dx, void* dhidden, int n_events, int Tin, int H, cudaStream_t s);
/* host data path (train.py:71 int16 token matrices; train.py:169-176 x = batch[:, :-1], y = batch[:, 1:]):
   batch int16 [B, S1, T] -> x, y int64 [B*(S1-1), T] in one pass */
int b200_batch_to_xy_i16(const void* batch, int B, int S1, int T, long long* x, long long* y, cudaStream_t s);
size_t b200_embed_bwd_workspace_bytes(int n_ids, int V, int H);
/* id i reads gradient row (i / per_row) * row_stride + (i % per_row) * row_inner + row_off; pad row gets 0 */
int b200_embed_bwd(const long long* ids, int n_ids, const void* dout, void* dtable, int V, int H, int per_row,
                   int row_stride, int row_inner, int row_off, int pad_id, int accumulate, void* workspace,
                   size_t workspace_bytes, cudaStream_t s);

/* ---- RMSNorm (hf modeling_llama.py:62-67) --------------------------------------------------- */
int b200_rmsnorm_fwd(const void* x, const void* w, void* y, float* rstd /*may be NULL*/, int M, int H, float eps,
                     cudaStream_t s);
/* fused residual add + norm: h_out = bf16(x + res) (hf :325 / :331), y = RMSNorm(h_out) * w */
int b200_add_rmsnorm_fwd(const void* x, const void* res, const void* w, void* h_out, void* y, float* rstd /*may be NULL*/,
                         int M, int H, float eps, cudaStream_t s);
int b200_rmsnorm_bwd_parts(void);
/* dx = dres + d(norm)/dx ; dw (+)= column sums.  workspace: float[b200_rmsnorm_bwd_parts() * H]; its first H + 1 words
 * (fp32 accumulator row + arrival ticket of the fused column sum) must be ZERO when first handed in -- the kernel hands
 * them back zeroed, so one cudaMemset at allocation is enough */
int b200_rmsnorm_bwd(const void* dy, const void* x, const void* w, const float* rstd, const void* dres /*may be NULL*/,
                     void* dx, void* dw /*may be NULL*/, int M, int H, int accumulate_dw, void* workspace,
                     size_t workspace_bytes, cudaStream_t s);

/* ---- RoPE (hf modeling_llama.py:124-168), applied in place to the q,k thirds of packed qkv -------- */
int b200_rope_table(const float* inv_freq, int half, int n_pos, int pos0, const int* pos0_dev /*may be NULL*/,
                    void* cos_t, void* sin_t, cudaStream_t s);
/* row r sits at absolute position pos0 (+ *pos0_dev) + r % S; tables are indexed by absolute position */
int b200_rope_qk(void* qkv, const void* cos_t, const void* sin_t, int rows, int S, int H, int D, int ld, int backward,
                 int pos0, const int* pos0_dev /*may be NULL*/, cudaStream_t s);

/* ---- SwiGLU (hf modeling_llama.py:183) on packed [rows, 2I] = [gate | up] ------------------------- */
int b200_swiglu_fwd(const void* gu, void* act, long long rows, int I, cudaStream_t s);
int b200_swiglu_bwd(const void* gu, const void* dact, void* dgu, long long rows, int I, cudaStream_t s);

/* ---- LoRA scaling (train.py:439-449 -> peft lora/layer.py Linear.forward `* scaling`): y = bf16(x * scale) over n
 *      elements.  The adapter itself runs on b200_gemm_bf16: t = x A^T, y += (scale t) B^T through the residual
 *      epilogue, and the four gradient GEMMs (midi_b200/engine.py::StackEngine._lora_fwd/_lora_bwd). */
int b200_scale_bf16(const void* x, void* y, long long n, float scale, cudaStream_t s);

/* ---- tensor-core GEMM (tcgen05 / TMEM / TMA): every nn.Linear of hf modeling_llama.py:177-184,
 *      238-264, 288 and lm_head (midi_model.py:135), plus their dgrad / wgrad.
 *      C[M,N] = A . B^T, fp32 accumulate, bf16 out.  a_mn_major / b_mn_major = operand stored [K, rows].
 *      R != NULL: C = bf16(bf16(acc) + R) (residual add, hf :325 / :331).
 *      splits > 1 or accumulate: fp32 split-K partials in `workspace`, reduced (and added to C). */
size_t b200_gemm_workspace_bytes(int M, int N, int splits);
/* optional fp32 workspace that lets b200_gemm_bf16 cut the tiles of the last partial wave along K (0: not useful) */
size_t b200_gemm_tail_workspace_bytes(int M, int N, int K, int block_n);
int b200_gemm_suggest_splits(int M, int N, int K, int block_n);
/* cheapest (block_n in {128,256}, split-K factor) for an [M,N,K] problem on this device */
int b200_gemm_plan(int M, int N, int K, int allow_split, int* block_n_out, int* splits_out);
int b200_gemm_bf16(const void* A, const void* B, void* C, const void* R, int M, int N, int K, int lda, int ldb, int ldc,
                   int ldr, int a_mn_major, int b_mn_major, int accumulate, int block_n, int splits, void* workspace,
                   size_t workspace_bytes, cudaStream_t s);

/*      QKV projection with RoPE fused into the epilogue (hf modeling_llama.py:262-268): rows sit at positions
 *      r % S, columns [0, rope_cols) are rotated per head of width head_dim, the rest (v) is stored unrotated. */
int b200_gemm_bf16_rope(const void* A, const void* B, void* C, int M, int N, int K, int lda, int ldb, int ldc,
                        const void* rope_cos, const void* rope_sin, int S, int head_dim, int rope_cols, cudaStream_t s);

/*      gate|up projection with SwiGLU fused (hf modeling_llama.py:182-184): gu[M,2I] = A . Wgu^T is stored (backward
 *      needs g, u) and act[M,I] = bf16(bf16(silu(g)) * u) is produced by the same epilogue; I % 128 == 0 */
int b200_gemm_bf16_swiglu(const void* A, const void* Wgu, void* gu, void* act, int M, int I, int K, int lda, int ldw,
                          int ld_gu, int ld_act, cudaStream_t s);

/* ---- attention (hf integrations/sdpa_attention.py:41-104 via modeling_llama.py:251-289) ----------
 *      outer stack: causal flash attention, head_dim 64; strides are element strides {batch,row,head}. */
int b200_attn_causal_fwd(const void* q, const void* k, const void* v, void* o, float* lse /*may be NULL*/,
                         const long long* strides /*4x3: q,k,v,o*/, int batch, int n_heads, int Sq, int Sk, int head_dim,
                         float scale, cudaStream_t s);
/*      same contract on the tcgen05 tensor cores (TMA-staged 128-key K/V tiles, S and P.V accumulators in TMEM);
 *      heads must be contiguous blocks of 64 columns (strides[.h] == 64) */
int b200_attn_causal_fwd_tc(const void* q, const void* k, const void* v, void* o, float* lse /*may be NULL*/,
                            const long long* strides /*4x3: q,k,v,o*/, int batch, int n_heads, int Sq, int Sk, int head_dim,
                            float scale, cudaStream_t s);
int b200_attn_causal_bwd(const void* q, const void* k, const void* v, const void* o, const void* d_o, const float* lse,
                         float* delta /*float[batch*n_heads*Sq]*/, void* dq, void* dk, void* dv,
                         const long long* strides /*8x3: q,k,v,o,do,dq,dk,dv*/, int batch, int n_heads, int Sq, int Sk,
                         int head_dim, float scale, const void* rope_cos /*may be NULL: fuse RoPE backward into dq, dk*/,
                         const void* rope_sin, cudaStream_t s);
/*      backward on tcgen05 (5 UMMA groups per tile pair, dQ tiles added into an fp32 accumulator by TMA reduce-add);
 *      training shapes only */
size_t b200_attn_causal_bwd_tc_workspace_bytes(int batch, int n_heads, int Sq);
int b200_attn_causal_bwd_tc(const void* q, const void* k, const void* v, const void* o, const void* d_o, const float* lse,
                            void* dq, void* dk, void* dv, const long long* strides /*8x3: q,k,v,o,do,dq,dk,dv*/, int batch,
                            int n_heads, int Sq, int Sk, int head_dim, float scale, const void* rope_cos /*may be NULL*/,
                            const void* rope_sin, void* workspace, size_t workspace_bytes, cudaStream_t s);
/*      tuning hook, device buffer of 128 int64 (NULL = off): while set, b200_attn_causal_fwd_tc launches its instrumented
        instantiation, which adds per-phase clock64 sums of the softmax warps into buf[group*16 + phase] (tools/attn_fwd_profile.py) */
void b200_attn_debug_trace(long long* buf);
/*      inner stack: L <= 8 positions per event, head_dim 256, packed qkv rows [n_events*L, ld_qkv]. */
/*      rope_cos/sin != NULL: qkv holds PRE-RoPE projections; q and k are rotated in place (fused RoPE) before use */
int b200_attn_tiny_fwd(void* qkv, void* out, int n_events, int L, int n_heads, int head_dim, int ld_qkv, int ld_out,
                       float scale, const void* rope_cos /*may be NULL*/, const void* rope_sin, cudaStream_t s);
int b200_attn_tiny_bwd(const void* qkv, const void* d_out, void* dqkv, int n_events, int L, int n_heads, int head_dim,
                       int ld_qkv, int ld_out, float scale, const void* rope_cos /*may be NULL*/, const void* rope_sin,
                       cudaStream_t s);

/* ---- loss (train.py:180-185: mean CE, ignore_index = pad) ----------------------------------------- */
int b200_ce_fwd(const void* logits, const long long* targets, float* lse, float* row_loss,
                float* loss_and_count /*float[2]: mean loss, #targets*/, long long rows, int V, int ld,
                long long ignore_index, cudaStream_t s);
int b200_ce_bwd(void* logits_inout, const long long* targets, const float* lse, const float* loss_and_count,
                long long rows, int V, int ld, long long ignore_index, float grad_scale,
                const void* grad_scale_dev /*may be NULL: device scalar multiplied into grad_scale*/,
                int grad_scale_is_bf16, cudaStream_t s);

/* ---- optimizer (train.py:121-138 AdamW groups; :464 gradient_clip_val) ----------------------------- */
int b200_gradnorm_parts(void);
int b200_grad_clip_coef(const void* grads, long long n, float max_norm, float* norm_and_coef /*float[2]*/,
                        void* workspace, size_t workspace_bytes, cudaStream_t s);
int b200_adamw_step(void* params, const void* grads, float* exp_avg, float* exp_avg_sq,
                    const unsigned char* nodecay_blocks /*[n/256]*/, long long n, float lr, float beta1, float beta2,
                    float eps, float weight_decay, int step, const float* norm_and_coef /*may be NULL*/, cudaStream_t s);

/* ---- generate() loop (midi_model.py:167-250) ------------------------------------------------------ */
int b200_gemv_bf16(const void* x, const void* W, const void* res /*may be NULL*/, void* y, int B, int N, int K, int ldx,
                   int ldw, int ldr, int ldy, cudaStream_t s);
/*      fused decode-step projection: y = [swiglu]([rmsnorm_w](x or table[ids]) . W^T) [+ res]; N_out = rows of W
 *      (half of them when swiglu: W = [gate | up]) */
int b200_gemv_fused(const void* x /*or NULL*/, const long long* ids /*or NULL*/, int ids_stride, const void* table, int V,
                    const void* norm_w /*may be NULL*/, float eps, const void* W, const void* res /*may be NULL*/, void* y,
                    int B, int N_out, int K, int ldx, int ldw, int ldr, int ldy, int swiglu, cudaStream_t s);
/*      paged KV cache replacing DynamicCache.update's torch.cat (hf cache_utils.py:102-121):
 *      pools [n_pages][n_heads][page][head_dim], block_table [batch][max_pages] */
int b200_kv_append(const void* qkv, void* k_pool, void* v_pool, const int* block_table, int max_pages, int page,
                   int n_heads, int head_dim, int batch, int s_new, int pos0, const int* pos0_dev, int ld, cudaStream_t s);
size_t b200_attn_decode_workspace_bytes(int rows, int n_heads, int head_dim, int n_split);
int b200_attn_decode(const void* q, const void* k_pool, const void* v_pool, const int* block_table, int max_pages, int page,
                     void* out, int batch, int s_q, int n_heads, int head_dim, int past, const int* past_dev, int max_T,
                     int ldq, int ldo, float scale, int n_split, void* workspace, size_t workspace_bytes, cudaStream_t s);
/*      one new token per row: RoPE(q, k) + KV append + attention over positions 0..pos0(+*pos_dev) in one launch */
int b200_attn_decode_fused(const void* qkv, void* k_pool, void* v_pool, const int* block_table, int max_pages, int page,
                           const void* cos_t, const void* sin_t, void* out, int batch, int n_heads, int head_dim, int pos0,
                           const int* pos_dev, int max_T, int ldq, int ldo, float scale, int n_split, void* workspace,
                           size_t workspace_bytes, cudaStream_t s);
/*      sampler: MIDIModel.sample_top_p_k (midi_model.py:152-165) on given probabilities ...            */
int b200_sample_topp_topk(const void* probs, int is_bf16, int rows, int V, int ld, float top_p, int top_k,
                          const float* uniforms, long long* out, cudaStream_t s);
/*      ... and fused with temperature-softmax + grammar mask (midi_model.py:202-223)                    */
int b200_sample_from_logits(const void* logits, int rows, int V, int ld, float temp, float top_p, int top_k, int step,
                            const long long* event_tok, const int* lut, int n_event_types, int eos_id, int pad_id,
                            const unsigned char* dense_mask /*may be NULL*/, const float* uniforms, long long* out,
                            int out_stride, cudaStream_t s);
/* state_dev = {call counter (incremented), device-side seed}: u[i] = hash(seed ^ state[1], state[0], i) */
int b200_uniform_fill(float* u, int n, unsigned long long seed, unsigned long long* state_dev, cudaStream_t s);
int b200_add_int(int* p, int v, cudaStream_t s);
/* graph-captured generate loop: commit the event sampled into ev_t [T][B] to seq[:, *pos+1] and ev_next; (*pos)++ */
int b200_event_commit(const long long* ev_t, long long* seq, long long* ev_next, int* pos_dev, int B, int T, int max_len,
                      cudaStream_t s);


/* ---- persistent generate kernel (midi_model.py:192-248: one generated event = event-level decode step + up to 8
 *      token-level decode steps with grammar-masked sampling + commit) -------------------------------------------
 *      ONE cooperative launch runs `n_events` whole events on one CTA per SM with grid-wide barriers between the
 *      dependent phases (csrc/decode_persist.cu).  All pointers are device pointers; the descriptor itself is host
 *      memory.  State (`pos`, `ev_in`, `seq`, `rng_state`) is the same device-resident state the launch-per-phase loop
 *      (b200_gemv_fused / b200_attn_decode_fused / b200_sample_from_logits / b200_event_commit) works on, so the two
 *      loops are interchangeable event by event. */
typedef struct b200_decode_desc {
    const long long* outer_w;   /* device table [n_outer][6] of device addresses: qkv [3H,H], o [H,H], gate|up [2I,H],
                                   down [H,I], input_layernorm [H], post_attention_layernorm [H]  (hf :303-332) */
    const long long* inner_w;   /* same for the token-level stack, [n_inner][6] */
    int n_outer, n_inner;
    const void *outer_norm, *inner_norm, *lm_head /*[V,H]*/, *emb_outer /*[V,H]*/, *emb_inner /*[V,H]*/;
    int H, I_outer, I_inner, nh_outer, nh_inner, V, pitch /* logits row pitch >= V */;
    float eps;
    const long long* kv_outer;  /* device table [n_outer][2]: k pool, v pool ([pages][heads][page][64], b200_kv_append layout) */
    const int* block_table;     /* [batch][max_pages] */
    int max_pages, page;
    const void *cos_outer, *sin_outer /*[>= max_len][32]*/, *cos_inner, *sin_inner /*[>= 8][128]*/;
    int* pos;                   /* events already in the KV cache = index of the event fed next (incremented) */
    long long* ev_in;           /* [batch][8] the event fed next (rewritten with every generated event) */
    long long* seq;             /* [batch][max_len][8] output; event pos+1 is written */
    int max_len;
    unsigned long long* rng_state;   /* {counter (advanced by 8 per event), seed}: as b200_uniform_fill */
    const unsigned char* dense_mask; /* may be NULL: [batch][V] extra sampling mask ANDed with the grammar */
    const int* lut;             /* [n_event_types][8][2] parameter id ranges (midi_tokenizer.py:517-535) */
    int n_event_types, eos_id, pad_id;
    float temp, top_p;
    int top_k, batch;
    unsigned long long* prof;   /* may be NULL.  Tuning hook: device array of 128 counters; [i] += SM cycles CTA 0 spent in phase i
                                   (incl. the closing barrier), [32 + i] += 1; phases: qkv, attention, combine, o_proj, gate|up,
                                   down of the event-level stack (0-5) and of the token-level stack (6-10, no combine),
                                   lm_head (11), sample (12), commit (13); [64 + 2i] / [65 + 2i] += the part of phase i
                                   spent staging activations / doing the phase's own work (the rest = barrier wait) */
} b200_decode_desc;
size_t b200_decode_desc_bytes(void);            /* sizeof(b200_decode_desc): lets a binding check its struct mirror */
size_t b200_decode_events_workspace_bytes(const b200_decode_desc* d);
int b200_decode_events(const b200_decode_desc* d, int n_events, void* workspace /*256-byte aligned*/,
                       size_t workspace_bytes, cudaStream_t s);

#ifdef __cplusplus
}
#endif
#endif /* MIDI_B200_H */
