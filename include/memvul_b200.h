/* memvul_b200 -- C ABI of the B200-native MemVul batch-inference hot path.
 *
 * The reference (panshengyi/MemVul) is pure Python: its "FFI" for this path is the set of
 * PyTorch module calls made by
 *     MemVul/custom_PTM_embedder.py:224-235   PretrainedTransformerEmbedder.forward -> HF BertModel
 *     MemVul/model_memory.py:90-103           ModelMemory._instance_forward (BertPooler + header)
 *     MemVul/model_memory.py:105-115          ModelMemory.forward_gold_instances (anchor bank)
 *     MemVul/model_memory.py:133-147          ModelMemory.forward test branch (match/softmax/argmax)
 *     MemVul/model_single.py:84-92            ModelSingle.forward (MemVul-m head)
 * Each entry point below names the call it replaces.  Conventions (SURVEY.md section 8b):
 *   - plain C types only; every pointer is a DEVICE pointer unless the name says host;
 *   - the library borrows pointers for the duration of the call, allocates nothing on the
 *     device, and enqueues all work on `stream` (a cudaStream_t passed as void*), asynchronously;
 *   - return 0 on success, a negative MEMVUL_E_* code on failure; memvul_last_error() gives the
 *     text of the calling thread's last failure.  No C++ exception crosses the boundary.
 *   - fp32 = float, fp16 = IEEE binary16 (passed as void*), token ids int64 as AllenNLP emits them.
 */
#ifndef MEMVUL_B200_H
#define MEMVUL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MEMVUL_ABI_VERSION 3

enum {
  MEMVUL_OK = 0,
  MEMVUL_E_INVALID = -1,   /* bad argument / unsupported shape */
  MEMVUL_E_CUDA = -2,      /* CUDA runtime / driver error      */
  MEMVUL_E_WORKSPACE = -3  /* workspace too small              */
};

/* memvul_encoder_forward flags */
enum {
  MEMVUL_ENC_CLS_ONLY = 1,  /* only the [CLS] row of every sequence is the last layer's output          */
  MEMVUL_ENC_PACKED = 2,    /* token-major var-len execution: padded tokens are never computed (needs row_start) */
  MEMVUL_ENC_PRECISE = 4    /* accuracy mode: split-fp16 operands (3 partial products per GEMM), fp32 between GEMMs */
};

/* GEMM epilogues (memvul_gemm_f16) */
enum {
  MEMVUL_EPI_BIAS_F16 = 0,       /* out fp16 = A W^T + bias                    */
  MEMVUL_EPI_BIAS_GELU_F16 = 1,  /* out fp16 = gelu_erf(A W^T + bias)          */
  MEMVUL_EPI_BIAS_RESID_F32 = 2, /* out fp32 = A W^T + bias + resid (fp32)     */
  MEMVUL_EPI_BIAS_F32 = 3        /* out fp32 = A W^T + bias                    */
};

/* pool/match phases (memvul_pool_match phase_mask); MEMVUL_PM_ALL runs as one cooperative launch */
enum {
  MEMVUL_PM_POOL = 1, MEMVUL_PM_HEADER = 2, MEMVUL_PM_UTERM = 4, MEMVUL_PM_MATCH = 8, MEMVUL_PM_FINAL = 16,
  MEMVUL_PM_ALL = 31
};

/* One BERT encoder layer; GEMM kernels are fp16 [out,in] row-major (nn.Linear layout), the rest fp32. */
typedef struct memvul_bert_layer {
  const void* w_qkv;  const float* b_qkv;   /* [3H,H] rows = query|key|value, [3H] */
  const void* w_ao;   const float* b_ao;    /* attention.output.dense [H,H], [H]   */
  const float* ln1_g; const float* ln1_b;   /* attention.output.LayerNorm          */
  const void* w_ff1;  const float* b_ff1;   /* intermediate.dense [I,H], [I]       */
  const void* w_ff2;  const float* b_ff2;   /* output.dense [H,I], [H]             */
  const float* ln2_g; const float* ln2_b;   /* output.LayerNorm                    */
} memvul_bert_layer;

typedef struct memvul_bert_weights {
  int32_t hidden, layers, heads, intermediate, vocab, max_pos, type_vocab;
  float ln_eps;
  const float* word_emb; const float* pos_emb; const float* type_emb;   /* fp32 tables */
  const float* emb_ln_g; const float* emb_ln_b;
  const memvul_bert_layer* layer;           /* HOST array of `layers` entries */
} memvul_bert_weights;

int memvul_abi_version(void);
const char* memvul_last_error(void);

/* Bytes of scratch memvul_encoder_forward needs for B sequences padded to S tokens with these flags.  The workspace
 * needs no initialisation and may be reused for batches of any shape: every row a call reads is first written by that
 * call (with MEMVUL_ENC_PACKED, the rows past the last token that partially filled tiles and the last sequence's key
 * block read are zero-filled by the call's embedding kernel). */
size_t memvul_encoder_workspace_bytes(const memvul_bert_weights* w, int B, int S, int flags);

/* Replaces PretrainedTransformerEmbedder.forward / HF BertModel.forward
 * (custom_PTM_embedder.py:224-235; SURVEY 2.2 K1-K6).
 *   token_ids [B,S] int64; type_ids [B,S] int64 or NULL (all zero, custom_PTM_embedder.py:199-202);
 *   lens [B] int32 = number of unmasked (prefix) tokens per sequence, 1 <= len <= S;
 *   row_start [B+1] int32 = exclusive prefix sum of lens (memvul_mask_to_lens fills it), or NULL without
 *     MEMVUL_ENC_PACKED;
 *   hidden_out [B*S, H] fp32 = last_hidden_state in the PADDED layout (row b*S + s); rows of padded tokens are
 *     zero with MEMVUL_ENC_PACKED and unspecified-but-finite without it;
 *   bad_flag: device int32 (or NULL), bit 1 is set when a token id / type id was out of range (the reference's
 *     torch.embedding raises; custom_PTM_embedder.py:205 raises for type ids) -- the host reads it with its results.
 * flags: MEMVUL_ENC_CLS_ONLY -- only hidden_out[b*S + 0] (the [CLS] row BertPooler reads, model_memory.py:99) is the
 *   last layer's output; the last layer then runs its attention on the first query tile and its output projection /
 *   FFN / LayerNorms on B rows instead of B*S (identical arithmetic per row; ~1/12 of the encoder's work saved).
 *   MEMVUL_ENC_PACKED -- the reference pads every batch to its longest member (config_memory.json:50-57) and pays
 *   for the padding in every GEMM; here the embedding kernel writes the valid tokens of all sequences back to back
 *   (token-major, sequence b at rows row_start[b]..row_start[b+1]) and every kernel reads the row count from
 *   row_start[B] ON THE DEVICE, so no host synchronisation is needed and padded tokens cost nothing.
 *   MEMVUL_ENC_PRECISE -- opt-in accuracy mode for checkpoints whose heads amplify the fp16-operand error beyond the
 *   1e-3 logit tolerance (profiles/r02h_precision.json): every GEMM operand is split into two fp16 numbers
 *   (a = a_hi + a_lo) and the three significant partial products are computed by the same tcgen05 kernels on
 *   K-concatenated operands; the caller passes the layers' GEMM kernels as [N, 3K] fp16 = [W_hi | W_hi | W_lo]
 *   (memvul_b200/native.py PackedBert(precise=True)).  Activations stay fp32 between the GEMMs and the attention runs
 *   in fp32 on the CUDA cores: ~5.5x slower than the default path, max |d logit| ~7e-6 instead of ~2.7e-4 against the
 *   fp32 reference (profiles/r02n_precision_split.json; the floor is the tensor core's own fp32 accumulation).
 *   MEMVUL_ENC_CLS_ONLY is accepted (all rows are computed; hidden_out[b*S] is the guaranteed output).
 * Supported: H in {128, 768} (H % 128 == 0, head_dim == 64), S <= 512, S <= max_pos. */
int memvul_encoder_forward(const memvul_bert_weights* w, const int64_t* token_ids, const int64_t* type_ids,
                           const int32_t* lens, const int32_t* row_start, int B, int S, float* hidden_out,
                           void* workspace, size_t workspace_bytes, int flags, int32_t* bad_flag, void* stream);

/* bool mask [B,S] (1 byte each, AllenNLP `mask`) -> lens[B] and (if non-NULL) row_start[B+1] = exclusive prefix sum;
 * *bad_flag (device int32) gets bit 0 set if a mask is not a non-empty prefix mask.
 * (custom_PTM_embedder.py:215-216 consumes the mask.) */
int memvul_mask_to_lens(const uint8_t* mask, int B, int S, int32_t* lens, int32_t* row_start, int32_t* bad_flag,
                        void* stream);

/* Anchor-bank side term: vterm[g,c] = Wv[c] . bank[g]  (the v third of Linear(1536->2),
 * model_memory.py:141), computed once per bank build (model_memory.py:105-115). */
int memvul_bank_prepare(const float* bank, const float* w_proj, int G, int D, float* vterm, void* stream);

/* Replaces BertPooler + FeedForward header + match + softmax + argmax + gather
 * (model_memory.py:99,102,135-147; SURVEY 2.2 K7-K10).  cls row b is read at cls + b*cls_stride.
 * Outputs: u [B,D]; logits, probs [B,G,2]; best_idx [B] int32 (first maximum of probs[:, :, same_idx]);
 * best_probs [B,2].  Scratch: pooled [B,H], uterm [B,2], best_key [B] (8 bytes each).
 * phase_mask selects phases (tests); MEMVUL_PM_ALL is the fused single launch.  G may be 0 only when
 * phase_mask has neither MATCH nor FINAL (bank building uses POOL|HEADER). */
int memvul_pool_match(const float* cls, int64_t cls_stride, const float* w_pool, const float* b_pool,
                      const float* w_head, const float* b_head, const float* w_proj, const float* bank,
                      const float* vterm, int B, int G, int H, int D, int same_idx, float* pooled, float* u,
                      float* uterm, uint64_t* best_key, float* logits, float* probs, int32_t* best_idx,
                      float* best_probs, int phase_mask, void* stream);

/* MemVul-m classifier (model_single.py:62-65,88-90): logits = feat Wc^T, probs = softmax. */
int memvul_single_head(const float* feat, const float* w_cls, int B, int D, float* logits, float* probs,
                       void* stream);

/* ---- building blocks, exported for the parity tests and the profiler harness ---- */
/* out = epilogue(A[M,K] fp16 x W[N,K]^T fp16); K % 64 == 0, N % 128 == 0; resid/out leading dim = N. */
int memvul_gemm_f16(const void* a, const void* w, const float* bias, const float* resid, void* out, int M, int N,
                    int K, int epilogue, void* stream);
/* x32 (fp32) and x16 (fp16) = LayerNorm(A[M,K] W[768,K]^T + bias + resid) in one kernel (six-CTA clusters exchange the
 * row statistics through distributed shared memory); N must be 768, M >= 256.  In place (x32 == resid) is allowed. */
int memvul_gemm_ln_f16(const void* a, const void* w, const float* bias, const float* resid, const float* gamma,
                       const float* beta, float eps, float* x32, void* x16, int M, int N, int K, void* stream);
/* ctx[B*S,H] fp16 = softmax(QK^T/8 + mask)V per head from qkv [B*S,3H] fp16; head_dim 64, S <= 512.
 * row_start NULL: padded layout (sequence b at rows b*S..); else packed layout (rows row_start[b]..+lens[b]). */
int memvul_attention_f16(const void* qkv, const int32_t* lens, const int32_t* row_start, void* ctx, int B, int S,
                         int H, void* stream);
/* Accuracy-mode building blocks (MEMVUL_ENC_PRECISE): the fp32 attention (qkv fp32 [rows,3H] -> ctx fp32 [rows,H], same
 * layouts and masking as memvul_attention_f16) and the operand split out fp16 [M,3K] = [hi | lo | hi] of x fp32 [M,K]
 * (gelu != 0: of gelu_erf(x)). */
int memvul_attention_f32(const float* qkv, const int32_t* lens, const int32_t* row_start, float* ctx, int B, int S,
                         int H, void* stream);
int memvul_split3_f16(const float* x, void* out, int M, int K, int gelu, void* stream);
/* x32/x16 = LayerNorm(y) rows; x32 or x16 may be NULL; in-place x32 == y allowed. */
int memvul_layernorm(const float* y, const float* gamma, const float* beta, float eps, float* x32, void* x16,
                     int M, int H, void* stream);
/* K1: LayerNorm(word[ids] + pos + type) -> x32, x16 (token ids are always the padded [B,S] matrix).  row_start NULL:
 * padded output rows b*S+s; else packed output rows row_start[b]+s for s < lens[b].  bad_flag (nullable): bit 1 is
 * set on an out-of-range token / type id. */
int memvul_embed_layernorm(const memvul_bert_weights* w, const int64_t* token_ids, const int64_t* type_ids,
                           const int32_t* lens, const int32_t* row_start, int B, int S, float* x32, void* x16,
                           int32_t* bad_flag, void* stream);

/* ---- measurement hooks (bench.py) ----
 * Kernel classes, in the order memvul_profile_read fills them:
 *   0 embed_ln, 1 gemm_qkv, 2 attention, 3 gemm_attn_out, 4 layernorm, 5 gemm_ffn_up, 6 gemm_ffn_down,
 *   7 pool_match, 8 other, 9 attention_cls (first query tile of the CLS-only last layer), 10 cls_tail (the B-row
 *   GEMMs / LayerNorms of the CLS-only last layer). */
#define MEMVUL_KERNEL_CLASSES 11
/* Number of kernels this library has launched in the calling process (all threads). */
long long memvul_launch_count(void);
/* When enabled, every launch is bracketed by CUDA events on its stream (adds ~2 us per launch). */
int memvul_profile_enable(int on);
/* cudaDeviceSynchronize(), then per-class summed device milliseconds and launch counts since the last
 * read; returns MEMVUL_KERNEL_CLASSES (or a negative error). */
int memvul_profile_read(int n_classes, double* ms_out, long long* count_out);

#ifdef __cplusplus
}
#endif
#endif /* MEMVUL_B200_H */
