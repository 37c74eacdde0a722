/* mmsum_b200 — C-ABI of the B200-native MultimodalSum training-step kernels.
 *
 * The reference (nc-ai/MultimodalSum) has no FFI layer: its hot path reaches native code only
 * through torch (ATen/cuBLAS/apex).  Each entry point below therefore replaces a torch call site
 * of the reference; the file:line cited is relative to /root/reference.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller; the library never allocates or frees
 *   - `stream` is a cudaStream_t passed as void*; all calls are asynchronous, no host sync
 *   - return value: 0 ok; < 0 invalid argument / driver problem detected on the host before launch;
 *     > 0 a cudaError_t from the launch.  No C++ exception crosses this boundary.
 *   - activations / weights are bf16 (uint16 storage), statistics / master gradients fp32,
 *     token ids int64, masks uint8 (1 = valid)
 */
#ifndef MMSUM_B200_H_
#define MMSUM_B200_H_
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* ---- dense contraction (tcgen05/TMEM/TMA) -----------------------------------------------------
 * D[M,N] (+)= epi(alpha * sum_k A(m,k) B(n,k)).  Replaces nn.Linear/F.linear forward and the dgrad /
 * wgrad GEMMs autograd derives from them: src/transformer/modeling_multimodalsum.py:272-273 (fc1/fc2),
 * :695-704 (q/k/v/out/alpha/beta_proj), :2281 (LM head), src/img_encoder.py:40, src/table_encoder.py:70-72. */
typedef struct MmsumGemmArgs {
  const void* A;      /* bf16. K-major: [M,K] row-major (lda = row pitch in elements); MN-major: [K,M] row-major */
  const void* B;      /* bf16. K-major: [N,K] row-major; MN-major: [K,N] row-major */
  void* D;            /* [M,N] row-major, bf16 or fp32 (out_f32) */
  int64_t lda, ldb, ldd;
  int32_t M, N, K;
  int32_t a_mn_major, b_mn_major;
  int32_t out_f32;    /* 1: D is fp32 */
  int32_t accumulate; /* 1: D += (fp32 only; TMA reduce-add) */
  int32_t splits;     /* split-K factor; 0 = auto (only >1 when accumulate) */
  int32_t block_n;    /* 0 = auto, 128 or 256 */
  int32_t raster_m_fast;
  float alpha;
  const float* bias;  /* fp32 [N] or NULL, added after alpha */
  int32_t act;        /* 0 none, 1 GELU(erf), 2 ReLU */
  int32_t aux_mode;   /* 0 none, 1 store pre-activation (bf16) to aux, 2 multiply result by act'(aux),
                         3 store act'(pre-activation) to aux (GELU only), 4 multiply result by aux;
                         1..4 need bf16 output and a row-major A (a_mn_major = 0) */
  void* aux;          /* bf16 [M,N] */
  int64_t ld_aux;
  const void* A2;     /* optional: A = [A | A2] concatenated along K at k_split (K-major A only), else NULL */
  int64_t lda2;
  int32_t k_split;    /* multiple of 64 */
} MmsumGemmArgs;
int mmsum_gemm_bf16(const MmsumGemmArgs* args, void* stream);


/* ---- multi-entity attention ----------------------------------------------------------------------
 * Replaces SelfAttention.forward / get_head_output (src/transformer/modeling_multimodalsum.py:722-886) for the
 * encoder self-attention, the decoder causal self-attention and the multi-modal multi-entity cross-attention
 * (per-entity softmax, mean over valid entities, leave-one-out target exclusion of src/multimodal_train.py:150-163),
 * and the backward autograd derives from them.  128 query positions per sequence, head_dim 64.
 * Query sequence `qseq` belongs to business `qseq / R` and is leave-one-out target `qseq % R`. */
typedef struct MmsumAttnMod {
  int64_t kv_row_base; /* first KV row of this modality; entity (biz,e) starts at kv_row_base + (biz*E+e)*ent_stride */
  int64_t o_off;       /* element offset of this modality's [n_qseq*128, ldo] output (fwd) / upstream grad (bwd) */
  int32_t E;           /* entities per business */
  int32_t Sk;          /* keys per entity */
  int32_t loo;         /* 1: entity e is skipped for target e */
  int32_t ent_base;    /* index of entity 0 of this modality in the [.., E_total] arrays */
  int32_t ent_stride;  /* KV rows between consecutive entities (0 = Sk); > Sk when entity frames are padded */
  int32_t reserved;
} MmsumAttnMod;

typedef struct MmsumAttnArgs {
  const void* Q;  int64_t ldq;  int32_t q_col;               /* bf16 [n_qseq*128, ldq], head h at q_col + 64h */
  const void* KV; int64_t ldkv; int32_t k_col; int32_t v_col; /* bf16 memory rows; K head h at k_col+64h, V at v_col+64h */
  void* O; int64_t ldo;            /* fwd: out (bf16); bwd: upstream gradient of the per-modality outputs */
  float* LSE;                      /* [n_qseq, H, E_total, 128] log2-domain log-sum-exp (fwd out, bwd in) */
  float* DELTA;                    /* [n_qseq, H, E_total, 128] bwd scratch */
  const uint8_t* key_valid;        /* per KV row, 1 = attend; NULL = all valid */
  const uint8_t* ent_valid;        /* [n_biz, E_total]; NULL = all valid */
  const float* inv_n;              /* [n_qseq, n_mod] 1/#valid entities (0 when none); NULL = 1 */
  void* dQ;  int64_t lddq;  int32_t dq_col;                   /* bwd out, bf16 */
  void* dKV; int64_t lddkv; int32_t dk_col; int32_t dv_col;    /* bwd out, bf16, same row indexing as KV */
  int32_t n_qseq, H, R, causal, n_mod, E_total;
  float scale;
  int32_t q_rows;      /* rows of Q / O / dQ per query sequence (the frame stride), 0 = 128; a multiple of 16 <= 128.  Rows beyond
                          q_rows of a sequence's 128-row query tile belong to the next sequence: they are computed and dropped
                          (forward / dQ) or masked (dK/dV).  LSE / DELTA keep 128 slots per sequence. */
  MmsumAttnMod mods[3];
} MmsumAttnArgs;
int mmsum_attn_fwd(const MmsumAttnArgs* args, void* stream);
int mmsum_attn_bwd(const MmsumAttnArgs* args, void* stream); /* dQ/DELTA pass, then dK/dV pass */
/* Test aid: one CTA per SM fills its shared memory and all 512 tensor-memory columns with NaN bit patterns.  A kernel that
 * consumes stale on-chip state (0 * stale, unwritten accumulator columns) produces non-finite or run-dependent results when it
 * is launched after this one (tests/test_kernels_gpu.py::test_kernels_ignore_stale_onchip_state). */
int mmsum_debug_poison(void* stream);

/* ---- decode-step attention (beam search, BASELINE config 5) ------------------------------------------
 * Replaces the cached branch of SelfAttention.get_head_output (src/transformer/modeling_multimodalsum.py:774-815, 889-920)
 * and the cache re-gathering of _reorder_cache (:3103-3115, :663-669).
 * mmsum_attn_decode_cross: MmsumAttnArgs with ONE query row per hypothesis: Q [n_qseq, ldq], O per modality [n_qseq, ldo] at
 *   mods[m].o_off; R = hypotheses (beams, <= 8) per business, adjacent; they attend to the same un-expanded per-business memory
 *   rows of KV (K|V read once per business and head).  inv_n [n_qseq, n_mod]; LSE / DELTA / dQ / dKV unused; loo must be 0.
 * mmsum_attn_decode_self: qkv [n_hyp, ldqkv] = q | k | v of the newest position (heads of 64); appends k, v to
 *   cache [n_hyp, 128, 2*H*64] at row (n, pos) and sets hist[n][pos] = n; attends to positions 0..pos where position j < pos of
 *   hypothesis n is read from cache row (hist[n][j], j).  Re-ranking the beams is `hist = hist[beam_idx]` (int32 [n_hyp, 128]);
 *   the caches never move.  pos_dev: device scalar.  out [n_hyp, ldo] bf16. */
int mmsum_attn_decode_cross(const MmsumAttnArgs* args, void* stream);
int mmsum_attn_decode_self(const void* qkv, int64_t ldqkv, void* cache, int32_t* hist, const int32_t* pos_dev, void* out,
                           int64_t ldo, int32_t n_hyp, int32_t H, float scale, void* stream);

/* Candidate selection of one beam-search token, per hypothesis row: forced BOS / EOS (adjust_logits_during_generation,
 * modeling_multimodalsum.py:3084-3101), log_softmax, EOS ban below min_length and n-gram ban from the row's own history
 * (generation_utils.py:57-99, 848-868), + beam_scores, top-K (:2919-2925).  logits fp32 [rows, ld]; ids int64 [rows, L] token
 * history; cur_dev: device scalar, current length; K in {2,4,8,16}; out_val / out_tok [rows, K] sorted by descending score. */
int mmsum_beam_topk(const float* logits, int64_t ld, int32_t rows, int32_t V, const float* beam_scores, const int64_t* ids,
                    int32_t L, const int64_t* cur_dev, int32_t min_length, int32_t ngram, int32_t bos, int32_t eos, int32_t K,
                    float* out_val, int32_t* out_tok, void* stream);

/* Per-business beam update after mmsum_beam_topk (_generate_beam_search :2933-3010, BeamHypotheses.add / is_done
 * generation_utils.py:962-993): merges the k x K row candidates, admits finished ones (rank < k) to the business' pool, selects
 * the next k beams, permutes the token histories `ids` in place, writes beam_scores / beam_idx / next_tok.  All state is device
 * memory (done: 1 byte per business; pool_* as in generation.BeamSearch).  Optional decoder hooks: next_tok32 [B*k] (token input
 * of the next decode step), hist [B*k, 128] (self-attention slot table, permuted like ids = _reorder_cache :3103-3115). */
int mmsum_beam_update(const float* cand_val, const int32_t* cand_tok, int64_t* ids, float* beam_scores, uint8_t* done,
                      float* pool_score, int64_t* pool_tok, int64_t* pool_len, int64_t* pool_n, const int64_t* cur_dev,
                      int64_t* beam_idx, int64_t* next_tok, int32_t* next_tok32, int32_t* hist, int32_t B, int32_t k, int32_t K,
                      int32_t L, int32_t eos, int32_t pad, int32_t early_stopping, float length_penalty, void* stream);

/* ---- HBM-bound row kernels (d_model = 1024) ----------------------------------------------------- */
/* fp32 -> bf16 (weight arena cast, feature cast) */
int mmsum_cast_f32_bf16(const float* src, void* dst, int64_t n, void* stream);

/* out = dropout(LN(E[ids] + P[t+2] + rating_diff[seq]*remb)): BartEncoder.forward modeling_multimodalsum.py:368-372,
 * BartDecoder.forward :588-597, LearnedPositionalEmbedding :961-969.  rating_diff/remb NULL for the encoder. */
/* Dropout masks are a pure function of (seed, stream_id + 4096 * step, element index); `step_dev` (optional) points to a
 * device-resident step counter read inside the kernel, so a recorded CUDA graph of the step draws fresh masks at every replay. */
int mmsum_embed_ln_fwd(const int32_t* ids, const float* E, const float* P, const float* rating_diff, const float* remb,
                       const float* gamma, const float* beta, void* out, float* mean, float* rstd, int32_t rows,
                       int32_t S, int32_t d_model, float p_drop, uint64_t seed, uint32_t stream_id, const uint32_t* step_dev,
                       void* stream);
/* decode step (eval, one token per hypothesis): as above with S = 1, every row at decoder position pos_dev[0] (device
 * memory, so the launch can be replayed from a CUDA graph); the cached branch of BartDecoder.forward :583-597, :964-965 */
int mmsum_embed_ln_decode(const int32_t* ids, const float* E, const float* P, const float* rating_diff, const float* remb,
                          const float* gamma, const float* beta, void* out, float* mean, float* rstd, int32_t rows,
                          int32_t d_model, const int32_t* pos_dev, void* stream);
/* backward: scatter-add into dE (pad id skipped, nn.Embedding(padding_idx=1) :1001), dP, dremb, dgamma, dbeta (all +=) */
int mmsum_embed_ln_bwd(const void* dout, const void* dout2 /* optional addend */, const int32_t* ids, const float* E, const float* P, const float* rating_diff,
                       const float* remb, const float* gamma, const float* mean, const float* rstd, float* dE, float* dP,
                       float* dremb, float* dgamma, float* dbeta, float* dz_scratch, int32_t rows, int32_t S,
                       int32_t d_model, int32_t pad_id, float p_drop, uint64_t seed, uint32_t stream_id, const uint32_t* step_dev,
                       void* stream);

/* out = LN(res + dropout(y)): the post-LN residual blocks of EncoderLayer.forward :288-308 / DecoderLayer.forward :442-489
 * (LayerNorm factory :972-980, eps 1e-5).  Dropout masks are a pure function of (seed, stream_id, element). */
int mmsum_add_ln_fwd(const void* res, const void* y, const float* gamma, const float* beta, void* out, float* mean,
                     float* rstd, int32_t rows, int32_t d_model, float p_drop, uint64_t seed, uint32_t stream_id,
                     const uint32_t* step_dev, void* stream);
/* backward: upstream = d1 (+ d2 if not NULL); dres = dz, dy = dz * mask (may alias dres when p_drop == 0); dgamma/dbeta += */
int mmsum_add_ln_bwd(const void* d1, const void* d2, const void* res, const void* y, const float* gamma, const float* mean,
                     const float* rstd, void* dres, void* dy, float* dgamma, float* dbeta, int32_t rows, int32_t d_model,
                     float p_drop, uint64_t seed, uint32_t stream_id, const uint32_t* step_dev, void* stream);

/* out[n] += sum_r x[r,n]  (bias gradients) */
int mmsum_colsum(const void* x, int64_t ld, int32_t rows, int32_t N, float* out, void* stream);

/* gate fusion of the three modalities, SelfAttention.forward :732-744.  o3 = [3][rows,D] (text, table, img out_proj
 * outputs), u = [2][rows,D] (alpha/beta pre-activations), pres = [n_biz][2] modality presence, ab = [2][rows,D] gates out */
int mmsum_gate_fwd(const void* o3, const void* u, const uint8_t* pres, void* y, void* ab, int32_t rows,
                   int32_t rows_per_biz, int32_t d_model, void* stream);
int mmsum_gate_bwd_u(const void* dy, const void* o3, const void* ab, void* du, int32_t rows, int32_t d_model, void* stream);
int mmsum_gate_bwd_o(const void* dy, const void* ab, const void* dca, const void* dcb, void* do3, int32_t rows,
                     int32_t d_model, void* stream);

/* label-smoothed CE over bf16 logits [rows, ld] (src/utils.py:32-38; eps < 0: plain CE, src/text_pretrain.py:97);
 * loss_rows[r] per-row loss (computed before the row is overwritten); loss_out (optional) = loss_scale * sum(loss_rows);
 * write_grad: logits := dlogits * gscale.  lse_rows (optional fp32 [rows]): written by the loss pass (write_grad = 0), read by
 * the gradient pass (write_grad = 1), which then reads the logits once instead of twice and leaves loss_rows untouched */
int mmsum_ce_fwd_bwd(void* logits, int64_t ld, int32_t rows, int32_t V, const int32_t* target, float eps, float gscale,
                     const float* gscale_dev /* optional device scalar multiplied into gscale */, float* loss_rows, float* loss_out,
                     float loss_scale, float* lse_rows, int32_t write_grad, void* stream);

/* integer bookkeeping of one step: decoder inputs (shift_tokens_right :225-246), pad masks (:249-254), rating_diff
 * (src/multimodal_train.py:154-156), memory key/entity validity, 1/#valid entities, modality presence */
typedef struct MmsumPrepArgs {
  int32_t B, R, S, F, n_img, img_keys, n_mod, pad_id, bos_id, eos_id;
  int32_t S_enc;       /* encoder frame: the first S_enc <= S tokens of every review (0 = S); every token beyond it must be pad.
                          enc_ids / enc_valid / the text region of mem_valid then have B*R*S_enc entries */
  int32_t* enc_ids;    /* [B*R*S] */
  int32_t* dec_ids;    /* [B*R*S] */
  int32_t* labels;     /* [B*R*S] */
  uint8_t* enc_valid;  /* [B*R*S] */
  uint8_t* dec_valid;  /* [B*R*S] */
  uint8_t* mem_valid;  /* [B*R*S + B*F + B*n_img*img_keys] */
  uint8_t* ent_valid;  /* [B, R + (F>0) + n_img] */
  uint8_t* pres;       /* [B, 2] or NULL */
  float* rating_diff;  /* [B*R] */
  float* inv_n;        /* [B*R, n_mod] */
} MmsumPrepArgs;
int mmsum_prep_step(const int64_t* reviews, const int64_t* reviews_mask, const float* rating, const uint8_t* table_valid,
                    const uint8_t* img_mask, const MmsumPrepArgs* args, void* stream);

/* table-encoder front end: src/table_encoder.py:27-82 (yelp, dataset 0: v0..v5 = name, category, str_categorical,
 * str_boolean, rating, hours; W0 = rating_embedding.weight, W1 = hours_embedding.weight) and :108-166 (amazon, dataset 1:
 * v0..v5 = price, rating, brand, name, category, description; W0 = price_embedding.weight, W1 = rating_embedding.weight).
 * X = [B, F, 2*1024] bf16 (names | values), valid = [B, F]. */
typedef struct MmsumTableArgs {
  int32_t dataset, B;
  const float* E;
  const int64_t* field;
  const int64_t* v0; const int64_t* v1; const int64_t* v2; const int64_t* v3; const int64_t* v4; const int64_t* v5;
  const float* W0; const float* W1;
  void* X;
  uint8_t* valid;
} MmsumTableArgs;
int mmsum_table_fwd(const MmsumTableArgs* args, void* stream);
/* dW[c,j] += sum bits[b,row,j] * dX[b, f0+row, 1024 + c]   (rating / hours / price embedding gradients) */
int mmsum_table_bits_bwd(const void* dX, const int64_t* bits, float* dW, int32_t B, int32_t F, int32_t f0, int32_t nrows,
                         int32_t nb, void* stream);

/* ---- optimizer over the flat arenas ---------------------------------------------------------------
 * mmsum_grad_sumsq: out[0] = sum g^2 (two deterministic stages; partial needs >= 1184 floats) — the global norm of
 * torch.nn.utils.clip_grad_norm_ (src/multimodal_train.py:361-362).
 * mmsum_adamw_step: transformers-3.0.2 AdamW.step (src/transformer/optimization.py:208-267) with the clip coefficient
 * min(1, max_norm / (sqrt(sumsq) + 1e-6)) folded in; step_size = lr * sqrt(1 - beta2^t) / (1 - beta1^t); flags[i/64]
 * bit0 = update, bit1 = weight decay; also writes the bf16 compute copy. */
int mmsum_grad_sumsq(const float* g, int64_t n, float* partial, int32_t n_partial, float* out, void* stream);
int mmsum_adamw_step(float* w32, void* w16, const float* g, float* m, float* v, const uint8_t* flags, int64_t n, float lr,
                     float beta1, float beta2, float eps, float weight_decay, float step_size, const float* sumsq,
                     float max_norm, void* stream);

#ifdef __cplusplus
}
#endif
#endif
