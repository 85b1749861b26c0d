/*
 * leaf_b200.h - C ABI of the B200-native engine for LEAF's inner attack loop.
 *
 * The reference (LIONS-EPFL/LEAF) has no FFI layer: its seam is the Python call
 *   attack_text_leaf(model, tokenizer, sentences, anchor_features, device, objective, n, k, V, constrain)
 *   (utils_attacks.py:297-393) plus model.encode_text (src/open_clip/model.py:269-284) and
 *   tokenizer(list[str]) (src/open_clip/tokenizer.py:226-265).
 * Every entry point below states which reference lines it replaces. The Python mirror of the
 * reference interface (leaf_b200/attack.py) binds these with ctypes; INTEGRATION.md shows the stub.
 *
 * Conventions
 *   - every function returns LEAF_OK (0) or a negative leaf_status_t; nothing throws across the ABI;
 *     leaf_last_error() returns a thread-local UTF-8 message for the last failure;
 *   - all tensor pointers are DEVICE pointers owned by the caller (PyTorch); the engine owns only
 *     its workspace and its bf16 weight copies; int32 unless stated otherwise;
 *   - work is enqueued on the given cudaStream_t (passed as void*) and is asynchronous;
 *   - one handle per (device, stream user); a handle is not thread-safe;
 *   - there is no CPU path: every call fails with LEAF_ERR_CUDA when no sm_100 device is present.
 */
#ifndef LEAF_B200_H_
#define LEAF_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
  LEAF_OK = 0,
  LEAF_ERR_INVALID = -1,      /* bad argument / shape */
  LEAF_ERR_CUDA = -2,         /* CUDA runtime or driver failure, or no sm_100 device */
  LEAF_ERR_STATE = -3,        /* call order (weights not bound, tables not loaded, workspace too small) */
  LEAF_ERR_UNSUPPORTED = -4   /* input outside the tokenizer's closed domain (see leaf_tokenize_status) */
} leaf_status_t;

typedef struct leaf_engine* leaf_handle_t;

enum { LEAF_ACT_GELU_ERF = 0, LEAF_ACT_QUICK_GELU = 1 };
enum { LEAF_OBJ_L2 = 0, LEAF_OBJ_NEGL2 = 1, LEAF_OBJ_SIM = 2, LEAF_OBJ_DISSIM = 3 };
enum { LEAF_CTX = 77, LEAF_SOT = 49406, LEAF_EOT = 49407, LEAF_VOCAB = 49408, LEAF_N_MERGES = 48894 };
enum { LEAF_MAX_CAPTION_BYTES = 1000, LEAF_MAX_CAPTION_BYTES_LONG = 3560 };

/* Text-tower shape: src/open_clip/model_configs/ViT-{L,H,g,bigG}-14.json "text_cfg" + "embed_dim". */
typedef struct {
  int32_t width;        /* W, multiple of 128 */
  int32_t layers;       /* L */
  int32_t heads;        /* H, head_dim = W / H must be 64 */
  int32_t embed_dim;    /* E */
  int32_t activation;   /* LEAF_ACT_* : nn.GELU (model.py:192) or QuickGELU (transformer.py:33-36) */
  float ln_eps;         /* 1e-5, torch default used by transformer.py:24-30 */
} leaf_cfg_t;

/* Per-layer fp32 parameter pointers, open_clip layout (SURVEY.md appendix C; transformer.py:210-252).
 * For the HF CLIPTextModel layout the host wrapper passes q/k/v separately (in_proj_* == NULL). */
typedef struct {
  const float* ln1_w; const float* ln1_b;
  const float* in_proj_w;  /* [3W, W] rows q;k;v, or NULL when q_w/k_w/v_w are given */
  const float* in_proj_b;  /* [3W] */
  const float* q_w; const float* k_w; const float* v_w;   /* [W, W] each (HF layout) */
  const float* q_b; const float* k_b; const float* v_b;   /* [W] each */
  const float* out_w; const float* out_b;                 /* [W, W], [W] */
  const float* ln2_w; const float* ln2_b;
  const float* fc1_w; const float* fc1_b;                 /* [4W, W], [4W] */
  const float* fc2_w; const float* fc2_b;                 /* [W, 4W], [W] */
} leaf_layer_ptrs_t;

typedef struct {
  const float* token_embedding;       /* [49408, W]   model.py:272 */
  const float* positional_embedding;  /* [77, W]      model.py:274 */
  const float* lnf_w; const float* lnf_b;   /* ln_final, model.py:279 */
  const float* text_projection;       /* open_clip: [W, E] used as x @ P (model.py:282); HF: [E, W] */
  int32_t projection_is_ew;           /* 0 = [W, E] (open_clip), 1 = [E, W] (HF text_projection.weight) */
  const leaf_layer_ptrs_t* layers;    /* [L] host array */
} leaf_weight_ptrs_t;

/* ---- lifetime ------------------------------------------------------------------------------- */
int leaf_create(const leaf_cfg_t* cfg, leaf_handle_t* out);
int leaf_destroy(leaf_handle_t h);
const char* leaf_last_error(void);
const char* leaf_version(void);

/* CLIP BPE merge table: merge_pairs[r] = (left_id << 16) | right_id for rank r, merged id = 512 + r
 * (what SimpleTokenizer.__init__ builds from bpe_simple_vocab_16e6.txt.gz, tokenizer.py:142-158).
 * HOST pointer; copied into a device hash table. */
int leaf_load_bpe(leaf_handle_t h, const uint32_t* merge_pairs_host, int32_t n_merges);

/* Bind the live fp32 parameters (device pointers stay owned by torch) and make the engine's bf16
 * operand copies. leaf_refresh_weights re-casts after each optimizer step (the attacked tower is the
 * trained tower, utils_AT.py:307 vs :339-362). */
int leaf_bind_weights(leaf_handle_t h, const leaf_weight_ptrs_t* w, void* stream);
int leaf_refresh_weights(leaf_handle_t h, void* stream);

/* Workspace for up to max_seqs token rows per call (worst case 77 positions each). */
int leaf_reserve(leaf_handle_t h, int32_t max_seqs);

/* ---- K1: candidate expansion + CLIP tokenization ---------------------------------------------
 * Replaces generate_all_sentences / generate_random_sentences_at_z (utils_attacks.py:215-236,
 * 275-295, called at :318 and :357), the constraint substitution (:321-325, :360-364) and
 * tokenizer(SS) (:327, :366 -> tokenizer.py:226-265).
 *   caps/cap_off : B captions, concatenated bytes and [B+1] offsets (ASCII, each <= LEAF_MAX_CAPTION_BYTES)
 *   pos  [B,n]   : edit position z in [0, 2*len] per candidate; if sel != NULL the position of every
 *                  candidate of sample b is pos[b*n + sel[b]] (phase 2: best position of phase 1, :350-353)
 *   chr  [B,n]   : code point to write, -1 = delete (V[u], train_AT_text_only.py:93)
 *   valid[B,n]   : 0 => candidate is replaced by the unedited caption (:325); NULL = all valid
 *   n == 0       : tokenize the B captions themselves (tokenizer(texts), utils_AT.py:296,312)
 *   tok_out [R,77] int32 zero padded; len_out[R] = argmax(ids)+1 (transformer.py:661).
 *                  n == 0: R = B. n > 0: R = B*n + B - the B*n candidates (sample-major) followed by the B unedited
 *                  captions, whose hidden states the candidates share up to the edited word (see leaf_encode);
 *   base_out [R] : (may be NULL) for candidate rows the index of their sample's caption row (B*n + b), else -1
 * Token ids equal SimpleTokenizer's bit for bit. status_out (device int32[1], may be NULL) gets
 * OR-ed flags: 1 = an html entity expanded outside U+0000..U+024F (or entity text ftfy would unescape differently), 2 = text
 * outside the domain (code point > U+024F, a capital whose lower case leaves it, a sequence ftfy would rewrite; any non-ASCII byte in
 * HF-tokenizer mode), 4 = caption too long / edit position out of range. Captions are UTF-8. */
int leaf_expand_tokenize(leaf_handle_t h, const uint8_t* caps, const int32_t* cap_off, int32_t B, int32_t n,
                         const int32_t* pos, const int32_t* chr, const int32_t* sel, const uint8_t* valid,
                         int32_t* tok_out, int32_t* len_out, int32_t* base_out, int32_t* status_out, void* stream);

/* Which tokenizer leaf_expand_tokenize reproduces: 0 = open_clip's SimpleTokenizer (default; tokenizer.py:133-265),
 * 1 = transformers' CLIPTokenizer as the reference's HF evaluation path wraps it (utils_attacks.py:67-71,
 * eval_textfare.py:127): same BPE, no html.unescape, special tokens spelled <|startoftext|> / <|endoftext|>. */
int leaf_set_tokenizer_mode(leaf_handle_t h, int32_t mode);
/* Largest caption (UTF-8 bytes) the next leaf_expand_tokenize calls will see. Up to LEAF_MAX_CAPTION_BYTES (the default) the
 * kernel runs three candidates per CTA; beyond, up to LEAF_MAX_CAPTION_BYTES_LONG, its long-text variant (one per CTA) is used.
 * The reference's tokenizer takes text of any length (tokenizer.py:226-265); longer captions are flagged (status bit 4). */
int leaf_set_max_caption_bytes(leaf_handle_t h, int32_t bytes);

/* ---- the `--constrain` filter on the device ---------------------------------------------------------
 * Replaces valid_sentence_batched (utils_attacks.py:110-143; applied at :321-325, :360-364, :478-481, :532-537):
 * valid[b,j] = len(W & set(word_tokenize(candidate.lower()))) < len(W & set(word_tokenize(sentence_b.lower()))).
 * leaf_load_words takes W (the reference: nltk.corpus.words.words()) and, optionally, Punkt's abbreviation types, as
 * HOST byte blobs with [n+1] offsets, and keeps them as hash sets on the device. leaf_constrain_mask has
 * leaf_expand_tokenize's candidate arguments; valid_out [B,n] uint8 feeds leaf_expand_tokenize's `valid`;
 * count_out [B*n+B] (may be NULL) receives the dictionary-word counts (candidates, then the B sentences).
 * word_tokenize is NLTK's: the Treebank substitutions are restated one by one (exact by construction), Punkt's sentence
 * split is approximated - PARITY UNPINNED against NLTK, which cannot be installed here (csrc/constrain_core.cuh). */
int leaf_load_words(leaf_handle_t h, const uint8_t* words_blob, const int32_t* words_off, int32_t n_words,
                    const uint8_t* abbrev_blob, const int32_t* abbrev_off, int32_t n_abbrev);
int leaf_constrain_mask(leaf_handle_t h, const uint8_t* caps, const int32_t* cap_off, int32_t B, int32_t n,
                        const int32_t* pos, const int32_t* chr, const int32_t* sel, uint8_t* valid_out,
                        int32_t* count_out, int32_t* status_out, void* stream);

/* ---- K2: text tower forward -------------------------------------------------------------------
 * Replaces CLIP.encode_text(tokens, normalize) (model.py:269-284; transformer.py:254-265,355-366,
 * 653-665). tok [N,77] int32, len [N] (positions after argmax(ids) are dead under the causal mask and
 * are not computed). feat_out [N,E] fp32. bf16 tensor-core GEMMs, fp32 accumulate/residual/LN/softmax.
 * base [N] (may be NULL): base[i] = j >= 0 names another row of this batch (with base[j] = -1) that row i was
 * derived from; positions where both token rows agree have identical hidden states under the causal mask, so
 * they are computed once (on row j) and row i's attention reads row j's keys/values for them. Results are
 * bit-identical to base == NULL.
 * dedup_group > 1: rows [0, dedup_rows) come in groups of dedup_group consecutive rows (the n candidates of a sample);
 * a row whose tokens equal an EARLIER row of its group is not encoded again - it receives that row's features (bit
 * identical, so exact ties keep resolving to the first index). dedup_group <= 1 disables it.
 * trim_providers != 0 (with base and 0 < dedup_rows < N): the caller does not read feat_out of the rows [dedup_rows, N) that
 * other rows name as base (the unedited captions of an attack phase: utils_attacks.py never encodes them at all, here they
 * exist so that their prefixes are computed once). They are computed only as far as some row reads them and their feat_out
 * rows are UNDEFINED; every other row is unchanged, bit for bit. */
int leaf_encode(leaf_handle_t h, const int32_t* tok, const int32_t* len, const int32_t* base, int32_t N,
                int32_t dedup_rows, int32_t dedup_group, int32_t trim_providers, int32_t normalize, float* feat_out, void* stream);

/* ---- K3: TextFARE score + per-sample argmax ----------------------------------------------------
 * Replaces utils_attacks.py:332-348 / :370-386 / :393. feat [B*n,E] fp32, anchor [B,E] fp32.
 * loss_out [B,n] (may be NULL); best_out [B] = first index of the maximum (torch.argmax);
 * best_feat_out [B,E] (may be NULL) = features of the winner. */
int leaf_score(leaf_handle_t h, const float* feat, const float* anchor, int32_t B, int32_t n, int32_t objective,
               float* loss_out, int32_t* best_out, float* best_feat_out, void* stream);

/* Top-k of a score vector, for the single-sentence evaluation attacks built on K1-K3 (attack_text_charmer_inference,
 * utils_attacks.py:451-580: torch.topk of the position scores :519 and torch.argmax over the whole candidate list
 * :575; attack_text_bruteforce :447). score_a [m] fp32; score_b (may be NULL) a second tower's scores of the same
 * candidates, averaged as (a+b)/2 (:498-513). idx_out [k] int32, val_out [k] (may be NULL): value descending, ties by
 * ascending index (k = 1 is torch.argmax's first-index rule). */
int leaf_topk(leaf_handle_t h, const float* score_a, const float* score_b, int32_t m, int32_t k, int32_t* idx_out,
              float* val_out, void* stream);

/* ---- K4: train-mode forward + backward of the selected adversarial batch -----------------------
 * Replaces model.encode_text(adv_tokens) under autograd and loss.backward() of utils_AT.py:317-337 (the loss itself,
 * mse(...).sum(-1).mean() on [B,E], stays a two-line torch expression on top of feat_out / dfeat).
 * leaf_train_reserve sizes the activation store (and makes the [in,out] bf16 weight copies the dgrad products need);
 * leaf_forward_train computes feat_out [N,E] fp32 and keeps every layer's activations. The packed row count sizes the
 * weight-gradient contractions on the host: pass rows_hint = sum(len) and max_len_hint >= max(len) when the host knows them
 * (checked on the device: a wrong hint traps) and nothing synchronises; with 0 / 0 the stream is synchronised once to learn them; leaf_backward consumes dfeat [N,E] fp32 and ACCUMULATES (+=) the parameter
 * gradients into the fp32 device buffers named by `grads` (same struct and layouts as leaf_bind_weights; a NULL
 * pointer marks a frozen parameter). bf16 operands, fp32 accumulation, fp32 LayerNorm/softmax/activation math. By default
 * some gradients are atomic sums and not bit-reproducible run to run; leaf_set_deterministic(h, 1) makes all of them so.
 * ONE forward, ONE backward: the engine keeps a single activation store. Every leaf_forward_train gets a generation
 * number (> 0, written to *generation_out when that is not NULL); leaf_backward(generation != 0) fails with
 * LEAF_ERR_STATE when the store holds a different forward (a second encode_text ran before this output's backward -
 * torch autograd would differentiate each output through its own graph, utils_AT.py:317-337 has exactly one), and with
 * LEAF_ERR_INVALID when dfeat_rows is not the N of that forward. The store is consumed by a successful backward. */
int leaf_train_reserve(leaf_handle_t h, int32_t max_seqs);
int leaf_forward_train(leaf_handle_t h, const int32_t* tok, const int32_t* len, int32_t N, float* feat_out,
                       int32_t rows_hint, int32_t max_len_hint, int64_t* generation_out, void* stream);
int leaf_backward(leaf_handle_t h, int64_t generation, const float* dfeat, int32_t dfeat_rows, const leaf_weight_ptrs_t* grads,
                  void* stream);

/* Host callback of leaf_backward, the hook the data-parallel gradient exchange hangs on (what DDP's bucketed all-reduce does
 * for the reference, train_AT_text_only.py:310-317): called on the calling thread, in stream order, with
 *   layer == L (the layer count)  after the text_projection / ln_final gradients have been enqueued,
 *   layer == L-1 ... 0            after ALL weight gradients of that layer have been enqueued (the bias and LayerNorm
 *                                 gradients of the layers above it are complete at that point as well),
 *   layer == -1                   at the end (embedding gradients enqueued).
 * "Enqueued" means: an event recorded on `stream` inside the callback completes after those gradients are final, so a
 * second stream can all-reduce that slice while the backward of the layers below still runs. fn == NULL removes it. */
typedef void (*leaf_backward_hook_t)(int32_t layer, void* user);
int leaf_set_backward_hook(leaf_handle_t h, leaf_backward_hook_t fn, void* user);
/* Cap the persistent GEMM grids at n_sms SMs (0 = the whole device) so that a collective's CTAs find SMs of their own while
 * it runs next to the backward. */
int leaf_set_sm_budget(leaf_handle_t h, int32_t n_sms);
/* Deterministic mode (off by default; PyTorch's torch.use_deterministic_algorithms(True) turns it on through
 * leaf_b200.LeafEngine). The forward is deterministic in either mode. Off, leaf_backward sums several gradients with fp32
 * atomics in arrival order and they are not bit-reproducible run to run: the split-K weight gradients (out-proj, QKV, HF q/k/v,
 * the [E,W] projection, any weight gradient with fewer output tiles than CTA pairs), the fc1 / fc2 / out-proj / in-projection
 * biases, the LayerNorm gains and biases, the token and positional embeddings; leaf_sumsq adds its block sums with atomics too.
 * On, every one of these is a fixed-order reduction: each gradient leaf_backward writes and the value leaf_sumsq adds are
 * functions of the inputs alone, bit for bit - whatever the run, leaf_set_sm_budget, LEAF_PDL or the order in which blocks
 * finish. The two modes sum in different orders, so they agree to rounding, not to the bit. Turning it on allocates its
 * workspace (a few tens of MB; synchronises the device) for the current leaf_train_reserve size, and leaf_train_reserve
 * sizes it from then on. The deterministic reductions of one handle share that workspace and their arrival counters: in this
 * mode its leaf_backward and leaf_sumsq calls must be stream-ordered (one stream, or ordered by events); two of them running
 * at the same time on different streams would corrupt each other's sums. */
int leaf_set_deterministic(leaf_handle_t h, int32_t on);

/* AdamW (torch.optim.AdamW semantics, decoupled weight decay) over the tower's parameters held in ONE flat fp32 buffer
 * (train_AT_text_only.py:326-341: the gain / bias / LayerNorm group with weight_decay 0 is laid out first, elements
 * [0, n_nodecay); utils_AT.py:358-362). grads are multiplied by grad_scale first (1/accum_freq, or a clipping
 * coefficient). step >= 1 is the bias-correction step count. One launch, 28 B of HBM traffic per parameter.
 * leaf_sumsq adds the sum of squares of a flat buffer into out[0] (gradient-norm clipping, utils_AT.py:349-357). */
int leaf_adamw(leaf_handle_t h, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n,
               int64_t n_nodecay, float lr, float beta1, float beta2, float eps, float weight_decay, int32_t step,
               float grad_scale, void* stream);
int leaf_sumsq(leaf_handle_t h, const float* g, int64_t n, float* out, void* stream);
/* g[0, n) *= s in place (n a multiple of 4): the rescale of torch.nn.utils.clip_grad_norm_ on the ACCUMULATED gradients
 * after a micro-batch that is not followed by an optimizer step - utils_AT.py:356-357 clips after every micro-batch. */
int leaf_scale(leaf_handle_t h, float* g, int64_t n, float s, void* stream);

/* ---- test / bench hooks (used by tests/ and bench.py only) ------------------------------------ */
/* C[M,N] = A[M,K] . Bt[N,K]^T (+bias[N]) with the tower's tcgen05 kernel. epilogue: 0 = bf16 store,
 * 1 = bf16 store after activation `act`, 2 = fp32 C += result (residual), 3 = fp32 store.
 * A, Bt bf16 row-major; m_dev (device int32, may be NULL) overrides M at run time. */
int leaf_gemm_bf16(leaf_handle_t h, const void* A, const void* Bt, const float* bias, void* C,
                   int32_t M, int32_t N, int32_t K, int32_t epilogue, int32_t act, const int32_t* m_dev,
                   void* stream);
/* The same kernel with MN-major operands: B is [K,N] row-major; A is [K,M] row-major when a_mn != 0 (C = A^T . B, the shape
 * of a weight gradient dW[out,in] = dY[rows,out]^T . X[rows,in], read as the activations lie), else [M,K] (C = A . B, the
 * shape of a data gradient dX = dY . W with W [out,in] as it lies). M (when a_mn) and N multiples of 8; epilogue as above. */
int leaf_gemm_bf16_mn(leaf_handle_t h, const void* A, const void* B, const float* bias, void* C, int32_t M, int32_t N,
                      int32_t K, int32_t epilogue, int32_t a_mn, void* stream);
/* y[rows,W] (bf16) = LayerNorm(x[rows,W] fp32) with the tower's kernel; W = cfg.width. */
int leaf_test_layernorm(leaf_handle_t h, const float* x, int32_t rows, const float* gamma, const float* beta, void* y,
                        void* stream);
/* out[rows,W] (bf16) = causal attention over packed qkv[rows,3W] (bf16); meta [N,4] int32 = {own_row, t, p, base_row}
 * per sequence (positions [p,t) are rows own_row.., keys/values of [0,p) are rows base_row..). */
int leaf_test_attention(leaf_handle_t h, const void* qkv, const int32_t* meta, int32_t N, void* out, void* stream);
/* K4's attention backward alone: qkv [rows,3W] bf16, o [rows,W] bf16 (the forward output), dout [rows,W] fp32, meta as above
 * with p = 0 (training batches share no prefixes), T >= the longest sequence; dqkv [rows,3W] bf16 = (dQ | dK | dV). */
int leaf_test_attention_bwd(leaf_handle_t h, const void* qkv, const void* o, const float* dout, const int32_t* meta, int32_t N,
                            int32_t T, void* dqkv, void* stream);
/* leaf_encode computes the final layer's out-proj / LayerNorm / MLP on the pooled EOS row of every sequence only (the
 * one row transformer.py:661 reads); on by default, results are bit-identical either way. on = 0 computes every row. */
int leaf_set_prune_last(leaf_handle_t h, int32_t on);
/* Number of kernels the engine has launched since the last call with reset != 0. */
int64_t leaf_launch_count(leaf_handle_t h, int32_t reset);
/* Packed-row count (sum of len) of the last leaf_encode; synchronises the device. */
int64_t leaf_last_rows(leaf_handle_t h);
/* Accumulated device time (ms) of the launches of class `which` between CUDA events recorded on the launching stream, since
 * timing was last enabled with leaf_set_timing(h, 1): 0 = every GEMM, 1 = LayerNorm, 2 = attention, 3 = row packing +
 * embedding, 4 + e = the GEMM launches with epilogue e (0 bf16 store with N != K: QKV; 1 activation: fc1; 2 residual; 3 fp32
 * store: projection), 8 = the residual GEMMs with K > N (fc2; counted in class 6 as well), 9 = bf16 store with N == K
 * (out-proj). Synchronises on the recorded events. */
int leaf_set_timing(leaf_handle_t h, int32_t on);
double leaf_timing_ms(leaf_handle_t h, int32_t which, int32_t* launches);

#ifdef __cplusplus
}
#endif
#endif /* LEAF_B200_H_ */
