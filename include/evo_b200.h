/* evo_b200 — C ABI of the B200-native StripedHyena forward engine.
 *
 * The reference (evo-design/evo) has no FFI: its boundary is the Python duck-type
 * of stripedhyena.model.StripedHyena (evo/models.py:141-150, evo/scoring.py:81,
 * evo/generation.py:117,152).  Everything that object computes is executed by the
 * entry points below; evo_b200/stripedhyena/model.py binds them with ctypes and
 * mirrors the Python protocol on top.  Each entry point cites the reference
 * operation it replaces (names inside stripedhyena==0.2.2 / flash_attn, which the
 * reference pins in requirements.txt:1 and README.md:47-48).
 *
 * Conventions
 *   - every pointer is a raw DEVICE pointer owned by the caller (a torch tensor);
 *     the library never allocates device memory except one small per-device cache
 *     (the SM -> die table and claim words of the GEMM's die-aware tile walk, csrc/die_map.cu);
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it;
 *   - bf16 tensors are row-major with the innermost dimension contiguous;
 *   - return value 0 = ok, negative = error; evo_last_error() has the message;
 *   - no exceptions cross the boundary, no torch types appear in signatures.
 */
#ifndef EVO_B200_H
#define EVO_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* evo_last_error(void);
int evo_abi_version(void);
/* #launches of evo_b200 kernels since the last evo_reset_launch_count() (bench: gpu_launches) */
int64_t evo_launch_count(void);
void evo_reset_launch_count(void);
/* a CUDA-graph replay launches the kernels captured in it without passing through this library: the host adds the
 * number of launches recorded at capture time, once per replay (and subtracts the ones counted while capturing,
 * when nothing ran), so that evo_launch_count() stays truthful */
void evo_note_graph_replay(int64_t launches);

/* ---- embedding gather: VocabParallelEmbedding.embed (evo/models.py:136 pins the key) ----
 * ids: int32 or int64 (ids_are_i64), n tokens; table (vocab, D) bf16; out (n, D) bf16. */
int evo_embed(const void* ids, int ids_are_i64, const void* table, void* out,
              int64_t n_tokens, int D, int vocab, void* stream);

/* ---- RMSNorm, non-flash branch of stripedhyena layers.RMSNorm.forward:
 * y = scale * x / (||x||_2 * D^-1/2 + eps), every intermediate rounded to bf16 as the
 * reference's bf16 tensor ops do.  x,out (rows, D) bf16; scale (D) bf16. */
int evo_rmsnorm(const void* x, const void* scale, void* out, int64_t rows, int D, float eps, void* stream);

/* ---- tensor-core linear layers (nn.Linear / ParallelGatedMLP / unembed) ----
 * C[M,N] = epilogue(A[M,K] . W[N,K]^T), bf16 in, fp32 accumulate (tcgen05, TMEM), bf16 out.
 * Requirements: K % 64 == 0, N % 256 == 0 (weights are re-packed once at load time,
 * see evo_b200/stripedhyena/model.py), lda/ldc/ldr in elements. */
enum {
  EVO_EPI_NONE = 0,       /* C = bf16(acc)                                              */
  EVO_EPI_BIAS = 1,       /* C = bf16(acc + bias[n])                nn.Linear(bias=True) */
  EVO_EPI_BIAS_RESID = 2, /* C = bf16(bf16(acc + bias[n]) + R[m,n]) out_filter_dense(z)+u, out_proj(ctx)+u */
  EVO_EPI_RESID = 3,      /* C = bf16(bf16(acc) + R[m,n])           l3(...) + u           */
  EVO_EPI_GELU_GATE = 4,  /* W rows interleaved in 128-row groups [l1 | l2]; C[M,N/2] =
                             bf16(gelu(bf16(acc1)) * bf16(acc2))    act(l1 x) * l2 x      */
  EVO_EPI_HYENA_STEP = 7, /* evo_gemm_smallm only: the Hyena in-projection (N = 3D, bias) with the decode step of the operator
                             (engine.step_fir + step_iir == evo_hyena_step) applied in the epilogue: a tile is one head's
                             [x2 | x1 | v] rows, C is y (M, D); fir_state / state are updated in place; z is never stored */
  EVO_EPI_BIAS_ROPE = 6   /* Wqkv projection with the rotary embedding applied where flash_attn applies it
                             (MHA.forward, mha.py:635-648): x = bf16(acc + bias[n]); columns n < rope_cols (q and k,
                             heads of 128) are rotated NeoX-style with the cos/sin row of the token's position
                             (row m -> table row m % rope_L; the caller offsets the tables by the first position),
                             fp32 arithmetic, one rounding on store -- evo_rotary_qk's result without a second pass */
};
typedef struct {
  const void* A; int64_t lda;
  const void* W;                 /* (N, K) row-major */
  void* C; int64_t ldc;
  const void* bias;              /* (N) bf16 or NULL */
  const void* residual; int64_t ldr;
  int64_t M, N, K;
  int epilogue;
  int variant;                   /* 0 = 2-CTA 256x256 tiles; 1 = 1-CTA 128x256 tiles; 2 = 1-CTA 128x64 weight-streaming tiles (small M);
                                    3 = like 2 with W given tile-major: (N/64, K/64, 64, 64), i.e. W.view(N/64,64,K/64,64).permute(0,2,1,3) */
  const void* rope_cos; const void* rope_sin;   /* EVO_EPI_BIAS_ROPE: (positions, 64) bf16 tables (evo_rope_tables) */
  int64_t rope_L;                /* tokens per sequence: row m uses table row m % rope_L */
  int64_t rope_cols;             /* columns [0, rope_cols) are rotated (2*H*128 for a qkv projection), the rest only get the bias */
  /* Peer-scattered output (n_c_peers > 0): the epilogue stores straight into up to 8 peer-mapped buffers over NVLink, i.e.
   * the Ulysses head<->sequence all-to-all of a sequence-parallel attention layer fused into the Wqkv GEMM (no NCCL, no
   * permute): column n of row m goes to c_peers[(n % peer_period) / peer_inner], element
   * (peer_row0 + m) * ldc + (n / peer_period) * peer_inner + n % peer_inner.  For qkv (3, H, 128) and P ranks:
   * peer_period = H*128, peer_inner = H/P*128, ldc = 3*peer_inner, peer_row0 = rank * rows.  C is ignored. */
  void* const* c_peers;          /* HOST array of n_c_peers device pointers */
  int n_c_peers; int64_t peer_period, peer_inner, peer_row0;
} evo_gemm_params;
int evo_gemm(const evo_gemm_params* p, void* stream);
/* Decode-step linear layer (M <= 64 rows): the same C = epilogue(A . W^T) with the same rounding points, as a
 * weight-streaming kernel (csrc/gemm_smallm.cu): swap-AB tcgen05 tiles (128 W rows x M), stream-K over all SMs,
 * deterministic fix-up through `workspace`, weight prefetch ahead of the programmatic-dependent-launch wait.
 * EVO_EPI_GELU_GATE is fused here (C is (M, N/2)); replaces ParallelGatedMLP / nn.Linear at L == 1
 * (evo/generation.py:152 step path).  workspace: evo_gemm_smallm_workspace() bytes, zero-filled ONCE by the caller
 * (the per-tile counters in it reset themselves); one workspace may serve every call on a stream. */
typedef struct {
  const void* A; int64_t lda;
  const void* W;                 /* (N, K) row-major; GELU_GATE: rows interleaved [l1 | l2] per 256 */
  void* C; int64_t ldc;
  const void* bias;
  const void* residual; int64_t ldr;
  int64_t M, N, K;               /* M <= 64, N % 256 == 0, K % 64 == 0 */
  int epilogue;                  /* EVO_EPI_* */
  void* workspace; size_t workspace_bytes;
  /* EVO_EPI_HYENA_STEP only (same tensors as evo_hyena_step): */
  void* fir_state; float* state;                 /* (M, 3D, 2) bf16, (M, D, 8, 2) fp32: in/out */
  const void* fir_w; const void* fir_b; const void* Dskip;
  const float* poles; const float* residues;
} evo_gemm_smallm_params;
size_t evo_gemm_smallm_workspace(int64_t M, int64_t N, int64_t K, int epilogue);
int evo_gemm_smallm(const evo_gemm_smallm_params* p, void* stream);
/* Programmatic dependent launch for the decode step.  0 = off (default); 1 = every decode-step kernel is launched with
 * programmatic stream serialization; 2 = only evo_gemm_smallm is (its weight prefetch then overlaps the small kernel or
 * the GEMM tail in front of it); 3 = evo_gemm_smallm and the few-row evo_rmsnorm; 4 = those and
 * evo_hyena_step (which fetches its filter parameters and states ahead of the wait).  Every decode-step kernel begins with griddepcontrol.launch_dependents and waits
 * (griddepcontrol.wait) before it first touches dependent data.  Process-wide switch; returns the previous value. */
int evo_set_pdl(int level);

/* ---- fused Hyena operator: HyenaInferenceEngine.parallel_fir + ParallelHyenaFilter.
 * compute_filter + parallel_iir (+ prefill_via_modal_fft) of stripedhyena 0.2.2, as one
 * modal scan.  z (B, L, 3D) bf16 -> y (B, L, D) bf16.
 *   fir_w (3D, 3) bf16 taps [t-2, t-1, t]; fir_b (3D) bf16; Dskip (D) bf16;
 *   poles, residues (D, S, 2) fp32 (re, im), S == 8; nheads: column-split head count.
 * Optional (NULL to skip):
 *   halo (B, 2, 3D) bf16: the two z rows preceding row 0 (sequence-sharded rank > 0, or
 *        a continued prefill); zero history otherwise.
 *   state_in (B, D, S, 2) fp32: modal state entering row 0.
 *   state_out (B, D, S, 2) fp32: modal state after the last row (== inference_params.
 *        state_dict[layer] of the reference, complex64).
 *   fir_state_out (B, 3D, 2) bf16: last two z rows (== fir_state_dict[layer]).
 * workspace: evo_hyena_fwd_workspace() bytes (segment carries when L is split). */
typedef struct {
  const void* z; void* y;
  const void* fir_w; const void* fir_b; const void* Dskip;
  const float* poles; const float* residues;
  int B; int64_t L; int D; int S; int nheads;
  const void* halo; const float* state_in;
  float* state_out; void* fir_state_out;
  int force_segments;            /* 0 = auto; >0 forces the number of L segments (tests) */
  int state_only;                /* 1 = compute state_out only (sequence-parallel carry pass); y may be NULL */
  int reuse_segment_states;      /* 1 = workspace already holds the zero-start segment end states of a preceding
                                    state_only call on the same z / halo / geometry: skip recomputing them */
} evo_hyena_params;
size_t evo_hyena_fwd_workspace(const evo_hyena_params* p);
int evo_hyena_fwd(const evo_hyena_params* p, void* workspace, size_t workspace_bytes, void* stream);
/* the same operator on a right-padded batch: row b holds lengths_dev[b] (int32, DEVICE, clamped to [0, L]) valid tokens,
 * rows stay L apart in z and y.  state_out is the modal state after row b's own last token, fir_state_out the two z rows
 * before lengths_dev[b] (zero when there are fewer); y past a row's length is left unwritten.  With every length == L the
 * result is bit-identical to evo_hyena_fwd.  Mode-split scan only (head_dim 128, D % 256 == 0, EVO_B200_HYENA_VARIANT=1);
 * halo, state_in and reuse_segment_states are rejected.  workspace: evo_hyena_fwd_ragged_workspace() bytes. */
size_t evo_hyena_fwd_ragged_workspace(const evo_hyena_params* p);
int evo_hyena_fwd_ragged(const evo_hyena_params* p, const int32_t* lengths_dev, void* workspace, size_t workspace_bytes, void* stream);

/* decode step: engine.step_fir + step_iir.  u (B, 3D) bf16 -> y (B, D) bf16;
 * fir_state (B, 3D, 2) bf16 and state (B, D, S, 2) fp32 are updated in place. */
int evo_hyena_step(const void* u, void* y, void* fir_state, float* state,
                   const void* fir_w, const void* fir_b, const void* Dskip,
                   const float* poles, const float* residues,
                   int B, int D, int S, int nheads, void* stream);

/* combine per-rank end states into the state entering rank `rank`'s shard:
 * S_in = sum_{q<rank} p^{(rank-1-q)*seg_len} * ends[q].  ends (nranks, B, D, S, 2) fp32. */
int evo_hyena_combine_states(const float* ends, float* state_in, const float* poles,
                             int rank, int nranks, int64_t seg_len, int B, int D, int S, void* stream);

/* ---- peer-memory exchange for the sequence-parallel Hyena carry (NVLink stores + flags, no collective):
 * evo_peer_publish copies `bytes` from src into slot `rank` (slot_stride_bytes apart) of each peer buffer
 * peer_dsts[first_peer..last_peer] (device array of peer-mapped pointers) and then sets peer_flags[p][rank] = epoch
 * with system-scope release; evo_peer_wait blocks the stream until flags[first..last] >= epoch (acquire).
 * block_counter: one zero-initialised int of scratch on the calling device. */
int evo_peer_publish(const void* src, int64_t bytes, void* const* peer_dsts, int* const* peer_flags, int64_t slot_stride_bytes,
                     int rank, int first_peer, int last_peer, int epoch, int* block_counter, void* stream);
int evo_peer_wait(const int* flags, int first, int last, int epoch, void* stream);

/* ---- rotary tables + application (flash_attn layers/rotary.py:382-416,
 * ops/triton/rotary.py; stripedhyena LinearlyScaledRotaryEmbedding for 131k) ----
 * cos/sin (n_pos, hd/2) bf16 for positions pos0 .. pos0+n_pos-1, angle = (pos/scaling) * inv_freq[i]. */
int evo_rope_tables(void* cos_out, void* sin_out, const float* inv_freq, int64_t pos0, int64_t n_pos,
                    int half_dim, float scaling_factor, void* stream);
/* in-place NeoX rotary on q and k of qkv (B, L, 3, H, 128) bf16; cos/sin rows index the
 * position of row l directly (caller offsets the table for decode). */
int evo_rotary_qk(void* qkv, const void* cos, const void* sin, int B, int64_t L, int H, int hd, void* stream);

/* ---- causal attention core: flash_attn_qkvpacked_func (mha.py:122) ----
 * q: (B, Lq, H, 128) with row stride q_stride elements between tokens; k, v likewise over Lk
 * keys; query i attends keys j <= q_pos0 + i.  out (B, Lq, H*128) bf16 contiguous. */
typedef struct {
  const void* q; const void* k; const void* v; void* out;
  int64_t q_tok_stride, kv_tok_stride;     /* elements between consecutive tokens */
  int64_t q_batch_stride, kv_batch_stride; /* elements between batches */
  int B; int64_t Lq, Lk; int H; int hd;
  int64_t q_pos0;
  float softmax_scale;
  /* Peer-scattered output (n_out_peers > 0; variant 2, B == 1): query row i is stored into
   * out_peers[i / out_rows_per_peer] at element (i % out_rows_per_peer) * out_row_stride + out_col0 + h*128 -- the return
   * all-to-all of a sequence-parallel attention layer fused into the attention epilogue.  `out` is ignored. */
  void* const* out_peers;        /* HOST array of device pointers */
  int n_out_peers; int64_t out_rows_per_peer, out_row_stride, out_col0;
} evo_attn_params;
/* variant 0: V is transposed into the workspace first and consumed as a K-major operand;
 * variant 1: V is consumed in place as an MN-major operand (no workspace);
 * variant 2: ping-pong kernel: two query tiles per CTA, P kept in TMEM (A operand from TMEM), V in place;
 * variant 3: variant 2 with packed softmax arithmetic and 3 of every 8 exponentials evaluated on the FMA pipe (cubic). */
size_t evo_attn_fwd_workspace(const evo_attn_params* p, int variant);
int evo_attn_fwd_ws(const evo_attn_params* p, int variant, void* workspace, size_t workspace_bytes, void* stream);

/* append k,v of qkv (B, L, 3, H, hd) at rows [pos0, pos0+L) of the KV cache
 * (max_B, max_seqlen, 2, H, hd) bf16 — MHA._update_kv_cache (mha.py:344-370). */
int evo_kv_append(const void* qkv, void* cache, int B, int64_t L, int H, int hd,
                  int64_t pos0, int64_t max_seqlen, void* stream);

/* ---- decode step (L == 1), CUDA-graph friendly: the sequence position is read from DEVICE memory ----
 * evo_gelu_gate_interleaved: out[m, g*128+c] = bf16(gelu(t[m, g*256+c])) * t[m, g*256+128+c]; t (M, 2*ipad) is the
 *   plain GEMM output against the [l1 | l2]-interleaved weights (small-M tiles have no fused gate epilogue).
 * evo_decode_qkv_prep: rotary on q,k of qkv (B, 3, H, 128) at position *pos and append of k,v at cache row *pos
 *   (flash_attn_with_kvcache's rotary + cache-append half, mha.py:502-540).
 * evo_decode_attn: one query per sequence over cache keys [0, *pos] (the attention half); split-K over nsplit.
 * evo_advance_position: *pos += delta on the stream. */
int evo_gelu_gate_interleaved(const void* t, void* out, int64_t M, int ipad, void* stream);
int evo_decode_qkv_prep(void* qkv, void* cache, const void* cos, const void* sin, const int64_t* pos,
                        int B, int H, int hd, int64_t max_seqlen, void* stream);
size_t evo_decode_attn_workspace(int B, int H, int nsplit);
int evo_decode_attn(const void* qkv, const void* cache, void* out, const int64_t* pos, int B, int H, int hd,
                    int64_t max_seqlen, int nsplit, float softmax_scale, void* workspace, size_t workspace_bytes, void* stream);
int evo_advance_position(int64_t* pos, int64_t delta, void* stream);
/* the same two steps for a batch whose rows sit at different positions: pos is a DEVICE vector (B) int64 and row b's
 * rotary row, cache slot and key range [0, pos[b]] come from pos[b].  With every entry equal they compute exactly what
 * evo_decode_qkv_prep / evo_decode_attn compute. */
int evo_decode_qkv_prep_rows(void* qkv, void* cache, const void* cos, const void* sin, const int64_t* pos,
                             int B, int H, int hd, int64_t max_seqlen, void* stream);
int evo_decode_attn_rows(const void* qkv, const void* cache, void* out, const int64_t* pos, int B, int H, int hd,
                         int64_t max_seqlen, int nsplit, float softmax_scale, void* workspace, size_t workspace_bytes, void* stream);

/* ---- device-side sampler and generation loop: stripedhyena.sample.sample (evo/generation.py:162-167) and the host half
 * of the token loop (evo/generation.py:131-189) ----
 * evo_sample: logits (B, V) bf16 -> out (B) int64.  top_k == 1: argmax (first maximum); otherwise top-k (top_k <= 0:
 *   whole vocabulary) -> / temperature (bf16-rounded like the reference's tensor op) -> top-p tail mask (entries whose
 *   cumulative mass counted from the smallest up is <= 1 - top_p) -> multinomial.  Randomness: Philox4x32-10 keyed by
 *   (seed, step, row) -- reproducible, independent of launch order, CUDA-graph friendly.  V <= 1024.
 * evo_sample_step: the same inside the on-device loop.  Step index i = *step_dev (device); while i < n_forced the
 *   token is forced[row, i] (teacher-forced prompt tail), afterwards it is sampled with RNG step step0 + i and recorded:
 *   picked[row, i - n_forced] = token, kept_logits[row, i - n_forced, :] = float(logits[row]).  The token is also
 *   written to x[row], the next step's input.  All of evo_loop_params lives in DEVICE memory, so one captured graph
 *   serves every generate() call.
 * evo_advance_counters: *a += delta, *b += delta (either may be NULL). */
typedef struct {
  const int64_t* forced; int64_t n_forced; int64_t forced_stride;   /* (B, n_forced) int64 */
  int64_t* picked; int64_t picked_stride;                          /* (B, n_out) int64 or NULL */
  float* kept_logits; int64_t n_out;                               /* (B, n_out, V) fp32 or NULL */
  int32_t top_k; float top_p; float temperature;
  uint64_t seed; int64_t step0;
} evo_loop_params;
int evo_sample(const void* logits, int64_t* out, int B, int V, int top_k, float top_p, float temperature,
               uint64_t seed, uint64_t step, void* stream);
int evo_sample_step(const void* logits, int64_t* x, int B, int V, const evo_loop_params* loop_params_dev,
                    const int64_t* step_dev, void* stream);
int evo_advance_counters(int64_t* a, int64_t* b, int64_t delta, void* stream);
/* the loop for prompts of different lengths (one batch, one captured graph per step).  Row b's token at step i is
 *   forced[b, i] while i < n_forced[b]; afterwards it is sampled (RNG counter (seed, i, b)) and recorded at column
 *   out_cols - n_out[b] + (i - n_forced[b]) of picked (B, out_cols) int64 and kept_logits (B, out_cols, V) fp32 while
 *   i - n_forced[b] < n_out[b]; a row past its n_forced[b] + n_out[b] steps records nothing and keeps its input token.
 * evo_ragged_advance: *step += 1; pos[b] = start[b] + min(*step, n_forced[b] + n_out[b] - 1) (clamped at start[b]), so a
 *   finished row keeps the position of its last step.  B <= 1024.
 * The struct and every array it points to live in DEVICE memory. */
typedef struct {
  const int64_t* n_forced; const int64_t* n_out; const int64_t* start;   /* (B) each */
  const int64_t* forced; int64_t forced_stride;                         /* (B, forced_stride) int64 or NULL */
  int64_t* picked; float* kept_logits; int64_t out_cols;                /* (B, out_cols) int64, (B, out_cols, V) fp32; either may be NULL */
  int32_t top_k; float top_p; float temperature;
  uint64_t seed;
} evo_ragged_loop_params;
int evo_sample_step_rows(const void* logits, int64_t* x, int B, int V, const evo_ragged_loop_params* loop_params_dev,
                         const int64_t* step_dev, void* stream);
int evo_ragged_advance(int64_t* pos, int64_t* step, const evo_ragged_loop_params* loop_params_dev, int B, void* stream);

/* (test comparators -- cuBLASLt GEMM, CUDA-core attention, bf16 add -- live in tests/support/libevo_b200_test.so,
 *  not in this library) */

/* ---- scoring epilogue: evo/scoring.py:36-59 logits_to_logprobs ----
 * logits (rows, V) bf16; targets (rows) int64 (-1 = skip -> 0); out (rows) fp32 =
 * log_softmax(logits)[target], fp32 statistics. */
int evo_logprobs(const void* logits, const int64_t* targets, float* out, int64_t rows, int V, void* stream);


/* ---- batch front-end: evo/scoring.py:9-33 prepare_batch on the device ----
 * bytes: the sequences' raw bytes back to back (uint8, device); offsets (B+1) int64 (device): sequence b is
 * bytes[offsets[b] : offsets[b+1]].  ids_out (B, width) int32/int64 = [bos_id if prepend_bos] + bytes + pad_id ...
 * (CharLevelTokenizer.tokenize is the identity on bytes, evo/tokenizer.py:41).  width >= prepend_bos + max length. */
int evo_tokenize_pad(const void* bytes, const int64_t* offsets, void* ids_out, int ids_are_i64, int B, int64_t width,
                     int prepend_bos, int bos_id, int pad_id, void* stream);

/* ---- fused scoring head: unembed (tied embedding, N = vocab) + log_softmax + gather + entropy in one pass; the
 * (rows, V) logits never reach HBM (evo/scoring.py:36-59 logits_to_logprobs, :119-121 positional_entropies).
 * x (M, K) bf16 = final-norm output; W (V, K) bf16; targets (M) int64 (-1 = none -> logprob 0) or NULL.
 * logprobs[r] = bf16(x_r . W_t) - logsumexp_v(bf16(x_r . W_v)) in fp32 -- the logits are rounded to bf16 exactly where
 * the reference's logits tensor is, the statistics are fp32 (the reference's own log_softmax runs in bf16, quirk Q4);
 * entropy[r] = -sum_v p_v log p_v over the same distribution.  Either output may be NULL.  V % 256 == 0, K % 64 == 0. */
typedef struct {
  const void* x; const void* W;
  const int64_t* targets;
  float* logprobs; float* entropy;
  int64_t M; int V; int64_t K;
  void* workspace; size_t workspace_bytes;     /* evo_unembed_score_workspace(M, V) bytes */
} evo_score_params;
size_t evo_unembed_score_workspace(int64_t M, int V);
int evo_unembed_score(const evo_score_params* p, void* stream);

#ifdef __cplusplus
}
#endif
#endif
