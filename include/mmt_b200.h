/*
 * mmt_b200.h -- C ABI of the B200-native MMT candidate-generation engine.
 *
 * Drop-in boundary for ONE path of mpriessner/MultiModalSpectralTransformer:
 * spectra -> encoder memory -> greedy / multinomial SMILES token ids.
 * The reference has no FFI of its own (pure Python); each entry point below
 * names the reference function whose arithmetic it replaces (paths relative to
 * the reference's utils_MMT/).  The Python host in
 * multimodalspectraltransformer_b200/ binds these with ctypes and re-exposes the
 * reference's Python signatures (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer named d_* is DEVICE memory on
 *     the engine's device, h_* is HOST memory.
 *   - every call is stream-ordered on `stream` (a cudaStream_t passed as void*)
 *     and never synchronises unless documented.
 *   - threads and streams: an engine owns ONE workspace, so calls on one handle
 *     are serialised -- the library takes a per-engine mutex for the duration of
 *     each call (callers may use a handle from several threads), and a call
 *     issued on a different stream than the previous call on that handle first
 *     waits, on the device, for the previous call's work (an event recorded at
 *     the end of every call).  Two handles never share state.
 *   - return value: 0 on success, non-zero on failure; mmt_last_error() then
 *     returns a thread-local, NUL-terminated description.  There is no CPU
 *     fallback: without a usable sm_100 device mmt_create fails.
 */
#ifndef MMT_B200_H
#define MMT_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MMT_ABI_VERSION 2

typedef struct mmt_engine mmt_engine;

/* Hyper-parameters read from the reference's config (config_V8.json). */
typedef struct mmt_model_desc {
    int32_t d_model;        /* hidden_size        = 128 (only value supported) */
    int32_t n_heads;        /* num_heads          = 16  (modality encoders, decoder) */
    int32_t n_heads_cross;  /* int(num_heads / 4) = 4   (encoder_cross, models_MMT_v15_4.py:532) */
    int32_t d_ff;           /* 2048, torch default dim_feedforward (never overridden, :510-541) */
    int32_t n_enc_layers;   /* num_encoder_layers = 6 */
    int32_t n_dec_layers;   /* num_decoder_layers = 6 */
    int32_t vocab;          /* in_size = out_size = 43 */
    int32_t max_len;        /* rows of pe_trg     = 128 */
    int32_t mf_vocab;       /* MF_vocab_size      = 212 */
    int32_t ms_vocab;       /* MS_vocab_size      = 43 */
    int32_t ir_bins;        /* input_dim_IR       = 1000 */
    int32_t fp_size;        /* fingerprint_size   = 512 */
    int32_t pad_points;     /* padding_points_number = 64 */
} mmt_model_desc;

/* training_mode -> bit set ("1H" in config.training_mode, ...). */
enum {
    MMT_MODE_1H = 1 << 0, MMT_MODE_13C = 1 << 1, MMT_MODE_HSQC = 1 << 2, MMT_MODE_COSY = 1 << 3,
    MMT_MODE_IR = 1 << 4, MMT_MODE_MF = 1 << 5, MMT_MODE_MS = 1 << 6, MMT_MODE_MW = 1 << 7
};

/* Arithmetic of the GEMM-shaped work.  FP32 = SIMT FMA "check mode" (greedy ids
 * reproduce the reference's fp32 path); BF16 = tcgen05 tensor-core mode (bf16
 * operands, fp32 accumulate / residual stream / LayerNorm / softmax). */
enum { MMT_PREC_FP32 = 0, MMT_PREC_BF16 = 1 };

enum { MMT_SAMPLE_GREEDY = 0, MMT_SAMPLE_MULTINOMIAL = 1 };

/* Collated spectra, the tensor contract of dataloaders_pl_v15_4.py:665-712
 * (SURVEY.md A.1).  A pointer may be NULL iff its modality bit is not set. */
typedef struct mmt_spectra {
    const float*   d_src_1H;   const float* d_mask_1H;    /* (B,64,2) , (B,64) 0 valid / non-zero pad */
    const float*   d_src_13C;  const float* d_mask_13C;   /* (B,64)   , (B,64) */
    const float*   d_src_HSQC; const float* d_mask_HSQC;  /* (B,64,2) , (B,64) */
    const float*   d_src_COSY; const float* d_mask_COSY;  /* (B,64,2) , (B,64) */
    const float*   d_src_IR;                              /* (B,ir_bins); mask_IR is ignored by the model (:766) */
    const int64_t* d_src_MF;   const uint8_t* d_mask_MF;  /* (B,64) ids, (B,64) 1 = pad */
    const int64_t* d_src_MS;   const uint8_t* d_mask_MS;  /* (B,64) ids, (B,64) 1 = pad */
    const float*   d_trg_MW;                              /* (B) */
} mmt_spectra;

/* ---- lifetime ------------------------------------------------------------- */

int32_t mmt_abi_version(void);
const char* mmt_last_error(void);

/* Weight slots of the fp32 blob.  Names are the reference's state_dict keys
 * (models_MMT_v15_4.py:494-546; SURVEY.md A.3) so the host packs a checkpoint by
 * name: blob[mmt_weight_offset(i) : +mmt_weight_numel(i)] =
 * state_dict[mmt_weight_name(i)].float().flatten(); gaps (alignment) are ignored. */
int32_t     mmt_weight_count(const mmt_model_desc* desc);
const char* mmt_weight_name(const mmt_model_desc* desc, int32_t i);
int64_t     mmt_weight_numel(const mmt_model_desc* desc, int32_t i);
int64_t     mmt_weight_offset(const mmt_model_desc* desc, int32_t i);
int64_t     mmt_weight_total(const mmt_model_desc* desc);

/* Replaces: MultimodalTransformer.__init__ + load_MMT_model (.to("cuda"))
 * (models_MMT_v15_4.py:488-546, mmt_result_test_functions_15_4.py:467-475).
 * Copies the fp32 blob (h_weights, n_floats == mmt_weight_total) to `device`
 * and derives the bf16 operand copies.  Synchronous. */
int32_t mmt_create(const mmt_model_desc* desc, const float* h_weights, int64_t n_floats,
                   int32_t device, mmt_engine** out);
void    mmt_destroy(mmt_engine* e);

/* ---- encoder ---------------------------------------------------------------- */

/* Length S of the encoder memory for a mode (582 for all five spectra + MF + MW;
 * blank-modality and MS rules of models_MMT_v15_4.py:834-939). */
int32_t mmt_memory_len(const mmt_model_desc* desc, uint32_t mode_bits);
/* 1 when the reference's concatenated key-padding mask is promoted to float
 * (a 1H/13C/HSQC/COSY modality absent from training_mode, SURVEY.md B.2). */
int32_t mmt_mask_is_float(uint32_t mode_bits);

/* Replaces: vgmmt.run_model / MultimodalTransformer.forward(trg=None)
 * (validate_generate_MMT_v15_4.py:95-267, models_MMT_v15_4.py:803-953):
 * embedders -> 5 modality encoders -> encoder_cross -> mean -> fp1.
 *   d_memory        out (S,B,128) f32, sequence-first like the reference
 *   d_embedding_src out (S,B,128) f32 or NULL (forward()'s 2nd return)
 *   d_key_bias      out (B,S) f32: additive attention bias of each memory row,
 *                   0 valid, -inf padded, or the float mask value (0 / 1) in
 *                   float-mask modes
 *   d_pad_mask      out (B,S) u8: 1 where the reference's mask is True / 1.0
 *   d_fingerprint   out (B,fp_size) f32
 *   d_avg_memory    out (B,128) f32 or NULL (mean over S, input of fp1)        */
int32_t mmt_encode(mmt_engine* e, const mmt_spectra* in, int32_t B, uint32_t mode_bits,
                   int32_t precision, float* d_memory, float* d_embedding_src, float* d_key_bias,
                   uint8_t* d_pad_mask, float* d_fingerprint, float* d_avg_memory, void* stream);

/* Bitwise equality of the collated inputs of two encode calls (all arrays of the modalities in mode_bits, B spectra).
 * Serves the repeated-encode pattern of the callers -- CLIP's forward(trg=None) on a batch run_model has just encoded
 * (models_CLIP_v15_4.py:278-285, 337-347; SURVEY.md 8 f4): the host keeps the last encode's inputs and outputs and
 * skips the second encode when this returns 1.  One small kernel, a 4-byte device-to-host read, synchronises `stream`.
 * mmt_encode itself accepts d_memory == NULL with d_embedding_src != NULL for an embedding-only pass (forward()'s
 * second output when the rest comes from the cache). */
int32_t mmt_spectra_equal(mmt_engine* e, const mmt_spectra* a, const mmt_spectra* b, int32_t B, uint32_t mode_bits,
                          int32_t* h_equal, void* stream);

/* ---- decoder ---------------------------------------------------------------- */

typedef struct mmt_decode_args {
    /* encoder memory as the reference hands it to the decode loops: element
     * (s,b,d) at d_memory[s*stride_s + b*stride_b + d]; any caller slicing /
     * duplication is expressible (validate_generate_MMT_v15_4.py:1083-1084). */
    const float* d_memory; int64_t stride_s; int64_t stride_b;
    const float* d_key_bias;       /* (Bm,S) additive bias, row stride S */
    int32_t S;                     /* memory rows */
    int32_t Bm;                    /* distinct memories */
    int32_t n_cand;                /* sequences per memory; sequence n reads memory n / n_cand.
                                      The reference gets 128 by tensor duplication
                                      (run_batch_gen_val_MMT_v15_4.py:93-107); here K/V are shared. */
    int32_t max_len;               /* config.max_len at call time (<= desc.max_len) */
    float   temperature;           /* config.temperature at call time */
    int32_t sampling;              /* MMT_SAMPLE_* */
    int32_t stop_on_all_pad;       /* greedy_sequence's early exit (validate_generate_MMT_v15_4.py:763) */
    int32_t precision;             /* MMT_PREC_* */
    /* Philox state of torch's CUDA generator for torch.multinomial parity
     * (SURVEY.md appendix D).  One "torch.multinomial((N_total,43),1)" call per
     * step: step t uses offset philox_offset + t*mmt_philox_increment(N_total*vocab).
     * seq_index_base / N_total place this call's sequences inside a larger
     * logical batch so that sharded runs draw the numbers of the unsharded run. */
    uint64_t philox_seed; uint64_t philox_offset;
    int64_t  seq_index_base; int64_t N_total;
    int32_t  rng_sm_count; int32_t rng_max_threads_per_sm;   /* 0 = this device's */
} mmt_decode_args;

/* Replaces the decode loops greedy_sequence / multinomial_sequence /
 * multinomial_sequence_multi (validate_generate_MMT_v15_4.py:723-775, 841-880;
 * run_batch_gen_val_MMT_v15_4.py:121-158): KV-cached, one step per position.
 *   d_tokens out (max_len, N) i64  -- generated ids, WITHOUT the <SOS> row
 *   d_probs  out (max_len, N) f32  -- softmax(logits/T) of the chosen id, every step
 *   h_steps  out host int: steps executed (max_len, or the step at which every
 *            sequence emitted <PAD> when stop_on_all_pad).  Synchronises `stream`
 *            once at the end when h_steps != NULL and stop_on_all_pad is set.   */
int32_t mmt_decode(mmt_engine* e, const mmt_decode_args* a, int64_t* d_tokens, float* d_probs,
                   int32_t* h_steps, void* stream);

/* mmt_decode with the multinomial draws in PER-MEMORY streams: the n_cand candidates of memory column b draw what one
 * torch.multinomial((n_cand, vocab), 1) call per step would, the columns' calls taken in order, as the reference's
 * per-spectrum loop does (multinomial_sequence_multi on n_cand duplicates, spectrum after spectrum).  With
 * B0 = seq_index_base / n_cand and inc = mmt_philox_increment(n_cand*vocab): column b at step t uses offset
 * philox_offset + ((B0 + b)*max_len + t)*inc, candidate j its elements j*vocab .. of that call.  A caller's generator
 * ends advanced by Bm_total*max_len*inc.  Fails unless a->sampling is multinomial and seq_index_base is a multiple of
 * n_cand; N_total is ignored. */
int32_t mmt_decode_memory_streams(mmt_engine* e, const mmt_decode_args* a, int64_t* d_tokens, float* d_probs,
                                  int32_t* h_steps, void* stream);

/* mmt_decode (per_memory_rng == 0) or mmt_decode_memory_streams (per_memory_rng != 0) that stops computing a sequence
 * once it has emitted `eos`: same arguments, preconditions and draws (every sequence keeps its Philox elements, a
 * caller's generator is advanced by the same amount).  With L_n the position of the first `eos` the plain call writes
 * for sequence n (max_len if none):
 *   d_tokens / d_probs  (max_len, N): bit-identical to the plain call at t <= L_n; <PAD> (0) / 0.0f after L_n and at
 *                       t >= *h_steps
 *   d_len   out (N) i32: L_n (mmt_first_eos of the plain call's ids)
 *   h_steps out host int or NULL: positions up to the one at which every sequence had finished (greedy with
 *           stop_on_all_pad: finished or emitted <PAD>), else max_len
 *   h_rows  out host (max_len) i64 or NULL: decode-step rows computed at each position, summed over waves and lanes
 *           (0 where no step ran)
 * Large (un-fused) waves drop finished rows at 8-position group boundaries, from counts the host reads one group
 * behind the launches; small waves keep their rows and only stop early.  Fails when `eos` is outside [0, vocab). */
int32_t mmt_decode_until_eos(mmt_engine* e, const mmt_decode_args* a, int32_t per_memory_rng, int64_t eos,
                             int64_t* d_tokens, float* d_probs, int32_t* d_len, int32_t* h_steps, int64_t* h_rows,
                             void* stream);

/* Per-memory-column sampling controls for multinomial decoding.  Each non-NULL array holds `count` (== the call's
 * columns) host values; column b (one spectrum, all its n_cand candidates) samples at every step as follows:
 *   p = softmax(logits / temperature[b])            (bit-identical to the plain call's p where temperature[b] equals it)
 *   rank: token i before j iff p_i > p_j, or p_i == p_j and i < j
 *   top-k: keep rank < top_k[b]                     (0 or vocab: off)
 *   top-p: of the top-k survivors keep the rank-0 token and every i with before_i < top_p[b] * mass, mass = fp32 sum of
 *          the survivors' p, before_i = that of the survivors ranked before i, both summed in ascending token index
 *          (top_p[b] == 1: off, not evaluated)
 *   draw:  the first arg-max of p_i / q_i over the kept tokens, q the Exp(1) variates of the plain call (either RNG
 *          mapping), so a draw the plain call makes inside the kept set is unchanged; the generator advance is the plain
 *          call's whatever the controls
 *   reported probability: p of the chosen token, NOT renormalised over the kept set (equal to the plain call's wherever
 *          the draw is, and comparable across columns with different truncation).
 * Ranges, checked on the host: temperature > 0 and finite, top_k in [0, vocab], top_p in (0, 1]. */
typedef struct mmt_sampling_controls {
    int64_t        count;           /* entries in each non-NULL array */
    const float*   h_temperature;   /* (count) host, or NULL: a->temperature for every column */
    const int32_t* h_top_k;         /* (count) host, or NULL: off */
    const float*   h_top_p;         /* (count) host, or NULL: off */
} mmt_sampling_controls;

/* mmt_decode / mmt_decode_memory_streams (eos < 0) or mmt_decode_until_eos (eos >= 0; d_len, h_steps, h_rows as there,
 * ignored when eos < 0) with per-column sampling controls (count == a->Bm).  Multinomial only.  Neutral controls (every
 * temperature a->temperature, top-k and top-p off) give the plain call's output bit for bit.  The values are copied to
 * the device before the first step and are not part of a cached decode graph. */
int32_t mmt_decode_controlled(mmt_engine* e, const mmt_decode_args* a, int32_t per_memory_rng, int64_t eos,
                              const mmt_sampling_controls* c, int64_t* d_tokens, float* d_probs, int32_t* d_len,
                              int32_t* h_steps, int64_t* h_rows, void* stream);

/* Replaces the decoder tail of MultimodalTransformer.forward(..., trg_SMI_input)
 * (models_MMT_v15_4.py:955-976) and the teacher-forced scorers' inner call:
 * d_trg (T,N) i64 -> d_logits (T,N,vocab) f32 (fc_out, before softmax). */
int32_t mmt_teacher_forced(mmt_engine* e, const mmt_decode_args* a, const int64_t* d_trg, int32_t T,
                           float* d_logits, void* stream);

/* Replaces the teacher-forced scorers predict_prop_correct_max_sequence(_2) (validate_generate_MMT_v15_4.py:309-509)
 * and mrtf.predict_prop_correct_max_sequence_3 (mmt_result_test_functions_15_4.py:340-400): T positions with the given
 * input tokens d_trg_in (T,N) (row 0 = <SOS>), one KV-cached step per position instead of a full-prefix decoder run
 * per position.  At every position: d_pick / d_pick_prob (T,N) = the greedy (a->sampling == GREEDY: argmax, first max)
 * or multinomial (Philox contract of mmt_decode) pick under softmax(logits / a->temperature) and its probability --
 * never fed back; d_target_prob (T,N) = probability of d_target (T,N) (both NULL to skip).  a->stop_on_all_pad is
 * ignored. */
int32_t mmt_teacher_forced_scores(mmt_engine* e, const mmt_decode_args* a, const int64_t* d_trg_in, const int64_t* d_target,
                                  int32_t T, int64_t* d_pick, float* d_pick_prob, float* d_target_prob, void* stream);

/* Replaces vgmmt.beam_search / beam_search_step (validate_generate_MMT_v15_4.py:995-1086), batched: the
 * beam_size beams of each of the a->Bm memory columns are slots of one KV-cached decode wave (a->n_cand, max_len,
 * temperature and sampling are ignored: the reference ranks with softmax(logits) without temperature, :1038).
 * gen_len steps (config.gen_len) from the single [<SOS>] beam; beams ending in `eos` are carried unchanged;
 * score = product of the chosen probabilities in double (Python floats); per step a stable sort by score.
 * Slot n = column * beam_size + rank (rank 0 = best):
 *   d_seq   out (N, gen_len+1) i64  sequence incl. <SOS>, zero-filled past d_len
 *   d_len   out (N) i32             tokens in the sequence (<SOS> included)
 *   d_score out (N) f64
 *   d_probs out (N, gen_len) f32    probability of every chosen token, zero-filled past d_len-1
 *   h_steps out host int or NULL: steps executed (fewer than gen_len once every beam has finished; the skipped
 *           steps are fixed points of the reference's loop).  Synchronises `stream` every 16 steps. */
int32_t mmt_beam_search(mmt_engine* e, const mmt_decode_args* a, int32_t beam_size, int32_t gen_len, int32_t eos,
                        int64_t* d_seq, int32_t* d_len, double* d_score, float* d_probs, int32_t* h_steps, void* stream);

/* Sampling without replacement by stochastic beam search (Kool, van Hoof & Welling, ICML 2019): per memory column b the
 * k = a->n_cand (1..128) slots hold k DISTINCT sequences that are an exact sample without replacement from the engine's
 * ancestral-sampling distribution at temperature tau_b (the leaves of the tree of <SOS>-prefixes: sequences ending in
 * `eos` or holding max_len tokens), in the order of a Gumbel-top-k: slot 0 is an ancestral sample, slot 1 a sample from
 * the rest, ...  Per step, each live slot of rank r perturbs its children's log-probabilities phi + log p_i
 * (p = softmax(logits / tau_b) in fp32, as the multinomial sampler computes it) with -log E_i, E_i the Exp(1) variate at
 * element r * V + i of one torch exponential_ call of k * V elements at generator offset
 * philox_offset + ((seq_index_base / k + b) * max_len + t) * increment(k * V) (per-memory streams); children's keys
 * are conditioned on the parent's key in double; the k largest keys of all children and carried finished slots become
 * the new slots (ties: parent rank, then token id).  Slots without a sequence (fewer than k leaves exist) are empty.
 * Uses a->n_cand, max_len, philox_seed / philox_offset, seq_index_base (a multiple of n_cand), N_total (0, or a multiple
 * of n_cand: the caller advances its generator by (N_total or Bm * n_cand) / n_cand * max_len * increment(k * V)),
 * rng_sm_count / rng_max_threads_per_sm and precision; a->sampling is ignored.  h_temperature: (Bm) host, or NULL for
 * a->temperature everywhere; each > 0 and finite.  Slot n = column * n_cand + rank:
 *   d_tokens   out (max_len, N) i64  ids without <SOS>, <PAD> after <EOS> and in empty slots
 *   d_probs    out (max_len, N) f32  p of each chosen token, 0 after <EOS>
 *   d_len      out (N) i32           generated tokens including <EOS> (0: empty slot)
 *   d_log_prob out (N) f64           sum of log((double)p) (-inf: empty slot)
 *   d_key      out (N) f64           Gumbel key, descending within a column (-inf: empty slot)
 *   h_steps    out host int or NULL: steps executed (fewer than max_len once every slot has finished).
 * Synchronises `stream` every 16 steps and between waves. */
int32_t mmt_sample_without_replacement(mmt_engine* e, const mmt_decode_args* a, const float* h_temperature, int32_t eos,
                                       int64_t* d_tokens, float* d_probs, int32_t* d_len, double* d_log_prob, double* d_key,
                                       int32_t* h_steps, void* stream);

/* One selection step of mmt_sample_without_replacement on given logits and state (unit-test hook): Bm columns of k
 * slots, V tokens, step `step` of T.  In: d_logits (Bm*k, V) f32, slot state d_phi / d_key (Bm*k) f64 (-inf: empty),
 * d_len (Bm*k) i32, d_hist (Bm*k, T) u8 token ids, d_probs (Bm*k, T) f32; h_temperature (Bm) host.  Out: the new state
 * in the *_out buffers (positions past `step` of hist / probs copied from the input); d_p_out (Bm*k, V) f32 optional:
 * softmax(logits / tau) of every live, unfinished slot (other rows untouched).  RNG as above with seq_index_base / k
 * the global index of column 0. */
int32_t mmt_sbs_select_step(mmt_engine* e, const float* d_logits, int32_t Bm, int32_t k, int32_t V, int32_t T, int32_t step, int32_t eos,
                            const float* h_temperature, uint64_t philox_seed, uint64_t philox_offset, int64_t seq_index_base,
                            int32_t rng_sm_count, int32_t rng_max_threads_per_sm,
                            const double* d_phi, const double* d_key, const int32_t* d_len, const uint8_t* d_hist, const float* d_probs,
                            double* d_phi_out, double* d_key_out, int32_t* d_len_out, uint8_t* d_hist_out, float* d_probs_out, float* d_p_out,
                            void* stream);

/* Offset increment torch applies to its Philox generator for one
 * exponential_() over `numel` elements (DistributionTemplates.h calc_execution_policy). */
uint64_t mmt_philox_increment(int64_t numel, int32_t sm_count, int32_t max_threads_per_sm);

/* Device-to-device gather of token ids into bytes: (T,N) i64 -> (T,N) u8
 * (vocab 43 < 256); the payload the data-parallel scheduler all-gathers. */
int32_t mmt_pack_tokens_u8(const int64_t* d_tokens, int64_t n, uint8_t* d_out, void* stream);
int32_t mmt_unpack_tokens_u8(const uint8_t* d_in, int64_t n, int64_t* d_tokens, void* stream);

/* The same payload in SEQUENCE-MAJOR order: (T,N) i64 ids -> (N,T) u8, and back.  Ranks own contiguous blocks of
 * sequences, so an all-gather of (N_local,T) blocks lands directly in the final (N_total,T) order -- no re-layout copy
 * after the collective (the time-major form interleaves the ranks' columns).  The inverse reads `N` rows of the
 * gathered (>= N, T) buffer and writes the caller-facing (T,N) i64 tensor (tiled transposes through shared memory). */
int32_t mmt_pack_tokens_u8_seqmajor(const int64_t* d_tokens, int32_t T, int64_t N, uint8_t* d_out, void* stream);
int32_t mmt_unpack_tokens_u8_seqmajor(const uint8_t* d_in, int32_t T, int64_t N, int64_t* d_tokens, void* stream);

/* ---- ragged ingest (the data format in front of the path) -------------------------- */

/* Replaces MultimodalData._zero_pad + the per-modality normalisation of __getitem__
 * (dataloaders_pl_v15_4.py:267-299, 352-365, 456-460, 481-485, 505-509, 546-550): CSR peak lists
 * (d_values: nnz x cols doubles, d_offsets: B+1 int64) -> d_src (B,P[,cols]) f32 = value / div_c rounded like
 * torch.tensor(python floats), zero padded, truncated at P; d_mask (B,P) f32, 0 valid / 1 pad.  cols == 1
 * reproduces the reference's all-ones mask for lists with >= P entries (SURVEY A.1). */
int32_t mmt_ingest_peaks(const double* d_values, const int64_t* d_offsets, int32_t B, int32_t cols,
                         double div0, double div1, int32_t pad_points, float* d_src, float* d_mask, void* stream);
/* Replaces MultimodalData._load_IR_data's binning (dataloaders_pl_v15_4.py:324-346): every spectrum of
 * arbitrary length -> `bins` mean-binned values divided by the spectrum's maximum, (B,bins) f32. */
int32_t mmt_ingest_ir(const double* d_values, const int64_t* d_offsets, int32_t B, int32_t bins,
                      float* d_src_IR, void* stream);

/* Replaces the per-element .item() scans of tensor_to_smiles / tensor_to_smiles_and_prob(_2)
 * (helper_functions_pl_v15_4.py:255-301, 390-419): d_len[n] = position of the first `eos` id in column n
 * of d_tokens (T,N) i64, or T if the sequence never emits it.  The host then slices tokens / probabilities
 * and joins the strings after ONE device-to-host copy. */
int32_t mmt_first_eos(const int64_t* d_tokens, int32_t T, int64_t N, int32_t eos, int32_t* d_len, void* stream);

/* Distinct strings per memory column of candidate ids d_tokens (T,N) i64, N = Bm*n_cand: for column b, the distinct
 * values of tensor_to_smiles(tokens[:, b*n_cand:(b+1)*n_cand], itos) in first-occurrence order (dict.fromkeys), each
 * with the index of its first candidate and its multiplicity.  A string is the byte concatenation of the itos entries
 * of the ids before the first `eos`; strings are compared byte by byte.  itos as a table: d_itos_entries (n_itos, 2)
 * i32 {byte start, byte length} into d_itos_bytes (UTF-8), length -1 where an id has no entry; itos_max_bytes = the
 * longest entry.  With d_work NULL: *work_bytes = the device workspace these sizes need.  Otherwise runs, synchronises
 * `stream` once and returns h_result[6] = {distinct strings D, their bytes, offset and size of the output in d_work,
 * 1 if an id before <EOS> has no itos entry, that id}.  The output (int64 unless noted): col_off[Bm+1], first[D],
 * count[D], ntok[D] (ids before <EOS>), boff[D+1], then the strings' bytes (u8) -- string d = bytes[boff[d], boff[d+1]). */
int32_t mmt_distinct_smiles(const int64_t* d_tokens, int32_t T, int64_t N, int32_t n_cand, int64_t eos,
                            const uint8_t* d_itos_bytes, const int32_t* d_itos_entries, int32_t n_itos, int32_t itos_max_bytes,
                            void* d_work, int64_t* work_bytes, int64_t* h_result, void* stream);

/* ---- building blocks exported for unit parity tests --------------------------- */

/* fused fc_out + softmax(logits/T) + greedy|multinomial pick on hidden states
 * d_x (N,128): the sampling kernel of the decode step, stand-alone.
 * d_logits_out (N,vocab) optional. */
int32_t mmt_sample(mmt_engine* e, const float* d_x, int64_t N, float temperature, int32_t sampling,
                   uint64_t philox_seed, uint64_t philox_offset, int64_t seq_index_base, int64_t N_total,
                   int32_t rng_sm_count, int32_t rng_max_threads_per_sm,
                   int64_t* d_token, float* d_prob, float* d_logits_out, void* stream);

/* The Exp(1) variates torch's CUDA `exponential_` writes (ATen DistributionTemplates.h:427-441 through
 * torch.multinomial's fast path, SURVEY.md App. D): d_q[i] = the variate at linear element elem_base + i of a
 * tensor of numel_total elements under generator state (seed, offset) on a device with sm_count SMs of
 * max_threads_per_sm threads.  Lets a test assert BIT equality with torch.empty(...).exponential_(). */
int32_t mmt_exponential(uint64_t philox_seed, uint64_t philox_offset, int64_t elem_base, int64_t n, int64_t numel_total,
                        int32_t sm_count, int32_t max_threads_per_sm, float* d_q, void* stream);

/* torch.multinomial(p, 1) on caller-supplied probabilities d_p (N,V) f32: token = first arg-max of p / q with q as
 * above (rows seq_index_base .. seq_index_base+N of a logical (N_total,V) call).  With torch's own p as input the
 * ids must equal torch.multinomial's exactly -- separates the RNG stream from probability round-off. */
int32_t mmt_sample_probs(const float* d_p, int64_t N, int32_t V, uint64_t philox_seed, uint64_t philox_offset,
                         int64_t seq_index_base, int64_t N_total, int32_t sm_count, int32_t max_threads_per_sm,
                         int64_t* d_token, void* stream);

/* The per-memory mapping of mmt_decode_memory_streams at one step, stand-alone: rows n of a call placed at
 * seq_index_base (a multiple of n_cand) draw as candidate (seq_index_base+n) mod n_cand of column
 * (seq_index_base+n) / n_cand at step `step` of max_len.  Exactly one of d_x (N,128) hidden states (the decode
 * step's fused fc_out + softmax(logits/temperature) + pick, d_prob optional) and d_p (N,vocab) caller probabilities
 * (the stream alone, as mmt_sample_probs; d_prob unused). */
int32_t mmt_sample_memory_streams(mmt_engine* e, const float* d_x, const float* d_p, int64_t N, int32_t n_cand, int32_t max_len,
                                  int32_t step, float temperature, uint64_t philox_seed, uint64_t philox_offset,
                                  int64_t seq_index_base, int32_t rng_sm_count, int32_t rng_max_threads_per_sm,
                                  int64_t* d_token, float* d_prob, void* stream);

/* The controlled pick (mmt_sampling_controls) at step `step` of max_len, stand-alone, for N rows; row n belongs to control
 * column n / n_cand (c->count == ceil(N / n_cand)).  Exactly one of d_x (N,128) hidden states (the decode step's fc_out +
 * softmax(logits / temperature) + pick; d_logits_out (N,vocab) optional) and d_p (N,vocab) caller probabilities
 * (temperatures ignored).  RNG: per_memory_rng as mmt_sample_memory_streams, else the global mapping of mmt_sample
 * (rows seq_index_base .. of an N_total-row call, step `step` at offset philox_offset + step * increment).
 * d_prob (N) optional: p of the chosen token; d_kept (N,vocab) u8 optional: 1 where the token is kept. */
int32_t mmt_sample_controlled(mmt_engine* e, const float* d_x, const float* d_p, int64_t N, int32_t n_cand,
                              const mmt_sampling_controls* c, int32_t per_memory_rng, int32_t max_len, int32_t step,
                              uint64_t philox_seed, uint64_t philox_offset, int64_t seq_index_base, int64_t N_total,
                              int32_t rng_sm_count, int32_t rng_max_threads_per_sm,
                              int64_t* d_token, float* d_prob, float* d_logits_out, uint8_t* d_kept, void* stream);

/* C[M,N] = act(A[M,K] . W[N,K]^T + bias) in the requested precision
 * (fp32 SIMT or bf16 tcgen05); act: 0 none, 1 ReLU. */
int32_t mmt_linear(mmt_engine* e, const float* d_A, const float* d_W, const float* d_bias, float* d_C,
                   int64_t M, int32_t N, int32_t K, int32_t act, int32_t precision, void* stream);

/* The fused feed-forward block of one transformer layer (linear1 -> ReLU -> linear2 -> +residual
 * -> LayerNorm; torch TransformerEncoderLayer._ff_block + norm2, models_MMT_v15_4.py:510-541) in
 * the bf16 tensor-core mode:  d_out = LN(d_x + W2 relu(W1 bf16(d_x) + b1) + b2) * gamma + beta,
 * d_x / d_out (M,128) f32, W1 (F,128), W2 (128,F).  splits > 1 exercises the split-F partial path
 * the small-batch decoder uses.  weight_terms: 2 = W as the two-term bf16 split W_hi + W_lo (encoder layers),
 * 1 = W_hi alone (decoder layers; the kernel variant with the deeper GEMM1 / convert / GEMM2 pipeline). */
int32_t mmt_ffn(mmt_engine* e, const float* d_x, const float* d_w1, const float* d_b1, const float* d_w2,
                const float* d_b2, const float* d_gamma, const float* d_beta, float* d_out,
                int64_t M, int32_t F, int32_t splits, int32_t weight_terms, void* stream);

/* The self-attention half of one decoder layer of the un-fused (large-wave) decode step, stand-alone, with the code the
 * step runs: QKV projection of layer `layer` (bf16: tcgen05 on W_hi, K | V appended to the paged cache by the GEMM's
 * epilogue or by the attention kernel, as the engine's MMT_KV_HEAD_MAJOR / MMT_NO_KV_EPILOGUE knobs select; fp32: SIMT
 * GEMM) followed by the matching paged self-attention kernel, for positions t = 0 .. T-1 of N sequences in one wave
 * (slot-major page map).  d_x (T,N,128) f32: the layer's input rows at every position (rounded to bf16 in the bf16 mode);
 * d_out (T,N,128) f32: the attention output (before out_proj) of position t over keys 0..t, widened from bf16 in the
 * bf16 mode.  Unwritten cache slots hold NaN. */
int32_t mmt_decode_self_attention(mmt_engine* e, int32_t layer, const float* d_x, int64_t N, int32_t T, int32_t precision,
                                  float* d_out, void* stream);

/* The cross-attention of one decoder layer of the un-fused decode step, stand-alone: the memory of a->Bm spectra is
 * prepared as one decode wave (memory index, K/V projection with the two-term weights), then the queries d_q
 * (Bm*n_cand,128) f32 attend to it -- the tensor-core kernel for a->n_cand >= 8 in the bf16 mode (MMT_NO_TC_ATTENTION: the
 * SIMT kernel), the SIMT kernel otherwise.  d_out (Bm*n_cand,128) f32: the attention output (before out_proj), widened
 * from bf16 in the bf16 mode.  Memory, key_bias, S, Bm, n_cand and precision come from `a`; the rest of it is ignored. */
int32_t mmt_decode_cross_attention(mmt_engine* e, const mmt_decode_args* a, int32_t layer, const float* d_q, float* d_out,
                                   void* stream);

/* The rest of one decoder layer of the un-fused decode step after its two attentions, stand-alone, with the code the step
 * runs: R sequences in one wave, the variants chosen as the step chooses them (from R and the engine's MMT_NO_GEMM_CHAIN,
 * MMT_NO_FFN_PROLOGUE, MMT_DEC_PROJ_TWO_TERM and MMT_DEC_FFN_TWO_TERM knobs).  Inputs (R,128) f32: d_x the layer's input
 * rows (the fp32 residual), d_att_self / d_att_cross the self- and cross-attention outputs before their out_proj (rounded
 * to bf16 in the bf16 mode, as the step stores them).  Outputs (R,128) f32:
 *   d_x1  = norm1(x + out_proj(att_self)),
 *   d_qc  = the cross-attention query projection of x1,
 *   d_x2  = norm2(x1 + ca_out_proj(att_cross)) -- optional (may be NULL), and written only where the step stores it: not
 *           when the FFN kernel's prologue computes it (bf16 mode, R >= 2048, no MMT_NO_FFN_PROLOGUE),
 *   d_out = norm3(x2 + FFN(x2)), the layer's output. */
int32_t mmt_decode_layer_tail(mmt_engine* e, int32_t layer, const float* d_x, const float* d_att_self, const float* d_att_cross,
                              int64_t R, int32_t precision, float* d_x1, float* d_qc, float* d_x2, float* d_out, void* stream);

/* Layer `layer` of encoder stack `stack` (0-4: encoder_1H / 13C / HSQC / COSY / IR, 16 heads; 5: encoder_cross, n_heads_cross
 * heads), stand-alone, with the code the encoder runs: encoder_layer_bf16 (tcgen05 projections on the two-term weights, the
 * fused FFN) or encoder_layer_fp32, and the encoder attention kernel the engine's MMT_NO_TC_ATTENTION / MMT_TC5_ATTENTION /
 * MMT_TC_ATTENTION_FP32 knobs select.  d_x (rows,128) f32 input rows, B sequences in one of two layouts:
 *   dense  (d_key_bias != NULL): rows == B*S, sequence b owns rows b*S .. b*S+S-1; d_key_bias (B,S) additive (-inf: not a
 *          key; float masks: 0 / +1.0); the keys are compacted as the dense encoder does; row_start .. kstride ignored.
 *   ragged (d_key_bias == NULL): sequence b owns rows row_start[b] .. row_start[b]+cnt[b]-1 (cnt[b] <= S) and attends, with
 *          bias 0, the nk[b] rows kidx[b*kstride + j] (j < nk[b], row numbers relative to row_start[b]); all int32 on the
 *          device.  The attention CTAs are sized by max nk and max cnt, as the ragged encoder sizes them.
 * Outputs (rows,128) f32: d_qkv (rows,384, optional) the QKV projection the attention reads, d_att (optional) the attention
 * output before out_proj (widened from bf16 in the bf16 mode), d_out the layer output after norm2. */
int32_t mmt_encoder_layer(mmt_engine* e, int32_t stack, int32_t layer, const float* d_x, int64_t rows, int32_t B, int32_t S,
                          const float* d_key_bias, const int32_t* d_row_start, const int32_t* d_cnt, const int32_t* d_kidx,
                          const int32_t* d_nk, int32_t kstride, int32_t precision, float* d_qkv, float* d_att, float* d_out,
                          void* stream);

/* launches issued by this engine since creation (bench.py's gpu_launches). */
int64_t mmt_launch_count(const mmt_engine* e);

/* Per-kernel-class device time for the roofline report: while enabled, every
 * launch is bracketed by CUDA events recorded on the launching stream.
 * mmt_profile_report synchronises the device and writes a JSON object
 * {"kernel": {"launches": n, "ms": total, "flops": algorithmic GEMM flops}, ...}. */
int32_t mmt_profile_enable(mmt_engine* e, int32_t on);
int32_t mmt_profile_report(mmt_engine* e, char* buf, int64_t buf_len);

#ifdef __cplusplus
}
#endif
#endif /* MMT_B200_H */
