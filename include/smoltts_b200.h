/*
 * smoltts_b200 — C ABI of the B200-native DualAR / RQ-Transformer decode step.
 *
 * The reference (EndlessReform/smoltts) is pure Python and has no FFI; this header
 * is the boundary a maintainer would bind instead of the Python functions cited on
 * each entry point (paths relative to the reference checkout;  P = modeling/model/
 * rq_transformer.py,  M = mlx_inference/src/smoltts_mlx/lm/rq_transformer.py,
 * G = mlx_inference/src/smoltts_mlx/lm/generate.py,  K = .../lm/cache.py).
 * INTEGRATION.md shows the ctypes stub.
 *
 * Conventions
 *  - plain C types only; every pointer named d_* / inside the structs below is a
 *    DEVICE pointer owned by the caller and must outlive the model;
 *  - every compute call is asynchronous on the given cudaStream_t (passed as
 *    void*), never synchronises the device, never allocates: graph-capturable;
 *  - returns 0 on success, a negative SMOL_ERR_* otherwise; smol_last_error()
 *    gives a thread-local message;
 *  - one SmolModel per device; calls on one model are serialised by the caller.
 */
#ifndef SMOLTTS_B200_H
#define SMOLTTS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMOL_ABI_VERSION 2
#define SMOL_MAX_LAYERS 64
#define SMOL_MAX_FAST_LAYERS 16

enum {
    SMOL_OK = 0,
    SMOL_ERR_INVALID = -1,     /* bad argument / unsupported shape */
    SMOL_ERR_UNBOUND = -2,     /* weights / workspace / KV pool not bound yet */
    SMOL_ERR_CUDA = -3,        /* a CUDA runtime call failed (message has the reason) */
    SMOL_ERR_UNSUPPORTED = -4, /* config feature outside the decode path built so far */
    SMOL_ERR_CAPACITY = -5     /* batch / context exceeds what was configured */
};

/* Model shape: RQTransformerModelArgs (P:25-114; M:10-48) + token ids (TokenConfig M:51-89). */
typedef struct SmolConfig {
    int32_t dim, n_layer, n_head, n_local_heads, head_dim, intermediate_size, vocab_size;
    int32_t fast_dim, n_fast_layer, fast_n_head, fast_n_local_heads, fast_head_dim, fast_intermediate_size;
    int32_t codebook_size, num_codebooks;
    int32_t duplicate_code_0, depthwise_wte, depthwise_output, tie_word_embeddings;
    int32_t max_seq_len;       /* rows of the RoPE table / max cached positions per sequence */
    int32_t max_batch;         /* sequences per decode call */
    int32_t page_size;         /* KV page, positions (16 or 32) */
    int32_t semantic_start_id, semantic_end_id, im_end_id;
    int32_t mlx_embed_mask;    /* 0: PyTorch rule P:219 (default);  1: MLX rule M:162-169 */
    float norm_eps;
} SmolConfig;

/* One transformer block's parameters: state-dict keys `{layers|fast_layers}.{l}.*` (SURVEY §8(b)). All bf16. */
typedef struct SmolLayerWeights {
    const void* wqkv;           /* attention.wqkv.weight   [(H+2Hkv)*64, D]  rows q|k|v */
    const void* wo;             /* attention.wo.weight     [D, D] */
    const void* w1;             /* feed_forward.w1.weight  [F, D] */
    const void* w3;             /* feed_forward.w3.weight  [F, D] */
    const void* w2;             /* feed_forward.w2.weight  [D, F] */
    const void* attention_norm; /* [D] */
    const void* ffn_norm;       /* [D] */
} SmolLayerWeights;

/* Checkpoint tensors in the layout of train/convert_safetensors.py:6-16 plus the two
 * non-persistent RoPE buffers the loader rebuilds (P:180-188,389-397). All bf16. */
typedef struct SmolWeights {
    const void* embeddings;          /* [V, D] (also the tied LM head, P:252-253) */
    const void* codebook_embeddings; /* [N*C, D] */
    const void* norm;                /* [D] */
    const void* output;              /* [V, D] or NULL when tie_word_embeddings */
    const void* fast_embeddings;     /* [(N-1)*C, Df] (depthwise_wte) or [C, Df] */
    const void* fast_norm;           /* [Df] */
    const void* fast_output;         /* flattened [(i*C + k), Df] (M:212-217) or [C, Df] */
    const void* rope;                /* [max_seq_len, 32, 2] (cos,sin) rounded to bf16 (P:616-624) */
    const void* fast_rope;           /* [depth, 32, 2] */
    SmolLayerWeights layers[SMOL_MAX_LAYERS];
    SmolLayerWeights fast_layers[SMOL_MAX_FAST_LAYERS];
} SmolWeights;

/* One sequence's sampling parameters (SmolBatch.row_sampling): the fields of SmolSampling below that may differ
 * between the rows of one call.  temp == 0 -> argmax slow id, fast_temp == 0 -> argmax depth codes.  32 bytes. */
typedef struct SmolRowSampling {
    float temp, fast_temp;
    int32_t top_k;       /* slow token only; 0 = off */
    float top_p;         /* slow token only; >= 1 = off */
    float min_p;         /* "intended" min-p; 0 = off */
    uint32_t pad;
    uint64_t seed;
} SmolRowSampling;

/* Per-batch device state (the reference keeps these in Python: G:25-57, K:6-22). */
typedef struct SmolBatch {
    int32_t* tokens;        /* [B, R] current input column: row 0 vocab id, rows 1.. depth codes (G:143-145) */
    int32_t* seq_len;       /* [B] cached positions (KVCache.offset, K:10,21) */
    const int32_t* block_table; /* [B, max_pages] page ids into the KV pool */
    int32_t max_pages;
    uint8_t* finished;      /* [B] 1 once <|im_end|> was emitted under audio_only (G:162-166) */
    const int32_t* seq_id;  /* [B] global utterance id: RNG counter word, independent of sharding */
    int32_t* step;          /* [B] frames emitted so far (RNG counter word, index into out_codes) */
    int32_t* out_codes;     /* [B, max_frames, R] every emitted column, or NULL */
    int32_t max_frames;
    const SmolRowSampling* row_sampling; /* [B] device, or NULL: every row samples with the call's SmolSampling.  When set,
                                            row b samples with row_sampling[b] and the call's SmolSampling supplies only
                                            audio_only / ignore_stop.  Read by every launch that samples, never written:
                                            new contents between calls need no other change (no graph recapture).
                                            Forced ids (smol_set_force) still win. */
} SmolBatch;

/* GenerationSettings (G:12-16) + the north-star's top-k / top-p / seed. temp == 0 -> argmax. */
typedef struct SmolSampling {
    float temp;          /* slow token temperature (default_temp) */
    float fast_temp;     /* depth-code temperature (default_fast_temp; 0 -> argmax) */
    int32_t top_k;       /* slow token only; 0 = off */
    float top_p;         /* slow token only; >= 1 = off */
    float min_p;         /* "intended" min-p; 0 = off (the reference's min-p is a no-op, samplers.py:24-28) */
    uint64_t seed;
    int32_t audio_only;  /* stop rule G:162-166 */
    int32_t ignore_stop; /* benchmarks: never set finished */
} SmolSampling;

typedef struct SmolModel SmolModel;

int smol_abi_version(void);
const char* smol_last_error(void);

/* RQTransformer.__init__ (P:332-399 / M:92-148): shape checks, no device allocation. */
int smol_create(const SmolConfig* cfg, SmolModel** out);
void smol_destroy(SmolModel* m);

/* load_weights / load_state_dict (P:316; mlx __init__.py:49): borrow caller-owned tensors. */
int smol_bind_weights(SmolModel* m, const SmolWeights* w);

/* Activation workspace the caller allocates once (the reference allocates per op). */
size_t smol_workspace_bytes(const SmolModel* m);
int smol_bind_workspace(SmolModel* m, void* d_workspace, size_t bytes);

/* make_prompt_cache (K:25-33): paged pool replaces the grow-by-concat KVCache (K:12-22).
 * Pool layout: [n_pages][n_layer][2][n_local_heads][page_size][64] bf16. */
size_t smol_kv_page_bytes(const SmolModel* m);
int smol_kv_bind(SmolModel* m, void* d_kv_pool, int32_t n_pages);

/* Prefill (first next() of SingleBatchGenerator, G:66-73 with S > 1): pushes prompt
 * columns [0, len-1) of every sequence through the slow transformer into the KV pool,
 * leaves seq_len = len-1 and tokens = last prompt column so that the first
 * smol_decode_frame reproduces the reference's first sampled frame.
 * d_prompt [B, R, s_max] int32, d_prompt_len [B]. */
int smol_prefill(SmolModel* m, const SmolBatch* b, int32_t batch, const int32_t* d_prompt,
                 const int32_t* d_prompt_len, int32_t s_max, void* stream);

/* forward_generate with S == 1 (M:173-192): embed(tokens) -> slow layers (KV append at
 * seq_len) -> norm -> LM head.  Writes fp32 token logits [B, V] (bf16-rounded values) and
 * leaves the pre-norm hidden state [B, D] bf16 in the stream buffer.  advance != 0 also
 * increments seq_len. */
int smol_slow_step(SmolModel* m, const SmolBatch* b, int32_t batch, int32_t advance, void* stream);

/* forward_generate_fast (M:194-220): one depth step at position depth_pos; writes fp32 codebook
 * logits [B, C] into depth_logits[:, depth_pos].  Input of the step: from_xf == 0 -> the slow
 * hidden state (depth_pos 0) or the embedding of the code stored by smol_fast_embed for
 * depth_pos-1 (G:136-140);  from_xf != 0 -> whatever the caller put in the "xf" buffer
 * (the MLX signature passes x explicitly). */
int smol_fast_step(SmolModel* m, const SmolBatch* b, int32_t batch, int32_t depth_pos, int32_t from_xf,
                   void* stream);

/* fast_embeddings lookup feeding the next depth step (G:136-140): d_codes [B] int32. */
int smol_fast_embed(SmolModel* m, int32_t batch, const int32_t* d_codes, int32_t depth_pos, void* stream);

/* Sampling on caller-provided logits (G:88-99,118-132): d_logits [B, n] fp32 -> d_out [B]. stream_id:
 * 0 = slow token, 1+i = depth code i (RNG counter word).  b may be NULL; b->row_sampling, when set, replaces s per row. */
int smol_sample(SmolModel* m, const SmolBatch* b, int32_t batch, const float* d_logits, int32_t n,
                const SmolSampling* s, int32_t stream_id, int32_t* d_out, void* stream);

/* One whole frame for B sequences = one SingleBatchGenerator.__next__ (G:59-171) per
 * sequence: slow step, slow sample, depth loop with sampling, frame assembly, stop rule. */
int smol_decode_frame(SmolModel* m, const SmolBatch* b, int32_t batch, const SmolSampling* s, void* stream);

/* The loop of generate_blocking (G:200-205) without host round trips.  mode 2 / 0: ONE persistent
 * launch walks n_frames frames;  mode 1: the frame's per-phase launches are captured in a CUDA
 * graph (re-captured when batch / sampling / state pointers change) and replayed n_frames times. */
int smol_decode_frames(SmolModel* m, const SmolBatch* b, int32_t batch, const SmolSampling* s,
                       int32_t n_frames, void* stream);

/* Teacher forcing / greedy-with-resync: d_force [B, R] int32 ids that replace the sampled ones
 * after their logits were produced (NULL switches it off).  Borrowed pointer. */
int smol_set_force(SmolModel* m, const int32_t* d_force);

/* Runs phases [phase_begin, phase_end) of one frame's program (see smol_phase_count and DESIGN.md
 * "Phase program") - op-level parity tests and per-phase profiling. */
int smol_run_phases(SmolModel* m, const SmolBatch* b, int32_t batch, const SmolSampling* s,
                    int32_t phase_begin, int32_t phase_end, void* stream);
int32_t smol_phase_count(const SmolModel* m);

/* Per-phase timing (profiling aid): d_phase_ns [2 * 512 + 64] uint64 accumulators, zeroed by the
 * caller; CTA 0 adds [2p] = ns it spent inside phase p and [2p+1] = ns it then waited at the grid
 * barrier; [1024 + 4 * (kind + 8 * fast) + s] = ns in segment s (prologue, weight-stage wait,
 * GEMV + epilogue, closing block barrier) of the weight phases.  NULL switches it off. */
int smol_set_profile(SmolModel* m, uint64_t* d_phase_ns);

/* Per-frame clock (the "p50 per-frame latency at bs=1" of BASELINE.json): d_frame_ns [capacity] uint64; after frame f of
 * sequence 0 (f = its SmolBatch.step before the frame) the kernel stores %globaltimer (ns) in d_frame_ns[f].  Differences
 * of consecutive entries are per-frame latencies measured on the device.  NULL switches it off. */
int smol_set_frame_clock(SmolModel* m, uint64_t* d_frame_ns, int32_t capacity);

/* Options: "mode" 2 (default) = data-flow persistent kernel (flag-carrying activation words, TMA
 * producer warp; whole frames at batch 1, larger batches fall back to mode 0),
 * 0 = persistent cooperative kernel with a grid barrier per phase, 1 = one launch per phase, a frame
 * captured in a CUDA graph;  "n_ctas" = grid size (default: one CTA per SM);  "ll_flags" = A/B switches of the
 * data-flow kernel used by tools/ll_ncu.py (0 = the shipped configuration);
 * "tc_min_batch" (default 9: the measured crossover) = rows (sequences of a decode call, sequences x prompt positions of a prefill iteration)
 * from which the tcgen05 variant runs, 0 = never;  "prefill_tile" = cap on the prompt positions per prefill iteration
 * (0 = as many as fit: 128 rows on the tensor-core variant, 8 on the CUDA-core variants).
 * smol_get_option also answers "n_sms", "smem_bytes", "ll_ready", "tc_ready" (1 once the tcgen05 variant has been set up). */
int smol_set_option(SmolModel* m, const char* name, int64_t value);
int64_t smol_get_option(const SmolModel* m, const char* name);

/* Introspection for parity tests and benchmarks. name: "x" (slow stream [B,D] bf16), "h" [B,D] bf16,
 * "xf" (fast stream [B,Df] bf16), "q" [B,H*64] bf16, "attn" [B,D] bf16, "act" [B,F] bf16, "fkv"
 * [B,Lf,2,depth,Hkv*64] bf16, "token_logits" [B,V] f32, "depth_logits" [B,Nf,C] f32,
 * "frame_tokens" [B,R] i32. Returns NULL if unknown. */
void* smol_debug_buffer(SmolModel* m, const char* name);
/* Kernel launches issued for one frame in the current mode (mode 0: one launch covers all the
 * frames of a call). */
int32_t smol_launches_per_frame(const SmolModel* m);
/* Total kernel launches issued by this model so far. */
int64_t smol_launch_count(const SmolModel* m);

#ifdef __cplusplus
}
#endif
#endif /* SMOLTTS_B200_H */
