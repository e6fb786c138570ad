/*
 * smoltts_b200 — C ABI of the B200-native Mimi streaming decoder (codes -> PCM), the step AFTER the DualAR decode
 * step (SURVEY §8(f)-2), and of the Mimi encoder (PCM -> codes) that builds voice-clone prompts from audio.  Same
 * library (libsmoltts_b200.so) and conventions as smoltts_b200.h: plain C types, every pointer inside the structs / named d_* is a DEVICE pointer owned by the caller, every compute call is asynchronous
 * on the given cudaStream_t (passed as void*), no allocation after create, 0 / negative SMOL_ERR_* return codes with
 * smol_last_error().
 *
 * The reference has no FFI; each entry point cites the Python it replaces, paths relative to
 * mlx_inference/src/smoltts_mlx/ of the reference checkout (C = codec/).  All weights are fp32 in the layouts of
 * kyutai/mimi's model.safetensors (torch: Conv1d [out, in, k], ConvTranspose1d [in, out, k]) -- the file load_mimi()
 * reads (C/mimi.py:107-156).
 */
#ifndef SMOLTTS_B200_MIMI_H
#define SMOLTTS_B200_MIMI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMOL_MIMI_MAX_LAYERS 16
#define SMOL_MIMI_MAX_RATIOS 8
#define SMOL_MIMI_MAX_Q 32

/* MimiConfig = SeanetConfig (C/conv.py:8-22) + MimiTransformerConfig (C/transformer.py:10-33) + RVQConfig (C/rvq.py:7-13),
 * plus the capacities of this engine. */
typedef struct SmolMimiConfig {
    int32_t n_q;               /* codebooks per frame actually decoded: 1 semantic + (n_q - 1) acoustic */
    int32_t codebook_size, codebook_dim;
    int32_t dim;               /* seanet.dimension = transformer.d_model = rvq.hidden_dim (512) */
    int32_t n_layers, n_heads, head_dim, ffn;
    int32_t n_filters, n_ratios;
    int32_t ratios[SMOL_MIMI_MAX_RATIOS];
    int32_t kernel, res_kernel, last_kernel;
    int32_t max_streams;       /* concurrent streams (state slots) */
    int32_t max_positions;     /* transformer positions per stream = 2 x frames; rows of the RoPE table */
    int32_t window;            /* 0: attend to the whole history, as the reference's KVCache does (__init__.py:86);
                                  n > 0: kyutai's sliding window of n positions (transformer.context, unused by the reference) */
    int32_t upsample_carry;    /* 0: decode_step's rule -- every frame upsampled alone (C/mimi.py:73-86, C/conv.py:271-282);
                                  1: carry the transposed convolution's trailing taps: a run of steps == decode() of the sequence */
    int32_t use_graph;         /* 1: a step's launches are captured once per (batch, pointers) and replayed as a CUDA graph;
                                  0: plain launches (programmatic dependent launch), e.g. inside the caller's own capture */
    float norm_eps, codebook_eps;
} SmolMimiConfig;

/* decoder_transformer.layers.{l}.* (C/transformer.py:36-130) */
typedef struct SmolMimiLayerWeights {
    const float *q_proj, *k_proj, *v_proj, *o_proj;   /* self_attn.*.weight [dim, dim] */
    const float *fc1, *fc2;                           /* mlp.fc1.weight [ffn, dim], mlp.fc2.weight [dim, ffn] */
    const float *ln1_w, *ln1_b, *ln2_w, *ln2_b;       /* input_layernorm / post_attention_layernorm */
    const float *scale_attn, *scale_mlp;              /* self_attn_layer_scale.scale, mlp_layer_scale.scale [dim] */
} SmolMimiLayerWeights;

typedef struct SmolMimiConv {
    const float* weight;
    const float* bias;
} SmolMimiConv;

typedef struct SmolMimiWeights {
    /* quantizer.{semantic,acoustic}_residual_vector_quantizer.layers.{i}.codebook.* : index 0 = the semantic codebook,
     * 1 .. n_q-1 = acoustic codebooks 0 .. n_q-2 (C/rvq.py:27-45) */
    const float* embed_sum[SMOL_MIMI_MAX_Q];       /* [codebook_size, codebook_dim] */
    const float* cluster_usage[SMOL_MIMI_MAX_Q];   /* [codebook_size] */
    const float* semantic_output_proj;             /* ...output_proj.weight [dim, codebook_dim, 1] (C/rvq.py:95-97) */
    const float* acoustic_output_proj;
    const float* upsample;                         /* upsample.conv.weight [dim, 1, 4] (C/mimi.py:46-55) */
    SmolMimiLayerWeights layers[SMOL_MIMI_MAX_LAYERS];
    SmolMimiConv conv_in;                          /* decoder.layers.0 (C/seanet.py:107-112) */
    SmolMimiConv convtr[SMOL_MIMI_MAX_RATIOS];     /* decoder.layers.{2 + 3 i}: ConvTranspose1d (C/seanet.py:117-125) */
    SmolMimiConv res_conv1[SMOL_MIMI_MAX_RATIOS];  /* decoder.layers.{3 + 3 i}.block.1 (C/seanet.py:9-27) */
    SmolMimiConv res_conv2[SMOL_MIMI_MAX_RATIOS];  /* decoder.layers.{3 + 3 i}.block.3 */
    SmolMimiConv conv_out;                         /* decoder.layers.{2 + 3 n_ratios} (C/seanet.py:134-139) */
    const float* rope;                             /* [max_positions][head_dim]: cos (first half) | sin of pos * theta^(-2i/hd) */
} SmolMimiWeights;

typedef struct SmolMimi SmolMimi;

/* MimiModel.__init__ (C/mimi.py:32-62), decode half: shape checks only, pure host code. */
int smol_mimi_create(const SmolMimiConfig* cfg, SmolMimi** out);
void smol_mimi_destroy(SmolMimi* m);
int32_t smol_mimi_samples_per_frame(const SmolMimi* m);   /* 2 x prod(ratios) = 1920 */
size_t smol_mimi_workspace_bytes(const SmolMimi* m);

/* load_mimi() (C/mimi.py:107-156): borrows nothing -- every weight is repacked into the caller's workspace (GEMV rows,
 * normalised codebooks, fused q|k|v) by kernels on `stream`; all stream slots are reset. */
int smol_mimi_bind(SmolMimi* m, const SmolMimiWeights* w, void* d_workspace, size_t workspace_bytes, void* stream);

/* make_prompt_cache(codec.decoder_transformer) + MimiDecoder.reset() (__init__.py:86, C/seanet.py:156-161): back to the
 * start of a stream for the n slots listed in d_slots (device int32; NULL = slots 0 .. n-1). */
int smol_mimi_reset(SmolMimi* m, const int32_t* d_slots, int32_t n, void* stream);

/* MimiModel.decode_step(codes, cache) (C/mimi.py:102-104) for `batch` streams at once: d_codes int32 [batch][n_q]
 * (row b: the frame's codes of the stream in slot d_slots[b], NULL = slot b), d_pcm fp32 [batch][samples_per_frame]. */
int smol_mimi_decode_step(SmolMimi* m, const int32_t* d_codes, const int32_t* d_slots, int32_t batch, float* d_pcm,
                          void* stream);

/* Test / profiling hooks: intermediate buffers by name ("emb": upsampled embeddings, "xf": transformer output; slot-major),
 * kernel launches per step, device-side error word (nonzero: a stream ran past max_positions). */
void* smol_mimi_debug_buffer(SmolMimi* m, const char* name, int64_t* slot_stride_floats);
int32_t smol_mimi_launches_per_step(const SmolMimi* m);
int32_t* smol_mimi_error_word(SmolMimi* m);

/* ---- the encode half: PCM -> codes (MimiModel.encode of transformers' MimiModel, which the reference's codec mirrors) ----
 *
 * A separate handle: a decode-only engine allocates nothing for it.  Whole clips, not a stream: every call encodes n clips
 * (24 kHz mono fp32, concatenated) from their first sample, each exactly as if it were alone -- same kernels, same
 * summation orders whatever shares the call.  All fp32. */
typedef struct SmolMimiEncoderConfig {
    int32_t n_q;               /* codebooks per frame produced: 1 semantic + (n_q - 1) acoustic */
    int32_t codebook_size, codebook_dim;
    int32_t dim;               /* seanet.dimension = transformer.d_model = rvq.hidden_dim (512) */
    int32_t n_layers, n_heads, head_dim, ffn;
    int32_t n_filters, n_ratios;
    int32_t ratios[SMOL_MIMI_MAX_RATIOS];   /* as the decoder lists them (8, 6, 5, 4); the encoder applies them in reverse */
    int32_t kernel, res_kernel, last_kernel;
    int32_t max_clips;         /* clips per call, 1 .. 256 */
    int32_t max_samples;       /* total samples per call (all clips) */
    int32_t window;            /* the encoder transformer's causal sliding window: query i sees keys i - window < j <= i (250) */
    float norm_eps, codebook_eps;
} SmolMimiEncoderConfig;

typedef struct SmolMimiEncoderWeights {
    /* codebooks as in SmolMimiWeights: index 0 = semantic, 1 .. n_q-1 = acoustic 0 .. n_q-2 */
    const float* embed_sum[SMOL_MIMI_MAX_Q];       /* [codebook_size, codebook_dim] */
    const float* cluster_usage[SMOL_MIMI_MAX_Q];   /* [codebook_size] */
    const float* semantic_input_proj;              /* quantizer.semantic_residual_vector_quantizer.input_proj.weight [codebook_dim, dim, 1] */
    const float* acoustic_input_proj;              /* quantizer.acoustic_residual_vector_quantizer.input_proj.weight */
    const float* downsample;                       /* downsample.conv.weight [dim, dim, 4] (stride 2, replicate padding, no bias) */
    SmolMimiLayerWeights layers[SMOL_MIMI_MAX_LAYERS];   /* encoder_transformer.layers.{l}.* */
    SmolMimiConv conv_in;                          /* encoder.layers.0 [n_filters, 1, kernel] */
    SmolMimiConv res_conv1[SMOL_MIMI_MAX_RATIOS];  /* stage i (ratio ratios[n_ratios - 1 - i]): encoder.layers.{1 + 3 i}.block.1 */
    SmolMimiConv res_conv2[SMOL_MIMI_MAX_RATIOS];  /* encoder.layers.{1 + 3 i}.block.3 */
    SmolMimiConv conv_down[SMOL_MIMI_MAX_RATIOS];  /* encoder.layers.{3 + 3 i}: kernel 2 r, stride r, C -> 2 C */
    SmolMimiConv conv_out;                         /* encoder.layers.{2 + 3 n_ratios} [dim, n_filters 2^n_ratios, last_kernel] */
    const float* rope;                             /* [ceil(max_samples / prod(ratios))][head_dim]: cos | sin, as SmolMimiWeights.rope */
} SmolMimiEncoderWeights;

typedef struct SmolMimiEncoder SmolMimiEncoder;

/* Shape and capacity checks only, pure host code. */
int smol_mimi_encoder_create(const SmolMimiEncoderConfig* cfg, SmolMimiEncoder** out);
void smol_mimi_encoder_destroy(SmolMimiEncoder* e);
int32_t smol_mimi_encoder_samples_per_frame(const SmolMimiEncoder* e);   /* 2 x prod(ratios) = 1920: a clip of L samples gives ceil(L / 1920) frames */
size_t smol_mimi_encoder_workspace_bytes(const SmolMimiEncoder* e);      /* grows with max_samples */

/* Every weight is repacked into the caller's workspace (256-byte aligned) by kernels on `stream`; nothing is borrowed. */
int smol_mimi_encoder_bind(SmolMimiEncoder* e, const SmolMimiEncoderWeights* w, void* d_workspace, size_t workspace_bytes,
                           void* stream);

/* MimiModel.encode of n clips: d_pcm fp32, the clips back to back (h_lengths: HOST int64[n], every length >= 1, sum <=
 * max_samples); d_codes int32 [sum_b ceil(L_b / 1920)][n_q], the frames of clip 0 first.  SMOL_ERR_CAPACITY over capacity,
 * SMOL_ERR_INVALID for a zero-length clip; nothing is launched then. */
int smol_mimi_encode(SmolMimiEncoder* e, const float* d_pcm, const int64_t* h_lengths, int32_t n, int32_t* d_codes, void* stream);

/* Test / profiling hook: "latent" = the pre-quantizer latent z of the last call, fp32 [sum_b T_b][dim]. */
void* smol_mimi_encoder_debug_buffer(SmolMimiEncoder* e, const char* name);
int32_t smol_mimi_encoder_launches(const SmolMimiEncoder* e);   /* kernel launches of the last call */

#ifdef __cplusplus
}
#endif
#endif
