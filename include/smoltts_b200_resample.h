/*
 * smoltts_b200 — C ABI of the sample-rate converter: PCM at one rate in, PCM at another out, for whole clips and for streams
 * fed a chunk at a time.  Same library (libsmoltts_b200.so) and conventions as smoltts_b200_mimi.h: plain C types, every
 * pointer named d_* is a DEVICE pointer owned by the caller, every compute call is asynchronous on the given cudaStream_t
 * (passed as void*), no allocation after create, 0 / negative SMOL_ERR_* return codes with smol_last_error().
 *
 * The arithmetic is scipy.signal.resample_poly(x, up, down) with its defaults (padtype='constant'):
 *   g = gcd(rate_in, rate_out), up = rate_out / g, down = rate_in / g, m = max(up, down), hl = 10 m,
 *   h = up * firwin(2 hl + 1, 1 / m, window=('kaiser', 5.0))            (designed by the caller, passed to bind)
 *   a clip x of L samples (zero outside [0, L)) gives ceil(L up / down) samples
 *   y[k] = sum over j = (k down + hl) mod up, step up, of h[j] x[(k down + hl - j) / up]
 * Every output is one fp32 sum over its phase's taps in ascending j, whatever the chunking, the other streams of a call and the
 * slot: a stream's output is bit-identical however its input was cut into chunks, and equals the whole-clip result.
 */
#ifndef SMOLTTS_B200_RESAMPLE_H
#define SMOLTTS_B200_RESAMPLE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SMOL_RESAMPLE_MAX_RATIO 320   /* largest max(up, down) accepted */
#define SMOL_RESAMPLE_MAX_CALL 256    /* streams per smol_resample call */

typedef struct SmolResampleConfig {
    int32_t rate_in, rate_out;   /* Hz, both >= 1; max(up, down) <= SMOL_RESAMPLE_MAX_RATIO */
    int32_t max_streams;         /* state slots, 1 .. 65536 */
} SmolResampleConfig;

typedef struct SmolResampler SmolResampler;

/* Ratio and capacity checks only, pure host code.  A ratio above the limit is SMOL_ERR_UNSUPPORTED. */
int smol_resampler_create(const SmolResampleConfig* cfg, SmolResampler** out);
void smol_resampler_destroy(SmolResampler* r);
int32_t smol_resampler_taps(const SmolResampler* r);            /* 2 hl + 1: the length of the filter bind takes */
size_t smol_resampler_workspace_bytes(const SmolResampler* r);  /* polyphase taps + two history rows per slot */

/* d_taps: fp32 [smol_resampler_taps()] (h above, gain up included).  Packed [phase][tap] into the caller's workspace
 * (256-byte aligned) by a kernel on `stream`; nothing is borrowed.  Every slot is reset. */
int smol_resampler_bind(SmolResampler* r, const float* d_taps, void* d_workspace, size_t workspace_bytes, void* stream);

/* Back to the start of a stream (zero history: the left zero padding) for the n slots listed in h_slots (HOST int32). */
int smol_resampler_reset(SmolResampler* r, const int32_t* h_slots, int32_t n, void* stream);

/* One step of n streams: stream b takes the next h_lengths[b] >= 0 samples (HOST int64; d_in holds the chunks back to back) of
 * the stream in slot h_slots[b] (HOST int32, distinct) and emits every output whose filter support is now complete.  With
 * finish = 1 the input after the chunk is zero: the rest of the outputs are emitted, ceil(L up / down) in all for a stream of
 * L samples, and the slot is back at the start.  A whole clip is one call on a fresh slot with finish = 1.  d_out receives the
 * outputs back to back in the order of h_slots; h_out_counts (HOST int64[n], may be NULL) their numbers, which depend only on
 * the lengths so far:
 *   streaming: S up <= hl ? 0 : (S up - 1 - hl) / down + 1 outputs in all after S samples;  finish: ceil(L up / down).
 * Nothing is launched on an error. */
int smol_resample(SmolResampler* r, const float* d_in, const int64_t* h_lengths, const int32_t* h_slots, int32_t n, int32_t finish,
                  float* d_out, int64_t* h_out_counts, void* stream);

#ifdef __cplusplus
}
#endif
#endif
