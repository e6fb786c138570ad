// Sample-rate conversion for sm_100a: scipy.signal.resample_poly's polyphase FIR (include/smoltts_b200_resample.h), one
// kernel for whole clips and streams.
//
// Output k of a stream reads phase p = (k down + hl) mod up of the filter and the inputs n0 - i, n0 = (k down + hl) / up,
// for i = 0 .. K_p - 1 (K_p = ceil((M - p) / up) taps of that phase, tap i = h[p + i up]).  The taps are packed [phase][K] at
// bind (K = ceil(M / up)), so a phase's taps are contiguous.
//
// A stream's state is its last K input samples (its "history", zero after a reset: the left zero padding) and two counters the
// host keeps: samples consumed S and outputs emitted E(S).  An output is complete once n0 <= S - 1; a step that brings S to S'
// emits outputs E(S) .. E(S') - 1, whose inputs reach back at most to S - K + 1, i.e. into the history.  With finish the input
// past the chunk is zero and the outputs up to ceil(S' up / down) - 1 follow.
//
// Launch: grid (output tiles, streams).  A CTA stages all packed taps and the input window of its tile (history, chunk or the
// right zero padding) in shared memory and writes one output per thread, each one fp32 FMA chain in ascending tap order.
// Nothing depends on the chunking or on what shares the launch, so a stream's samples are the same bits whatever the calls
// were.  Each slot has two history rows used in turn: tile 0 of a stream writes the new history into the row the next call
// reads while every tile of this call reads the other one, so one launch does the whole step.  No atomics.

#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <numeric>
#include <string>
#include <vector>

#include "../../include/smoltts_b200.h"
#include "../../include/smoltts_b200_resample.h"

namespace smol {
int capi_fail(int code, const std::string& msg);   // capi.cu: sets smol_last_error()
int capi_cuda_fail(cudaError_t e, const char* what);

namespace resample {

constexpr int kThreads = 256;
constexpr int kMaxTile = 256;                        // outputs per CTA
constexpr size_t kSmemCap = 160 * 1024;              // dynamic shared memory of a CTA at most (taps + input window)

struct Job {
    long long base;      // samples of the stream consumed before this call
    long long k0;        // outputs of the stream emitted before this call
    long long in_off;    // first sample of its chunk in d_in
    long long out_off;   // first output in d_out
    int in_len, n_out, slot, parity;
};

struct Params {
    const float* taps;   // [up][K]
    float* hist;         // [slots][2][K]
    const float* in;
    float* out;
    int up, down, hl, M, K, tile, finish;
    Job job[SMOL_RESAMPLE_MAX_CALL];
};

__global__ void __launch_bounds__(kThreads) resample_kernel(const __grid_constant__ Params p) {
    extern __shared__ float sm[];
    const Job& j = p.job[blockIdx.y];
    const int K = p.K, tid = threadIdx.x;
    const float* h_old = p.hist + ((size_t)j.slot * 2 + j.parity) * K;
    if (blockIdx.x == 0) {   // the next call's history: the last K samples of base + in_len, or zeros after a finish
        float* h_new = p.hist + ((size_t)j.slot * 2 + (j.parity ^ 1)) * K;
        for (int i = tid; i < K; i += kThreads) {
            const long long idx = (long long)j.in_len - K + i;   // relative to base
            h_new[i] = p.finish ? 0.f : (idx >= 0 ? p.in[j.in_off + idx] : h_old[K + idx]);
        }
    }
    const int t0 = blockIdx.x * p.tile;
    if (t0 >= j.n_out) return;
    const int cnt = min(p.tile, j.n_out - t0);
    const long long k_first = j.k0 + t0;
    const long long lo = (k_first * p.down + p.hl) / p.up - K + 1;                  // first input of the window (absolute)
    const long long hi = ((k_first + cnt - 1) * p.down + p.hl) / p.up;             // last one
    const int n_taps = p.up * K;
    float* s_taps = sm;
    float* s_win = sm + n_taps;
    for (int i = tid; i < n_taps; i += kThreads) s_taps[i] = p.taps[i];
    const int wlen = (int)(hi - lo + 1);
    for (int w = tid; w < wlen; w += kThreads) {
        const long long idx = lo + w - j.base;                                     // >= -K + 1 by construction
        s_win[w] = idx < 0 ? h_old[K + idx] : (idx < j.in_len ? p.in[j.in_off + idx] : 0.f);
    }
    __syncthreads();
    for (int o = tid; o < cnt; o += kThreads) {
        const long long t = (k_first + o) * p.down + p.hl;
        const int ph = (int)(t % p.up);
        const int kp = (p.M - ph + p.up - 1) / p.up;
        const float* h = s_taps + ph * K;
        const float* x = s_win + (t / p.up - lo);
        float acc = 0.f;
        for (int i = 0; i < kp; ++i) acc = fmaf(h[i], x[-i], acc);
        p.out[j.out_off + t0 + o] = acc;
    }
}

__global__ void pack_taps_kernel(float* __restrict__ dst, const float* __restrict__ h, int M, int up, int K) {
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < up * K; e += gridDim.x * blockDim.x) {
        const int ph = e / K, i = e % K;
        const long long src = (long long)ph + (long long)i * up;
        dst[e] = src < M ? h[src] : 0.f;
    }
}

}  // namespace resample
}  // namespace smol

using namespace smol::resample;

struct SmolResampler {
    SmolResampleConfig cfg{};
    int up = 0, down = 0, hl = 0, M = 0, K = 0, tile = 0;
    size_t smem = 0, o_hist = 0, total = 0;
    unsigned char* ws = nullptr;
    bool bound = false;
    std::vector<long long> consumed, emitted;   // per slot
    std::vector<unsigned char> parity;          // per slot: the history row the next call reads
};

#define RS_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return smol::capi_cuda_fail(e__, #call); } while (0)

static long long emitted_after(const SmolResampler* r, long long S, bool finish) {
    const long long a = S * r->up;
    if (finish) return (a + r->down - 1) / r->down;
    return a <= r->hl ? 0 : (a - 1 - r->hl) / r->down + 1;
}

static size_t window_floats(int tile, int up, int down, int K) { return (size_t)(tile - 1) * down / up + 2 + K; }

extern "C" int smol_resampler_create(const SmolResampleConfig* cfg, SmolResampler** out) {
    using smol::capi_fail;
    if (!cfg || !out) return capi_fail(SMOL_ERR_INVALID, "smol_resampler_create: null argument");
    const SmolResampleConfig& c = *cfg;
    if (c.rate_in < 1 || c.rate_out < 1) return capi_fail(SMOL_ERR_INVALID, "smol_resampler_create: rates must be >= 1 Hz");
    if (c.max_streams < 1 || c.max_streams > 65536) return capi_fail(SMOL_ERR_INVALID, "smol_resampler_create: max_streams must be 1 .. 65536");
    const int g = std::gcd(c.rate_in, c.rate_out);
    const int up = c.rate_out / g, down = c.rate_in / g;
    if (std::max(up, down) > SMOL_RESAMPLE_MAX_RATIO)
        return capi_fail(SMOL_ERR_UNSUPPORTED, "smol_resampler_create: " + std::to_string(c.rate_in) + " -> " + std::to_string(c.rate_out) +
                                                   " Hz is " + std::to_string(up) + "/" + std::to_string(down) +
                                                   ", max(up, down) above the limit of 320");
    SmolResampler* r = new SmolResampler();
    r->cfg = c;
    r->up = up;
    r->down = down;
    r->hl = 10 * std::max(up, down);
    r->M = 2 * r->hl + 1;
    r->K = (r->M + up - 1) / up;
    r->tile = kMaxTile;
    while (r->tile > 32 && ((size_t)up * r->K + window_floats(r->tile, up, down, r->K)) * 4 > kSmemCap) r->tile /= 2;
    r->smem = ((size_t)up * r->K + window_floats(r->tile, up, down, r->K)) * 4;   // within kSmemCap for every ratio up to 320
    r->o_hist = ((size_t)up * r->K * 4 + 255) / 256 * 256;
    r->total = r->o_hist + (size_t)c.max_streams * 2 * r->K * 4;
    r->consumed.assign(c.max_streams, 0);
    r->emitted.assign(c.max_streams, 0);
    r->parity.assign(c.max_streams, 0);
    *out = r;
    return SMOL_OK;
}

extern "C" void smol_resampler_destroy(SmolResampler* r) { delete r; }
extern "C" int32_t smol_resampler_taps(const SmolResampler* r) { return r ? r->M : 0; }
extern "C" size_t smol_resampler_workspace_bytes(const SmolResampler* r) { return r ? r->total : 0; }

static int reset_slots(SmolResampler* r, const int32_t* slots, int32_t n, cudaStream_t st) {
    for (int b = 0; b < n; ++b) {
        const int s = slots[b];
        RS_CUDA(cudaMemsetAsync(r->ws + r->o_hist + (size_t)s * 2 * r->K * 4, 0, (size_t)2 * r->K * 4, st));
        r->consumed[s] = r->emitted[s] = 0;
        r->parity[s] = 0;
    }
    return SMOL_OK;
}

extern "C" int smol_resampler_bind(SmolResampler* r, const float* d_taps, void* d_workspace, size_t workspace_bytes, void* stream) {
    using smol::capi_fail;
    if (!r || !d_taps || !d_workspace) return capi_fail(SMOL_ERR_INVALID, "smol_resampler_bind: null argument");
    if (workspace_bytes < r->total) return capi_fail(SMOL_ERR_CAPACITY, "smol_resampler_bind: workspace smaller than smol_resampler_workspace_bytes()");
    if ((uintptr_t)d_workspace % 256) return capi_fail(SMOL_ERR_INVALID, "smol_resampler_bind: workspace must be 256-byte aligned");
    // the limit belongs to the kernel, not to this handle: every handle sets the same kSmemCap (>= any handle's smem), so a
    // bind never lowers what an earlier handle's launches need
    RS_CUDA(cudaFuncSetAttribute(resample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemCap));
    cudaStream_t st = (cudaStream_t)stream;
    r->ws = reinterpret_cast<unsigned char*>(d_workspace);
    pack_taps_kernel<<<64, 256, 0, st>>>(reinterpret_cast<float*>(r->ws), d_taps, r->M, r->up, r->K);
    RS_CUDA(cudaGetLastError());
    RS_CUDA(cudaMemsetAsync(r->ws + r->o_hist, 0, r->total - r->o_hist, st));
    std::fill(r->consumed.begin(), r->consumed.end(), 0);
    std::fill(r->emitted.begin(), r->emitted.end(), 0);
    std::fill(r->parity.begin(), r->parity.end(), 0);
    r->bound = true;
    return SMOL_OK;
}

static int check_slots(const SmolResampler* r, const int32_t* slots, int32_t n, int32_t max_n, const char* fn) {
    using smol::capi_fail;
    if (n < 1 || n > max_n) return capi_fail(SMOL_ERR_CAPACITY, std::string(fn) + ": n outside 1 .. " + std::to_string(max_n));
    std::vector<char> seen(r->cfg.max_streams, 0);
    for (int b = 0; b < n; ++b) {
        const int s = slots[b];
        if (s < 0 || s >= r->cfg.max_streams) return capi_fail(SMOL_ERR_INVALID, std::string(fn) + ": slot " + std::to_string(s) + " outside 0 .. max_streams - 1");
        if (seen[s]++) return capi_fail(SMOL_ERR_INVALID, std::string(fn) + ": slot " + std::to_string(s) + " listed twice");
    }
    return SMOL_OK;
}

extern "C" int smol_resampler_reset(SmolResampler* r, const int32_t* h_slots, int32_t n, void* stream) {
    using smol::capi_fail;
    if (!r || !h_slots) return capi_fail(SMOL_ERR_INVALID, "smol_resampler_reset: null argument");
    if (!r->bound) return capi_fail(SMOL_ERR_UNBOUND, "smol_resampler_reset: taps / workspace not bound");
    const int rc = check_slots(r, h_slots, n, r->cfg.max_streams, "smol_resampler_reset");
    if (rc != SMOL_OK) return rc;
    return reset_slots(r, h_slots, n, (cudaStream_t)stream);
}

extern "C" int smol_resample(SmolResampler* r, const float* d_in, const int64_t* h_lengths, const int32_t* h_slots, int32_t n, int32_t finish,
                             float* d_out, int64_t* h_out_counts, void* stream) {
    using smol::capi_fail;
    if (!r || !h_lengths || !h_slots) return capi_fail(SMOL_ERR_INVALID, "smol_resample: null argument");
    if (!r->bound) return capi_fail(SMOL_ERR_UNBOUND, "smol_resample: taps / workspace not bound");
    int rc = check_slots(r, h_slots, n, std::min(r->cfg.max_streams, SMOL_RESAMPLE_MAX_CALL), "smol_resample");
    if (rc != SMOL_OK) return rc;
    static thread_local Params p;   // 12 KB: kept off the stack
    long long in_off = 0, out_off = 0, max_out = 0;
    for (int b = 0; b < n; ++b) {
        if (h_lengths[b] < 0) return capi_fail(SMOL_ERR_INVALID, "smol_resample: stream " + std::to_string(b) + " has a negative length");
        const int s = h_slots[b];
        const long long S0 = r->consumed[s], S1 = S0 + h_lengths[b];
        if (h_lengths[b] > (1LL << 30) || S1 > (1LL << 52) / r->down)
            return capi_fail(SMOL_ERR_CAPACITY, "smol_resample: stream " + std::to_string(b) + " is too long");
        const long long n_out = emitted_after(r, S1, finish != 0) - r->emitted[s];
        if (n_out > (1LL << 30)) return capi_fail(SMOL_ERR_CAPACITY, "smol_resample: stream " + std::to_string(b) + " emits above 2^30 samples in one call");
        Job& j = p.job[b];
        j.base = S0;
        j.k0 = r->emitted[s];
        j.in_off = in_off;
        j.out_off = out_off;
        j.in_len = (int)h_lengths[b];
        j.n_out = (int)n_out;
        j.slot = s;
        j.parity = r->parity[s];
        in_off += h_lengths[b];
        out_off += n_out;
        max_out = std::max(max_out, n_out);
    }
    if ((in_off > 0 && !d_in) || (out_off > 0 && !d_out)) return capi_fail(SMOL_ERR_INVALID, "smol_resample: null d_in / d_out");
    p.taps = reinterpret_cast<const float*>(r->ws);
    p.hist = reinterpret_cast<float*>(r->ws + r->o_hist);
    p.in = d_in;
    p.out = d_out;
    p.up = r->up; p.down = r->down; p.hl = r->hl; p.M = r->M; p.K = r->K; p.tile = r->tile; p.finish = finish != 0;
    const dim3 grid((unsigned)std::max(1LL, (max_out + r->tile - 1) / r->tile), (unsigned)n);
    resample_kernel<<<grid, kThreads, r->smem, (cudaStream_t)stream>>>(p);
    RS_CUDA(cudaGetLastError());
    for (int b = 0; b < n; ++b) {
        const int s = h_slots[b];
        if (h_out_counts) h_out_counts[b] = p.job[b].n_out;
        r->parity[s] ^= 1;
        if (finish) { r->consumed[s] = r->emitted[s] = 0; }
        else { r->consumed[s] += h_lengths[b]; r->emitted[s] += p.job[b].n_out; }
    }
    return SMOL_OK;
}
