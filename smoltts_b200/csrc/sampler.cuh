// Fused temperature / top-k / top-p / min-p sampling with a counter-based RNG (Philox4x32-10).
//
// Replaces the reference's host-synchronous sampling (mlx lm/generate.py:88-99,118-132 and
// lm/utils/samplers.py:7-34).  The algorithm is the integer-weight specification restated on the
// CPU in oracle/sampler_oracle.py; after exp_det_weight() everything is exact integer arithmetic,
// so the chosen id is bit-identical to the oracle's for identical logits and counters.
//
// One CTA (kThreads threads) samples one row held in shared memory.
#pragma once

#include "common.cuh"
#include "dev_model.h"

// Block barrier over the kThreads sampling threads.  The data-flow kernel (ll2_kernel.cu) runs an extra
// producer warp next to them and substitutes a named barrier.
#ifndef SMOL_BLOCK_SYNC
#define SMOL_BLOCK_SYNC() __syncthreads()
#endif

namespace smol {

constexpr int kSampleMaxPerThread = 8;  // rows up to kThreads * 8 = 4096 entries

struct SampleScratch {
    unsigned long long u64[kWarps];
    float f32[kWarps];
    int i32[kWarps];
    unsigned long long bcast_u64;
    float bcast_f32;
    int bcast_i32;
};

template <int NT>
__device__ __forceinline__ unsigned long long block_sum_u64(unsigned long long v, SampleScratch& sc) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    SMOL_BLOCK_SYNC();
    if (lane == 0) sc.u64[warp] = v;
    SMOL_BLOCK_SYNC();
    unsigned long long t = 0;
#pragma unroll
    for (int w = 0; w < (NT / 32); ++w) t += sc.u64[w];
    return t;
}

template <int NT>
__device__ __forceinline__ float block_max_f32(float v, SampleScratch& sc) {
    v = warp_max(v);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    SMOL_BLOCK_SYNC();
    if (lane == 0) sc.f32[warp] = v;
    SMOL_BLOCK_SYNC();
    float t = sc.f32[0];
#pragma unroll
    for (int w = 1; w < (NT / 32); ++w) t = fmaxf(t, sc.f32[w]);
    return t;
}

// First index of the maximum (torch / mx argmax tie rule).  lg in shared memory.
template <int NT>
__device__ __forceinline__ int block_argmax(const float* lg, int n, SampleScratch& sc) {
    const int per = (n + NT - 1) / NT;
    const int i0 = threadIdx.x * per;
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int e = 0; e < per; ++e) {
        const int i = i0 + e;
        if (i < n) {
            const float v = lg[i];
            if (v > bv || bi == 0x7fffffff) { bv = v; bi = i; }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (oi != 0x7fffffff && (bi == 0x7fffffff || ov > bv || (ov == bv && oi < bi))) { bv = ov; bi = oi; }
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    SMOL_BLOCK_SYNC();
    if (lane == 0) { sc.f32[warp] = bv; sc.i32[warp] = bi; }
    SMOL_BLOCK_SYNC();
    float tv = sc.f32[0];
    int ti = sc.i32[0];
#pragma unroll
    for (int w = 1; w < (NT / 32); ++w) {
        const float ov = sc.f32[w];
        const int oi = sc.i32[w];
        if (oi != 0x7fffffff && (ti == 0x7fffffff || ov > tv || (ov == tv && oi < ti))) { tv = ov; ti = oi; }
    }
    return ti;
}

// All NT threads call this.  lg: shared memory, n <= NT * kSampleMaxPerThread (template parameter: entries per thread).
template <int NT, int kSampleMaxPerThread = smol::kSampleMaxPerThread>
static __device__ __forceinline__ int sample_row(const float* lg, int n, float temp, int top_k, float top_p, float min_p,
                          unsigned long long seed, uint32_t step, uint32_t seq_id, uint32_t stream,
                          SampleScratch& sc) {
    if (temp == 0.0f) return block_argmax<NT>(lg, n, sc);

    const int per = (n + NT - 1) / NT;
    const int i0 = threadIdx.x * per;
    const float inv_temp = __fdiv_rn(1.0f, temp);

    float z[kSampleMaxPerThread];
    float zmax = -INFINITY;
#pragma unroll
    for (int e = 0; e < kSampleMaxPerThread; ++e) {
        const int i = i0 + e;
        z[e] = -INFINITY;
        if (e < per && i < n) {
            z[e] = __fmul_rn(lg[i], inv_temp);
            zmax = fmaxf(zmax, z[e]);
        }
    }
    zmax = block_max_f32<NT>(zmax, sc);

    uint32_t w[kSampleMaxPerThread];
    bool keep[kSampleMaxPerThread];
#pragma unroll
    for (int e = 0; e < kSampleMaxPerThread; ++e) {
        const int i = i0 + e;
        const bool valid = (e < per && i < n);
        w[e] = valid ? exp_det_weight(__fsub_rn(z[e], zmax)) : 0u;
        keep[e] = valid;
    }

    if (top_k > 0 && top_k < n) {
        // k-th largest weight = max t with count(w >= t) >= k
        uint32_t lo = 0u, hi = (1u << 30) + 1u;
        while (hi - lo > 1u) {
            const uint32_t mid = lo + ((hi - lo) >> 1);
            unsigned long long c = 0;
#pragma unroll
            for (int e = 0; e < kSampleMaxPerThread; ++e) c += (keep[e] && w[e] >= mid) ? 1ull : 0ull;
            c = block_sum_u64<NT>(c, sc);
            if (c >= (unsigned long long)top_k) lo = mid; else hi = mid;
        }
#pragma unroll
        for (int e = 0; e < kSampleMaxPerThread; ++e) keep[e] = keep[e] && (w[e] >= lo);
    }

    if (top_p < 1.0f) {
        double pd = (double)top_p * 4294967296.0;
        if (pd < 0.0) pd = 0.0;
        const unsigned long long p32 = pd >= 4294967295.0 ? 4294967295ull : (unsigned long long)pd;
        unsigned long long tsum = 0;
#pragma unroll
        for (int e = 0; e < kSampleMaxPerThread; ++e) tsum += keep[e] ? (unsigned long long)w[e] : 0ull;
        tsum = block_sum_u64<NT>(tsum, sc);
        // need = max(1, (T * P32) >> 32) with a 96-bit product
        const unsigned long long hi64 = __umul64hi(tsum, p32), lo64 = tsum * p32;
        unsigned long long need = (hi64 << 32) | (lo64 >> 32);
        if (need < 1ull) need = 1ull;
        uint32_t lo = 0u, hi = (1u << 30) + 1u;
        while (hi - lo > 1u) {
            const uint32_t mid = lo + ((hi - lo) >> 1);
            unsigned long long s = 0;
#pragma unroll
            for (int e = 0; e < kSampleMaxPerThread; ++e) s += (keep[e] && w[e] >= mid) ? (unsigned long long)w[e] : 0ull;
            s = block_sum_u64<NT>(s, sc);
            if (s >= need) lo = mid; else hi = mid;
        }
#pragma unroll
        for (int e = 0; e < kSampleMaxPerThread; ++e) keep[e] = keep[e] && (w[e] >= lo);
    }

    if (min_p > 0.0f) {
        const uint32_t thr = __float2uint_rz(__fmul_rn(min_p, 1073741824.0f));
#pragma unroll
        for (int e = 0; e < kSampleMaxPerThread; ++e) keep[e] = keep[e] && (w[e] >= thr);
    }

    // draw: first index (in index order) whose inclusive running sum of kept weights exceeds target
    unsigned long long mine = 0;
#pragma unroll
    for (int e = 0; e < kSampleMaxPerThread; ++e) mine += keep[e] ? (unsigned long long)w[e] : 0ull;
    // exclusive scan over threads (threads own contiguous index ranges in thread order)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    unsigned long long incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long up = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += up;
    }
    SMOL_BLOCK_SYNC();
    if (lane == 31) sc.u64[warp] = incl;
    SMOL_BLOCK_SYNC();
    unsigned long long warp_base = 0, total = 0;
#pragma unroll
    for (int wi = 0; wi < (NT / 32); ++wi) {
        const unsigned long long t = sc.u64[wi];
        if (wi < warp) warp_base += t;
        total += t;
    }
    const unsigned long long excl = warp_base + incl - mine;

    uint32_t c[4] = {step, seq_id, stream, 0u};
    philox4x32_10(c, (uint32_t)(seed & 0xffffffffull), (uint32_t)(seed >> 32));
    const unsigned long long r64 = ((unsigned long long)c[0] << 32) | (unsigned long long)c[1];
    const unsigned long long target = __umul64hi(r64, total);

    if (threadIdx.x == 0) sc.bcast_i32 = n - 1;  // unreachable fallback (total > target always)
    SMOL_BLOCK_SYNC();
    if (mine > 0 && excl <= target && target < excl + mine) {
        unsigned long long run = excl;
        int pick = -1;
#pragma unroll
        for (int e = 0; e < kSampleMaxPerThread; ++e) {
            if (keep[e]) {
                run += (unsigned long long)w[e];
                if (pick < 0 && run > target) pick = i0 + e;
            }
        }
        sc.bcast_i32 = pick;
    }
    SMOL_BLOCK_SYNC();
    return sc.bcast_i32;
}

// The sampling parameters of row b: its entry of SmolBatch.row_sampling when the caller bound a table, the call's
// SmolSampling otherwise.  Every kernel that samples takes them from here and hands them to sample_row unchanged.
__device__ __forceinline__ SmolRowSampling row_sampling(const SmolSampling& s, const SmolRowSampling* table, int b) {
    if (table != nullptr) return table[b];
    SmolRowSampling r;
    r.temp = s.temp; r.fast_temp = s.fast_temp; r.top_k = s.top_k; r.top_p = s.top_p; r.min_p = s.min_p;
    r.pad = 0u; r.seed = s.seed;
    return r;
}

}  // namespace smol
