// The Mimi streaming decoder (codes -> PCM) for sm_100a: the step after the DualAR decode step (SURVEY §8(f)-2).
//
// One frame of one stream: 8 codes -> RVQ rows summed and projected (512) -> 2 upsampled positions -> 8 transformer
// layers against the stream's KV cache -> SEANet decoder (conv k7, then 4 x [ELU, transposed conv x8/x6/x5/x4, residual
// block], ELU, conv k3) with carried convolution state -> 1920 fp32 samples.  The reference computes all of it in fp32
// (load_mimi(format="fp32")), so do these kernels: fp32 FMA, fixed summation orders, no atomics -- a stream decodes to the
// same bits alone or in any batch.
//
// At streaming batch sizes every stage is a handful of rows (2 .. 1920 per stream) against a weight matrix that is read
// once: weight-streaming "row" products.  ONE kernel shape carries them all (rows_kernel): a CTA stages up to 16 input
// rows in shared memory -- gathered straight from the producer's buffer, im2col of a causal convolution = a contiguous run
// of (kernel x channels) floats that begins in the carried history rows; ELU or LayerNorm applied while staging -- and every
// warp streams one weight row (four from 64 rows on) with 16-byte loads against all staged rows, finishing with a shuffle
// reduction and a fused epilogue (bias, GELU, layer scale + residual, residual, or the upsampler).  Transposed convolutions
// (kernel = 2 stride) are the same product with K = (previous | current input row) x channels and N = (phase, channel): their
// outputs land contiguously.  From 12 streams on the SEANet's many-row stages run as 64 x 64 register tiles (tile_kernel) and
// the one-channel last convolution as one thread per sample (rowdot_kernel).  Attention: one CTA per (stream, head, split
// of 512 cached positions), partial softmaxes combined in split order.  Everything a stream carries (convolution history
// rows, the upsampler's previous embedding, KV cache, position) lives in per-slot arenas of the caller's workspace; a step is
// a program of 57 operations, one launch each, replayed as one CUDA graph.
//
// Reference map (C = mlx_inference/src/smoltts_mlx/codec/): RVQ decode C/rvq.py:118-130,171-186; upsample C/conv.py:225-282;
// transformer C/transformer.py:36-150; Conv1d.step C/conv.py:133-160; ConvTranspose1d.step C/conv.py:207-221; residual
// block C/seanet.py:9-50; decoder C/seanet.py:99-161; decode_step C/mimi.py:73-104.

#include <cuda_runtime.h>
#include <stdint.h>

#include <cstring>
#include <string>
#include <vector>

#include "../../include/smoltts_b200.h"
#include "../../include/smoltts_b200_mimi.h"
#include "mimi_common.cuh"

namespace smol {
namespace mimi {

constexpr int kStageFloats = 8192;   // shared-memory staging area of rows_kernel: R rows x (8192 / R) floats
constexpr int kMaxBufs = 24;

struct RowOp {
    // input rows: slot arena + in_off, `in_hs` history rows before the step's T rows, in_c floats per row;
    // element k of row (slot, t) = in[(in_hs + t + tap0 + (k / in_c) * tapstep) * in_c + k % in_c]
    const float* in; long long in_stride; int in_hs, in_c, tap0, tapstep, T;
    const float* W; const float* bias; int N, K, bias_mod;
    float* out; long long out_stride; int out_off0, out_by_row;
    const float* res; long long res_stride; int res_off0;
    int pro, epi;
    const float* ln_w; const float* ln_b; float eps;
    const float* scale;
    const float* wup; float* up_prev; int carry;   // EPI_UPSAMPLE
    const int32_t* slots; int batch;

    // tile_kernel's row map: row = b T + t of the batch's streams, b's stream in slot slots[b]
    struct Rows { int slot[kTM], t[kTM], b[kTM]; };
    __device__ void map_rows(Rows& s, int row0) const {   // (the slot table is constant during a step: read before the dependency wait)
        const int tid = threadIdx.x;
        if (tid < kTM) {
            const int row = row0 + tid;
            int b = 0, t = 0, slot = -1;
            if (row < batch * T) { b = row / T; t = row - b * T; slot = slots ? slots[b] : b; }
            s.slot[tid] = slot; s.t[tid] = t; s.b[tid] = b;
        }
        __syncthreads();
    }
    struct ARow { const float* base; int slot; };
    __device__ ARow a_row(const Rows& s, int, int m) const {
        const int slot = s.slot[m];
        return {in + (long long)(slot < 0 ? 0 : slot) * in_stride + (long long)(in_hs + s.t[m] + tap0) * in_c, slot};
    }
    __device__ float4 load_a(const ARow& a, int k) const {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (a.slot >= 0) {
            const int j = k / in_c, c = k - j * in_c;
            v = *reinterpret_cast<const float4*>(a.base + (long long)j * tapstep * in_c + c);
            if (pro == PRO_ELU) v = elu4(v);
        }
        return v;
    }
    __device__ bool out_row(const Rows& s, int, int m, long long& oe, long long& re) const {
        const int slot = s.slot[m];
        if (slot < 0) return false;
        oe = (long long)(out_by_row ? s.b[m] : slot) * out_stride + out_off0 + (long long)s.t[m] * N;
        re = (long long)slot * res_stride + res_off0 + (long long)s.t[m] * N;
        return true;
    }
    __device__ int bias_col(int n) const { return n % bias_mod; }   // (bias_mod: a channel count, a multiple of 4)
};

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Y[row][n] = epilogue( sum_k A(row, k) W[n][k] ): R staged rows per CTA, one weight row per warp (8 per CTA).
// Work item (bx, by) = (group of 8 weight rows, chunk of R input rows).
struct RowsSmem {
    float As[kStageFloats];
    float mean[16], rstd[16];
    int slot[16], t[16], b[16];   // slot, row inside the step and batch row of every staged row
};

// CPW weight rows per warp: 1 at streaming batch sizes; 4 from 64 rows on, where an operation is many CTAs deep and every
// CTA pays the same latency chain -- four rows per warp reuse the staged input rows (16 FMAs per shared-memory load instead of 4)
// and cut the CTA count by four.  A column's arithmetic (lane-interleaved sums, shuffle tree) is the same for any CPW.
template <int R, bool kPdl, int CPW>
__device__ __forceinline__ void rows_body(const RowOp& op, int bx, int by, RowsSmem& S) {
    constexpr int KC = kStageFloats / R;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int rows = op.batch * op.T;
    const int row0 = by * R;
    const int n0 = (bx * kWarps + warp) * CPW;         // first of this warp's CPW weight rows
    const bool n_ok = n0 < op.N;
    const int n = n0;
    if (tid < R) {   // (the slot table is constant during a step: read before the dependency wait)
        const int row = row0 + tid;
        int b = 0, t = 0, slot = -1;
        if (row < rows) { b = row / op.T; t = row - b * op.T; slot = op.slots ? op.slots[b] : b; }
        S.slot[tid] = slot; S.t[tid] = t; S.b[tid] = b;
    }
    // weights do not depend on the previous kernel / phase: the first four 16-byte pieces of this lane go straight into
    // registers (their latency overlaps the wait and the staging of the input rows) and the warp pulls its whole weight
    // row into L2
    if (kPdl && n_ok && by == 0) {
        const char* wr = reinterpret_cast<const char*>(op.W + (long long)n * op.K);
        const int lines = (min(CPW, op.N - n) * op.K * 4 + 127) >> 7;     // (the warp's rows are contiguous)
        for (int l = lane; l < lines; l += 32) prefetch_l2(wr + ((long long)l << 7));
    }
    constexpr int kPre = CPW == 1 ? 4 : 0;
    float4 wpre[kPre > 0 ? kPre : 1];
    {
        const int k0 = min(KC, op.K);
#pragma unroll
        for (int i = 0; i < kPre; ++i) {
            const int k4 = lane * 4 + i * 128;
            wpre[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (n_ok && k4 < k0) wpre[i] = __ldg(reinterpret_cast<const float4*>(op.W + (long long)n * op.K + k4));
        }
    }
    __syncthreads();
    if (kPdl) { pdl_wait(); pdl_go(); }
    float acc[CPW][R];
#pragma unroll
    for (int c = 0; c < CPW; ++c)
#pragma unroll
        for (int r = 0; r < R; ++r) acc[c][r] = 0.f;

    for (int kc = 0; kc < op.K; kc += KC) {
        const int kcur = min(KC, op.K - kc);
        // ---- stage R rows x kcur (16-byte pieces: in_c and K are multiples of 4) ----
        // (A division-free form of this loop -- one unrolled pass per row, contiguous im2col runs -- and LayerNorm statistics
        //  spread over all warps were measured: 500 -> 689 us per step at one stream; this is the faster form.)
        const int q4 = kcur >> 2;
        for (int idx = tid; idx < R * q4; idx += kThreads) {
            const int r = idx / q4, k = kc + ((idx - r * q4) << 2);
            const int slot = S.slot[r], t = S.t[r];
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (slot >= 0) {
                const int j = k / op.in_c, c = k - j * op.in_c;
                const float* src = op.in + (long long)slot * op.in_stride + (long long)(op.in_hs + t + op.tap0 + j * op.tapstep) * op.in_c + c;
                v = *reinterpret_cast<const float4*>(src);
                if (op.pro == PRO_ELU) { v.x = elu1(v.x); v.y = elu1(v.y); v.z = elu1(v.z); v.w = elu1(v.w); }
            }
            *reinterpret_cast<float4*>(&S.As[r * KC + ((idx - r * q4) << 2)]) = v;
        }
        __syncthreads();
        if (op.pro == PRO_LN) {   // LayerNorm over the whole row (K <= KC, checked on the host): two passes, as torch does
            for (int r = warp; r < R; r += kWarps) {
                float s = 0.f;
                for (int k = lane; k < kcur; k += 32) s += S.As[r * KC + k];
                const float mean = warp_sum(s) / (float)kcur;
                float d2 = 0.f;
                for (int k = lane; k < kcur; k += 32) { const float d = S.As[r * KC + k] - mean; d2 = fmaf(d, d, d2); }
                const float var = warp_sum(d2) / (float)kcur;
                if (lane == 0) { S.mean[r] = mean; S.rstd[r] = 1.0f / sqrtf(var + op.eps); }
            }
            __syncthreads();
            for (int k = tid; k < kcur; k += kThreads) {
                const float w = op.ln_w[k], bb = op.ln_b[k];
#pragma unroll
                for (int r = 0; r < R; ++r) S.As[r * KC + k] = (S.As[r * KC + k] - S.mean[r]) * S.rstd[r] * w + bb;
            }
            __syncthreads();
        }
        // ---- the weight row against all staged rows ----
        if (n_ok) {
            const float* wrow = op.W + (long long)n * op.K + kc;
            int k4 = lane * 4;
            if (kc == 0) {   // the pieces fetched before the wait (same order of additions as the loop below)
#pragma unroll
                for (int i = 0; i < kPre; ++i) {
                    if (k4 < kcur) {
#pragma unroll
                        for (int r = 0; r < R; ++r) {
                            const float4 a = *reinterpret_cast<const float4*>(&S.As[r * KC + k4]);
                            acc[0][r] = fmaf(a.x, wpre[i].x, acc[0][r]); acc[0][r] = fmaf(a.y, wpre[i].y, acc[0][r]);
                            acc[0][r] = fmaf(a.z, wpre[i].z, acc[0][r]); acc[0][r] = fmaf(a.w, wpre[i].w, acc[0][r]);
                        }
                        k4 += 128;
                    }
                }
            }
#pragma unroll(CPW == 1 ? 4 : 1)
            for (; k4 < kcur; k4 += 128) {
                float4 w[CPW];
#pragma unroll
                for (int c = 0; c < CPW; ++c)
                    w[c] = (n + c < op.N) ? __ldg(reinterpret_cast<const float4*>(wrow + (long long)c * op.K + k4)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int r = 0; r < R; ++r) {
                    const float4 a = *reinterpret_cast<const float4*>(&S.As[r * KC + k4]);
#pragma unroll
                    for (int c = 0; c < CPW; ++c) {
                        acc[c][r] = fmaf(a.x, w[c].x, acc[c][r]); acc[c][r] = fmaf(a.y, w[c].y, acc[c][r]);
                        acc[c][r] = fmaf(a.z, w[c].z, acc[c][r]); acc[c][r] = fmaf(a.w, w[c].w, acc[c][r]);
                    }
                }
            }
        }
        __syncthreads();
    }
    // ---- reduce over the lanes; lane r finishes row r ----
#pragma unroll
    for (int cc = 0; cc < CPW; ++cc) {
    const int n = n0 + cc;
    float mine = 0.f;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const float v = warp_sum(acc[cc][r]);
        if (lane == r) mine = v;
    }
    if (n < op.N && lane < R && S.slot[lane] >= 0) {
        const int b = S.b[lane], t = S.t[lane], slot = S.slot[lane];
        float y = mine + (op.bias ? op.bias[n % op.bias_mod] : 0.f);
        if (op.epi == EPI_UPSAMPLE) {
            // grouped transposed convolution, kernel 4, stride 2 (conv.py:271-282): outputs 2 t + j take tap j of this frame
            // and, with `carry`, tap 2 + j of the previous one; decode_step upsamples every frame alone (carry = 0)
            const float4 wu = *reinterpret_cast<const float4*>(op.wup + 4 * n);
            float o0 = y * wu.x, o1 = y * wu.y;
            if (op.carry) {
                float* pp = op.up_prev + (long long)slot * op.N + n;
                const float pv = *pp;
                o0 = fmaf(pv, wu.z, o0); o1 = fmaf(pv, wu.w, o1);
                *pp = y;
            }
            float* o = op.out + (long long)slot * op.out_stride + op.out_off0 + n;
            o[0] = o0; o[op.N] = o1;
        } else {
            const long long e = (long long)op.out_off0 + (long long)t * op.N + n;
            float* o = op.out + (long long)(op.out_by_row ? b : slot) * op.out_stride + e;
            if (op.epi == EPI_GELU) y = gelu_erf(y);
            else if (op.epi == EPI_SCALE_RES) y = op.res[(long long)slot * op.res_stride + op.res_off0 + (long long)t * op.N + n] + y * op.scale[n];
            else if (op.epi == EPI_RES) y = op.res[(long long)slot * op.res_stride + op.res_off0 + (long long)t * op.N + n] + y;
            *o = y;
        }
    }
    }
    __syncthreads();   // S is reused by the next work item
}

template <int R, int CPW>
__global__ void __launch_bounds__(kThreads) rows_kernel(const RowOp op) {
    __shared__ __align__(16) RowsSmem S;
    rows_body<R, true, CPW>(op, blockIdx.x, blockIdx.y, S);
}

// The two-row Linears of up to 8 streams (the 32 transformer operations of a step): rows_kernel<R, 1>'s arithmetic -- the same
// lane-interleaved sums, shuffle trees and LayerNorm loops, hence the same bits -- without its generality: a stream's two
// input rows are one contiguous run, no im2col, prologue and epilogue fixed at compile time.  An operation at streaming batch
// sizes is bound by the dependent instruction stream of its 8 warps (ncu: ~850 instructions per warp for rows_kernel<2, 1>),
// not by bytes: fewer instructions per warp is what shortens it (one stream: 492 -> 462 us per step).
template <int R, int PRO, int EPI>
__global__ void __launch_bounds__(kThreads) lin_kernel(const RowOp op) {
    constexpr int KC = kStageFloats / R;                                // floats between staged rows (K <= KC, host)
    __shared__ __align__(16) float As[kStageFloats];
    __shared__ float s_mean[R], s_rstd[R];
    __shared__ int s_slot[R / 2];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int K = op.K, n = blockIdx.x * kWarps + warp;                 // N is a multiple of 8 (host)
    const int rows = 2 * op.batch;
    const float* wrow = op.W + (long long)n * K;
    float4 wpre[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) wpre[i] = __ldg(reinterpret_cast<const float4*>(wrow + lane * 4 + i * 128));   // K >= 512 (host)
    {
        const char* wr = reinterpret_cast<const char*>(wrow);
        for (int l = lane; l < (K >> 5); l += 32) prefetch_l2(wr + ((long long)l << 7));
    }
    if (tid < R / 2) s_slot[tid] = tid < op.batch ? (op.slots ? op.slots[tid] : tid) : -1;
    __syncthreads();
    pdl_wait();
    pdl_go();
    const int q4 = K >> 2;
#pragma unroll
    for (int b = 0; b < R / 2; ++b) {                                   // a stream's two rows: 2 K contiguous floats
        const int slot = s_slot[b];
        const float4* a4 = reinterpret_cast<const float4*>(op.in + (long long)(slot < 0 ? 0 : slot) * op.in_stride + (long long)op.in_hs * K);
        for (int i = tid; i < 2 * q4; i += kThreads) {
            const int t = i >= q4 ? 1 : 0;
            *reinterpret_cast<float4*>(&As[(2 * b + t) * KC + ((i - t * q4) << 2)]) = slot < 0 ? make_float4(0.f, 0.f, 0.f, 0.f) : a4[i];
        }
    }
    __syncthreads();
    if (PRO == PRO_LN) {
        for (int r = warp; r < R; r += kWarps) {
            float s = 0.f;
            for (int k = lane; k < K; k += 32) s += As[r * KC + k];
            const float mean = warp_sum(s) / (float)K;
            float d2 = 0.f;
            for (int k = lane; k < K; k += 32) { const float d = As[r * KC + k] - mean; d2 = fmaf(d, d, d2); }
            const float var = warp_sum(d2) / (float)K;
            if (lane == 0) { s_mean[r] = mean; s_rstd[r] = 1.0f / sqrtf(var + op.eps); }
        }
        __syncthreads();
        for (int k = tid; k < K; k += kThreads) {
            const float w = op.ln_w[k], bb = op.ln_b[k];
#pragma unroll
            for (int r = 0; r < R; ++r) As[r * KC + k] = (As[r * KC + k] - s_mean[r]) * s_rstd[r] * w + bb;
        }
        __syncthreads();
    }
    float acc[R];
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = 0.f;
    int k4 = lane * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i, k4 += 128) {
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const float4 x = *reinterpret_cast<const float4*>(&As[r * KC + k4]);
            acc[r] = fmaf(x.x, wpre[i].x, acc[r]); acc[r] = fmaf(x.y, wpre[i].y, acc[r]); acc[r] = fmaf(x.z, wpre[i].z, acc[r]); acc[r] = fmaf(x.w, wpre[i].w, acc[r]);
        }
    }
#pragma unroll 4
    for (; k4 < K; k4 += 128) {
        const float4 w = __ldg(reinterpret_cast<const float4*>(wrow + k4));
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const float4 x = *reinterpret_cast<const float4*>(&As[r * KC + k4]);
            acc[r] = fmaf(x.x, w.x, acc[r]); acc[r] = fmaf(x.y, w.y, acc[r]); acc[r] = fmaf(x.z, w.z, acc[r]); acc[r] = fmaf(x.w, w.w, acc[r]);
        }
    }
    float mine = 0.f;
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const float v = warp_sum(acc[r]);
        if (lane == r) mine = v;
    }
    if (lane < rows) {
        const int slot = s_slot[lane >> 1], t = lane & 1;
        float y = mine;
        const long long e = (long long)slot * op.out_stride + op.out_off0 + (long long)t * op.N + n;
        if (EPI == EPI_GELU) y = gelu_erf(y);
        else if (EPI == EPI_SCALE_RES) y = op.res[(long long)slot * op.res_stride + op.res_off0 + (long long)t * op.N + n] + y * op.scale[n];
        op.out[e] = y;
    }
}

// The same product for MANY rows: the SEANet stages from 12 streams on (16 .. 1920 rows per stream) run through the shared
// tile_kernel<RowOp> (mimi_common.cuh), whose 4 x 4 outputs per thread make 16 FMAs per pair of 16-byte shared-memory loads
// instead of the 4 of rows_kernel, built for a handful of rows.  Every output there is one sequential FMA chain over k: a
// different order than rows_kernel's lane-interleaved sums, so which kernel runs is decided by the BATCH SIZE alone (12+
// streams) and a stream's bits are the same in any batch of the same class (< 12 streams, 12+).  It takes the ELU or no
// prologue and the bias or residual epilogue: the convolutions, transposed convolutions and residual-block convolutions.

// The last convolution (one output channel) for many rows: one thread per output sample, the weight vector in shared memory.
__global__ void __launch_bounds__(kThreads) rowdot_kernel(const RowOp op) {
    __shared__ __align__(16) float w[1024];
    const int tid = threadIdx.x;
    for (int k = tid; k < op.K; k += kThreads) w[k] = op.W[k];
    __syncthreads();
    pdl_wait();
    pdl_go();
    const int row = blockIdx.x * kThreads + tid;
    if (row >= op.batch * op.T) return;
    const int b = row / op.T, t = row - b * op.T;
    const int slot = op.slots ? op.slots[b] : b;
    const float* a = op.in + (long long)slot * op.in_stride + (long long)(op.in_hs + t + op.tap0) * op.in_c;   // contiguous im2col run
    float acc = 0.f;
    for (int k = 0; k < op.K; k += 4) {
        float4 v = *reinterpret_cast<const float4*>(a + k);
        if (op.pro == PRO_ELU) { v.x = elu1(v.x); v.y = elu1(v.y); v.z = elu1(v.z); v.w = elu1(v.w); }
        const float4 ww = *reinterpret_cast<const float4*>(&w[k]);
        acc = fmaf(v.x, ww.x, acc); acc = fmaf(v.y, ww.y, acc); acc = fmaf(v.z, ww.z, acc); acc = fmaf(v.w, ww.w, acc);
    }
    op.out[(long long)(op.out_by_row ? b : slot) * op.out_stride + op.out_off0 + t] = acc + (op.bias ? op.bias[0] : 0.f);
}

// RVQ decode (rvq.py:118-130, 171-186): the semantic codebook's row | the sum of the acoustic codebooks' rows, in order.
struct EmbedArgs {
    const float* books;   // [n_q][codebook_size][cdim], rows already divided by max(cluster_usage, eps)
    const int32_t* codes; const int32_t* slots; float* q; long long q_stride;
    int n_q, cb_size, cdim, batch;
};
__device__ __forceinline__ void embed_body(const EmbedArgs& a, int b) {
    const int slot = a.slots ? a.slots[b] : b;
    for (int k = threadIdx.x; k < 2 * a.cdim; k += blockDim.x) {
        float v;
        if (k < a.cdim) {
            int c = a.codes[b * a.n_q]; c = min(max(c, 0), a.cb_size - 1);
            v = a.books[(long long)c * a.cdim + k];
        } else {
            v = 0.f;
            for (int i = 1; i < a.n_q; ++i) {
                int c = a.codes[b * a.n_q + i]; c = min(max(c, 0), a.cb_size - 1);
                const float e = a.books[((long long)i * a.cb_size + c) * a.cdim + (k - a.cdim)];
                v = i == 1 ? e : v + e;
            }
        }
        a.q[(long long)slot * a.q_stride + k] = v;
    }
}
__global__ void embed_kernel(const EmbedArgs a) {
    pdl_wait();
    pdl_go();
    embed_body(a, blockIdx.x);
}

// Attention of one (stream, head): the step's two positions against the stream's cache (transformer.py:62-91).
// Half-split RoPE (nn.RoPE traditional=False) from the table, K/V appended, scores by one thread per position, softmax,
// P V by (dim, position class) threads; fixed orders throughout.  The reference's cache never forgets (no window), so a long
// stream's history is cut into SPLITS of kAttnChunk positions, one CTA each (grid z; CTAs past the stream's length leave at
// once): a split leaves (max, sum, unnormalised P V) per query, the last split to arrive combines them in split order.  A
// history of one split (<= 512 positions) writes its result directly.
constexpr int kAttnChunk = 512;
struct AttnArgs {
    const float* qkv; long long qkv_stride;      // [2][3 dim]
    float* att; long long att_stride;            // [2][dim]
    float* kv; long long kv_slot_stride, kv_layer_stride;   // [slot][layer][2][max_pos][dim]
    const float* rope; const int32_t* pos; const int32_t* slots; int32_t* err;
    float* part; unsigned int* arrive;           // [slot][head][split][2][hd + 2], [slot][head]
    int layer, dim, hd, max_pos, window, batch, heads, max_splits;
};
__device__ __forceinline__ void attn_body(const AttnArgs& a, int b, int h, int sp, float* sm) {
    __shared__ int s_last;
    const int tid = threadIdx.x;
    const int slot = a.slots ? a.slots[b] : b;
    const int hd = a.hd, half = hd >> 1;
    const int p0 = 2 * a.pos[slot];
    if (p0 + 2 > a.max_pos) { if (tid == 0 && sp == 0) *a.err = 1; return; }   // (uniform over the CTA)
    const int L = p0 + 2;
    // visible positions: query t sees lo_t .. p0 + t
    const int lo0 = a.window > 0 ? max(0, p0 + 1 - a.window) : 0;
    const int lo1 = a.window > 0 ? max(0, p0 + 2 - a.window) : 0;
    const int s_first = lo0 / kAttnChunk, s_end = (L + kAttnChunk - 1) / kAttnChunk;   // splits that hold visible positions
    if (sp < s_first || sp >= s_end) return;
    const int n_part = s_end - s_first;
    const int pa = max(lo0, sp * kAttnChunk), pe = min(L, (sp + 1) * kAttnChunk);       // this split's positions
    float* q = sm;                // [2][hd], pre-scaled
    float* red = sm + 2 * hd;     // [2 * kThreads] scratch
    float* S = red + 2 * kThreads;   // [2][kAttnChunk]
    float* kc = a.kv + (long long)slot * a.kv_slot_stride + (long long)a.layer * a.kv_layer_stride;
    float* vc = kc + (long long)a.max_pos * a.dim;
    const float* src = a.qkv + (long long)slot * a.qkv_stride;
    const float scale = rsqrtf((float)hd);
    const bool newest = sp == s_end - 1;          // the split that holds the step's own two positions appends them
    for (int i = tid; i < 2 * half; i += kThreads) {   // (position t, pair i)
        const int t = i / half, j = i - t * half;
        const float* row = src + (long long)t * 3 * a.dim + h * hd;
        const float cs = a.rope[(long long)(p0 + t) * hd + j], sn = a.rope[(long long)(p0 + t) * hd + half + j];
        const float q1 = row[j], q2 = row[j + half];
        q[t * hd + j] = (q1 * cs - q2 * sn) * scale;
        q[t * hd + j + half] = (q2 * cs + q1 * sn) * scale;
        if (newest) {
            const float k1 = row[a.dim + j], k2 = row[a.dim + j + half];
            float* kd = kc + (long long)(p0 + t) * a.dim + h * hd;
            kd[j] = k1 * cs - k2 * sn;
            kd[j + half] = k2 * cs + k1 * sn;
            float* vd = vc + (long long)(p0 + t) * a.dim + h * hd;
            vd[j] = row[2 * a.dim + j];
            vd[j + half] = row[2 * a.dim + j + half];
        }
    }
    __syncthreads();
    float m0 = -INFINITY, m1 = -INFINITY;
    for (int p = pa + tid; p < pe; p += kThreads) {
        const float4* kr = reinterpret_cast<const float4*>(kc + (long long)p * a.dim + h * hd);
        float s0 = 0.f, s1 = 0.f;
        for (int i = 0; i < hd / 4; ++i) {
            const float4 kk = kr[i];
            const float4 qa = *reinterpret_cast<const float4*>(q + 4 * i), qb = *reinterpret_cast<const float4*>(q + hd + 4 * i);
            s0 = fmaf(qa.x, kk.x, s0); s0 = fmaf(qa.y, kk.y, s0); s0 = fmaf(qa.z, kk.z, s0); s0 = fmaf(qa.w, kk.w, s0);
            s1 = fmaf(qb.x, kk.x, s1); s1 = fmaf(qb.y, kk.y, s1); s1 = fmaf(qb.z, kk.z, s1); s1 = fmaf(qb.w, kk.w, s1);
        }
        if (p > p0) s0 = -INFINITY;
        if (p < lo1) s1 = -INFINITY;
        S[p - pa] = s0; S[kAttnChunk + p - pa] = s1;
        m0 = fmaxf(m0, s0); m1 = fmaxf(m1, s1);
    }
    // block maximum: shuffles inside a warp, the eight warp values through shared memory (max is order-independent)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, o)); m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, o)); }
    if ((tid & 31) == 0) { red[tid >> 5] = m0; red[kWarps + (tid >> 5)] = m1; }
    __syncthreads();
    m0 = red[0]; m1 = red[kWarps];
#pragma unroll
    for (int w = 1; w < kWarps; ++w) { m0 = fmaxf(m0, red[w]); m1 = fmaxf(m1, red[kWarps + w]); }
    __syncthreads();
    float l0 = 0.f, l1 = 0.f;
    for (int p = pa + tid; p < pe; p += kThreads) {   // (a split in which a query sees nothing has max -inf: its terms are 0)
        const float e0 = m0 == -INFINITY ? 0.f : expf(S[p - pa] - m0), e1 = m1 == -INFINITY ? 0.f : expf(S[kAttnChunk + p - pa] - m1);
        S[p - pa] = e0; S[kAttnChunk + p - pa] = e1;
        l0 += e0; l1 += e1;
    }
    // block sum: fixed shuffle tree inside a warp, warp sums added in warp order
    l0 = warp_sum(l0); l1 = warp_sum(l1);
    if ((tid & 31) == 0) { red[tid >> 5] = l0; red[kWarps + (tid >> 5)] = l1; }
    __syncthreads();
    l0 = red[0]; l1 = red[kWarps];
#pragma unroll
    for (int w = 1; w < kWarps; ++w) { l0 += red[w]; l1 += red[kWarps + w]; }
    __syncthreads();
    // P V: thread = (dim d, position class g of kThreads / hd)
    const int G = kThreads / hd, d = tid % hd, g = tid / hd;
    float o0 = 0.f, o1 = 0.f;
    if (g < G) {
        for (int p = pa + g; p < pe; p += G) {
            const float v = vc[(long long)p * a.dim + h * hd + d];
            o0 = fmaf(S[p - pa], v, o0); o1 = fmaf(S[kAttnChunk + p - pa], v, o1);
        }
    }
    red[tid] = o0; red[kThreads + tid] = o1;
    __syncthreads();
    float* dst = a.att + (long long)slot * a.att_stride + h * hd;
    float* mypart = a.part + (((long long)slot * a.heads + h) * a.max_splits) * (2 * (hd + 2));
    if (tid < hd) {
        float s0 = 0.f, s1 = 0.f;
        for (int gg = 0; gg < G; ++gg) { s0 += red[gg * hd + tid]; s1 += red[kThreads + gg * hd + tid]; }
        if (n_part == 1) {
            dst[tid] = s0 / l0;
            dst[a.dim + tid] = s1 / l1;
        } else {
            float* pp = mypart + (long long)sp * (2 * (hd + 2));
            pp[2 + tid] = s0; pp[(hd + 2) + 2 + tid] = s1;
            if (tid == 0) { pp[0] = m0; pp[1] = l0; pp[hd + 2] = m1; pp[hd + 3] = l1; }
        }
    }
    if (n_part > 1) {   // one arrival per split; the last one combines all of them in split order
        __threadfence();
        __syncthreads();
        if (tid == 0) {
            const unsigned int old = atomicAdd(a.arrive + (long long)slot * a.heads + h, 1u);
            s_last = old == (unsigned int)(n_part - 1);
            if (s_last) a.arrive[(long long)slot * a.heads + h] = 0u;
        }
        __syncthreads();
        if (s_last) {
            __threadfence();
            if (tid < 2 * hd) {
                const int qi = tid / hd, dd = tid - qi * hd;
                float M = -INFINITY;
                for (int s = s_first; s < s_end; ++s) M = fmaxf(M, __ldcg(mypart + (long long)s * (2 * (hd + 2)) + qi * (hd + 2)));
                float Ls = 0.f, O = 0.f;
                for (int s = s_first; s < s_end; ++s) {
                    const float* pp = mypart + (long long)s * (2 * (hd + 2)) + qi * (hd + 2);
                    const float ms = __ldcg(pp);
                    const float c = ms == -INFINITY ? 0.f : expf(ms - M);
                    Ls = fmaf(__ldcg(pp + 1), c, Ls);
                    O = fmaf(__ldcg(pp + 2 + dd), c, O);
                }
                dst[qi * a.dim + dd] = O / Ls;
            }
        }
    }
    __syncthreads();   // sm is reused by the next work item
}
__global__ void __launch_bounds__(kThreads) attn_kernel(const AttnArgs a) {
    extern __shared__ __align__(16) float sm[];
    pdl_wait();
    pdl_go();
    attn_body(a, blockIdx.x, blockIdx.y, blockIdx.z, sm);
}

// End of a step: the last `hs` rows of every history-carrying buffer move to its front; the position advances.
struct BufDesc { int off, hs, T, C; };
struct ShiftArgs {
    float* arena; long long stride; const int32_t* slots; int32_t* pos; float* up_prev; int dim;
    int n_bufs; int reset;   // reset = 1: zero the history rows, the upsampler's carry and the position instead
    int batch, pad;
    BufDesc bufs[kMaxBufs];
};
__device__ __forceinline__ void shift_body(const ShiftArgs& a, int b, int i, float* tmp /* 4096 floats */) {
    const int tid = threadIdx.x;
    const int slot = a.slots ? a.slots[b] : b;
    if (i == a.n_bufs) {
        if (a.reset) {
            for (int k = tid; k < a.dim; k += kThreads) a.up_prev[(long long)slot * a.dim + k] = 0.f;
            if (tid == 0) a.pos[slot] = 0;
        } else if (tid == 0) a.pos[slot] += 1;
        return;
    }
    const BufDesc d = a.bufs[i];
    float* base = a.arena + (long long)slot * a.stride + d.off;
    const int n = d.hs * d.C;
    if (a.reset) { for (int k = tid; k < n; k += kThreads) base[k] = 0.f; return; }
    const float* src = base + (long long)d.T * d.C;   // rows T .. T + hs
    for (int k0 = 0; k0 < n; k0 += 4096) {   // (source and destination overlap when T < hs: staged through shared memory)
        const int m = min(4096, n - k0);
        for (int k = tid; k < m; k += kThreads) tmp[k] = src[k0 + k];
        __syncthreads();
        for (int k = tid; k < m; k += kThreads) base[k0 + k] = tmp[k];
        __syncthreads();
    }
}
__global__ void __launch_bounds__(kThreads) shift_kernel(const ShiftArgs a) {
    __shared__ float tmp[4096];
    pdl_wait();
    pdl_go();
    shift_body(a, blockIdx.x, blockIdx.y, tmp);
}

// A step = a program of operations, one launch each (replayed as a CUDA graph).
// (Measured and dropped: the whole program inside ONE persistent cooperative kernel -- 296 co-resident CTAs walking 512-byte
//  operation records, a grid barrier after every operation, the next operation's weight rows prefetched into L2 before the
//  barrier.  Bit-identical, but 760 us per step against 500 us for the graph at one stream, 1.79 vs 1.37 ms at 8, and worse
//  on 148 or 74 CTAs (1 102 / 1 509 us): an operation is a chain of dependent instructions and L2 round trips inside a
//  CTA, which a barrier does not shorten, while the graph's kernel boundaries cost less than a 296-CTA barrier.)
enum { OP_ROWS = 0, OP_ATTN = 1, OP_EMBED = 2, OP_SHIFT = 3 };
struct OpRec {
    int kind, R;
    union { RowOp row; AttnArgs attn; EmbedArgs emb; ShiftArgs shift; };
};

// ---- bind-time packing (codebooks and Conv1d: mimi_common.cuh) -----------------------------------------------------
// ConvTranspose1d [Ci][Co][2 s] -> [(r, co)][(u, ci)] = w[ci][co][r + u s]   (u = 0: this input row, u = 1: the previous one)
__global__ void pack_convtr_kernel(float* dst, const float* w, int Ci, int Co, int s) {
    const long long total = (long long)s * Co * 2 * Ci;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int ci = (int)(i % Ci); long long r = i / Ci; const int u = (int)(r % 2); r /= 2; const int co = (int)(r % Co); const int ph = (int)(r / Co);
        dst[i] = w[((long long)ci * Co + co) * (2 * s) + ph + u * s];
    }
}
// two [N][K1] matrices side by side -> [N][2 K1]
__global__ void pack_hcat_kernel(float* dst, const float* a, const float* b, int N, int K1) {
    const long long total = (long long)N * 2 * K1;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int k = (int)(i % (2 * K1)); const int n = (int)(i / (2 * K1));
        dst[i] = k < K1 ? a[(long long)n * K1 + k] : b[(long long)n * K1 + (k - K1)];
    }
}

}  // namespace mimi
}  // namespace smol

// ---- host side -------------------------------------------------------------------------------------------------------
using namespace smol::mimi;

struct MimiBuf { size_t off; int hs, T, C; };   // per-slot arena buffer (floats)

struct SmolMimi {
    SmolMimiConfig cfg{};
    int spf = 0;                       // samples per frame
    int ch0 = 0;                       // channels after conv_in
    // per-slot arena
    std::vector<MimiBuf> bufs;
    int bX0 = 0, bQ = 0, bQKV = 0, bATT = 0, bFF = 0, bA0 = 0;
    int bCT[SMOL_MIMI_MAX_RATIOS], bH[SMOL_MIMI_MAX_RATIOS], bR[SMOL_MIMI_MAX_RATIOS];
    size_t arena_floats = 0;
    // workspace layout (bytes)
    size_t o_books = 0, o_wcat = 0, o_up = 0, o_rope = 0, o_small = 0, o_conv_in = 0, o_conv_out = 0;
    LayerOffsets o_layer[SMOL_MIMI_MAX_LAYERS];
    size_t o_ct[SMOL_MIMI_MAX_RATIOS], o_r1[SMOL_MIMI_MAX_RATIOS], o_r2[SMOL_MIMI_MAX_RATIOS], o_bias = 0;
    size_t o_arena = 0, o_kv = 0, o_pos = 0, o_upprev = 0, o_err = 0, total = 0;
    unsigned char* ws = nullptr;
    bool bound = false;
    int launches = 0;
    size_t attn_smem = 0, o_part = 0, o_arrive = 0;
    int max_splits = 1;
    // cached graph of one step
    cudaStream_t cap_stream = nullptr;
    // captured steps, keyed by (batch, buffers): a serving loop alternates between a few batch sizes
    struct Step { const void* codes; const void* slots; const void* pcm; int batch; std::vector<OpRec> prog; cudaGraphExec_t graph; uint64_t used; };
    std::vector<Step> steps;
    uint64_t tick = 0;
    void drop_steps() { for (Step& s : steps) if (s.graph) cudaGraphExecDestroy(s.graph); steps.clear(); }
};
constexpr size_t kMaxSteps = 16;

static int mimi_plan(SmolMimi* m) {
    const SmolMimiConfig& c = m->cfg;
    m->bufs.clear();
    size_t off = 0;
    auto add = [&](int hs, int T, int C) { m->bufs.push_back({off, hs, T, C}); off += (size_t)(hs + T) * C; off = (off + 3) / 4 * 4; return (int)m->bufs.size() - 1; };
    m->ch0 = c.n_filters << c.n_ratios;
    m->bX0 = add(c.kernel - 1, 2, c.dim);
    m->bQ = add(0, 1, 2 * c.codebook_dim);
    m->bQKV = add(0, 2, 3 * c.dim);
    m->bATT = add(0, 2, c.dim);
    m->bFF = add(0, 2, c.ffn);
    m->bA0 = add(1, 2, m->ch0);
    int T = 2, ch = m->ch0;
    for (int i = 0; i < c.n_ratios; ++i) {
        T *= c.ratios[i]; ch /= 2;
        m->bCT[i] = add(c.res_kernel - 1, T, ch);
        m->bH[i] = add(0, T, ch / 2);
        m->bR[i] = add(i + 1 < c.n_ratios ? 1 : c.last_kernel - 1, T, ch);
    }
    m->spf = T;
    m->arena_floats = (off + 63) / 64 * 64;
    if ((int)m->bufs.size() > kMaxBufs) return -1;
    // workspace
    WsPlan p;
    m->o_books = p.take((size_t)c.n_q * c.codebook_size * c.codebook_dim);
    m->o_wcat = p.take((size_t)c.dim * 2 * c.codebook_dim);
    m->o_up = p.take((size_t)c.dim * 4);
    m->o_rope = p.take((size_t)c.max_positions * c.head_dim);
    for (int l = 0; l < c.n_layers; ++l) m->o_layer[l] = plan_layer(p, c.dim, c.ffn);
    m->o_conv_in = p.take((size_t)m->ch0 * c.dim * c.kernel);
    ch = m->ch0;
    for (int i = 0; i < c.n_ratios; ++i) {
        m->o_ct[i] = p.take((size_t)ch * (ch / 2) * 2 * c.ratios[i]);
        ch /= 2;
        m->o_r1[i] = p.take((size_t)(ch / 2) * ch * c.res_kernel);
        m->o_r2[i] = p.take((size_t)ch * (ch / 2));
    }
    m->o_conv_out = p.take((size_t)ch * c.last_kernel);
    m->o_bias = p.take((size_t)4 * m->ch0 + 16);   // all SEANet biases, back to back
    m->o_arena = p.take(m->arena_floats * (size_t)c.max_streams);
    m->o_kv = p.take((size_t)c.max_streams * c.n_layers * 2 * c.max_positions * c.dim);
    m->o_pos = p.take((size_t)c.max_streams);
    m->o_upprev = p.take((size_t)c.max_streams * c.dim);
    m->o_err = p.take(4);
    m->max_splits = (c.max_positions + kAttnChunk - 1) / kAttnChunk;
    m->o_part = p.take((size_t)c.max_streams * c.n_heads * m->max_splits * 2 * (c.head_dim + 2));
    m->o_arrive = p.take((size_t)c.max_streams * c.n_heads);
    m->total = p.total;
    m->attn_smem = (size_t)(2 * c.head_dim + 2 * kThreads + 2 * kAttnChunk) * 4;
    m->max_splits = (c.max_positions + kAttnChunk - 1) / kAttnChunk;
    return 0;
}

extern "C" int smol_mimi_create(const SmolMimiConfig* cfg, SmolMimi** out) {
    if (!cfg || !out) return smol::capi_fail(SMOL_ERR_INVALID, "smol_mimi_create: null argument");
    const SmolMimiConfig& c = *cfg;
    if (c.n_q < 2 || c.n_q > SMOL_MIMI_MAX_Q) return smol::capi_fail(SMOL_ERR_INVALID, "mimi: n_q must be 2 .. 32 (one semantic + acoustic codebooks)");
    if (c.n_layers < 1 || c.n_layers > SMOL_MIMI_MAX_LAYERS) return smol::capi_fail(SMOL_ERR_INVALID, "mimi: n_layers out of range");
    if (c.n_ratios < 1 || c.n_ratios > SMOL_MIMI_MAX_RATIOS) return smol::capi_fail(SMOL_ERR_INVALID, "mimi: n_ratios out of range");
    if (c.dim != c.n_heads * c.head_dim) return smol::capi_fail(SMOL_ERR_INVALID, "mimi: dim != n_heads * head_dim");
    if (c.head_dim % 8 || c.head_dim > kThreads || kThreads % c.head_dim) return smol::capi_fail(SMOL_ERR_UNSUPPORTED, "mimi: head_dim must divide 256 and be a multiple of 8");
    if (c.dim % 4 || c.ffn % 4 || c.codebook_dim % 4 || (c.n_filters % 8)) return smol::capi_fail(SMOL_ERR_UNSUPPORTED, "mimi: channel counts must be multiples of 4 (n_filters of 8)");
    if (c.dim > kStageFloats / 16) return smol::capi_fail(SMOL_ERR_UNSUPPORTED, "mimi: dim above 512 does not fit the LayerNorm staging");
    if (c.kernel < 1 || c.res_kernel < 1 || c.last_kernel < 1) return smol::capi_fail(SMOL_ERR_INVALID, "mimi: kernel sizes");
    for (int i = 0; i < c.n_ratios; ++i) if (c.ratios[i] < 1) return smol::capi_fail(SMOL_ERR_INVALID, "mimi: ratios must be positive");
    if (c.max_streams < 1 || c.max_positions < 2 || (c.max_positions & 1)) return smol::capi_fail(SMOL_ERR_INVALID, "mimi: max_streams >= 1, max_positions even and >= 2");
    SmolMimi* m = new SmolMimi();
    m->cfg = c;
    if (mimi_plan(m) != 0) { delete m; return smol::capi_fail(SMOL_ERR_UNSUPPORTED, "mimi: too many buffers"); }
    if (c.max_positions > (1 << 20)) { delete m; return smol::capi_fail(SMOL_ERR_CAPACITY, "mimi: max_positions above 1 048 576"); }
    *out = m;
    return SMOL_OK;
}

extern "C" void smol_mimi_destroy(SmolMimi* m) {
    if (!m) return;
    m->drop_steps();
    if (m->cap_stream) cudaStreamDestroy(m->cap_stream);
    delete m;
}
extern "C" int32_t smol_mimi_samples_per_frame(const SmolMimi* m) { return m ? m->spf : 0; }
extern "C" size_t smol_mimi_workspace_bytes(const SmolMimi* m) { return m ? m->total : 0; }
extern "C" int32_t smol_mimi_launches_per_step(const SmolMimi* m) { return m ? m->launches : 0; }
extern "C" int32_t* smol_mimi_error_word(SmolMimi* m) { return (m && m->bound) ? reinterpret_cast<int32_t*>(m->ws + m->o_err) : nullptr; }

static float* wsf(SmolMimi* m, size_t off) { return reinterpret_cast<float*>(m->ws + off); }

static ShiftArgs shift_args(SmolMimi* m, const int32_t* slots, int reset) {
    ShiftArgs a{};
    a.arena = wsf(m, m->o_arena); a.stride = (long long)m->arena_floats; a.slots = slots;
    a.pos = reinterpret_cast<int32_t*>(m->ws + m->o_pos); a.up_prev = wsf(m, m->o_upprev); a.dim = m->cfg.dim;
    a.n_bufs = 0; a.reset = reset;
    for (const MimiBuf& b : m->bufs) if (b.hs > 0) a.bufs[a.n_bufs++] = BufDesc{(int)b.off, b.hs, b.T, b.C};
    return a;
}

extern "C" int smol_mimi_reset(SmolMimi* m, const int32_t* d_slots, int32_t n, void* stream) {
    if (!m) return smol::capi_fail(SMOL_ERR_INVALID, "smol_mimi_reset: null model");
    if (!m->bound) return smol::capi_fail(SMOL_ERR_UNBOUND, "smol_mimi_reset: weights / workspace not bound");
    if (n < 1 || n > m->cfg.max_streams) return smol::capi_fail(SMOL_ERR_CAPACITY, "smol_mimi_reset: n outside 1 .. max_streams");
    ShiftArgs a = shift_args(m, d_slots, 1);
    a.batch = n;
    shift_kernel<<<dim3(n, a.n_bufs + 1), kThreads, 0, (cudaStream_t)stream>>>(a);
    MIMI_CUDA(cudaGetLastError());
    return SMOL_OK;
}

extern "C" int smol_mimi_bind(SmolMimi* m, const SmolMimiWeights* w, void* d_workspace, size_t workspace_bytes, void* stream) {
    if (!m || !w || !d_workspace) return smol::capi_fail(SMOL_ERR_INVALID, "smol_mimi_bind: null argument");
    if (workspace_bytes < m->total) return smol::capi_fail(SMOL_ERR_CAPACITY, "smol_mimi_bind: workspace smaller than smol_mimi_workspace_bytes()");
    if ((uintptr_t)d_workspace % 256) return smol::capi_fail(SMOL_ERR_INVALID, "smol_mimi_bind: workspace must be 256-byte aligned");
    const SmolMimiConfig& c = m->cfg;
    cudaStream_t st = (cudaStream_t)stream;
    auto need = [&](const void* p) { return p != nullptr; };
    bool ok = need(w->semantic_output_proj) && need(w->acoustic_output_proj) && need(w->upsample) && need(w->rope) &&
              need(w->conv_in.weight) && need(w->conv_in.bias) && need(w->conv_out.weight) && need(w->conv_out.bias);
    for (int i = 0; i < c.n_q; ++i) ok = ok && need(w->embed_sum[i]) && need(w->cluster_usage[i]);
    for (int l = 0; l < c.n_layers; ++l) ok = ok && layer_weights_ok(w->layers[l]);
    for (int i = 0; i < c.n_ratios; ++i)
        ok = ok && need(w->convtr[i].weight) && need(w->convtr[i].bias) && need(w->res_conv1[i].weight) && need(w->res_conv1[i].bias) &&
             need(w->res_conv2[i].weight) && need(w->res_conv2[i].bias);
    if (!ok) return smol::capi_fail(SMOL_ERR_INVALID, "smol_mimi_bind: a weight pointer is null");
    m->ws = reinterpret_cast<unsigned char*>(d_workspace);
    m->drop_steps();
    const size_t f4 = sizeof(float);
    auto d2d = [&](size_t off, const float* src, size_t floats) { return cudaMemcpyAsync(m->ws + off, src, floats * f4, cudaMemcpyDeviceToDevice, st); };
    for (int i = 0; i < c.n_q; ++i)
        pack_codebook_kernel<<<256, 256, 0, st>>>(wsf(m, m->o_books) + (size_t)i * c.codebook_size * c.codebook_dim, w->embed_sum[i],
                                                   w->cluster_usage[i], c.codebook_size, c.codebook_dim, c.codebook_eps);
    pack_hcat_kernel<<<256, 256, 0, st>>>(wsf(m, m->o_wcat), w->semantic_output_proj, w->acoustic_output_proj, c.dim, c.codebook_dim);
    MIMI_CUDA(d2d(m->o_up, w->upsample, (size_t)c.dim * 4));
    MIMI_CUDA(d2d(m->o_rope, w->rope, (size_t)c.max_positions * c.head_dim));
    for (int l = 0; l < c.n_layers; ++l) {
        const int rc = bind_layer(m->ws, m->o_layer[l], w->layers[l], c.dim, c.ffn, st);
        if (rc != SMOL_OK) return rc;
    }
    pack_conv_kernel<<<512, 256, 0, st>>>(wsf(m, m->o_conv_in), w->conv_in.weight, m->ch0, c.dim, c.kernel);
    size_t bo = m->o_bias;
    MIMI_CUDA(d2d(bo, w->conv_in.bias, m->ch0)); bo += (size_t)m->ch0 * f4;
    int ch = m->ch0;
    for (int i = 0; i < c.n_ratios; ++i) {
        pack_convtr_kernel<<<512, 256, 0, st>>>(wsf(m, m->o_ct[i]), w->convtr[i].weight, ch, ch / 2, c.ratios[i]);
        ch /= 2;
        pack_conv_kernel<<<256, 256, 0, st>>>(wsf(m, m->o_r1[i]), w->res_conv1[i].weight, ch / 2, ch, c.res_kernel);
        MIMI_CUDA(d2d(m->o_r2[i], w->res_conv2[i].weight, (size_t)ch * (ch / 2)));
        MIMI_CUDA(d2d(bo, w->convtr[i].bias, ch)); bo += (size_t)ch * f4;
        MIMI_CUDA(d2d(bo, w->res_conv1[i].bias, ch / 2)); bo += (size_t)(ch / 2) * f4;
        MIMI_CUDA(d2d(bo, w->res_conv2[i].bias, ch)); bo += (size_t)ch * f4;
    }
    pack_conv_kernel<<<16, 256, 0, st>>>(wsf(m, m->o_conv_out), w->conv_out.weight, 1, ch, c.last_kernel);
    MIMI_CUDA(d2d(bo, w->conv_out.bias, 1));
    MIMI_CUDA(cudaGetLastError());
    MIMI_CUDA(cudaMemsetAsync(m->ws + m->o_err, 0, 16, st));
    MIMI_CUDA(cudaMemsetAsync(m->ws + m->o_arrive, 0, (size_t)c.max_streams * c.n_heads * 4, st));
    if (m->attn_smem > 48 * 1024) MIMI_CUDA(cudaFuncSetAttribute(attn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)m->attn_smem));
    m->bound = true;
    return smol_mimi_reset(m, nullptr, c.max_streams, stream);
}

// Launch with the programmatic-serialization attribute (see pdl_wait) if `pdl`, plainly otherwise.
template <class Args>
static cudaError_t launch_pdl(bool pdl, void (*kern)(const Args), dim3 grid, dim3 block, size_t smem, cudaStream_t st, const Args& a) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, a);
}
// (Measured and dropped: splitting a weight row over 2 .. 8 warps to get 256+ CTAs per operation changed nothing at one
//  stream -- 510 vs 513 us per step: the operations are latency chains, not bandwidth -- and cost 20 .. 45 % at 8 .. 64
//  streams, where every extra CTA re-stages the same input rows.)

static int rows_R(int rows) { return rows <= 2 ? 2 : rows <= 4 ? 4 : rows <= 8 ? 8 : 16; }

// 12+ streams: the many-row stages go through the tile kernel (decided by the batch size alone, see tile_kernel)
constexpr int kTileMinBatch = 12;   // measured: 8 streams 1.13 ms per step on rows_kernel vs 1.23 on the tiles; 12 streams 1.35 vs 1.30
static bool use_tile(const RowOp& op) {
    return op.batch >= kTileMinBatch && op.T >= 16 && op.N >= 16 && op.N % 4 == 0 && op.K % kTK == 0 &&
           (op.pro == PRO_NONE || op.pro == PRO_ELU) && (op.epi == EPI_BIAS || op.epi == EPI_RES);
}
static bool use_rowdot(const RowOp& op) {
    return op.batch >= kTileMinBatch && op.N == 1 && op.K <= 1024 && op.K % 4 == 0 && op.tapstep > 0 && op.epi == EPI_BIAS && op.pro != PRO_LN;
}

// the two-row Linears of up to 8 streams: the lean form of rows_kernel<R, 1> (same bits)
static bool use_lin(const RowOp& op) {
    const int R = rows_R(op.batch * op.T);
    return op.batch <= 8 && op.T == 2 && op.K == op.in_c && op.tapstep > 0 && op.tap0 == 0 && op.N % kWarps == 0 && op.K >= 512 &&
           op.K <= kStageFloats / R && op.K % 128 == 0 && op.bias == nullptr && op.out_by_row == 0 &&
           ((op.pro == PRO_LN && (op.epi == EPI_BIAS || op.epi == EPI_GELU)) || (op.pro == PRO_NONE && op.epi == EPI_SCALE_RES));
}
template <int R>
static cudaError_t launch_lin(const RowOp& op, cudaStream_t st, bool pdl) {
    const dim3 grid(op.N / kWarps);
    if (op.pro == PRO_LN && op.epi == EPI_BIAS) return launch_pdl(pdl, lin_kernel<R, PRO_LN, EPI_BIAS>, grid, dim3(kThreads), 0, st, op);
    if (op.pro == PRO_LN) return launch_pdl(pdl, lin_kernel<R, PRO_LN, EPI_GELU>, grid, dim3(kThreads), 0, st, op);
    return launch_pdl(pdl, lin_kernel<R, PRO_NONE, EPI_SCALE_RES>, grid, dim3(kThreads), 0, st, op);
}

static cudaError_t launch_rows(const RowOp& op, cudaStream_t st, bool pdl) {
    if (use_lin(op)) {
        switch (rows_R(op.batch * op.T)) {
            case 2: return launch_lin<2>(op, st, pdl);
            case 4: return launch_lin<4>(op, st, pdl);
            case 8: return launch_lin<8>(op, st, pdl);
            default: return launch_lin<16>(op, st, pdl);
        }
    }
    if (use_tile(op)) {
        const dim3 grid((op.batch * op.T + kTM - 1) / kTM, (op.N + kTN - 1) / kTN);
        return launch_pdl(pdl, tile_kernel<RowOp>, grid, dim3(kThreads), 0, st, op);
    }
    if (use_rowdot(op)) return launch_pdl(pdl, rowdot_kernel, dim3((op.batch * op.T + kThreads - 1) / kThreads), dim3(kThreads), 0, st, op);
    const int rows = op.batch * op.T;
    const int R = rows_R(rows);
    // 64+ rows (the SEANet stages below 12 streams, the two-row operations from 32 streams on): four weight rows per warp -- the
    // same bits, fewer and fatter CTAs.  Measured per step: 4 streams 825 -> 748 us, 32 streams 1.99 -> 1.73 ms, 64 streams
    // 3.22 -> 2.41 ms; operations of 16 rows (8 streams' Linears) lose 12 % with it, hence the bar.
    if (R == 16 && rows >= 64 && op.N >= 64) {
        const dim3 grid4((op.N + 4 * kWarps - 1) / (4 * kWarps), (rows + R - 1) / R);
        return launch_pdl(pdl, rows_kernel<16, 4>, grid4, dim3(kThreads), 0, st, op);
    }
    const dim3 grid((op.N + kWarps - 1) / kWarps, (rows + R - 1) / R);
    switch (R) {
        case 2: return launch_pdl(pdl, rows_kernel<2, 1>, grid, dim3(kThreads), 0, st, op);
        case 4: return launch_pdl(pdl, rows_kernel<4, 1>, grid, dim3(kThreads), 0, st, op);
        case 8: return launch_pdl(pdl, rows_kernel<8, 1>, grid, dim3(kThreads), 0, st, op);
        default: return launch_pdl(pdl, rows_kernel<16, 1>, grid, dim3(kThreads), 0, st, op);
    }
}

// The step as a program: every operation in order (executed by one launch each, or by the persistent kernel).
static void mimi_program(SmolMimi* m, const int32_t* d_codes, const int32_t* d_slots, int batch, float* d_pcm, std::vector<OpRec>& prog) {
    const SmolMimiConfig& c = m->cfg;
    float* arena = wsf(m, m->o_arena);
    const long long AS = (long long)m->arena_floats;
    prog.clear();
    auto buf = [&](int i) -> const MimiBuf& { return m->bufs[i]; };
    auto base_op = [&]() { RowOp op{}; op.slots = d_slots; op.batch = batch; op.in_stride = AS; op.out_stride = AS; op.res_stride = AS; op.bias_mod = 1; op.tapstep = 1; return op; };
    // input of an op: buffer bi, `taps` rows ending at the current one (conv) or {current, previous} (transposed conv)
    auto set_in = [&](RowOp& op, int bi, int taps, bool transposed) {
        const MimiBuf& b = buf(bi);
        op.in = arena + b.off; op.in_hs = b.hs; op.in_c = b.C; op.T = b.T; op.K = taps * b.C;
        op.tap0 = transposed ? 0 : -(taps - 1); op.tapstep = transposed ? -1 : 1;
    };
    auto set_out = [&](RowOp& op, int bi) { const MimiBuf& b = buf(bi); op.out = arena + b.off; op.out_off0 = b.hs * b.C; };
    auto set_res = [&](RowOp& op, int bi) { const MimiBuf& b = buf(bi); op.res = arena + b.off; op.res_off0 = b.hs * b.C; };
    auto push_rows = [&](const RowOp& op) { OpRec r{}; r.kind = OP_ROWS; r.R = rows_R(op.batch * op.T); r.row = op; prog.push_back(r); };

    {   // RVQ rows -> Q; projection + upsample -> the residual stream (current rows of X0)
        OpRec r{}; r.kind = OP_EMBED;
        r.emb = EmbedArgs{wsf(m, m->o_books), d_codes, d_slots, arena + buf(m->bQ).off, AS, c.n_q, c.codebook_size, c.codebook_dim, batch};
        prog.push_back(r);
        RowOp op = base_op();
        set_in(op, m->bQ, 1, false);
        op.W = wsf(m, m->o_wcat); op.N = c.dim; op.epi = EPI_UPSAMPLE; op.wup = wsf(m, m->o_up);
        op.up_prev = wsf(m, m->o_upprev); op.carry = c.upsample_carry;
        set_out(op, m->bX0);
        push_rows(op);
    }
    for (int l = 0; l < c.n_layers; ++l) {
        const LayerOffsets& lo = m->o_layer[l];
        const float* vec = wsf(m, lo.vec);
        {   // LayerNorm -> q | k | v
            RowOp op = base_op();
            set_in(op, m->bX0, 1, false);
            op.pro = PRO_LN; op.ln_w = vec; op.ln_b = vec + c.dim; op.eps = c.norm_eps;
            op.W = wsf(m, lo.qkv); op.N = 3 * c.dim; op.epi = EPI_BIAS;
            set_out(op, m->bQKV);
            push_rows(op);
        }
        {
            OpRec r{}; r.kind = OP_ATTN;
            AttnArgs& a = r.attn;
            a.qkv = arena + buf(m->bQKV).off; a.qkv_stride = AS; a.att = arena + buf(m->bATT).off; a.att_stride = AS;
            a.kv = wsf(m, m->o_kv); a.kv_layer_stride = (long long)2 * c.max_positions * c.dim; a.kv_slot_stride = a.kv_layer_stride * c.n_layers;
            a.rope = wsf(m, m->o_rope); a.pos = reinterpret_cast<const int32_t*>(m->ws + m->o_pos); a.slots = d_slots;
            a.err = reinterpret_cast<int32_t*>(m->ws + m->o_err);
            a.part = wsf(m, m->o_part); a.arrive = reinterpret_cast<unsigned int*>(m->ws + m->o_arrive); a.max_splits = m->max_splits;
            a.layer = l; a.dim = c.dim; a.hd = c.head_dim; a.max_pos = c.max_positions; a.window = c.window; a.batch = batch; a.heads = c.n_heads;
            prog.push_back(r);
        }
        {   // o_proj, layer scale, residual (in place on the stream)
            RowOp op = base_op();
            set_in(op, m->bATT, 1, false);
            op.W = wsf(m, lo.o); op.N = c.dim; op.epi = EPI_SCALE_RES; op.scale = vec + 4 * c.dim;
            set_out(op, m->bX0); set_res(op, m->bX0);
            push_rows(op);
        }
        {   // LayerNorm -> fc1 -> GELU
            RowOp op = base_op();
            set_in(op, m->bX0, 1, false);
            op.pro = PRO_LN; op.ln_w = vec + 2 * c.dim; op.ln_b = vec + 3 * c.dim; op.eps = c.norm_eps;
            op.W = wsf(m, lo.fc1); op.N = c.ffn; op.epi = EPI_GELU;
            set_out(op, m->bFF);
            push_rows(op);
        }
        {   // fc2, layer scale, residual
            RowOp op = base_op();
            set_in(op, m->bFF, 1, false);
            op.W = wsf(m, lo.fc2); op.N = c.dim; op.epi = EPI_SCALE_RES; op.scale = vec + 5 * c.dim;
            set_out(op, m->bX0); set_res(op, m->bX0);
            push_rows(op);
        }
    }
    // ---- SEANet decoder ----
    const float* bias = wsf(m, m->o_bias);
    {
        RowOp op = base_op();
        set_in(op, m->bX0, c.kernel, false);
        op.W = wsf(m, m->o_conv_in); op.N = m->ch0; op.bias = bias; op.bias_mod = m->ch0; op.epi = EPI_BIAS;
        set_out(op, m->bA0);
        push_rows(op);
        bias += m->ch0;
    }
    int ch = m->ch0, prev = m->bA0;
    for (int i = 0; i < c.n_ratios; ++i) {
        const int r = c.ratios[i];
        ch /= 2;
        {   // ELU -> transposed convolution (kernel 2 r, stride r): row t -> r output rows, contiguous
            RowOp op = base_op();
            set_in(op, prev, 2, true);
            op.pro = PRO_ELU; op.W = wsf(m, m->o_ct[i]); op.N = r * ch; op.bias = bias; op.bias_mod = ch; op.epi = EPI_BIAS;
            set_out(op, m->bCT[i]);
            push_rows(op);
            bias += ch;
        }
        {   // residual block: ELU -> conv k3 -> ELU -> conv k1, + skip
            RowOp op = base_op();
            set_in(op, m->bCT[i], c.res_kernel, false);
            op.pro = PRO_ELU; op.W = wsf(m, m->o_r1[i]); op.N = ch / 2; op.bias = bias; op.bias_mod = ch / 2; op.epi = EPI_BIAS;
            set_out(op, m->bH[i]);
            push_rows(op);
            bias += ch / 2;
            RowOp o2 = base_op();
            set_in(o2, m->bH[i], 1, false);
            o2.pro = PRO_ELU; o2.W = wsf(m, m->o_r2[i]); o2.N = ch; o2.bias = bias; o2.bias_mod = ch; o2.epi = EPI_RES;
            set_out(o2, m->bR[i]); set_res(o2, m->bCT[i]);
            push_rows(o2);
            bias += ch;
        }
        prev = m->bR[i];
    }
    {   // ELU -> conv k3 -> PCM (the caller's buffer, row b)
        RowOp op = base_op();
        set_in(op, prev, c.last_kernel, false);
        op.pro = PRO_ELU; op.W = wsf(m, m->o_conv_out); op.N = 1; op.bias = bias; op.bias_mod = 1; op.epi = EPI_BIAS;
        op.out = d_pcm; op.out_stride = m->spf; op.out_off0 = 0; op.out_by_row = 1;
        push_rows(op);
    }
    {
        OpRec r{}; r.kind = OP_SHIFT;
        r.shift = shift_args(m, d_slots, 0);
        r.shift.batch = batch;
        prog.push_back(r);
    }
}

// one launch per operation, in order, with programmatic dependent launch if `pdl`
static int mimi_enqueue(SmolMimi* m, const std::vector<OpRec>& prog, cudaStream_t st, bool pdl) {
    for (const OpRec& r : prog) {
        switch (r.kind) {
            case OP_ROWS: MIMI_CUDA(launch_rows(r.row, st, pdl)); break;
            case OP_ATTN: MIMI_CUDA(launch_pdl(pdl, attn_kernel, dim3(r.attn.batch, r.attn.heads, r.attn.max_splits), dim3(kThreads), m->attn_smem, st, r.attn)); break;
            case OP_EMBED: MIMI_CUDA(launch_pdl(pdl, embed_kernel, dim3(r.emb.batch), dim3(256), 0, st, r.emb)); break;
            default: MIMI_CUDA(launch_pdl(pdl, shift_kernel, dim3(r.shift.batch, r.shift.n_bufs + 1), dim3(kThreads), 0, st, r.shift)); break;
        }
    }
    m->launches = (int)prog.size();
    return SMOL_OK;
}

extern "C" int smol_mimi_decode_step(SmolMimi* m, const int32_t* d_codes, const int32_t* d_slots, int32_t batch, float* d_pcm, void* stream) {
    if (!m || !d_codes || !d_pcm) return smol::capi_fail(SMOL_ERR_INVALID, "smol_mimi_decode_step: null argument");
    if (!m->bound) return smol::capi_fail(SMOL_ERR_UNBOUND, "smol_mimi_decode_step: weights / workspace not bound");
    if (batch < 1 || batch > m->cfg.max_streams) return smol::capi_fail(SMOL_ERR_CAPACITY, "smol_mimi_decode_step: batch outside 1 .. max_streams");
    cudaStream_t st = (cudaStream_t)stream;
    const int mode = m->cfg.use_graph;   // 0: one launch per operation; 1: those launches replayed as a CUDA graph
    // programmatic dependent launch: every kernel fetches its first weights and prefetches its rows into L2 before the
    // dependency wait.  Measured per step at one stream: plain launches 632 -> 549 us; inside the replayed graph 462 -> 434 us
    // with the final kernels (an earlier, heavier kernel prologue had made it 510 -> 536); at 64 streams it costs 5 % inside the graph
    // (2.40 -> 2.52 ms; nothing either way at 10 streams), so from 12 streams on it is off there
    const bool pdl = mode == 0 || batch < kTileMinBatch;
    SmolMimi::Step* step = nullptr;
    for (SmolMimi::Step& c : m->steps)
        if (c.codes == d_codes && c.slots == d_slots && c.pcm == d_pcm && c.batch == batch) { step = &c; break; }
    if (!step) {
        if (m->steps.size() >= kMaxSteps) {   // evict the least recently used
            size_t lru = 0;
            for (size_t i = 1; i < m->steps.size(); ++i) if (m->steps[i].used < m->steps[lru].used) lru = i;
            if (m->steps[lru].graph) cudaGraphExecDestroy(m->steps[lru].graph);
            m->steps.erase(m->steps.begin() + lru);
        }
        m->steps.push_back(SmolMimi::Step{d_codes, d_slots, d_pcm, batch, {}, nullptr, 0});
        step = &m->steps.back();
        mimi_program(m, d_codes, d_slots, batch, d_pcm, step->prog);
    }
    step->used = ++m->tick;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    const bool capturing = st != nullptr && cudaStreamIsCapturing(st, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone;
    if (mode == 0 || capturing) return mimi_enqueue(m, step->prog, st, pdl);   // (capturing: become part of the caller's graph)
    if (!step->graph) {
        if (!m->cap_stream) MIMI_CUDA(cudaStreamCreateWithFlags(&m->cap_stream, cudaStreamNonBlocking));
        MIMI_CUDA(cudaStreamBeginCapture(m->cap_stream, cudaStreamCaptureModeThreadLocal));
        const int rc = mimi_enqueue(m, step->prog, m->cap_stream, pdl);
        cudaGraph_t g = nullptr;
        const cudaError_t ee = cudaStreamEndCapture(m->cap_stream, &g);
        if (rc != SMOL_OK) { if (g) cudaGraphDestroy(g); return rc; }
        MIMI_CUDA(ee);
        const cudaError_t ei = cudaGraphInstantiate(&step->graph, g, 0);
        cudaGraphDestroy(g);
        MIMI_CUDA(ei);
    }
    MIMI_CUDA(cudaGraphLaunch(step->graph, st));
    return SMOL_OK;
}

extern "C" void* smol_mimi_debug_buffer(SmolMimi* m, const char* name, int64_t* slot_stride_floats) {
    if (!m || !m->bound || !name) return nullptr;
    if (slot_stride_floats) *slot_stride_floats = (int64_t)m->arena_floats;
    float* arena = wsf(m, m->o_arena);
    auto cur = [&](int bi) { const MimiBuf& b = m->bufs[bi]; return (void*)(arena + b.off + (size_t)b.hs * b.C); };
    if (!strcmp(name, "xf") || !strcmp(name, "emb")) return cur(m->bX0);   // (emb: valid with n_layers' launches skipped; see tests)
    if (!strcmp(name, "q")) return cur(m->bQ);
    if (!strcmp(name, "conv_in")) return cur(m->bA0);
    if (!strcmp(name, "res_last")) return cur(m->bR[m->cfg.n_ratios - 1]);
    if (!strcmp(name, "pos")) return (void*)(m->ws + m->o_pos);
    return nullptr;
}
