// What the Mimi decoder (mimi_kernels.cu) and encoder (mimi_encoder.cu) share: device helpers, the 64 x 64 fp32 tile
// GEMM, the bind-time packing kernels and the host-side plan and bind of the transformer layers.  Both files include it,
// so its non-template kernels and host functions are `static` (one private copy per translation unit).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/smoltts_b200_mimi.h"

namespace smol {
int capi_fail(int code, const std::string& msg);              // capi.cu: sets smol_last_error()
int capi_cuda_fail(cudaError_t e, const char* what);

namespace mimi {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;

enum { PRO_NONE = 0, PRO_ELU = 1, PRO_LN = 2 };
enum { EPI_BIAS = 0, EPI_GELU = 1, EPI_SCALE_RES = 2, EPI_RES = 3, EPI_UPSAMPLE = 4 };

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float elu1(float x) { return x > 0.f ? x : expm1f(x); }
__device__ __forceinline__ float4 elu4(float4 v) { return make_float4(elu1(v.x), elu1(v.y), elu1(v.z), elu1(v.w)); }
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }

// Programmatic dependent launch: the decoder launches every kernel of a step with the programmatic-serialization
// attribute, so its CTAs may start while the previous kernel still runs.  Before pdl_wait() a kernel touches only what no
// kernel of the step writes (weights: prefetched into L2); pdl_wait() returns when the previous kernel has completed and
// its writes are visible; pdl_go() lets the next kernel's CTAs start their own prefetch.  Under a plain launch both
// return at once.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_go() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Y[row][n] = epilogue( sum_k A(row, k) W[n][k] ) for MANY rows: a 64 x 64 output tile per CTA (rows on blockIdx.x, which
// allows millions of rows; N on blockIdx.y), K in steps of 16 through shared memory, 4 x 4 outputs per thread -- 16 FMAs
// per pair of 16-byte shared-memory loads.  Every output is one sequential FMA chain over k = 0 .. K-1: deterministic and
// independent of what shares the launch.  Epilogues: bias, then residual | layer scale + residual | GELU.  N is a
// multiple of 4, K of 16.
//
// The operation type says where the rows are (the decoder's slot arena, the encoder's ragged clips):
//   struct Rows;                                   shared-memory row table of a tile
//   void map_rows(Rows&, int row0) const;          every thread calls it before the dependency wait; fills the table and
//                                                  makes it visible to the CTA
//   struct ARow;  ARow a_row(const Rows&, int row0, int m) const;        gather state of tile row m
//   float4 load_a(const ARow&, int k) const;       A(row, k .. k + 3), prologue applied, 0 outside the input
//   bool out_row(const Rows&, int row0, int m, long long& out, long long& res) const;
//                                                  element offsets of (tile row m, n = 0) in `out` and `res`; false: no row
//   int bias_col(int n) const;                     the bias element of column n; for n a multiple of 4, n + 1 .. n + 3
//                                                  take the next three
//   W, K, N, bias, epi, out, res, scale
constexpr int kTM = 64, kTN = 64, kTK = 16;
// (K steps of 32: the decoder's many-row stages 15 .. 30 % slower -- fewer resident CTAs -- measured at 64 streams.)
template <class Op>
__global__ void __launch_bounds__(kThreads, 2) tile_kernel(const Op op) {
    __shared__ __align__(16) float As[kTK][kTM + 4];
    __shared__ __align__(16) float Ws[kTK][kTN + 4];
    __shared__ typename Op::Rows rows;
    const int tid = threadIdx.x;
    const int row0 = blockIdx.x * kTM, n0 = blockIdx.y * kTN;
    op.map_rows(rows, row0);
    pdl_wait();
    pdl_go();
    const int lm = tid >> 2, lk = (tid & 3) << 2;      // this thread's row (of A and of W) and k offset of the 16-byte pieces it loads
    const typename Op::ARow ar = op.a_row(rows, row0, lm);
    const bool w_ok = n0 + lm < op.N;
    const float* w_base = op.W + (long long)(n0 + lm) * op.K;
    auto load_w = [&](int k) -> float4 {
        return w_ok ? __ldg(reinterpret_cast<const float4*>(w_base + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    const int ty = tid >> 4, tx = tid & 15;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    float4 ra = op.load_a(ar, lk), rw = load_w(lk);
    for (int k0 = 0; k0 < op.K; k0 += kTK) {
        As[lk + 0][lm] = ra.x; As[lk + 1][lm] = ra.y; As[lk + 2][lm] = ra.z; As[lk + 3][lm] = ra.w;
        Ws[lk + 0][lm] = rw.x; Ws[lk + 1][lm] = rw.y; Ws[lk + 2][lm] = rw.z; Ws[lk + 3][lm] = rw.w;
        __syncthreads();
        if (k0 + kTK < op.K) { ra = op.load_a(ar, k0 + kTK + lk); rw = load_w(k0 + kTK + lk); }   // next step's pieces in flight during the FMAs
#pragma unroll
        for (int k = 0; k < kTK; ++k) {
            const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
            const float4 w = *reinterpret_cast<const float4*>(&Ws[k][tx * 4]);
            acc[0][0] = fmaf(a.x, w.x, acc[0][0]); acc[0][1] = fmaf(a.x, w.y, acc[0][1]); acc[0][2] = fmaf(a.x, w.z, acc[0][2]); acc[0][3] = fmaf(a.x, w.w, acc[0][3]);
            acc[1][0] = fmaf(a.y, w.x, acc[1][0]); acc[1][1] = fmaf(a.y, w.y, acc[1][1]); acc[1][2] = fmaf(a.y, w.z, acc[1][2]); acc[1][3] = fmaf(a.y, w.w, acc[1][3]);
            acc[2][0] = fmaf(a.z, w.x, acc[2][0]); acc[2][1] = fmaf(a.z, w.y, acc[2][1]); acc[2][2] = fmaf(a.z, w.z, acc[2][2]); acc[2][3] = fmaf(a.z, w.w, acc[2][3]);
            acc[3][0] = fmaf(a.w, w.x, acc[3][0]); acc[3][1] = fmaf(a.w, w.y, acc[3][1]); acc[3][2] = fmaf(a.w, w.z, acc[3][2]); acc[3][3] = fmaf(a.w, w.w, acc[3][3]);
        }
        __syncthreads();
    }
    const int n = n0 + tx * 4;
    if (n >= op.N) return;                      // (N is a multiple of 4: the four columns of a thread are all in or all out)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        long long oe, re;
        if (!op.out_row(rows, row0, ty * 4 + i, oe, re)) continue;
        float4 y = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        if (op.bias) {
            const float* b = op.bias + op.bias_col(n);
            y.x += b[0]; y.y += b[1]; y.z += b[2]; y.w += b[3];
        }
        if (op.epi == EPI_RES) {
            const float4 r = *reinterpret_cast<const float4*>(op.res + re + n);
            y.x = r.x + y.x; y.y = r.y + y.y; y.z = r.z + y.z; y.w = r.w + y.w;
        } else if (op.epi == EPI_SCALE_RES) {
            const float4 r = *reinterpret_cast<const float4*>(op.res + re + n);
            y.x = r.x + y.x * op.scale[n]; y.y = r.y + y.y * op.scale[n + 1]; y.z = r.z + y.z * op.scale[n + 2]; y.w = r.w + y.w * op.scale[n + 3];
        } else if (op.epi == EPI_GELU) {
            y.x = gelu_erf(y.x); y.y = gelu_erf(y.y); y.z = gelu_erf(y.z); y.w = gelu_erf(y.w);
        }
        *reinterpret_cast<float4*>(op.out + oe + n) = y;
    }
}

// ---- bind-time packing -----------------------------------------------------------------------------------------------
static __global__ void pack_codebook_kernel(float* dst, const float* es, const float* cu, int rows, int dim, float eps) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)rows * dim; i += (long long)gridDim.x * blockDim.x)
        dst[i] = es[i] / fmaxf(cu[i / dim], eps);
}
// Conv1d [Co][Ci][k] -> [Co][j * Ci + ci]
static __global__ void pack_conv_kernel(float* dst, const float* w, int Co, int Ci, int k) {
    const long long total = (long long)Co * Ci * k;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
        const int ci = (int)(i % Ci); const long long r = i / Ci; const int j = (int)(r % k); const int co = (int)(r / k);
        dst[i] = w[((long long)co * Ci + ci) * k + j];
    }
}

// ---- host: workspace plan and the transformer layers' bind -----------------------------------------------------------
#define MIMI_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return smol::capi_cuda_fail(e__, #call); } while (0)

// Offsets (bytes) of consecutive 256-byte-aligned regions of a workspace.
struct WsPlan {
    size_t total = 0;
    size_t take(size_t floats) { const size_t r = total; total = (total + floats * 4 + 255) / 256 * 256; return r; }
};

// One transformer layer packed in a workspace: q|k|v fused [3 dim][dim], o [dim][dim], fc1 [ffn][dim], fc2 [dim][ffn],
// vec = ln1 w|b, ln2 w|b, scale_attn, scale_mlp [6][dim].
struct LayerOffsets { size_t qkv, o, fc1, fc2, vec; };

static LayerOffsets plan_layer(WsPlan& p, int dim, int ffn) {
    LayerOffsets L;
    L.qkv = p.take((size_t)3 * dim * dim);
    L.o = p.take((size_t)dim * dim);
    L.fc1 = p.take((size_t)ffn * dim);
    L.fc2 = p.take((size_t)dim * ffn);
    L.vec = p.take((size_t)6 * dim);
    return L;
}

static bool layer_weights_ok(const SmolMimiLayerWeights& L) {
    return L.q_proj && L.k_proj && L.v_proj && L.o_proj && L.fc1 && L.fc2 && L.ln1_w && L.ln1_b && L.ln2_w && L.ln2_b &&
           L.scale_attn && L.scale_mlp;
}

static int bind_layer(unsigned char* ws, const LayerOffsets& o, const SmolMimiLayerWeights& L, int dim, int ffn, cudaStream_t st) {
    auto d2d = [&](size_t off, const float* src, size_t floats) { return cudaMemcpyAsync(ws + off, src, floats * sizeof(float), cudaMemcpyDeviceToDevice, st); };
    const size_t dd = (size_t)dim * dim;
    MIMI_CUDA(d2d(o.qkv, L.q_proj, dd));
    MIMI_CUDA(d2d(o.qkv + dd * sizeof(float), L.k_proj, dd));
    MIMI_CUDA(d2d(o.qkv + 2 * dd * sizeof(float), L.v_proj, dd));
    MIMI_CUDA(d2d(o.o, L.o_proj, dd));
    MIMI_CUDA(d2d(o.fc1, L.fc1, (size_t)ffn * dim));
    MIMI_CUDA(d2d(o.fc2, L.fc2, (size_t)ffn * dim));
    const float* vecs[6] = {L.ln1_w, L.ln1_b, L.ln2_w, L.ln2_b, L.scale_attn, L.scale_mlp};
    for (int i = 0; i < 6; ++i) MIMI_CUDA(d2d(o.vec + (size_t)i * dim * sizeof(float), vecs[i], dim));
    return SMOL_OK;
}

}  // namespace mimi
}  // namespace smol
