// The Mimi encoder (PCM -> codes) for sm_100a, pinned to transformers' MimiModel.encode (the model the reference's codec
// mirrors).  A whole-clip program over all clips of a call at once, not a streaming step:
//
//   SEANet encoder   conv k7 (1 -> 64); per ratio 4, 5, 6, 8: [residual block: ELU, conv k3 C -> C/2, ELU, conv k1 C/2 -> C,
//                    + skip], ELU, conv k = 2 r stride r (C -> 2 C); ELU, conv k3 (1024 -> 512)         -> 25 Hz rows
//   transformer      8 layers: LayerNorm, q|k|v, half-split RoPE (positions from 0 per clip), causal attention over a
//                    sliding window of 250 positions, o_proj + layer scale, LayerNorm, fc1, exact GELU, fc2 + layer scale
//   downsample       conv k4 stride 2, no bias, REPLICATE padding                                      -> 12.5 Hz latent z
//   split RVQ        the semantic codebook on P_s z; 7 acoustic codebooks in sequence on a residual that starts from P_a z:
//                    first-index argmin of |e|^2 - 2 r.e (|r|^2 is the same for every row), r -= e_idx
//
// Every causal convolution pads k - stride zero rows on the left of ITS input; a strided one also pads zero rows on the
// right up to a multiple of its stride (T_out = ceil(T_in / r)).  Those rows are never stored: the tile kernel's gather
// returns 0 (or, for the downsample, the clip's edge row) for a source row outside the clip.  A clip's rows are a
// contiguous run of every level's buffer; a row's clip is found in the per-call table of row offsets (`Segs`, passed by
// value, so a call needs no host-to-device copy).
//
// One kernel per kind of operation, whatever the batch: every output is one sequential FMA chain (convolutions,
// Linears, RVQ distances), attention sums in a fixed order per query, and nothing depends on which rows share a launch --
// a clip's codes and latent are the same bits alone or in any batch.  No atomics.
//
// Convolutions are the decoder's "(previous | current rows)" product: in the row-major [T][C] layout the k taps of a
// causal convolution at output row t are the contiguous run of k C floats starting at input row t s - (k - s), so the
// packed weight [out][tap C + c] is a plain GEMM operand.

#include <cuda_runtime.h>
#include <stdint.h>

#include <algorithm>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "../../include/smoltts_b200.h"
#include "../../include/smoltts_b200_mimi.h"
#include "mimi_common.cuh"

namespace smol {
namespace mimi_enc {
using namespace smol::mimi;

constexpr int kMaxClips = 256;
constexpr int kMaxWindow = 1024;

// Row offsets of the clips of one call at one level: clip b owns output rows out_off[b] .. out_off[b + 1] and reads input
// rows in_off[b] .. in_off[b + 1].  n = 0: one sequence (a Linear: output row = input row).
struct Segs {
    int n;
    int in_off[kMaxClips + 1];
    int out_off[kMaxClips + 1];
};

__device__ __forceinline__ int seg_find(const Segs& s, int row) {   // the clip of output row `row` (n >= 1)
    int lo = 0, hi = s.n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (s.out_off[mid] <= row) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// out[row][n] = epilogue( sum_k A(row, k) W[n][k] ), A(row, tap j * cin + c) = prologue( in[clip row t stride - pad + j][c] ):
// the rows of tile_kernel<EncOp>.  A source row outside its clip reads 0, or with `replicate` the clip's edge row.
struct EncOp {
    const float* in; int cin, stride, pad, replicate, pro;
    const float* W; const float* bias; int N, K;
    float* out; int epi; const float* res; const float* scale;
    int rows;
    Segs seg;

    struct Rows {};                                     // (a row's clip is found per thread: no shared row table)
    __device__ void map_rows(Rows&, int) const {}
    struct ARow { long long base; int t0, tin; bool ok; };   // clip base row, first tap's source row, clip length
    __device__ ARow a_row(const Rows&, int row0, int m) const {
        const int arow = row0 + m;
        ARow a{0, 0, 1, arow < rows};
        if (a.ok) {
            if (seg.n == 0) { a.t0 = arow * stride - pad; a.tin = rows; }
            else {
                const int b = seg_find(seg, arow);
                a.base = seg.in_off[b];
                a.t0 = (arow - seg.out_off[b]) * stride - pad;
                a.tin = seg.in_off[b + 1] - seg.in_off[b];
            }
        }
        return a;
    }
    __device__ float4 load_a(const ARow& a, int k) const {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (a.ok) {
            const int j = k / cin, c = k - j * cin;
            int sr = a.t0 + j;
            if (replicate) sr = min(max(sr, 0), a.tin - 1);
            if (sr >= 0 && sr < a.tin) {
                v = *reinterpret_cast<const float4*>(in + (a.base + sr) * cin + c);
                if (pro == PRO_ELU) v = elu4(v);
            }
        }
        return v;
    }
    __device__ bool out_row(const Rows&, int row0, int m, long long& oe, long long& re) const {
        const int row = row0 + m;
        if (row >= rows) return false;
        oe = re = (long long)row * N;
        return true;
    }
    __device__ int bias_col(int n) const { return n; }
};

// The one-channel first convolution (K = kernel does not fit the tiles): one thread per (sample row, output channel).
__global__ void __launch_bounds__(kThreads) enc_conv_in_kernel(const float* __restrict__ pcm, const float* __restrict__ w,
                                                               const float* __restrict__ bias, float* __restrict__ out, int rows,
                                                               int C, int k, const Segs seg) {
    const long long i = (long long)blockIdx.x * kThreads + threadIdx.x;
    if (i >= (long long)rows * C) return;
    const int row = (int)(i / C), c = (int)(i - (long long)row * C);
    const int b = seg_find(seg, row);
    const int t = row - seg.out_off[b], base = seg.in_off[b];
    float acc = 0.f;
    for (int j = 0; j < k; ++j) {
        const int sr = t - (k - 1) + j;
        const float x = sr >= 0 ? pcm[base + sr] : 0.f;
        acc = fmaf(x, w[c * k + j], acc);
    }
    out[i] = acc + bias[c];
}

// LayerNorm of every row (one warp per row; two passes, as torch does).
__global__ void __launch_bounds__(kThreads) enc_ln_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                          const float* __restrict__ b, float* __restrict__ out, int rows, int D, float eps) {
    const int row = blockIdx.x * kWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= rows) return;
    const float* xr = x + (long long)row * D;
    float s = 0.f;
    for (int k = lane; k < D; k += 32) s += xr[k];
    const float mean = warp_sum(s) / (float)D;
    float d2 = 0.f;
    for (int k = lane; k < D; k += 32) { const float d = xr[k] - mean; d2 = fmaf(d, d, d2); }
    const float rstd = 1.0f / sqrtf(warp_sum(d2) / (float)D + eps);
    float* o = out + (long long)row * D;
    for (int k = lane; k < D; k += 32) o[k] = (xr[k] - mean) * rstd * w[k] + b[k];
}

// Half-split RoPE of q and k in place (qkv rows [q | k | v]); a row's position is its index inside its clip.
__global__ void __launch_bounds__(kThreads) enc_rope_kernel(float* __restrict__ qkv, const float* __restrict__ rope, int rows, int dim,
                                                            int hd, const Segs seg) {
    const int half = hd >> 1, per_row = dim / 2;   // (head, pair) per row
    const long long i = (long long)blockIdx.x * kThreads + threadIdx.x;
    if (i >= (long long)rows * per_row) return;
    const int row = (int)(i / per_row), p = (int)(i - (long long)row * per_row);
    const int h = p / half, j = p - h * half;
    const int t = row - seg.out_off[seg_find(seg, row)];
    const float cs = rope[(long long)t * hd + j], sn = rope[(long long)t * hd + half + j];
    float* r = qkv + (long long)row * 3 * dim + h * hd;
#pragma unroll
    for (int u = 0; u < 2; ++u) {   // q, then k
        float* v = r + u * dim;
        const float a = v[j], c = v[j + half];
        v[j] = a * cs - c * sn;
        v[j + half] = c * cs + a * sn;
    }
}

// Causal sliding-window attention, one warp per (query row, head): query t of a clip sees its positions t - window < j <= t.
// Scores by one lane per key (a sequential 4-wide dot product), the maximum and the sum of exponentials by a fixed shuffle
// tree, then P V with hd / 32 dims per lane, keys in order.
__global__ void __launch_bounds__(kThreads) enc_attn_kernel(const float* __restrict__ qkv, float* __restrict__ att, int rows, int dim,
                                                            int hd, int window, const Segs seg) {
    extern __shared__ __align__(16) float sm[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int row = blockIdx.x * kWarps + warp, h = blockIdx.y;
    float* q = sm + warp * (hd + ((window + 3) & ~3));   // (16-byte aligned per warp: q is read as float4)
    float* p = q + hd;
    if (row >= rows) return;                     // (a warp's work is its own: no block-wide barrier below)
    const int b = seg_find(seg, row);
    const int first = max(seg.out_off[b], row - window + 1), nk = row - first + 1;
    const float scale = rsqrtf((float)hd);
    for (int d = lane; d < hd; d += 32) q[d] = qkv[(long long)row * 3 * dim + h * hd + d] * scale;
    __syncwarp();
    float m = -INFINITY;
    for (int i = lane; i < nk; i += 32) {
        const float4* kr = reinterpret_cast<const float4*>(qkv + (long long)(first + i) * 3 * dim + dim + h * hd);
        float s = 0.f;
        for (int d4 = 0; d4 < hd / 4; ++d4) {
            const float4 kk = kr[d4];
            const float4 qq = *reinterpret_cast<const float4*>(q + 4 * d4);
            s = fmaf(qq.x, kk.x, s); s = fmaf(qq.y, kk.y, s); s = fmaf(qq.z, kk.z, s); s = fmaf(qq.w, kk.w, s);
        }
        p[i] = s;
        m = fmaxf(m, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    float l = 0.f;
    for (int i = lane; i < nk; i += 32) { const float e = expf(p[i] - m); p[i] = e; l += e; }
    l = warp_sum(l);
    __syncwarp();
    float o[4] = {0.f, 0.f, 0.f, 0.f};
    const float* vb = qkv + 2 * dim + h * hd;
    for (int i = 0; i < nk; ++i) {
        const float pi = p[i];
        const float* vr = vb + (long long)(first + i) * 3 * dim;
#pragma unroll
        for (int u = 0; u < 4; ++u) if (u * 32 < hd) o[u] = fmaf(pi, vr[u * 32 + lane], o[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) if (u * 32 < hd) att[(long long)row * dim + h * hd + u * 32 + lane] = o[u] / l;
}

// One codebook of the RVQ for every frame (one warp per frame): d_j = |e_j|^2 - 2 r.e_j from the scores of the tile kernel,
// first-index argmin (each lane scans its indices in order, the shuffle tree keeps the smaller index on a tie), the code,
// and the residual update r -= e_idx.
__global__ void __launch_bounds__(kThreads) enc_argmin_kernel(const float* __restrict__ scores, const float* __restrict__ norms,
                                                              const float* __restrict__ book, float* __restrict__ resid,
                                                              int32_t* __restrict__ codes, int frames, int cs, int cd, int n_q, int q) {
    const int f = blockIdx.x * kWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (f >= frames) return;
    const float* s = scores + (long long)f * cs;
    float best = INFINITY;
    int idx = 0x7fffffff;
    for (int j = lane; j < cs; j += 32) {
        const float d = fmaf(-2.f, s[j], norms[j]);
        if (d < best) { best = d; idx = j; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ob = __shfl_xor_sync(0xffffffffu, best, o);
        const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
        if (ob < best || (ob == best && oi < idx)) { best = ob; idx = oi; }
    }
    if (idx == 0x7fffffff) idx = 0;   // (only for non-finite scores)
    if (lane == 0) codes[(long long)f * n_q + q] = idx;
    const float* e = book + (long long)idx * cd;
    float* r = resid + (long long)f * cd;
    for (int c = lane; c < cd; c += 32) r[c] = r[c] - e[c];
}

// ---- bind-time packing (codebooks and Conv1d: mimi_common.cuh) ------------------------------------------------------
// |e_j|^2 of the packed rows, a sequential sum per row
__global__ void enc_row_norm_kernel(float* dst, const float* rows_, int rows, int dim) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= rows) return;
    const float* r = rows_ + (long long)j * dim;
    float s = 0.f;
    for (int c = 0; c < dim; ++c) s = fmaf(r[c], r[c], s);
    dst[j] = s;
}
}  // namespace mimi_enc
}  // namespace smol

// ---- host side -------------------------------------------------------------------------------------------------------
using namespace smol::mimi_enc;

struct SmolMimiEncoder {
    SmolMimiEncoderConfig cfg{};
    int n_st = 0;                                   // SEANet stages
    int ratio[SMOL_MIMI_MAX_RATIOS];                // ratio of stage i (the config's list reversed)
    long long hop = 1;                              // samples per 25 Hz row = prod(ratios)
    long long cap_rows[SMOL_MIMI_MAX_RATIOS + 1];   // row capacity of level i (samples / prod of the first i ratios + max_clips)
    long long cap_frames = 0, max_pos = 0;
    // workspace layout (bytes)
    size_t o_conv_in = 0, o_r1[SMOL_MIMI_MAX_RATIOS], o_r2[SMOL_MIMI_MAX_RATIOS], o_dn[SMOL_MIMI_MAX_RATIOS], o_conv_out = 0, o_bias = 0;
    LayerOffsets o_layer[SMOL_MIMI_MAX_LAYERS];
    size_t o_ds = 0, o_proj = 0, o_books = 0, o_norms = 0, o_rope = 0;
    size_t o_P = 0, o_Q = 0, o_H = 0, o_X = 0, o_Hn = 0, o_QKV = 0, o_ATT = 0, o_FF = 0, o_Z = 0, o_RS = 0, o_RA = 0, o_S = 0, total = 0;
    unsigned char* ws = nullptr;
    bool bound = false;
    int launches = 0;
};

static void enc_plan(SmolMimiEncoder* e) {
    const SmolMimiEncoderConfig& c = e->cfg;
    e->n_st = c.n_ratios;
    long long div = 1;
    for (int i = 0; i < c.n_ratios; ++i) { e->ratio[i] = c.ratios[c.n_ratios - 1 - i]; }
    e->cap_rows[0] = c.max_samples;
    size_t big = (size_t)c.max_samples * c.n_filters, half = big / 2;
    for (int i = 0; i < c.n_ratios; ++i) {
        div *= e->ratio[i];
        e->cap_rows[i + 1] = c.max_samples / div + c.max_clips;
        const size_t ch = (size_t)c.n_filters << (i + 1);
        big = std::max(big, (size_t)e->cap_rows[i + 1] * ch);
        if (i + 1 < c.n_ratios) half = std::max(half, (size_t)e->cap_rows[i + 1] * ch / 2);
    }
    e->hop = div;
    e->max_pos = (c.max_samples + div - 1) / div;
    e->cap_frames = c.max_samples / (2 * div) + c.max_clips;
    const long long R = e->cap_rows[c.n_ratios];
    WsPlan p;
    e->o_conv_in = p.take((size_t)c.n_filters * c.kernel);
    int ch = c.n_filters;
    size_t nb = c.n_filters;
    for (int i = 0; i < c.n_ratios; ++i) {
        e->o_r1[i] = p.take((size_t)(ch / 2) * ch * c.res_kernel);
        e->o_r2[i] = p.take((size_t)ch * (ch / 2));
        e->o_dn[i] = p.take((size_t)2 * ch * ch * 2 * e->ratio[i]);
        nb += (size_t)ch / 2 + ch + 2 * ch;
        ch *= 2;
    }
    e->o_conv_out = p.take((size_t)c.dim * ch * c.last_kernel);
    nb += c.dim;
    e->o_bias = p.take(nb);
    for (int l = 0; l < c.n_layers; ++l) e->o_layer[l] = plan_layer(p, c.dim, c.ffn);
    e->o_ds = p.take((size_t)c.dim * c.dim * 4);
    e->o_proj = p.take((size_t)2 * c.codebook_dim * c.dim);
    e->o_books = p.take((size_t)c.n_q * c.codebook_size * c.codebook_dim);
    e->o_norms = p.take((size_t)c.n_q * c.codebook_size);
    e->o_rope = p.take((size_t)e->max_pos * c.head_dim);
    // activations: SEANet ping-pong (P, Q) and residual hidden rows (H); transformer rows; latent and RVQ
    e->o_P = p.take(big);
    e->o_Q = p.take(big);
    e->o_H = p.take(half);
    e->o_X = p.take((size_t)R * c.dim);
    e->o_Hn = p.take((size_t)R * c.dim);
    e->o_QKV = p.take((size_t)R * 3 * c.dim);
    e->o_ATT = p.take((size_t)R * c.dim);
    e->o_FF = p.take((size_t)R * c.ffn);
    e->o_Z = p.take((size_t)e->cap_frames * c.dim);
    e->o_RS = p.take((size_t)e->cap_frames * c.codebook_dim);
    e->o_RA = p.take((size_t)e->cap_frames * c.codebook_dim);
    e->o_S = p.take((size_t)e->cap_frames * c.codebook_size);
    e->total = p.total;
}

extern "C" int smol_mimi_encoder_create(const SmolMimiEncoderConfig* cfg, SmolMimiEncoder** out) {
    using smol::capi_fail;
    if (!cfg || !out) return capi_fail(SMOL_ERR_INVALID, "smol_mimi_encoder_create: null argument");
    const SmolMimiEncoderConfig& c = *cfg;
    if (c.n_q < 2 || c.n_q > SMOL_MIMI_MAX_Q) return capi_fail(SMOL_ERR_INVALID, "mimi encoder: n_q must be 2 .. 32");
    if (c.n_layers < 1 || c.n_layers > SMOL_MIMI_MAX_LAYERS) return capi_fail(SMOL_ERR_INVALID, "mimi encoder: n_layers out of range");
    if (c.n_ratios < 1 || c.n_ratios > SMOL_MIMI_MAX_RATIOS) return capi_fail(SMOL_ERR_INVALID, "mimi encoder: n_ratios out of range");
    if (c.dim != c.n_heads * c.head_dim || c.n_heads < 1) return capi_fail(SMOL_ERR_INVALID, "mimi encoder: dim != n_heads * head_dim");
    if (c.head_dim % 32 || c.head_dim > 128) return capi_fail(SMOL_ERR_UNSUPPORTED, "mimi encoder: head_dim must be 32, 64, 96 or 128");
    if (c.dim % 16 || c.ffn % 16 || c.codebook_dim % 16 || c.n_filters % 32 || c.codebook_size % 4 || c.codebook_size < 1)
        return capi_fail(SMOL_ERR_UNSUPPORTED, "mimi encoder: dim, ffn and codebook_dim must be multiples of 16, n_filters of 32, codebook_size of 4");
    if (c.kernel < 1 || c.res_kernel < 1 || c.last_kernel < 1) return capi_fail(SMOL_ERR_INVALID, "mimi encoder: kernel sizes");
    for (int i = 0; i < c.n_ratios; ++i) if (c.ratios[i] < 1) return capi_fail(SMOL_ERR_INVALID, "mimi encoder: ratios must be positive");
    if (c.window < 1 || c.window > kMaxWindow) return capi_fail(SMOL_ERR_UNSUPPORTED, "mimi encoder: window must be 1 .. 1024");
    if (c.max_clips < 1 || c.max_samples < 1) return capi_fail(SMOL_ERR_INVALID, "mimi encoder: max_clips and max_samples must be >= 1");
    if (c.max_clips > kMaxClips) return capi_fail(SMOL_ERR_CAPACITY, "mimi encoder: max_clips above 256");
    if (c.max_samples > (1 << 30) / c.n_filters) return capi_fail(SMOL_ERR_CAPACITY, "mimi encoder: max_samples x n_filters above 2^30");
    SmolMimiEncoder* e = new SmolMimiEncoder();
    e->cfg = c;
    enc_plan(e);
    *out = e;
    return SMOL_OK;
}

extern "C" void smol_mimi_encoder_destroy(SmolMimiEncoder* e) { delete e; }
extern "C" int32_t smol_mimi_encoder_samples_per_frame(const SmolMimiEncoder* e) { return e ? (int32_t)(2 * e->hop) : 0; }
extern "C" size_t smol_mimi_encoder_workspace_bytes(const SmolMimiEncoder* e) { return e ? e->total : 0; }
extern "C" int32_t smol_mimi_encoder_launches(const SmolMimiEncoder* e) { return e ? e->launches : 0; }

static float* ews(SmolMimiEncoder* e, size_t off) { return reinterpret_cast<float*>(e->ws + off); }

extern "C" int smol_mimi_encoder_bind(SmolMimiEncoder* e, const SmolMimiEncoderWeights* w, void* d_workspace, size_t workspace_bytes,
                                      void* stream) {
    using smol::capi_fail;
    if (!e || !w || !d_workspace) return capi_fail(SMOL_ERR_INVALID, "smol_mimi_encoder_bind: null argument");
    if (workspace_bytes < e->total) return capi_fail(SMOL_ERR_CAPACITY, "smol_mimi_encoder_bind: workspace smaller than smol_mimi_encoder_workspace_bytes()");
    if ((uintptr_t)d_workspace % 256) return capi_fail(SMOL_ERR_INVALID, "smol_mimi_encoder_bind: workspace must be 256-byte aligned");
    const SmolMimiEncoderConfig& c = e->cfg;
    bool ok = w->semantic_input_proj && w->acoustic_input_proj && w->downsample && w->rope && w->conv_in.weight && w->conv_in.bias &&
              w->conv_out.weight && w->conv_out.bias;
    for (int i = 0; i < c.n_q; ++i) ok = ok && w->embed_sum[i] && w->cluster_usage[i];
    for (int l = 0; l < c.n_layers; ++l) ok = ok && layer_weights_ok(w->layers[l]);
    for (int i = 0; i < c.n_ratios; ++i)
        ok = ok && w->res_conv1[i].weight && w->res_conv1[i].bias && w->res_conv2[i].weight && w->res_conv2[i].bias &&
             w->conv_down[i].weight && w->conv_down[i].bias;
    if (!ok) return capi_fail(SMOL_ERR_INVALID, "smol_mimi_encoder_bind: a weight pointer is null");
    e->ws = reinterpret_cast<unsigned char*>(d_workspace);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t f4 = sizeof(float);
    auto d2d = [&](size_t off, const float* src, size_t floats) { return cudaMemcpyAsync(e->ws + off, src, floats * f4, cudaMemcpyDeviceToDevice, st); };
    MIMI_CUDA(d2d(e->o_conv_in, w->conv_in.weight, (size_t)c.n_filters * c.kernel));
    size_t bo = e->o_bias;
    MIMI_CUDA(d2d(bo, w->conv_in.bias, c.n_filters)); bo += (size_t)c.n_filters * f4;
    int ch = c.n_filters;
    for (int i = 0; i < c.n_ratios; ++i) {
        pack_conv_kernel<<<256, 256, 0, st>>>(ews(e, e->o_r1[i]), w->res_conv1[i].weight, ch / 2, ch, c.res_kernel);
        MIMI_CUDA(d2d(e->o_r2[i], w->res_conv2[i].weight, (size_t)ch * (ch / 2)));
        pack_conv_kernel<<<512, 256, 0, st>>>(ews(e, e->o_dn[i]), w->conv_down[i].weight, 2 * ch, ch, 2 * e->ratio[i]);
        MIMI_CUDA(d2d(bo, w->res_conv1[i].bias, ch / 2)); bo += (size_t)(ch / 2) * f4;
        MIMI_CUDA(d2d(bo, w->res_conv2[i].bias, ch)); bo += (size_t)ch * f4;
        MIMI_CUDA(d2d(bo, w->conv_down[i].bias, 2 * ch)); bo += (size_t)2 * ch * f4;
        ch *= 2;
    }
    pack_conv_kernel<<<512, 256, 0, st>>>(ews(e, e->o_conv_out), w->conv_out.weight, c.dim, ch, c.last_kernel);
    MIMI_CUDA(d2d(bo, w->conv_out.bias, c.dim));
    for (int l = 0; l < c.n_layers; ++l) {
        const int rc = bind_layer(e->ws, e->o_layer[l], w->layers[l], c.dim, c.ffn, st);
        if (rc != SMOL_OK) return rc;
    }
    pack_conv_kernel<<<512, 256, 0, st>>>(ews(e, e->o_ds), w->downsample, c.dim, c.dim, 4);
    MIMI_CUDA(d2d(e->o_proj, w->semantic_input_proj, (size_t)c.codebook_dim * c.dim));
    MIMI_CUDA(d2d(e->o_proj + (size_t)c.codebook_dim * c.dim * f4, w->acoustic_input_proj, (size_t)c.codebook_dim * c.dim));
    const size_t book = (size_t)c.codebook_size * c.codebook_dim;
    for (int i = 0; i < c.n_q; ++i) {
        pack_codebook_kernel<<<256, 256, 0, st>>>(ews(e, e->o_books) + i * book, w->embed_sum[i], w->cluster_usage[i], c.codebook_size,
                                                      c.codebook_dim, c.codebook_eps);
        enc_row_norm_kernel<<<(c.codebook_size + 255) / 256, 256, 0, st>>>(ews(e, e->o_norms) + (size_t)i * c.codebook_size,
                                                                           ews(e, e->o_books) + i * book, c.codebook_size, c.codebook_dim);
    }
    MIMI_CUDA(d2d(e->o_rope, w->rope, (size_t)e->max_pos * c.head_dim));
    MIMI_CUDA(cudaGetLastError());
    e->bound = true;
    return SMOL_OK;
}

extern "C" int smol_mimi_encode(SmolMimiEncoder* e, const float* d_pcm, const int64_t* h_lengths, int32_t n, int32_t* d_codes, void* stream) {
    using smol::capi_fail;
    if (!e || !d_pcm || !h_lengths || !d_codes) return capi_fail(SMOL_ERR_INVALID, "smol_mimi_encode: null argument");
    if (!e->bound) return capi_fail(SMOL_ERR_UNBOUND, "smol_mimi_encode: weights / workspace not bound");
    const SmolMimiEncoderConfig& c = e->cfg;
    if (n < 1 || n > c.max_clips) return capi_fail(SMOL_ERR_CAPACITY, "smol_mimi_encode: n outside 1 .. max_clips");
    long long total = 0;
    for (int b = 0; b < n; ++b) {
        if (h_lengths[b] < 1) return capi_fail(SMOL_ERR_INVALID, "smol_mimi_encode: clip " + std::to_string(b) + " has no samples");
        total += h_lengths[b];
    }
    if (total > c.max_samples)
        return capi_fail(SMOL_ERR_CAPACITY, "smol_mimi_encode: " + std::to_string(total) + " samples above max_samples = " + std::to_string(c.max_samples));
    cudaStream_t st = (cudaStream_t)stream;
    // row offsets of every level: 0 = samples, i + 1 = after stage i (ceil(T / r) rows), then the 12.5 Hz frames
    std::vector<std::vector<int>> lvl(e->n_st + 2, std::vector<int>(n + 1, 0));
    for (int b = 0; b < n; ++b) {
        long long T = h_lengths[b];
        lvl[0][b + 1] = lvl[0][b] + (int)T;
        for (int i = 0; i < e->n_st; ++i) { T = (T + e->ratio[i] - 1) / e->ratio[i]; lvl[i + 1][b + 1] = lvl[i + 1][b] + (int)T; }
        T = (T + 1) / 2;
        lvl[e->n_st + 1][b + 1] = lvl[e->n_st + 1][b] + (int)T;
    }
    auto segs = [&](int li, int lo) { Segs s; s.n = n; for (int b = 0; b <= n; ++b) { s.in_off[b] = lvl[li][b]; s.out_off[b] = lvl[lo][b]; } return s; };
    int launches = 0;
    auto tile = [&](const EncOp& op) -> cudaError_t {
        const dim3 grid((op.rows + kTM - 1) / kTM, (op.N + kTN - 1) / kTN);
        tile_kernel<EncOp><<<grid, kThreads, 0, st>>>(op);
        ++launches;
        return cudaGetLastError();
    };
    auto conv = [&](const float* in, int cin, int k, int stride, int replicate, int pro, const float* W, const float* bias, int N, float* out,
                    int epi, const float* res, int li, int lo) {
        EncOp op{};
        op.in = in; op.cin = cin; op.stride = stride; op.pad = k - stride; op.replicate = replicate; op.pro = pro;
        op.W = W; op.bias = bias; op.N = N; op.K = k * cin; op.out = out; op.epi = epi; op.res = res;
        op.seg = segs(li, lo); op.rows = lvl[lo][n];
        return tile(op);
    };
    auto linear = [&](const float* in, int K, const float* W, int N, float* out, int epi, const float* res, const float* scale, int rows) {
        EncOp op{};
        op.in = in; op.cin = K; op.stride = 1; op.W = W; op.N = N; op.K = K; op.out = out; op.epi = epi; op.res = res; op.scale = scale;
        op.rows = rows; op.seg.n = 0;
        return tile(op);
    };
    float *P = ews(e, e->o_P), *Q = ews(e, e->o_Q), *H = ews(e, e->o_H);
    const float* bias = ews(e, e->o_bias);
    {   // conv k7, one channel in
        const long long cnt = (long long)lvl[0][n] * c.n_filters;
        enc_conv_in_kernel<<<(unsigned)((cnt + kThreads - 1) / kThreads), kThreads, 0, st>>>(d_pcm, ews(e, e->o_conv_in), bias, P, lvl[0][n],
                                                                                           c.n_filters, c.kernel, segs(0, 0));
        ++launches;
        MIMI_CUDA(cudaGetLastError());
        bias += c.n_filters;
    }
    int ch = c.n_filters;
    for (int i = 0; i < e->n_st; ++i) {
        // residual block: ELU -> conv k3 (C -> C/2) -> ELU -> conv k1 (C/2 -> C), + skip (in place on P)
        MIMI_CUDA(conv(P, ch, c.res_kernel, 1, 0, PRO_ELU, ews(e, e->o_r1[i]), bias, ch / 2, H, EPI_BIAS, nullptr, i, i));
        bias += ch / 2;
        MIMI_CUDA(conv(H, ch / 2, 1, 1, 0, PRO_ELU, ews(e, e->o_r2[i]), bias, ch, P, EPI_RES, P, i, i));
        bias += ch;
        // ELU -> conv k = 2 r, stride r (C -> 2 C)
        MIMI_CUDA(conv(P, ch, 2 * e->ratio[i], e->ratio[i], 0, PRO_ELU, ews(e, e->o_dn[i]), bias, 2 * ch, Q, EPI_BIAS, nullptr, i, i + 1));
        bias += 2 * ch;
        ch *= 2;
        std::swap(P, Q);
    }
    const int L = e->n_st;          // the 25 Hz level
    const int R = lvl[L][n];
    float *X = ews(e, e->o_X), *Hn = ews(e, e->o_Hn), *QKV = ews(e, e->o_QKV), *ATT = ews(e, e->o_ATT), *FF = ews(e, e->o_FF);
    MIMI_CUDA(conv(P, ch, c.last_kernel, 1, 0, PRO_ELU, ews(e, e->o_conv_out), bias, c.dim, X, EPI_BIAS, nullptr, L, L));
    // ---- encoder transformer ----
    const Segs rows_seg = segs(L, L);
    const size_t attn_smem = (size_t)kWarps * (c.head_dim + ((c.window + 3) & ~3)) * 4;
    for (int l = 0; l < c.n_layers; ++l) {
        const LayerOffsets& lo = e->o_layer[l];
        const float* vec = ews(e, lo.vec);
        enc_ln_kernel<<<(R + kWarps - 1) / kWarps, kThreads, 0, st>>>(X, vec, vec + c.dim, Hn, R, c.dim, c.norm_eps);
        ++launches;
        MIMI_CUDA(linear(Hn, c.dim, ews(e, lo.qkv), 3 * c.dim, QKV, EPI_BIAS, nullptr, nullptr, R));
        const long long pairs = (long long)R * (c.dim / 2);
        enc_rope_kernel<<<(unsigned)((pairs + kThreads - 1) / kThreads), kThreads, 0, st>>>(QKV, ews(e, e->o_rope), R, c.dim, c.head_dim, rows_seg);
        enc_attn_kernel<<<dim3((R + kWarps - 1) / kWarps, c.n_heads), kThreads, attn_smem, st>>>(QKV, ATT, R, c.dim, c.head_dim, c.window, rows_seg);
        launches += 3;
        MIMI_CUDA(cudaGetLastError());
        MIMI_CUDA(linear(ATT, c.dim, ews(e, lo.o), c.dim, X, EPI_SCALE_RES, X, vec + 4 * c.dim, R));
        enc_ln_kernel<<<(R + kWarps - 1) / kWarps, kThreads, 0, st>>>(X, vec + 2 * c.dim, vec + 3 * c.dim, Hn, R, c.dim, c.norm_eps);
        ++launches;
        MIMI_CUDA(linear(Hn, c.dim, ews(e, lo.fc1), c.ffn, FF, EPI_GELU, nullptr, nullptr, R));
        MIMI_CUDA(linear(FF, c.ffn, ews(e, lo.fc2), c.dim, X, EPI_SCALE_RES, X, vec + 5 * c.dim, R));
    }
    // ---- downsample (replicate padding, no bias) -> z ----
    const int Fr = lvl[L + 1][n];
    float *Z = ews(e, e->o_Z), *RS = ews(e, e->o_RS), *RA = ews(e, e->o_RA), *S = ews(e, e->o_S);
    MIMI_CUDA(conv(X, c.dim, 4, 2, 1, PRO_NONE, ews(e, e->o_ds), nullptr, c.dim, Z, EPI_BIAS, nullptr, L, L + 1));
    // ---- split RVQ ----
    const float* proj = ews(e, e->o_proj);
    MIMI_CUDA(linear(Z, c.dim, proj, c.codebook_dim, RS, EPI_BIAS, nullptr, nullptr, Fr));
    MIMI_CUDA(linear(Z, c.dim, proj + (size_t)c.codebook_dim * c.dim, c.codebook_dim, RA, EPI_BIAS, nullptr, nullptr, Fr));
    const size_t book = (size_t)c.codebook_size * c.codebook_dim;
    for (int q = 0; q < c.n_q; ++q) {
        float* r = q == 0 ? RS : RA;
        const float* bk = ews(e, e->o_books) + q * book;
        MIMI_CUDA(linear(r, c.codebook_dim, bk, c.codebook_size, S, EPI_BIAS, nullptr, nullptr, Fr));
        enc_argmin_kernel<<<(Fr + kWarps - 1) / kWarps, kThreads, 0, st>>>(S, ews(e, e->o_norms) + (size_t)q * c.codebook_size, bk, r, d_codes,
                                                                          Fr, c.codebook_size, c.codebook_dim, c.n_q, q);
        ++launches;
        MIMI_CUDA(cudaGetLastError());
    }
    e->launches = launches;
    return SMOL_OK;
}

extern "C" void* smol_mimi_encoder_debug_buffer(SmolMimiEncoder* e, const char* name) {
    if (!e || !e->bound || !name) return nullptr;
    if (!strcmp(name, "latent")) return (void*)ews(e, e->o_Z);
    return nullptr;
}
