// The DualAR decode step as ONE persistent kernel (sm_100a).
//
// One CTA per SM (148 on B200), 16 warps each.  A frame is a fixed program of phases
// (dev_model.h: decode_phase); every CTA walks the same program and the CTAs meet at a
// release/acquire grid barrier between phases, so one cooperative launch runs any number of
// frames (or prompt positions) without returning to the host:
//
//   slow layer l :  QKV   [embed ->] RMSNorm -> wqkv GEMV -> RoPE -> paged KV append      (P:205-221,535-552,601-640; K:12-22)
//                   ATTN  split-KV decode attention over the paged cache, GQA             (P:556-566)
//                   WO    wo GEMV + residual                                               (P:570,499)
//                   W13   RMSNorm -> w1/w3 GEMV -> silu(a)*b                                (P:581-582)
//                   W2    w2 GEMV + residual                                               (P:582,500)
//   HEAD / SAMPLE   final norm -> tied LM head -> argmax | top-k/top-p/temperature          (P:250-255; G:88-99)
//   depth step i :  per fast layer QKV, WO (attention over <= depth on-chip positions fused in),
//                   W13, W2; then HEAD (fast_norm + W_i) and SAMPLE                       (P:409-448,585-598; M:194-220; G:110-141)
//
// (P = modeling/model/rq_transformer.py, M = mlx lm/rq_transformer.py, G = mlx lm/generate.py,
//  K = mlx lm/cache.py of the reference.)
//
// Weight streaming.  At this batch size every matrix op is a GEMV bounded by HBM latency/bandwidth,
// and weights do not depend on activations.  So each CTA owns a fixed set of weight rows per phase
// and fetches them ONE PHASE AHEAD: as soon as a phase's math is done, one lane per warp issues
// TMA bulk copies (cp.async.bulk global->shared, completion on a per-warp mbarrier) for the rows the
// warp needs in the next weight phase.  The copies fly while the CTA sits in the grid barrier and
// runs the next phase's prologue (activation gather + RMSNorm), so the GEMV itself reads weights
// and activations from shared memory only.
//
// Rounding points follow the reference's eager bf16 forward exactly (bf16 after every Linear, each
// RMSNorm stage, RoPE, SDPA, silu, the product and each residual add; fp32 inside), so only
// summation order differs.

#include "common.cuh"
#include "dev_model.h"
#include "sampler.cuh"
#include "umma.cuh"

namespace smol {

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldcg_v4(const void* p) { return __ldcg(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ uint32_t ldcg_u32(const void* p) { return __ldcg(reinterpret_cast<const unsigned int*>(p)); }
__device__ __forceinline__ int ldcg_i32(const void* p) { return __ldcg(reinterpret_cast<const int*>(p)); }
__device__ __forceinline__ float ldcg_f32(const void* p) { return __ldcg(reinterpret_cast<const float*>(p)); }
__device__ __forceinline__ float bf_to_f(uint16_t v) { return __uint_as_float(((uint32_t)v) << 16); }
__device__ __forceinline__ uint16_t f_to_bf(float v) { return __bfloat16_as_ushort(__float2bfloat16_rn(v)); }
__device__ __forceinline__ uint16_t ldcg_u16(const uint16_t* p) {
    return __ldcg(reinterpret_cast<const unsigned short*>(p));
}

// Position of element k of a K-vector inside the shared-memory activation row.  Elements are kept
// as two half-rows (first / second float4 of every 8-element chunk) so that the 16-byte reads of
// 32 consecutive lanes are contiguous and bank-conflict free.
__device__ __forceinline__ int xs_index(int k, int K) {
    const int c = k >> 3, e = k & 7;
    return (e < 4) ? (c * 4 + e) : ((K >> 1) + c * 4 + (e - 4));
}

__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
    f[0] = bf_lo(v.x); f[1] = bf_hi(v.x); f[2] = bf_lo(v.y); f[3] = bf_hi(v.y);
    f[4] = bf_lo(v.z); f[5] = bf_hi(v.z); f[6] = bf_lo(v.w); f[7] = bf_hi(v.w);
}

__device__ __forceinline__ void store_chunk(float* row, int K, int c, const float (&f)[8]) {
    *reinterpret_cast<float4*>(row + c * 4) = make_float4(f[0], f[1], f[2], f[3]);
    *reinterpret_cast<float4*>(row + (K >> 1) + c * 4) = make_float4(f[4], f[5], f[6], f[7]);
}

__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// Release/acquire grid barrier, split into arrive and wait so that work which does not depend on the
// other CTAs (issuing the next phase's weight copies) sits between the two.  All CTAs are co-resident
// (cooperative launch).  `target` is the cumulative arrival count this barrier completes at; it only ever grows
// (wrap-safe compare) and is the same number in every CTA.  One atomic counter, one polling thread per CTA.
// Measured alternatives on B200 (bs=256 step, 148 CTAs), all slower or equal:
//  * per-CTA flag words, every CTA polling all 148 flags with one thread each: 4.41 ms per step against 2.84 ms
//    (21 904 pollers slow the very stores they wait for -- the poll-pressure effect of the data-flow kernel);
//  * a two-level counter (12 group counters whose last arrivers arrive on the root): 3.3 us vs 2.2 us per barrier;
//  * relaxed polls + one acquire fence instead of acquiring polls: 2.95 vs 2.84 ms.
__device__ __forceinline__ void grid_arrive(uint32_t* ctr, uint32_t& target, uint32_t n_ctas) {
    target += n_ctas;
    __syncthreads();
    if (threadIdx.x == 0) asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(ctr), "r"(1u) : "memory");
}
__device__ __forceinline__ void grid_wait(uint32_t* ctr, uint32_t target) {
    if (threadIdx.x == 0) {
        uint32_t v;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ctr) : "memory");
        } while ((int32_t)(v - target) < 0);
    }
    __syncthreads();
}

// ---- mbarrier + TMA bulk copy (global -> shared) ---------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// Generic-proxy writes (st.global of activations) <-> async-proxy reads (TMA tensor loads of the same buffers by other
// CTAs): fenced on both sides of the grid barrier in the tensor-core variant.
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }

struct Ctx {
    int cta, n_ctas, warp, lane, tid;
    float* xs;            // activations of the batch tile, fp32 (dynamic shared memory)
    unsigned char* stage; // weight rows of the current / next weight phase (dynamic shared memory)
    int iter;             // frame (decode) or prompt position (prefill) inside this launch
};

__shared__ SampleScratch g_sc;
__shared__ int g_pos[kBatchTile];
__shared__ float g_part[kWarps];
__shared__ int g_flag;
__shared__ __align__(8) uint64_t g_mbar[kWarps];

// ------------------------------------------------------------------------------------------------
// weight plan of a phase and its staging
// ------------------------------------------------------------------------------------------------
// A phase's GEMV is `n_units` units of R weight rows of K elements; unit u lands in slot
// (u - cta) / n_ctas of the CTA's stage buffer as R contiguous rows.
struct Plan {
    const uint16_t* w0;
    const uint16_t* w1;  // second row source (w3) for the gated MLP, else nullptr
    int K, n_units, R;
};

__device__ __forceinline__ Plan phase_plan(const DevModel& M, const Phase& ph) {
    Plan pl;
    pl.w0 = nullptr; pl.w1 = nullptr; pl.K = 0; pl.n_units = 0; pl.R = 1;
    const bool fast = ph.fast != 0;
    const int D = fast ? M.fdim : M.dim, F = fast ? M.finter : M.inter;
    const DevLayer& L = fast ? M.fast_layers[ph.layer] : M.layers[ph.layer];
    switch (ph.kind) {
        case PH_QKV: {
            const int Hq = fast ? M.fn_head : M.n_head, Hkv = fast ? M.fn_kv : M.n_kv;
            pl.w0 = L.wqkv; pl.K = D; pl.R = 2; pl.n_units = (Hq + 2 * Hkv) * kHeadDim / 2;
        } break;
        case PH_WO: pl.w0 = L.wo; pl.K = D; pl.n_units = D; break;
        case PH_W13: pl.w0 = L.w1; pl.w1 = L.w3; pl.K = D; pl.R = 2; pl.n_units = F; break;
        case PH_W2: pl.w0 = L.w2; pl.K = F; pl.n_units = D; break;
        case PH_HEAD: {
            const int N = fast ? M.codebook_size : M.vocab;
            pl.w0 = fast ? M.fast_output + (M.depthwise_output ? (size_t)ph.depth_pos * N * D : 0) : M.head;
            pl.K = D; pl.n_units = N;
        } break;
        default: break;
    }
    return pl;
}

// One lane per warp issues the bulk copies of the warp's units; the bytes complete on the warp's
// own mbarrier.  Callers guarantee (block barrier) that nobody still reads the stage buffer.
__device__ __forceinline__ void stage_issue(const Ctx& c, const Plan& pl) {
    if (c.lane != 0 || pl.n_units == 0) return;
    const uint32_t row_bytes = (uint32_t)pl.K * 2u, slot_bytes = row_bytes * pl.R;
    int mine = 0;
    for (int u = c.cta + c.warp * c.n_ctas; u < pl.n_units; u += kWarps * c.n_ctas) ++mine;
    if (mine == 0) return;
    fence_proxy_async();
    mbar_expect_tx(&g_mbar[c.warp], (uint32_t)mine * slot_bytes);
    int j = c.warp;
    for (int u = c.cta + c.warp * c.n_ctas; u < pl.n_units; u += kWarps * c.n_ctas, j += kWarps) {
        unsigned char* dst = c.stage + (size_t)j * slot_bytes;
        if (pl.w1 != nullptr) {
            bulk_g2s(dst, pl.w0 + (size_t)u * pl.K, row_bytes, &g_mbar[c.warp]);
            bulk_g2s(dst + row_bytes, pl.w1 + (size_t)u * pl.K, row_bytes, &g_mbar[c.warp]);
        } else {
            bulk_g2s(dst, pl.w0 + (size_t)u * pl.R * pl.K, slot_bytes, &g_mbar[c.warp]);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// activation staging
// ------------------------------------------------------------------------------------------------

// xs[b][:] = rows[b][0:K] (bf16 in global, read through L2), b < nb; all threads cooperate.
template <class RowPtr>
__device__ __forceinline__ void fill_rows(const Ctx& c, int K, int nb, RowPtr rowptr) {
    const int nch = K >> 3;
    for (int idx = c.tid; idx < nb * nch; idx += kThreads) {
        const int b = idx / nch, ch = idx - b * nch;
        const uint16_t* src = rowptr(b);
        float f[8];
        unpack8(ldcg_v4(src + ch * 8), f);
        store_chunk(c.xs + (size_t)b * K, K, ch, f);
    }
}

// RMSNorm (reference RMSNorm.forward :607-613: fp32 normalise, round to bf16, multiply by the bf16
// weight, round again) of nb rows gathered by `load_chunk(b, ch, f)` straight into xs.  One thread per
// 16-byte chunk: a row occupies ceil(K/256) warps, the sum of squares goes through shuffles and one
// shared-memory hop, and the thread that loaded a chunk normalises and stores it -- one round trip to
// L2 and two block barriers, with only the warps that hold data issuing instructions.
// If `spill` is set (CTA 0 on layer 0) the raw row is also written to global as the residual stream.
template <class LoadChunk>
__device__ __forceinline__ void norm_rows(const Ctx& c, int K, int nb, LoadChunk load_chunk, const uint16_t* w, float eps,
                                          uint16_t* spill, int b0) {
    const int nch = K >> 3;
    const int wpr = (nch + 31) >> 5;         // warps per row (<= 3: K <= 768)
    const int rows_per_pass = kWarps / wpr;
    const int wr = c.warp / wpr, wi = c.warp - wr * wpr;
    const int ch = wi * 32 + c.lane;
    for (int bp = 0; bp < nb; bp += rows_per_pass) {
        const int b = bp + wr;
        const bool act = (wr < rows_per_pass) && (b < nb) && (ch < nch);
        float x[8];
        float ss = 0.f;
        uint4 wv = make_uint4(0u, 0u, 0u, 0u);
        if (act) {
            wv = __ldg(reinterpret_cast<const uint4*>(w + ch * 8));
            load_chunk(b, ch, x);
#pragma unroll
            for (int e = 0; e < 8; ++e) ss = fmaf(x[e], x[e], ss);
        }
        ss = warp_sum(ss);
        if (c.lane == 0) g_part[c.warp] = ss;
        __syncthreads();
        if (act) {
            float t = 0.f;
            for (int i = 0; i < wpr; ++i) t += g_part[wr * wpr + i];
            const float mean = __fdiv_rn(t, (float)K);
            const float r = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(mean, eps)));
            if (spill != nullptr) {
                uint4 pk;
                pk.x = pack_bf16(x[0], x[1]); pk.y = pack_bf16(x[2], x[3]);
                pk.z = pack_bf16(x[4], x[5]); pk.w = pack_bf16(x[6], x[7]);
                *reinterpret_cast<uint4*>(spill + (size_t)(b0 + b) * K + ch * 8) = pk;
            }
            float wf[8], o[8];
            unpack8(wv, wf);
#pragma unroll
            for (int e = 0; e < 8; ++e) o[e] = bf16_round(__fmul_rn(bf16_round(__fmul_rn(x[e], r)), wf[e]));
            store_chunk(c.xs + (size_t)b * K, K, ch, o);
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------
// GEMV over the units owned by this CTA, weights and activations both in shared memory
// ------------------------------------------------------------------------------------------------
// acc[r][b] = sum_k W_r[k] * xs[b][k], reduced over the warp; lane b receives sequence b's sums.
// Only <BT, R> are compile-time: the chunk loop is a runtime loop so that the whole frame program
// stays small enough for the instruction cache (every phase runs once per frame).
template <int BT, int R, class Epi>
__device__ __forceinline__ void gemv_units(const Ctx& c, int n_units, int K, Epi epi) {
    const int nchunks = K >> 3;
    const int half = K >> 1;
    const size_t slot_bytes = (size_t)K * 2 * R;
    int j = c.warp;
    for (int u = c.cta + c.warp * c.n_ctas; u < n_units; u += kWarps * c.n_ctas, j += kWarps) {
        const uint4* wrow = reinterpret_cast<const uint4*>(c.stage + (size_t)j * slot_bytes);
        // K is summed in slices of 128 chunks (1024 elements): inside a slice lane-strided chunks with two
        // accumulator chains and a butterfly warp sum, slices added in order.  (The data-flow kernel gives the
        // slices of a long row to different warps; the order of the additions is the same.)
        float tot[R][BT];
#pragma unroll
        for (int r = 0; r < R; ++r)
#pragma unroll
            for (int b = 0; b < BT; ++b) tot[r][b] = 0.f;
        for (int c0 = 0; c0 < nchunks; c0 += 128) {
            const int c1 = min(c0 + 128, nchunks);
            float acc0[R][BT], acc1[R][BT];
#pragma unroll
            for (int r = 0; r < R; ++r)
#pragma unroll
                for (int b = 0; b < BT; ++b) { acc0[r][b] = 0.f; acc1[r][b] = 0.f; }
#pragma unroll(BT <= 2 ? 3 : 1)
            for (int ch = c0 + c.lane; ch < c1; ch += 32) {
                float wf[R][8];
#pragma unroll
                for (int r = 0; r < R; ++r) unpack8(wrow[r * nchunks + ch], wf[r]);
#pragma unroll
                for (int b = 0; b < BT; ++b) {
                    const float* xr = c.xs + (size_t)b * K + ch * 4;
                    const float4 x0 = *reinterpret_cast<const float4*>(xr);
                    const float4 x1 = *reinterpret_cast<const float4*>(xr + half);
#pragma unroll
                    for (int r = 0; r < R; ++r) {
                        float a0 = acc0[r][b], a1 = acc1[r][b];
                        a0 = fmaf(wf[r][0], x0.x, a0); a1 = fmaf(wf[r][4], x1.x, a1);
                        a0 = fmaf(wf[r][1], x0.y, a0); a1 = fmaf(wf[r][5], x1.y, a1);
                        a0 = fmaf(wf[r][2], x0.z, a0); a1 = fmaf(wf[r][6], x1.z, a1);
                        a0 = fmaf(wf[r][3], x0.w, a0); a1 = fmaf(wf[r][7], x1.w, a1);
                        acc0[r][b] = a0; acc1[r][b] = a1;
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < R; ++r)
#pragma unroll
                for (int b = 0; b < BT; ++b) tot[r][b] = __fadd_rn(tot[r][b], warp_sum(acc0[r][b] + acc1[r][b]));
        }
        float mine[R];
#pragma unroll
        for (int r = 0; r < R; ++r) {
            mine[r] = 0.f;
#pragma unroll
            for (int b = 0; b < BT; ++b)
                if (c.lane == b) mine[r] = tot[r][b];
        }
        epi(u, mine);
    }
}

// Waits until this warp's staged weight rows have landed (if it owns any unit of the phase).
__device__ __forceinline__ void stage_wait(const Ctx& c, int n_units, uint32_t& parity) {
    if (c.cta + c.warp * c.n_ctas < n_units) {
        mbar_wait(&g_mbar[c.warp], parity);
        parity ^= 1u;
    }
}

// ------------------------------------------------------------------------------------------------
// phases
// ------------------------------------------------------------------------------------------------
// Prefill runs `tile_t` consecutive prompt positions of every sequence as rows of one iteration (they share the pass over
// the weights; causality comes from each row's own context length): row bg = sequence bg / tile_t, offset bg % tile_t.
__device__ __forceinline__ int row_seq(const CallArgs& A, int bg) { return A.tile_t > 1 ? bg / A.tile_t : bg; }
__device__ __forceinline__ int row_off(const CallArgs& A, int bg) { return A.tile_t > 1 ? bg % A.tile_t : 0; }
__device__ __forceinline__ int prefill_t(const CallArgs& A, const Ctx& c, int bg) {
    return A.iter_base + c.iter * (A.tile_t > 1 ? A.tile_t : 1) + row_off(A, bg);
}
__device__ __forceinline__ bool seq_active(const DevModel& M, const CallArgs& A, const Ctx& c, int bg) {
    if (A.prefill) return prefill_t(A, c, bg) < ldcg_i32(A.prompt_len + row_seq(A, bg)) - 1;
    return A.b.finished == nullptr || __ldcg(A.b.finished + bg) == 0;
}

// id of grid row r of sequence bg for the slow embedding
__device__ __forceinline__ int input_token(const DevModel& M, const CallArgs& A, const Ctx& c, int bg, int r) {
    if (A.prefill) {
        int t = prefill_t(A, c, bg);
        const int b = row_seq(A, bg);
        const int len = ldcg_i32(A.prompt_len + b);
        if (t > len - 1) t = len - 1;
        return ldcg_i32(A.prompt + ((size_t)b * M.n_rows + r) * A.s_max + t);
    }
    return ldcg_i32(A.b.tokens + (size_t)bg * M.n_rows + r);
}

// BaseTransformer.embed (P:205-221) for one 8-element chunk: text row + sum of the codebook rows,
// zeroed by the PyTorch rule (row-1 code == 0) or the MLX rule (row-0 id outside the semantic range,
// M:162-169).
__device__ __forceinline__ void embed_chunk(const DevModel& M, const CallArgs& A, const Ctx& c, int bg, int ch,
                                            float (&f)[8]) {
    const int D = M.dim;
    const int t0 = input_token(M, A, c, bg, 0);
    unpack8(ldcg_v4(M.embeddings + (size_t)t0 * D + ch * 8), f);
    bool use_vq;
    if (M.mlx_embed_mask) use_vq = (t0 >= M.semantic_start && t0 <= M.semantic_end);
    else use_vq = input_token(M, A, c, bg, 1) != 0;
    if (use_vq) {
        float s[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) s[e] = 0.f;
        for (int r = 1; r < M.n_rows; ++r) {
            const int code = input_token(M, A, c, bg, r);
            const int row = code + (M.dup0 ? (r - 1) : r) * M.codebook_size;
            float g[8];
            unpack8(ldcg_v4(M.codebook_embeddings + (size_t)row * D + ch * 8), g);
#pragma unroll
            for (int e = 0; e < 8; ++e) s[e] = __fadd_rn(s[e], g[e]);
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) f[e] = bf16_round(__fadd_rn(f[e], bf16_round(s[e])));
    }
}

// Attention of the fast transformer for the current batch tile, computed redundantly by every CTA
// straight into xs (the input of the wo GEMV): <= kMaxDepth cached positions per sequence.  One warp
// per (sequence, head).  Scores: 4 lanes per position (16 dims each), two positions per lane group
// when depth > 8.  One softmax with the global max; the probabilities are rounded to bf16 before the
// PV product while the row sum keeps the unrounded values -- what the reference's fused SDPA does
// for bf16 inputs (flash kernels, CPU and CUDA alike).
__device__ __forceinline__ void fast_attention_rows(const DevModel& M, const Ctx& c, int layer, int depth_pos,
                                                    int b0, int nb) {
    const int Hq = M.fn_head, Hkv = M.fn_kv, G = Hq / Hkv, D = M.fdim;
    const int kvw = Hkv * kHeadDim;
    const int jl = c.lane >> 2, part = c.lane & 3;
    for (int pair = c.warp; pair < nb * Hq; pair += kWarps) {
        const int b = pair / Hq, hq = pair - b * Hq, bg = b0 + b, kvh = hq / G;
        const uint16_t* qp = M.q + (size_t)bg * Hq * kHeadDim + hq * kHeadDim + part * 16;
        const uint16_t* kb = M.fkv + ((size_t)(bg * M.n_flayer + layer) * 2) * M.depth * kvw + kvh * kHeadDim;
        const uint16_t* vb = kb + (size_t)M.depth * kvw;
        float qf[16];
        {
            float t0[8], t1[8];
            unpack8(ldcg_v4(qp), t0);
            unpack8(ldcg_v4(qp + 8), t1);
#pragma unroll
            for (int e = 0; e < 8; ++e) { qf[e] = t0[e]; qf[8 + e] = t1[e]; }
        }
        const bool deep = depth_pos >= 8;  // warp-uniform: second position per lane group only then
        float sc[2];
        bool ok[2];
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {
            const int j = jl + 8 * h2;
            ok[h2] = j <= depth_pos;
            sc[h2] = -INFINITY;
            if (h2 == 0 || deep) {
                float s = 0.f;
                if (ok[h2]) {
                    float k0[8], k1[8];
                    unpack8(ldcg_v4(kb + (size_t)j * kvw + part * 16), k0);
                    unpack8(ldcg_v4(kb + (size_t)j * kvw + part * 16 + 8), k1);
#pragma unroll
                    for (int e = 0; e < 8; ++e) s = fmaf(qf[e], k0[e], s);
#pragma unroll
                    for (int e = 0; e < 8; ++e) s = fmaf(qf[8 + e], k1[e], s);
                }
                s += __shfl_xor_sync(0xffffffffu, s, 1);
                s += __shfl_xor_sync(0xffffffffu, s, 2);
                if (ok[h2]) sc[h2] = s * 0.125f;
            }
        }
        float m = fmaxf(sc[0], sc[1]);
        m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 4));
        m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 8));
        m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, 16));
        const float pe0 = ok[0] ? expf(sc[0] - m) : 0.f;
        const float pe1 = ok[1] ? expf(sc[1] - m) : 0.f;
        float l = pe0 + pe1;
        l += __shfl_xor_sync(0xffffffffu, l, 4);
        l += __shfl_xor_sync(0xffffffffu, l, 8);
        l += __shfl_xor_sync(0xffffffffu, l, 16);
        const float pb0 = bf16_round(pe0), pb1 = bf16_round(pe1);
        // PV: lane owns dims 2*lane, 2*lane+1
        float o0 = 0.f, o1 = 0.f;
        {
            uint32_t vv[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) vv[j] = (j <= depth_pos) ? ldcg_u32(vb + (size_t)j * kvw + 2 * c.lane) : 0u;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float p = __shfl_sync(0xffffffffu, pb0, j * 4);
                o0 = fmaf(p, bf_lo(vv[j]), o0);
                o1 = fmaf(p, bf_hi(vv[j]), o1);
            }
        }
        if (deep) {
            for (int j = 8; j < kMaxDepth; ++j) {
                const float p = __shfl_sync(0xffffffffu, pb1, (j & 7) * 4);
                if (j <= depth_pos) {
                    const uint32_t v = ldcg_u32(vb + (size_t)j * kvw + 2 * c.lane);
                    o0 = fmaf(p, bf_lo(v), o0);
                    o1 = fmaf(p, bf_hi(v), o1);
                }
            }
        }
        const float inv = 1.0f / l;
        float* row = c.xs + (size_t)b * D;
        const int k = hq * kHeadDim + 2 * c.lane;
        row[xs_index(k, D)] = bf16_round(o0 * inv);
        row[xs_index(k + 1, D)] = bf16_round(o1 * inv);
    }
}

// Split-KV decode attention over the paged cache.  Unit = (sequence, kv head, split); the G query
// heads of a kv head share every K/V read.  Each 8-lane group owns one cached position per step
// and keeps its own online-softmax state; states are merged across groups, warps and (through a
// last-arriver fix-up in global memory) splits, always in a fixed order.
__device__ void phase_attn_g(const DevModel& M, const CallArgs& A, const Ctx& c, const Phase& ph, int s_max) {
    constexpr int GM = kMaxGroup;
    const int Hq = M.n_head, Hkv = M.n_kv, ps = M.page_size, G = Hq / Hkv;
    const int dch = c.lane & 7, psub = c.lane >> 3;
    float* red = c.xs;  // [kWarps][G][kPartialStride]
    const int n_units = A.batch * Hkv * s_max;
    for (int u = c.cta; u < n_units; u += c.n_ctas) {
        const int s = u % s_max, kvh = (u / s_max) % Hkv, b = u / (s_max * Hkv);
        const int bs = row_seq(A, b);  // the sequence whose cache this row reads (prefill tiles: several rows per sequence)
        int Lb = ldcg_i32(A.b.seq_len + bs) + row_off(A, b) + 1;
        const int cap = A.b.max_pages * ps;
        if (Lb > cap) Lb = cap;
        int ns = (Lb + kSplitMin - 1) / kSplitMin;
        if (ns > s_max) ns = s_max;
        if (ns < 1) ns = 1;
        if (s >= ns) continue;
        const int chunk = (Lb + ns - 1) / ns;
        const int p0 = s * chunk, p1 = min(Lb, p0 + chunk);

        float qf[GM][8];
#pragma unroll
        for (int g = 0; g < GM; ++g) {
            if (g >= G) continue;
            unpack8(ldcg_v4(M.q + (size_t)b * Hq * kHeadDim + (kvh * G + g) * kHeadDim + dch * 8), qf[g]);
#pragma unroll
            for (int e = 0; e < 8; ++e) qf[g][e] *= 0.125f;  // 1/sqrt(64), exact
        }
        float m[GM], l[GM], acc[GM][8];
#pragma unroll
        for (int g = 0; g < GM; ++g) {
            if (g >= G) continue;
            m[g] = -INFINITY; l[g] = 0.f;
#pragma unroll
            for (int e = 0; e < 8; ++e) acc[g][e] = 0.f;
        }
        const int32_t* bt = A.b.block_table + (size_t)bs * A.b.max_pages;
        const size_t head_stride = (size_t)ps * kHeadDim;
        for (int pb = p0 + c.warp * 4; pb < p1; pb += kWarps * 4) {
            const int p = pb + psub;
            const bool valid = p < p1;
            uint4 kk = make_uint4(0u, 0u, 0u, 0u), vv = kk;
            if (valid) {
                const int page = ldcg_i32(bt + p / ps);
                const uint16_t* kp = M.kv_pool + ((((size_t)page * M.n_layer + ph.layer) * 2) * Hkv + kvh) * head_stride
                                     + (size_t)(p % ps) * kHeadDim + dch * 8;
                kk = ldcg_v4(kp);
                vv = ldcg_v4(kp + (size_t)Hkv * head_stride);
            }
            float kf[8], vf[8];
            unpack8(kk, kf);
            unpack8(vv, vf);
#pragma unroll
            for (int g = 0; g < GM; ++g) {
            if (g >= G) continue;
                float sc = 0.f;
#pragma unroll
                for (int e = 0; e < 8; ++e) sc = fmaf(qf[g][e], kf[e], sc);
                sc += __shfl_xor_sync(0xffffffffu, sc, 1);
                sc += __shfl_xor_sync(0xffffffffu, sc, 2);
                sc += __shfl_xor_sync(0xffffffffu, sc, 4);
                if (valid) {
                    const float mn = fmaxf(m[g], sc);
                    const float corr = (m[g] == -INFINITY) ? 0.f : expf(m[g] - mn);
                    const float pe = expf(sc - mn);
                    l[g] = fmaf(l[g], corr, pe);
                    // the reference's SDPA rounds P to bf16 for the PV product and sums the unrounded values (P:559-566)
                    const float pq = bf16_round(pe);
#pragma unroll
                    for (int e = 0; e < 8; ++e) acc[g][e] = fmaf(acc[g][e], corr, pq * vf[e]);
                    m[g] = mn;
                }
            }
        }
        // merge the four position groups of the warp
#pragma unroll
        for (int o = 8; o <= 16; o <<= 1) {
#pragma unroll
            for (int g = 0; g < GM; ++g) {
            if (g >= G) continue;
                const float mo = __shfl_xor_sync(0xffffffffu, m[g], o);
                const float lo = __shfl_xor_sync(0xffffffffu, l[g], o);
                const float mn = fmaxf(m[g], mo);
                const float c1 = (m[g] == -INFINITY) ? 0.f : expf(m[g] - mn);
                const float c2 = (mo == -INFINITY) ? 0.f : expf(mo - mn);
                l[g] = fmaf(l[g], c1, __fmul_rn(lo, c2));
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const float ao = __shfl_xor_sync(0xffffffffu, acc[g][e], o);
                    acc[g][e] = fmaf(acc[g][e], c1, __fmul_rn(ao, c2));
                }
                m[g] = mn;
            }
        }
        if (psub == 0) {
#pragma unroll
            for (int g = 0; g < GM; ++g) {
            if (g >= G) continue;
                float* dst = red + (c.warp * G + g) * kPartialStride;
                if (dch == 0) { dst[0] = m[g]; dst[1] = l[g]; }
#pragma unroll
                for (int e = 0; e < 8; ++e) dst[2 + dch * 8 + e] = acc[g][e];
            }
        }
        __syncthreads();
        // merge the warps (fixed order)
        float Mx = -INFINITY, Ls = 0.f, Os = 0.f;
        const int g = c.tid / kHeadDim, d = c.tid & (kHeadDim - 1);
        if (c.tid < G * kHeadDim) {
            for (int wi = 0; wi < kWarps; ++wi) Mx = fmaxf(Mx, red[(wi * G + g) * kPartialStride]);
            for (int wi = 0; wi < kWarps; ++wi) {
                const float* src = red + (wi * G + g) * kPartialStride;
                if (src[0] == -INFINITY) continue;
                const float sc = expf(src[0] - Mx);
                Ls = fmaf(src[1], sc, Ls);
                Os = fmaf(src[2 + d], sc, Os);
            }
        }
        const int hq = kvh * G + g;
        if (ns == 1) {
            if (c.tid < G * kHeadDim) M.attn[(size_t)b * Hq * kHeadDim + hq * kHeadDim + d] = f_to_bf(Os / Ls);
        } else {
            if (c.tid < G * kHeadDim) {
                float* dst = M.partial + (((size_t)b * Hq + hq) * kMaxSplits + s) * kPartialStride;
                if (d == 0) { dst[0] = Mx; dst[1] = Ls; }
                dst[2 + d] = Os;
            }
            __threadfence();
            __syncthreads();
            if (c.tid == 0) {
                const uint32_t old = atomicAdd(M.split_count + (size_t)b * Hkv + kvh, 1u);
                g_flag = (old == (uint32_t)(ns - 1)) ? 1 : 0;
            }
            __syncthreads();
            if (g_flag) {  // last split of this (sequence, kv head): combine all splits in split order
                __threadfence();
                if (c.tid < G * kHeadDim) {
                    const float* base = M.partial + ((size_t)b * Hq + hq) * kMaxSplits * kPartialStride;
                    float Mg = -INFINITY;
                    for (int si = 0; si < ns; ++si) Mg = fmaxf(Mg, ldcg_f32(base + si * kPartialStride));
                    float Lg = 0.f, Og = 0.f;
                    for (int si = 0; si < ns; ++si) {
                        const float* src = base + si * kPartialStride;
                        const float ms = ldcg_f32(src);
                        if (ms == -INFINITY) continue;
                        const float sc = expf(ms - Mg);
                        Lg = fmaf(ldcg_f32(src + 1), sc, Lg);
                        Og = fmaf(ldcg_f32(src + 2 + d), sc, Og);
                    }
                    M.attn[(size_t)b * Hq * kHeadDim + hq * kHeadDim + d] = f_to_bf(Og / Lg);
                }
                if (c.tid == 0) M.split_count[(size_t)b * Hkv + kvh] = 0u;
            }
        }
        __syncthreads();
    }
}

// Splits per (sequence, kv head): a function of the sequence's own length only (ceil(L / 64), at most kMaxSplits),
// never of the batch size or the grid -- a sequence must decode to the same bits alone, in any batch and on any shard.
__device__ int attn_splits(const DevModel& M, int batch, int n_ctas) {
    (void)M; (void)batch; (void)n_ctas;
    return kMaxSplits;
}

__device__ void phase_attn(const DevModel& M, const CallArgs& A, const Ctx& c, const Phase& ph) {
    phase_attn_g(M, A, c, ph, attn_splits(M, A.batch, c.n_ctas));
}

}  // namespace smol
#include "tc_phases.cuh"
namespace smol {

__shared__ __align__(8) umma::Bars g_tc_bars;

// Every phase that streams weights: [gather / RMSNorm / fast attention] -> staged-weight GEMV ->
// epilogue.  One function so that each building block is instantiated exactly once (code size is what
// the instruction cache sees: every phase runs once per frame).
template <int BT>
__device__ void phase_gemv(const DevModel& M, const CallArgs& A, const Ctx& c, const Phase& ph, uint32_t& parity) {
    const bool fast = ph.fast != 0;
    const int kind = ph.kind;
    const int D = fast ? M.fdim : M.dim, F = fast ? M.finter : M.inter;
    const int Hq = fast ? M.fn_head : M.n_head, Hkv = fast ? M.fn_kv : M.n_kv;
    const DevLayer& L = fast ? M.fast_layers[ph.layer] : M.layers[ph.layer];
    const int q_rows = Hq * kHeadDim, k_end = (Hq + Hkv) * kHeadDim;
    const int n_head_rows = fast ? M.codebook_size : M.vocab;
    const int K = (kind == PH_W2) ? F : D;
    const int n_units = kind == PH_QKV ? (Hq + 2 * Hkv) * kHeadDim / 2 : kind == PH_W13 ? F : kind == PH_HEAD ? n_head_rows : D;
    const bool normed = kind == PH_QKV || kind == PH_W13 || kind == PH_HEAD;
    const uint16_t* norm_w = kind == PH_QKV ? L.attention_norm : kind == PH_W13 ? L.ffn_norm : (fast ? M.fast_norm : M.norm);
    const uint16_t* table = fast ? M.fast_rope : M.rope;
    uint16_t* stream = fast ? M.xf : M.x;
    const bool prof = (M.prof != nullptr) && c.cta == 0 && c.tid == 0;
    unsigned long long* seg = M.prof + 2 * kMaxProg + (size_t)(kind + (fast ? 8 : 0)) * 4;
    unsigned long long ts = 0;
    if (prof) ts = globaltimer_ns();
    // A.repeat > 0 (profiling only): the idempotent body runs again with a warm instruction cache
    for (int rep = 0; rep <= A.repeat; ++rep)
    for (int b0 = 0; b0 < A.batch; b0 += BT) {
        const int nb = min(BT, A.batch - b0);
        if (kind == PH_QKV && c.tid < nb)
            g_pos[c.tid] = fast ? ph.depth_pos : ldcg_i32(A.b.seq_len + row_seq(A, b0 + c.tid)) + row_off(A, b0 + c.tid);
        if (normed) {
            // where the row of sequence b comes from: 0 token embedding (P:205-221), 1 slow hidden state,
            // 2 embedding of the previous depth code (G:136-140), 3 a stream buffer
            int src_kind = 3;
            const uint16_t* base = kind == PH_W13 ? M.h : stream;
            uint16_t* spill = nullptr;
            if (kind == PH_QKV && ph.layer == 0) {
                if (!fast) { src_kind = 0; spill = M.x; }
                else if (!A.fast_from_xf) { src_kind = ph.depth_pos == 0 ? 1 : 2; spill = M.xf; }
            }
            if (c.cta != 0) spill = nullptr;
            norm_rows(c, D, nb, [&](int b, int ch, float (&f)[8]) {
                if (src_kind == 0) { embed_chunk(M, A, c, b0 + b, ch, f); return; }
                const uint16_t* src;
                if (src_kind == 1) {
                    src = M.x + (size_t)(b0 + b) * D;
                } else if (src_kind == 2) {
                    const int code = ldcg_i32(M.frame_tokens + (size_t)(b0 + b) * M.n_rows + ph.depth_pos);
                    const int off = M.depthwise_wte ? (M.dup0 ? ph.depth_pos - 1 : ph.depth_pos) * M.codebook_size : 0;
                    src = M.fast_embeddings + (size_t)(code + off) * D;
                } else {
                    src = base + (size_t)(b0 + b) * D;
                }
                unpack8(ldcg_v4(src + ch * 8), f);
            }, norm_w, M.eps, spill, b0);
        } else if (kind == PH_WO && fast) {
            fast_attention_rows(M, c, ph.layer, ph.depth_pos, b0, nb);
            __syncthreads();
        } else {
            const uint16_t* src = kind == PH_WO ? M.attn : M.act;
            fill_rows(c, K, nb, [&](int b) { return src + (size_t)(b0 + b) * K; });
            __syncthreads();
        }
        if (prof) { const unsigned long long t = globaltimer_ns(); seg[0] += t - ts; ts = t; }
        if (b0 == 0 && rep == 0) stage_wait(c, n_units, parity);
        if (prof) { const unsigned long long t = globaltimer_ns(); seg[1] += t - ts; ts = t; }

        if (kind == PH_QKV || kind == PH_W13) {
            auto epi = [&](int u, const float (&acc)[2]) {
                if (c.lane >= nb) return;
                const int bg = b0 + c.lane;
                if (kind == PH_W13) {
                    const float a = bf16_round(acc[0]), g = bf16_round(acc[1]);
                    const float sg = bf16_round(__fdiv_rn(a, __fadd_rn(1.0f, expf(-a))));  // F.silu in fp32, bf16 out
                    M.act[(size_t)bg * F + u] = f_to_bf(__fmul_rn(sg, g));
                    return;
                }
                const int n0 = 2 * u, pos = g_pos[c.lane];
                float v0 = bf16_round(acc[0]), v1 = bf16_round(acc[1]);
                if (n0 < k_end) {  // q and k rows: interleaved-pair RoPE with the bf16 table (P:616-640)
                    const int j = (n0 & (kHeadDim - 1)) >> 1;
                    // (positions are bounded by the host's capacity checks; the clamp keeps a bad caller inside the table)
                    const int tp = fast ? pos : min(pos, M.max_seq_len - 1);
                    const uint32_t cs = __ldg(reinterpret_cast<const uint32_t*>(table + ((size_t)tp * (kHeadDim / 2) + j) * 2));
                    const float co = bf_lo(cs), si = bf_hi(cs);
                    const float r0 = bf16_round(__fsub_rn(__fmul_rn(v0, co), __fmul_rn(v1, si)));
                    const float r1 = bf16_round(__fadd_rn(__fmul_rn(v1, co), __fmul_rn(v0, si)));
                    v0 = r0; v1 = r1;
                }
                const uint32_t packed = pack_bf16(v0, v1);
                if (n0 < q_rows) {
                    *reinterpret_cast<uint32_t*>(M.q + (size_t)bg * q_rows + n0) = packed;
                    return;
                }
                const int is_v = n0 >= k_end ? 1 : 0;
                const int n1 = n0 - (is_v ? k_end : q_rows);
                const int kvh = n1 / kHeadDim, d = n1 & (kHeadDim - 1);
                if (fast) {
                    uint16_t* dst = M.fkv + (((size_t)(bg * M.n_flayer + ph.layer) * 2 + is_v) * M.depth + ph.depth_pos) * (Hkv * kHeadDim)
                                    + kvh * kHeadDim + d;
                    *reinterpret_cast<uint32_t*>(dst) = packed;
                } else {
                    if (!seq_active(M, A, c, bg)) return;
                    const int ps = M.page_size;
                    if (pos >= A.b.max_pages * ps) return;
                    const int page = ldcg_i32(A.b.block_table + (size_t)row_seq(A, bg) * A.b.max_pages + pos / ps);
                    uint16_t* dst = M.kv_pool + ((((size_t)page * M.n_layer + ph.layer) * 2 + is_v) * Hkv + kvh) * ((size_t)ps * kHeadDim)
                                    + (size_t)(pos % ps) * kHeadDim + d;
                    *reinterpret_cast<uint32_t*>(dst) = packed;
                }
            };
            gemv_units<BT, 2>(c, n_units, K, epi);
        } else {
            auto epi = [&](int u, const float (&acc)[1]) {
                if (c.lane >= nb) return;
                const int bg = b0 + c.lane;
                if (kind == PH_HEAD) {
                    float* out = fast ? M.depth_logits + ((size_t)bg * M.depth + ph.depth_pos) * n_head_rows
                                      : M.token_logits + (size_t)bg * n_head_rows;
                    out[u] = bf16_round(acc[0]);
                    return;
                }
                // wo: h = stream + wo(attn)   (P:499)      w2: stream = h + w2(act)   (P:500)
                const uint16_t* res = kind == PH_WO ? stream : M.h;
                uint16_t* dst = kind == PH_WO ? M.h : stream;
                const size_t o = (size_t)bg * D + u;
                dst[o] = f_to_bf(__fadd_rn(bf_to_f(ldcg_u16(res + o)), bf16_round(acc[0])));
            };
            gemv_units<BT, 1>(c, n_units, K, epi);
        }
        if (prof) { const unsigned long long t = globaltimer_ns(); seg[2] += t - ts; ts = t; }
        __syncthreads();
        if (prof) { const unsigned long long t = globaltimer_ns(); seg[3] += t - ts; ts = t; }
    }
}

// Sampling of one id per sequence (G:88-99 slow, G:118-132 depth) and, after the last depth code,
// frame assembly and the stop rule (G:143-166).
// tc_feed (tensor-core variant, cooperative launch, a depth step follows in the launch): the CTA that chose row b's id also
// writes the next depth step's input -- the slow hidden state after the slow id, the embedding of the code after a depth
// code (G:136-140) -- to the fast residual stream and its RMSNorm to M.xn, exactly as that step's own pre-step would
// (tc_row_step: same chunks per warp, same order of additions), which then is skipped.
__device__ void phase_sample(const DevModel& M, const CallArgs& A, const Ctx& c, const Phase& ph, bool tc_feed = false) {
    const bool fast = ph.fast != 0;
    const int N = fast ? M.codebook_size : M.vocab;
    const int r = fast ? 1 + ph.depth_pos : 0;
    const int R = M.n_rows;
    for (int b = c.cta; b < A.batch; b += c.n_ctas) {
        const float* src = fast ? M.depth_logits + ((size_t)b * M.depth + ph.depth_pos) * N : M.token_logits + (size_t)b * N;
        for (int i = c.tid; i < N; i += kThreads) c.xs[i] = ldcg_f32(src + i);
        __syncthreads();
        const uint32_t step = A.b.step ? (uint32_t)ldcg_i32(A.b.step + b) : 0u;
        const uint32_t seq_id = A.b.seq_id ? (uint32_t)ldcg_i32(A.b.seq_id + b) : (uint32_t)b;
        const SmolRowSampling prm = row_sampling(A.s, A.b.row_sampling, b);
        int tok = sample_row<kThreads>(c.xs, N, fast ? prm.fast_temp : prm.temp, fast ? 0 : prm.top_k, fast ? 1.0f : prm.top_p,
                             prm.min_p, prm.seed, step, seq_id, (uint32_t)r, g_sc);
        if (M.force != nullptr) tok = ldcg_i32(M.force + (size_t)b * R + r);
        if (c.tid == 0) {
            M.frame_tokens[(size_t)b * R + r] = tok;
            if (fast && ph.depth_pos == M.depth - 1) {
                const bool live = A.b.finished == nullptr || __ldcg(A.b.finished + b) == 0;
                if (live) {
                    const int st = A.b.step ? ldcg_i32(A.b.step + b) : 0;
                    int slow = 0;
                    for (int rr = 0; rr < R; ++rr) {
                        const int v = (rr == r) ? tok : ldcg_i32(M.frame_tokens + (size_t)b * R + rr);
                        if (rr == 0) slow = v;
                        A.b.tokens[(size_t)b * R + rr] = v;
                        if (A.b.out_codes != nullptr && st < A.b.max_frames)
                            A.b.out_codes[((size_t)b * A.b.max_frames + st) * R + rr] = v;
                    }
                    if (A.b.step) A.b.step[b] = st + 1;
                    if (b == 0 && M.frame_ns != nullptr && st < M.frame_ns_cap) M.frame_ns[st] = globaltimer_ns();
                    A.b.seq_len[b] = ldcg_i32(A.b.seq_len + b) + 1;
                    if (A.b.finished != nullptr && A.s.audio_only && !A.s.ignore_stop && slow == M.im_end)
                        A.b.finished[b] = 1;
                }
            }
        }
        if (tc_feed) {
            const int D = M.fdim, nch = D >> 3, ch = c.tid;
            const int next_pos = fast ? ph.depth_pos + 1 : 0;
            const uint16_t* row = !fast ? M.x + (size_t)b * D
                                        : M.fast_embeddings + (size_t)(tok + (M.depthwise_wte ? (M.dup0 ? next_pos - 1 : next_pos) * M.codebook_size : 0)) * D;
            const uint16_t* norm_w = M.fast_layers[0].attention_norm;
            float x[8];
            float ss = 0.f;
            uint4 wv = make_uint4(0u, 0u, 0u, 0u);
            if (ch < nch) {
                wv = __ldg(reinterpret_cast<const uint4*>(norm_w + ch * 8));
                unpack8(ldcg_v4(row + ch * 8), x);
#pragma unroll
                for (int e = 0; e < 8; ++e) ss = fmaf(x[e], x[e], ss);
            }
            ss = warp_sum(ss);
            if (c.lane == 0) g_part[c.warp] = ss;
            __syncthreads();
            if (ch < nch) {
                float t = 0.f;
                for (int i = 0; i < 3; ++i) t += g_part[i];
                const float mean = __fdiv_rn(t, (float)D);
                const float rs = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(mean, M.eps)));
                uint4 raw;
                raw.x = pack_bf16(x[0], x[1]); raw.y = pack_bf16(x[2], x[3]); raw.z = pack_bf16(x[4], x[5]); raw.w = pack_bf16(x[6], x[7]);
                *reinterpret_cast<uint4*>(M.xf + (size_t)b * D + ch * 8) = raw;
                float wf[8];
                unpack8(wv, wf);
                uint4 o;
                o.x = pack_bf16(__fmul_rn(bf16_round(__fmul_rn(x[0], rs)), wf[0]), __fmul_rn(bf16_round(__fmul_rn(x[1], rs)), wf[1]));
                o.y = pack_bf16(__fmul_rn(bf16_round(__fmul_rn(x[2], rs)), wf[2]), __fmul_rn(bf16_round(__fmul_rn(x[3], rs)), wf[3]));
                o.z = pack_bf16(__fmul_rn(bf16_round(__fmul_rn(x[4], rs)), wf[4]), __fmul_rn(bf16_round(__fmul_rn(x[5], rs)), wf[5]));
                o.w = pack_bf16(__fmul_rn(bf16_round(__fmul_rn(x[6], rs)), wf[6]), __fmul_rn(bf16_round(__fmul_rn(x[7], rs)), wf[7]));
                *reinterpret_cast<uint4*>(M.xn + (size_t)b * D + ch * 8) = o;
            }
        }
        __syncthreads();
    }
}

// BT == 0: the tensor-core variant (tc_phases.cuh) -- 128-row tiles, batch attention.
template <int BT>
__device__ __forceinline__ void run_phase(const DevModel& M, const CallArgs& A, const Ctx& c, const Phase& ph,
                                          uint32_t& parity, umma::Pipe& pipe, uint32_t& target, bool first_in_launch,
                                          bool next_in_launch) {
    if (BT == 0) {
        if (ph.kind == PH_ATTN) phase_attn_batch(M, A, c, ph);
        else if (ph.kind == PH_SAMPLE)
            phase_sample(M, A, c, ph, next_in_launch && !A.fast_from_xf && !(ph.fast && ph.depth_pos == M.depth - 1));
        else phase_gemm_tc(M, A, c, ph, &g_tc_bars, pipe, target, first_in_launch, next_in_launch);
        return;
    }
    if (ph.kind == PH_ATTN) phase_attn(M, A, c, ph);
    else if (ph.kind == PH_SAMPLE) phase_sample(M, A, c, ph);
    else phase_gemv<(BT > 0 ? BT : 1)>(M, A, c, ph, parity);
}

// Flat index (iteration, phase) of the next phase of this launch that streams weights, or -1.
__device__ __forceinline__ bool next_weight_phase(const DevModel& M, const CallArgs& A, int& it, int& p) {
    for (;;) {
        ++p;
        if (p >= A.phase_end) { p = A.phase_begin; ++it; }
        if (it >= A.n_iter) return false;
        const int k = (int)(M.prog[p] & 15u);
        if (k != PH_ATTN && k != PH_SAMPLE) return true;
    }
}

template <int BT>
__global__ void __launch_bounds__(kThreads, 1)
smol_decode_kernel(const __grid_constant__ DevModel M, const __grid_constant__ CallArgs A, const int xs_bytes) {
    extern __shared__ __align__(128) unsigned char smem_dyn[];
    Ctx c;
    c.cta = blockIdx.x; c.n_ctas = gridDim.x; c.tid = threadIdx.x;
    c.warp = threadIdx.x >> 5; c.lane = threadIdx.x & 31;
    c.xs = reinterpret_cast<float*>(smem_dyn);
    c.stage = smem_dyn + xs_bytes;
    c.iter = 0;

    if (c.tid == 0) {
        for (int w = 0; w < kWarps; ++w) mbar_init(&g_mbar[w], 1u);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    uint32_t target = ldcg_u32(M.barrier + 1);
    uint32_t parity = 0;
    umma::Pipe pipe;
    pipe.chunk = 0; pipe.tile = 0;
    if (BT == 0) umma::setup(&g_tc_bars, pipe, (uint32_t)umma::kAcc, 2u);
    const int per_iter = A.prefill ? phases_per_prefill_step(M.n_layer)
                                   : phases_per_frame(M.n_layer, M.n_flayer, M.depth);
    const bool prof_cta = (M.prof != nullptr) && c.cta == 0;  // CTA-uniform
    const bool prof = prof_cta && c.tid == 0;
    unsigned long long t0 = 0, t1 = 0;
    int st_it = -1, st_p = -1;  // (iteration, phase) whose weights are staged / in flight
    for (int it = 0; it < A.n_iter; ++it) {
        c.iter = it;
        for (int p = A.phase_begin; p < A.phase_end; ++p) {
            const Phase ph = unpack_phase(M.prog[p]);
            const bool has_w = BT != 0 && ph.kind != PH_ATTN && ph.kind != PH_SAMPLE;  // weights staged a phase ahead (GEMV variants)
            if (prof) t0 = globaltimer_ns();
            if (has_w && !(st_it == it && st_p == p)) {  // cold start of a launch
                stage_issue(c, phase_plan(M, ph));
                st_it = it; st_p = p;
            }
            run_phase<BT>(M, A, c, ph, parity, pipe, target, p == A.phase_begin, p + 1 < A.phase_end);
            if (prof_cta) {
                __syncthreads();
                if (prof) t1 = globaltimer_ns();
            }
            if (c.cta == 0 && p == per_iter - 1 && A.prefill) {
                // prefill bookkeeping: every sequence advances by the positions of this tile that lie inside its prompt
                const int T = A.tile_t > 1 ? A.tile_t : 1;
                for (int b = c.tid; b < A.real_batch; b += kThreads) {
                    int n_act = ldcg_i32(A.prompt_len + b) - 1 - (A.iter_base + c.iter * T);
                    n_act = n_act < 0 ? 0 : (n_act > T ? T : n_act);
                    if (n_act) A.b.seq_len[b] = ldcg_i32(A.b.seq_len + b) + n_act;
                }
            }
            if (c.cta == 0 && !A.prefill && A.advance && p == A.phase_end - 1) {
                for (int b = c.tid; b < A.batch; b += kThreads) A.b.seq_len[b] = ldcg_i32(A.b.seq_len + b) + 1;
            }
            const bool last = (it == A.n_iter - 1) && (p == A.phase_end - 1);
            if (!last) {
                if (BT == 0) fence_proxy_async_all();
                grid_arrive(M.barrier, target, (uint32_t)c.n_ctas);
            }
            if (has_w) {
                // Every warp is past its last read of the stage buffer (phases end with a block barrier):
                // stream the next weight phase in while the other CTAs arrive at the grid barrier.
                int nit = it, np = p;
                if (next_weight_phase(M, A, nit, np)) {
                    stage_issue(c, phase_plan(M, unpack_phase(M.prog[np])));
                    st_it = nit; st_p = np;
                }
            }
            if (!last) {
                grid_wait(M.barrier, target);
                if (BT == 0 && (c.tid == umma::kTmaProducerA || c.tid == umma::kTmaProducerB)) fence_proxy_async_all();   // the threads that issue TMA loads
            }
            if (prof) {  // [2p] CTA 0's own time in the phase, [2p+1] its wait at the barrier that follows
                const unsigned long long t2 = globaltimer_ns();
                M.prof[2 * p] += t1 - t0;
                M.prof[2 * p + 1] += t2 - t1;
            }
        }
    }
    if (A.prefill && A.finalize && c.cta == 0) {
        // leave the last prompt column as the pending input of the first decode frame (G:66-73)
        for (int i = c.tid; i < A.real_batch * M.n_rows; i += kThreads) {
            const int b = i / M.n_rows, r = i - b * M.n_rows;
            const int len = ldcg_i32(A.prompt_len + b);
            A.b.tokens[i] = ldcg_i32(A.prompt + ((size_t)b * M.n_rows + r) * A.s_max + (len - 1));
        }
    }
    if (c.cta == 0 && c.tid == 0) M.barrier[1] = target;
    if (BT == 0) umma::teardown(&g_tc_bars);
}

// Stand-alone sampler on caller-provided logits [B][n] (smol_sample): one CTA per sequence.
__global__ void __launch_bounds__(kThreads, 1)
smol_sample_kernel(const float* logits, int n, int batch, SmolSampling s, const SmolRowSampling* table, int stream_id,
                   const int32_t* seq_id, const int32_t* step, int32_t* out) {
    extern __shared__ __align__(16) float smem_sample[];
    float* smem_dyn = smem_sample;
    for (int b = blockIdx.x; b < batch; b += gridDim.x) {
        for (int i = threadIdx.x; i < n; i += kThreads) smem_dyn[i] = logits[(size_t)b * n + i];
        __syncthreads();
        const bool fast = stream_id != 0;
        const SmolRowSampling prm = row_sampling(s, table, b);
        const int tok = sample_row<kThreads>(smem_dyn, n, fast ? prm.fast_temp : prm.temp, fast ? 0 : prm.top_k, fast ? 1.0f : prm.top_p,
                                   prm.min_p, prm.seed, step ? (uint32_t)step[b] : 0u, seq_id ? (uint32_t)seq_id[b] : (uint32_t)b,
                                   (uint32_t)stream_id, g_sc);
        if (threadIdx.x == 0) out[b] = tok;
        __syncthreads();
    }
}

// smol_fast_embed: remember depth code `depth_pos` of every sequence; the next depth step embeds it.
__global__ void smol_store_codes_kernel(int32_t* frame_tokens, const int32_t* codes, int batch, int n_rows, int row) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < batch) frame_tokens[(size_t)b * n_rows + row] = codes[b];
}

cudaError_t sample_launch(const float* logits, int n, int batch, const SmolSampling& s, const SmolRowSampling* table,
                          int stream_id, const int32_t* seq_id, const int32_t* step, int32_t* out, cudaStream_t stream) {
    const size_t smem = (size_t)n * sizeof(float);
    cudaError_t e = cudaFuncSetAttribute(smol_sample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
    if (e != cudaSuccess) return e;
    smol_sample_kernel<<<batch < 1024 ? batch : 1024, kThreads, smem, stream>>>(logits, n, batch, s, table, stream_id, seq_id,
                                                                               step, out);
    return cudaGetLastError();
}

// silu over EVERY bf16 input, by the exact expression the GEMV epilogues use (F.silu in fp32, bf16 out; P:581): the
// tensor-core epilogue and the data-flow kernel look the result up instead of evaluating exp and a division per element,
// so all kernels round at the same points and agree bit for bit.
__global__ void smol_silu_lut_kernel(uint16_t* lut) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 65536u) return;
    const float a = __uint_as_float(i << 16);
    lut[i] = f_to_bf(__fdiv_rn(a, __fadd_rn(1.0f, expf(-a))));
}
cudaError_t silu_lut_launch(uint16_t* lut, cudaStream_t stream) {
    smol_silu_lut_kernel<<<256, 256, 0, stream>>>(lut);
    return cudaGetLastError();
}

cudaError_t store_codes_launch(int32_t* frame_tokens, const int32_t* codes, int batch, int n_rows, int row,
                               cudaStream_t stream) {
    smol_store_codes_kernel<<<(batch + 127) / 128, 128, 0, stream>>>(frame_tokens, codes, batch, n_rows, row);
    return cudaGetLastError();
}

// ---- host-side launch helpers (called from capi.cu) ----------------------------------------------
// Activation region: the batch tile's rows in fp32 (also the attention merge scratch and the
// sampler's logits row).  Sized for the batch the model was created for.
size_t decode_xs_bytes(const DevModel& M, int bt) {
    if (bt == 0) return (size_t)umma::kRingBytes + 2048 + kTcRows * 4;  // 1024-aligned ring + RoPE positions of the tile's rows
    int kmax = M.dim;
    if (M.inter > kmax) kmax = M.inter;
    if (M.fdim > kmax) kmax = M.fdim;
    if (M.finter > kmax) kmax = M.finter;
    size_t a = (size_t)bt * kmax * sizeof(float);
    size_t b = (size_t)kWarps * kMaxGroup * kPartialStride * sizeof(float);
    int nl = M.vocab > M.codebook_size ? M.vocab : M.codebook_size;
    size_t cbytes = (size_t)nl * sizeof(float);
    size_t m = a > b ? a : b;
    m = m > cbytes ? m : cbytes;
    return (m + 127) / 128 * 128;
}

// Stage region: the weight rows one CTA owns in the heaviest phase.
size_t decode_stage_bytes(const DevModel& M, int n_ctas) {
    auto per = [&](long units, long slot) { return (size_t)((units + n_ctas - 1) / n_ctas) * (size_t)slot; };
    size_t m = 0;
    auto upd = [&](size_t v) { if (v > m) m = v; };
    upd(per((M.n_head + 2 * M.n_kv) * kHeadDim / 2, 4L * M.dim));
    upd(per(M.dim, 2L * M.dim));
    upd(per(M.inter, 4L * M.dim));
    upd(per(M.dim, 2L * M.inter));
    upd(per(M.vocab, 2L * M.dim));
    upd(per((M.fn_head + 2 * M.fn_kv) * kHeadDim / 2, 4L * M.fdim));
    upd(per(M.fdim, 2L * M.fdim));
    upd(per(M.finter, 4L * M.fdim));
    upd(per(M.fdim, 2L * M.finter));
    upd(per(M.codebook_size, 2L * M.fdim));
    return (m + 127) / 128 * 128;
}

// Kernel variant by batch tile (sequences whose activations share one pass over the weights).
static int tile_index(int bt) { return bt <= 0 ? 4 : bt <= 1 ? 0 : bt <= 2 ? 1 : bt <= 4 ? 2 : 3; }  // bt 0: tensor-core variant
static const void* decode_fn(int bt) {
    switch (tile_index(bt)) {
        case 4: return (const void*)smol_decode_kernel<0>;
        case 0: return (const void*)smol_decode_kernel<1>;
        case 1: return (const void*)smol_decode_kernel<2>;
        case 2: return (const void*)smol_decode_kernel<4>;
        default: return (const void*)smol_decode_kernel<8>;
    }
}
int decode_batch_tile(int batch) { return batch <= 1 ? 1 : batch <= 2 ? 2 : batch <= 4 ? 4 : 8; }

// The attribute is per function, not per model: it only ever grows (several models may coexist).
static size_t g_smem_configured[5] = {0, 0, 0, 0, 0};
cudaError_t decode_configure(int bt, size_t smem) {
    size_t& cur = g_smem_configured[tile_index(bt)];
    if (smem <= cur) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(decode_fn(bt), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) cur = smem;
    return e;
}

cudaError_t decode_max_ctas(int bt, size_t smem, int* per_sm) {
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, decode_fn(bt), kThreads, smem);
}

cudaError_t decode_launch(const DevModel& M, const CallArgs& A, int bt, int n_ctas, size_t smem, int xs_bytes,
                          cudaStream_t stream) {
    void* args[3] = {(void*)&M, (void*)&A, (void*)&xs_bytes};
    return cudaLaunchCooperativeKernel(decode_fn(bt), dim3(n_ctas), dim3(kThreads), args, smem, stream);
}

}  // namespace smol
