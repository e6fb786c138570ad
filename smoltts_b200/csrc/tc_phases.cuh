// Batched decode on the tensor cores: the weight phases of decode_kernel.cu as tcgen05 tiles (umma.cuh) for batches of
// 9+ rows (sequences, or prompt positions of a prefill tile), plus the batch forms of the two attentions.
// Included by decode_kernel.cu (uses its Ctx, grid barrier, embedding and row bookkeeping helpers).
//
// A weight phase Y[rows][n_out] = f(X)[rows][K] * W[n_out][K]^T is cut into units (128-row tile, block of `blk` weight
// rows); blk is the smallest multiple of 16 that gives every CTA at most one unit.  A unit streams its 128 x K activation
// tile and blk x K weight rows through the cp.async ring in 64-element stages; RMSNorm is applied to the activation
// pieces in shared memory (row statistics from a first pass over the rows), the epilogues (RoPE + KV append, residual
// add, silu * up, logits) read the fp32 accumulator from TMEM -- same rounding points as the GEMV kernels (bf16 after
// every Linear / norm stage / RoPE / silu / product / residual add), only the summation order inside a dot product is
// the tensor core's.
#pragma once

// L2 policy of the weight boxes: 0 default, 1 evict_first, 2 evict_last.  Measured at bs=256 (profiles/r2_l2_policy_ab.txt):
// the hints (evict_last on the depth transformer, evict_first on the slow one) cost 9 % MORE DRAM traffic than no hint
// and no time either way, so the tiles carry none.  (The data-flow kernel keeps its hints: there they hold the depth
// weights in L2, 235 MB of DRAM traffic per frame against 271 MB of weights.)
#ifndef SMOL_TC_FAST_POLICY
#define SMOL_TC_FAST_POLICY umma::kWeightsDefault
#endif
#ifndef SMOL_TC_SLOW_POLICY
#define SMOL_TC_SLOW_POLICY umma::kWeightsDefault
#endif
// Unit -> CTA order: 1 = the row tiles that share a weight block run on neighbouring CTAs (prefill iterations of 4 row
// tiles: 20 % less DRAM traffic, same time), 0 = row tile major.
#ifndef SMOL_TC_UNIT_ORDER
#define SMOL_TC_UNIT_ORDER 1
#endif

namespace smol {

constexpr int kTcRows = umma::kM;
constexpr int kTcSplit = 128;  // cached positions per attention split of the batch attention (CallArgs.tc_split overrides it)
__device__ __forceinline__ float ex2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
    uint4 v;
    v.x = pack_bf16(f[0], f[1]); v.y = pack_bf16(f[2], f[3]); v.z = pack_bf16(f[4], f[5]); v.w = pack_bf16(f[6], f[7]);
    return v;
}

// Row steps of the tensor-core variant (pre-step of a normed phase, post-step of a split-K phase).  Three warps per row
// (one 16-byte chunk per lane: every load of a row is in flight at once), five rows per CTA and pass, rows spread over
// the grid.  load(bg, ch, x) produces chunk ch of row bg; the row goes to `raw` (if any) as it is and, if norm_w is given,
// through RMSNorm (P:601-613: fp32 normalise, round to bf16, multiply by the bf16 weight, round again) to M.xn.
constexpr int kRowWarps = 3;
constexpr int kRowsPerPass = kWarps / kRowWarps;

template <class Load>
__device__ __forceinline__ void tc_row_step(const DevModel& M, const CallArgs& A, const Ctx& c, int D, uint16_t* raw,
                                            const uint16_t* norm_w, Load load) {
    const int nch = D >> 3;
    const int slot = c.warp / kRowWarps, wi = c.warp - slot * kRowWarps;
    const int ch = wi * 32 + c.lane;
    for (int row0 = c.cta * kRowsPerPass; row0 < A.batch; row0 += c.n_ctas * kRowsPerPass) {
        const int bg = row0 + slot;
        const bool act = slot < kRowsPerPass && bg < A.batch && ch < nch;
        float x[8];
        float ss = 0.f;
        uint4 wv = make_uint4(0u, 0u, 0u, 0u);
        if (act) {
            if (norm_w != nullptr) wv = __ldg(reinterpret_cast<const uint4*>(norm_w + ch * 8));
            load(bg, ch, x);
#pragma unroll
            for (int e = 0; e < 8; ++e) ss = fmaf(x[e], x[e], ss);
        }
        ss = warp_sum(ss);
        if (c.lane == 0) g_part[c.warp] = ss;
        __syncthreads();
        if (act) {
            if (raw != nullptr) *reinterpret_cast<uint4*>(raw + (size_t)bg * D + ch * 8) = pack8(x);
            if (norm_w != nullptr) {
                float t = 0.f;
                for (int i = 0; i < kRowWarps; ++i) t += g_part[slot * kRowWarps + i];
                const float mean = __fdiv_rn(t, (float)D);
                const float r = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(mean, M.eps)));
                float wf[8], o[8];
                unpack8(wv, wf);
#pragma unroll
                for (int e = 0; e < 8; ++e) o[e] = __fmul_rn(bf16_round(__fmul_rn(x[e], r)), wf[e]);
                *reinterpret_cast<uint4*>(M.xn + (size_t)bg * D + ch * 8) = pack8(o);
            }
        }
        __syncthreads();
    }
}

// Input pre-step of a normed weight phase: gather the row (token embedding P:205-221, the slow hidden state or the
// previous depth code's embedding G:136-140, or a residual stream), keep the raw row as the residual stream where the
// phase starts one (`spill`), and write RMSNorm(row) to M.xn, which the phase's tiles read through TMA.
// src_kind: 0 token embedding, 1 slow hidden state, 2 embedding of the previous depth code, 3 `base` rows.
__device__ void tc_norm_rows(const DevModel& M, const CallArgs& A, const Ctx& c, const Phase& ph, int src_kind,
                             const uint16_t* base, uint16_t* spill, const uint16_t* norm_w, int D) {
    tc_row_step(M, A, c, D, spill, norm_w, [&](int bg, int ch, float (&x)[8]) {
        if (src_kind == 0) { embed_chunk(M, A, c, bg, ch, x); return; }
        const uint16_t* src = base + (size_t)bg * D;
        if (src_kind == 1) {
            src = M.x + (size_t)bg * D;
        } else if (src_kind == 2) {
            const int code = ldcg_i32(M.frame_tokens + (size_t)bg * M.n_rows + ph.depth_pos);
            const int off = M.depthwise_wte ? (M.dup0 ? ph.depth_pos - 1 : ph.depth_pos) * M.codebook_size : 0;
            src = M.fast_embeddings + (size_t)(code + off) * D;
        }
        unpack8(ldcg_v4(src + ch * 8), x);
    });
}

// Post-step of the split-K phases (wo, w2): dst = res + bf16(sum of the K-slice partials, in slice order) -- the Linear's
// bf16 output plus the residual (P:499-500) -- and, when the next phase of the launch is the normed phase that reads dst
// (w13 after wo; the next layer's QKV or the head after w2), its RMSNorm into M.xn, so that phase starts without a
// pre-step of its own.
__device__ void tc_residual_finish(const DevModel& M, const CallArgs& A, const Ctx& c, const uint16_t* res, uint16_t* dst,
                                   int D, int n_split, const uint16_t* norm_w) {
    tc_row_step(M, A, c, D, dst, norm_w, [&](int bg, int ch, float (&x)[8]) {
        const uint4 rv = ldcg_v4(res + (size_t)bg * D + ch * 8);
        float4 pa[kTcKSplit], pb[kTcKSplit];
#pragma unroll
        for (int sp = 0; sp < kTcKSplit; ++sp) {
            if (sp < n_split) {
                const float* pp = M.kpart + ((size_t)sp * M.ws_rows + bg) * D + ch * 8;
                pa[sp] = __ldcg(reinterpret_cast<const float4*>(pp));
                pb[sp] = __ldcg(reinterpret_cast<const float4*>(pp + 4));
            } else {
                pa[sp] = make_float4(0.f, 0.f, 0.f, 0.f);
                pb[sp] = pa[sp];
            }
        }
        float acc[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] = 0.f;
#pragma unroll
        for (int sp = 0; sp < kTcKSplit; ++sp) {
            if (sp < n_split) {
                acc[0] = __fadd_rn(acc[0], pa[sp].x); acc[1] = __fadd_rn(acc[1], pa[sp].y);
                acc[2] = __fadd_rn(acc[2], pa[sp].z); acc[3] = __fadd_rn(acc[3], pa[sp].w);
                acc[4] = __fadd_rn(acc[4], pb[sp].x); acc[5] = __fadd_rn(acc[5], pb[sp].y);
                acc[6] = __fadd_rn(acc[6], pb[sp].z); acc[7] = __fadd_rn(acc[7], pb[sp].w);
            }
        }
        float rf[8];
        unpack8(rv, rf);
#pragma unroll
        for (int e = 0; e < 8; ++e) x[e] = bf16_round(__fadd_rn(rf[e], bf16_round(acc[e])));
    });
}

// Attention of the fast transformer for every (row, head) of the batch, one warp per pair, spread over the grid; the
// result goes to M.attn (the wo tiles read it after a grid barrier).  Same arithmetic as fast_attention_rows.
__device__ void tc_fast_attention(const DevModel& M, const CallArgs& A, const Ctx& c, int layer, int depth_pos) {
    const int Hq = M.fn_head, Hkv = M.fn_kv, G = Hq / Hkv, D = M.fdim;
    const int kvw = Hkv * kHeadDim;
    const int jl = c.lane >> 2, part = c.lane & 3;
    for (int pair = c.cta * kWarps + c.warp; pair < A.batch * Hq; pair += c.n_ctas * kWarps) {
        const int bg = pair / Hq, hq = pair - bg * Hq, kvh = hq / G;
        const uint16_t* qp = M.q + (size_t)bg * Hq * kHeadDim + hq * kHeadDim + part * 16;
        const uint16_t* kb = M.fkv + ((size_t)(bg * M.n_flayer + layer) * 2) * M.depth * kvw + kvh * kHeadDim;
        const uint16_t* vb = kb + (size_t)M.depth * kvw;
        // every load of the pair is issued before the first use: q (16 dims per lane), the lane group's K rows, all V
        const bool ok0 = jl <= depth_pos, ok1 = jl + 8 <= depth_pos;
        const uint4 zero4 = make_uint4(0u, 0u, 0u, 0u);
        const uint4 q0 = ldcg_v4(qp), q1 = ldcg_v4(qp + 8);
        const uint4 ka0 = ok0 ? ldcg_v4(kb + (size_t)jl * kvw + part * 16) : zero4;
        const uint4 ka1 = ok0 ? ldcg_v4(kb + (size_t)jl * kvw + part * 16 + 8) : zero4;
        const uint4 kb0 = ok1 ? ldcg_v4(kb + (size_t)(jl + 8) * kvw + part * 16) : zero4;
        const uint4 kb1 = ok1 ? ldcg_v4(kb + (size_t)(jl + 8) * kvw + part * 16 + 8) : zero4;
        // V rows as 32-bit offsets from one per-lane base: a 64-bit address per position, each under its own j <= depth_pos
        // predicate, makes this prologue ~20 % longer and spills predicates (the fast wo pre-step at bs=256: +9 %)
        const uint32_t* vl = reinterpret_cast<const uint32_t*>(vb) + c.lane;   // V dims 2*lane, 2*lane+1 of position 0
        uint32_t vv[kMaxDepth];
#pragma unroll
        for (int j = 0; j < kMaxDepth; ++j) vv[j] = j <= depth_pos ? __ldcg(vl + j * (kvw / 2)) : 0u;
        float qf[16];
        unpack8(q0, *reinterpret_cast<float(*)[8]>(qf));
        unpack8(q1, *reinterpret_cast<float(*)[8]>(qf + 8));
        float sc[2];
        const bool ok[2] = {ok0, ok1};
#pragma unroll
        for (int h2 = 0; h2 < 2; ++h2) {
            sc[h2] = -INFINITY;
            float k0[8], k1[8];
            unpack8(h2 ? kb0 : ka0, k0);
            unpack8(h2 ? kb1 : ka1, k1);
            float s = 0.f;
#pragma unroll
            for (int e = 0; e < 8; ++e) s = fmaf(qf[e], k0[e], s);
#pragma unroll
            for (int e = 0; e < 8; ++e) s = fmaf(qf[8 + e], k1[e], s);
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            if (ok[h2]) sc[h2] = s * 0.125f;
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
        float o0 = 0.f, o1 = 0.f;  // lane owns dims 2*lane, 2*lane+1
#pragma unroll
        for (int j = 0; j < kMaxDepth; ++j) {
            const float p = __shfl_sync(0xffffffffu, j < 8 ? pb0 : pb1, (j & 7) * 4);
            o0 = fmaf(p, bf_lo(vv[j]), o0);   // positions past depth_pos: p = 0, v = 0
            o1 = fmaf(p, bf_hi(vv[j]), o1);
        }
        const float inv = 1.0f / l;
        *reinterpret_cast<uint32_t*>(M.attn + (size_t)bg * D + hq * kHeadDim + 2 * c.lane) = pack_bf16(o0 * inv, o1 * inv);
    }
}

// ---- batch attention on the tensor cores -------------------------------------------------------------------------
// mma.sync.m16n8k16 (bf16 x bf16 -> fp32): the 16 rows of the A operand are the query rows that share one kv head's
// cached K/V -- the G query heads of the kv head (GQA) times, in a prefill iteration, up to 16/G consecutive prompt
// positions of the sequence -- so one pass over a position's 256 bytes of K|V serves all of them.
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
    return r;
}

// Split schedule of the batch attention: ABSOLUTE position ranges, the same for every row whatever its length -- 16
// splits of s0 positions, then splits of 2*s0 -- so that rows of different lengths (the consecutive prompt positions of a
// prefill group) share their K/V passes and a row's result is still a function of its own context only (it combines, in
// split order, the splits that start below its length).  s0 = 128 covers 6144 positions with kMaxSplits = 32 splits.
struct SplitPlan {
    int s0, wide_from;   // splits [0, wide_from) hold s0 positions, later ones 2*s0
    __device__ __forceinline__ int lo(int k) const { return k <= wide_from ? k * s0 : wide_from * s0 + (k - wide_from) * 2 * s0; }
    __device__ __forceinline__ int count(int L) const {   // splits that start below position L
        if (L <= wide_from * s0) return (L + s0 - 1) / s0;
        return wide_from + (L - wide_from * s0 + 2 * s0 - 1) / (2 * s0);
    }
};
__device__ __forceinline__ SplitPlan split_plan(const CallArgs& A, int cap) {
    SplitPlan sp;
    if (A.tc_split >= 16) {   // the caller's override (tests): uniform splits, widened only if kMaxSplits would not cover cap
        sp.s0 = max(A.tc_split & ~15, (((cap + kMaxSplits - 1) / kMaxSplits) + 15) & ~15);
        sp.wide_from = kMaxSplits;
        return sp;
    }
    sp.s0 = kTcSplit;
    sp.wide_from = kMaxSplits / 2;
    while (sp.lo(kMaxSplits) < cap) sp.s0 *= 2;
    return sp;
}

// Decode / prefill attention over the paged cache for a batch.  Unit = one WARP per (query group, kv head, split); a
// query group is one decode row, or up to 16/G consecutive prompt positions of one sequence.  Per 16 cached positions:
// S = Q K^T (2 n-tiles x 4 k-steps), online softmax in base 2 with P rounded to bf16 for the PV product as the reference's
// SDPA does (P:559-566; the denominator sums the unrounded fp32 values), O += P V (8 n-tiles).  K, V and Q fragments are
// loaded straight from global memory with 16-byte loads: the k index of the QK product and the n index of the PV product
// are permuted so that every thread's fragment words are contiguous in memory (a dot product does not care about the
// order of its dims as long as both operands use the same one).
// Splits of a long row meet through M.partial / M.split_count; the last arriver combines them in split order.
__device__ void phase_attn_batch(const DevModel& M, const CallArgs& A, const Ctx& c, const Phase& ph) {
    const int Hq = M.n_head, Hkv = M.n_kv, ps = M.page_size, G = Hq / Hkv;
    const int cap = A.b.max_pages * ps;
    const int T = A.tile_t > 1 ? A.tile_t : 1;
    const int P = T > 1 ? 16 / G : 1;              // query positions per unit
    const int gps = (T + P - 1) / P;               // units (groups) per sequence
    const int n_groups = (A.batch / T) * gps;
    const int gq = c.lane >> 2, tq = c.lane & 3;   // fragment coordinates of this lane
    // splits to enumerate: enough for the longest row of the batch (one pass over seq_len; rows with fewer splits skip)
    if (c.tid == 0) g_flag = 1;
    __syncthreads();
    {
        int lmax = 1;
        for (int b = c.tid; b < A.batch; b += kThreads) lmax = max(lmax, ldcg_i32(A.b.seq_len + row_seq(A, b)) + row_off(A, b) + 1);
        lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, 16));
        lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, 8));
        lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, 4));
        lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, 2));
        lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, 1));
        if (c.lane == 0) atomicMax(&g_flag, lmax);
    }
    __syncthreads();
    const SplitPlan sp = split_plan(A, cap);
    const int s_cap = min(sp.count(min(g_flag, cap)), kMaxSplits);
    const int n_tasks = n_groups * Hkv * s_cap;
    const size_t head_stride = (size_t)ps * kHeadDim;
    const size_t page_stride = (size_t)M.n_layer * 2 * Hkv * head_stride;
    constexpr float kScale = 0.125f * 1.4426950408889634f;   // 1/sqrt(64) * log2(e): softmax in base 2

    for (int t = c.cta * kWarps + c.warp; t < n_tasks; t += c.n_ctas * kWarps) {
        const int s = t % s_cap, kvh = (t / s_cap) % Hkv, grp = t / (s_cap * Hkv);
        const int b0 = (grp / gps) * T + (grp % gps) * P;            // first batch row of the group
        const int nq = min(P, T - (grp % gps) * P);                   // its live query positions
        const int bs = row_seq(A, b0);
        const int len0 = ldcg_i32(A.b.seq_len + bs);
        const int L0 = len0 + row_off(A, b0) + 1;                     // context of the first row (its own position included)
        const int Lg = min(L0 + nq - 1, cap);                         // ... of the last one
        const int p0 = sp.lo(s);
        if (p0 >= Lg) continue;
        // cached positions that hold data: everything up to the group's last ACTIVE row (rows past the end of a prompt do
        // not append; their stale slots must not reach the PV product of the active rows as 0 x garbage)
        int Lload = Lg;
        if (A.prefill) {
            const int act = ldcg_i32(A.prompt_len + bs) - 1 - (A.iter_base + c.iter * T);
            Lload = min(Lg, len0 + max(0, min(act, T)));
        }
        const int p1 = min(Lg, sp.lo(s + 1));
        const int pl = min(p1, Lload);
        // the two query rows of this lane: row r = (query position r / G, head r % G)
        const int ra = gq, rb = gq + 8;
        const int ia = ra / G, ib = rb / G;
        const bool va = ia < nq, vb = ib < nq;
        const int La = min(L0 + ia, cap), Lb = min(L0 + ib, cap);     // causal limits (positions < L are visible)
        uint32_t qa[4][4];
        {
            const uint4 z = make_uint4(0u, 0u, 0u, 0u);
            const uint16_t* qpa = M.q + ((size_t)(b0 + ia) * Hq + kvh * G + (ra - ia * G)) * kHeadDim + tq * 8;
            const uint16_t* qpb = M.q + ((size_t)(b0 + ib) * Hq + kvh * G + (rb - ib * G)) * kHeadDim + tq * 8;
            const uint4 a0 = va ? ldcg_v4(qpa) : z, a1 = va ? ldcg_v4(qpa + 32) : z;
            const uint4 c0 = vb ? ldcg_v4(qpb) : z, c1 = vb ? ldcg_v4(qpb + 32) : z;
            // k-step ks covers the dims {32 (ks >> 1) + 8 tq + 4 (ks & 1) + 0..3} of this lane (K uses the same map)
            qa[0][0] = a0.x; qa[0][1] = c0.x; qa[0][2] = a0.y; qa[0][3] = c0.y;
            qa[1][0] = a0.z; qa[1][1] = c0.z; qa[1][2] = a0.w; qa[1][3] = c0.w;
            qa[2][0] = a1.x; qa[2][1] = c1.x; qa[2][2] = a1.y; qa[2][3] = c1.y;
            qa[3][0] = a1.z; qa[3][1] = c1.z; qa[3][2] = a1.w; qa[3][3] = c1.w;
        }
        float o[8][4];
#pragma unroll
        for (int n = 0; n < 8; ++n) { o[n][0] = 0.f; o[n][1] = 0.f; o[n][2] = 0.f; o[n][3] = 0.f; }
        float ma = -INFINITY, mb = -INFINITY, la = 0.f, lb = 0.f;      // running max (quad-uniform), this lane's share of the sums
        const int32_t* bt = A.b.block_table + (size_t)bs * A.b.max_pages;
        // page ids of the split: lane i holds the id of the i-th page the split touches (one coalesced load; a split longer
        // than 32 pages reloads).  A 16-position group never straddles a page (pages hold 16 or 32 positions).
        const int psh = ps == 32 ? 5 : 4;
        int pg_base = p0 >> psh;
        int my_page = ((pg_base + c.lane) << psh) < pl ? ldcg_i32(bt + pg_base + c.lane) : 0;
        // Addressing is the hot loop's other half (the phase is issue-bound): everything per-lane is a byte offset fixed
        // before the loop, a group costs one shuffle and one 64-bit multiply-add, full groups load without predicates.
        const char* pool = reinterpret_cast<const char*>(M.kv_pool) + ((size_t)ph.layer * 2 * Hkv + kvh) * head_stride * 2;
        const size_t page_bytes = page_stride * 2, v_delta = (size_t)Hkv * head_stride * 2;
        const uint32_t koff = (uint32_t)(gq * kHeadDim + tq * 8) * 2;        // K row gq (n-tile 1: + 8 rows), this lane's dims 8 tq .. (+ 32)
        const uint32_t voff = (uint32_t)(2 * tq * kHeadDim + gq * 8) * 2;    // V rows 2 tq (+ 1, + 8, + 9), dims 8 gq ..
        auto group_base = [&](int pb) -> const char* {
            const int pg = pb >> psh;
            if (pg - pg_base >= 32) {
                pg_base = pg;
                my_page = ((pg_base + c.lane) << psh) < pl ? ldcg_i32(bt + pg_base + c.lane) : 0;
            }
            const int page = __shfl_sync(0xffffffffu, my_page, (pg - pg_base) & 31);
            return pool + (size_t)page * page_bytes + ((size_t)(pb & (ps - 1)) << 7);
        };
        const uint4 z = make_uint4(0u, 0u, 0u, 0u);
        uint4 kk[2][2], vv[4];
        auto load_k = [&](const char* gb, int pb) {      // K rows of n-tile j: position pb + 8 j + gq, this lane's 2 x 8 dims
            const char* kp = gb + koff;
            if (pb + 16 <= pl) {
                kk[0][0] = ldcg_v4(kp); kk[0][1] = ldcg_v4(kp + 64);
                kk[1][0] = ldcg_v4(kp + 1024); kk[1][1] = ldcg_v4(kp + 1088);
            } else {
                const bool ok0 = pb + gq < pl, ok1 = pb + 8 + gq < pl;
                kk[0][0] = ok0 ? ldcg_v4(kp) : z; kk[0][1] = ok0 ? ldcg_v4(kp + 64) : z;
                kk[1][0] = ok1 ? ldcg_v4(kp + 1024) : z; kk[1][1] = ok1 ? ldcg_v4(kp + 1088) : z;
            }
        };
        auto load_v = [&](const char* gb, int pb) {      // V rows pb + {2 tq, 2 tq + 1, 2 tq + 8, 2 tq + 9}, dims 8 gq .. 8 gq + 7
            const char* vp = gb + v_delta + voff;
            if (pb + 16 <= pl) {
                vv[0] = ldcg_v4(vp); vv[1] = ldcg_v4(vp + 128); vv[2] = ldcg_v4(vp + 1024); vv[3] = ldcg_v4(vp + 1152);
            } else {
                const int r = pb + 2 * tq;
                vv[0] = r < pl ? ldcg_v4(vp) : z; vv[1] = r + 1 < pl ? ldcg_v4(vp + 128) : z;
                vv[2] = r + 8 < pl ? ldcg_v4(vp + 1024) : z; vv[3] = r + 9 < pl ? ldcg_v4(vp + 1152) : z;
            }
        };
        // software pipeline without extra registers: the K fragments are dead after the QK products and the V fragments
        // after the PV products, so the next group's K loads are issued right after QK (covered by the softmax and PV of
        // this group) and its V loads right after PV (covered by the next group's QK and softmax)
        const char* gb = group_base(p0);
        load_k(gb, p0);
        load_v(gb, p0);
        for (int pb = p0; pb < p1; pb += 16) {
            const bool more = pb + 16 < p1;
            float sc[2][4];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                sc[j][0] = 0.f; sc[j][1] = 0.f; sc[j][2] = 0.f; sc[j][3] = 0.f;
                mma16816(sc[j], qa[0], kk[j][0].x, kk[j][0].y);
                mma16816(sc[j], qa[1], kk[j][0].z, kk[j][0].w);
                mma16816(sc[j], qa[2], kk[j][1].x, kk[j][1].y);
                mma16816(sc[j], qa[3], kk[j][1].z, kk[j][1].w);
            }
            if (more) { gb = group_base(pb + 16); load_k(gb, pb + 16); }
            // scores in the log2 domain, causal mask per row, one running-max update per row and 16 positions
            float mna = ma, mnb = mb;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int pc = pb + 8 * j + 2 * tq;
                sc[j][0] = pc < La ? sc[j][0] * kScale : -INFINITY;
                sc[j][1] = pc + 1 < La ? sc[j][1] * kScale : -INFINITY;
                sc[j][2] = pc < Lb ? sc[j][2] * kScale : -INFINITY;
                sc[j][3] = pc + 1 < Lb ? sc[j][3] * kScale : -INFINITY;
                mna = fmaxf(mna, fmaxf(sc[j][0], sc[j][1]));
                mnb = fmaxf(mnb, fmaxf(sc[j][2], sc[j][3]));
            }
            mna = fmaxf(mna, __shfl_xor_sync(0xffffffffu, mna, 1));
            mna = fmaxf(mna, __shfl_xor_sync(0xffffffffu, mna, 2));
            mnb = fmaxf(mnb, __shfl_xor_sync(0xffffffffu, mnb, 1));
            mnb = fmaxf(mnb, __shfl_xor_sync(0xffffffffu, mnb, 2));
            const float refa = (mna == -INFINITY) ? 0.f : mna, refb = (mnb == -INFINITY) ? 0.f : mnb;   // nothing visible yet: all factors 0
            const float ca = ex2(ma - refa), cb = ex2(mb - refb);
            ma = mna; mb = mnb;
            float sa = 0.f, sb = 0.f;
            uint32_t pa[4];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const float e0 = ex2(sc[j][0] - refa), e1 = ex2(sc[j][1] - refa);
                const float e2 = ex2(sc[j][2] - refb), e3 = ex2(sc[j][3] - refb);
                sa += e0 + e1; sb += e2 + e3;
                pa[2 * j] = pack_bf16(e0, e1);       // row a, k = 8 j + 2 tq, + 1
                pa[2 * j + 1] = pack_bf16(e2, e3);   // row b
            }
            la = fmaf(la, ca, sa); lb = fmaf(lb, cb, sb);
            if (__any_sync(0xffffffffu, (ca != 1.f) | (cb != 1.f))) {   // a row's maximum moved (rare after the first groups)
#pragma unroll
                for (int n = 0; n < 8; ++n) { o[n][0] *= ca; o[n][1] *= ca; o[n][2] *= cb; o[n][3] *= cb; }
            }
            // O += P V: n-tile n, column gq of the B fragment = dim 8 gq + n; k pairs (2 tq, 2 tq + 1) and (2 tq + 8, 2 tq + 9)
            const uint32_t v0[4] = {vv[0].x, vv[0].y, vv[0].z, vv[0].w}, v1[4] = {vv[1].x, vv[1].y, vv[1].z, vv[1].w};
            const uint32_t v2[4] = {vv[2].x, vv[2].y, vv[2].z, vv[2].w}, v3[4] = {vv[3].x, vv[3].y, vv[3].z, vv[3].w};
#pragma unroll
            for (int n = 0; n < 8; ++n) {
                const uint32_t sel = (n & 1) ? 0x7632u : 0x5410u;
                mma16816(o[n], pa, prmt(v0[n >> 1], v1[n >> 1], sel), prmt(v2[n >> 1], v3[n >> 1], sel));
            }
            if (more) load_v(gb, pb + 16);
        }
        la += __shfl_xor_sync(0xffffffffu, la, 1); la += __shfl_xor_sync(0xffffffffu, la, 2);
        lb += __shfl_xor_sync(0xffffffffu, lb, 1); lb += __shfl_xor_sync(0xffffffffu, lb, 2);
        // this lane holds, for rows a and b, the dims 16 tq + n (o[n][0], o[n][2]) and 16 tq + 8 + n (o[n][1], o[n][3])
        bool need_count = false;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const bool valid = h ? vb : va;
            const int r = h ? rb : ra, i = h ? ib : ia, Lr = h ? Lb : La;
            if (!valid || Lr <= p0) continue;            // padding row, or a row that ends before this split starts
            const int row = b0 + i, hq = kvh * G + (r - i * G);
            const float lsum = h ? lb : la, mrow = h ? mb : ma;
            if (sp.count(Lr) == 1) {
                float x0[8], x1[8];
#pragma unroll
                for (int n = 0; n < 8; ++n) { x0[n] = o[n][2 * h] / lsum; x1[n] = o[n][2 * h + 1] / lsum; }
                uint16_t* dst = M.attn + (size_t)row * Hq * kHeadDim + hq * kHeadDim + 16 * tq;
                *reinterpret_cast<uint4*>(dst) = pack8(x0);
                *reinterpret_cast<uint4*>(dst + 8) = pack8(x1);
            } else {
                need_count = true;
                float* dst = M.partial + (((size_t)row * Hq + hq) * kMaxSplits + s) * kPartialStride;
                if (tq == 0) { dst[0] = mrow; dst[1] = lsum; }
#pragma unroll
                for (int n = 0; n < 8; n += 2) {
                    *reinterpret_cast<float2*>(dst + 2 + 16 * tq + n) = make_float2(o[n][2 * h], o[n + 1][2 * h]);
                    *reinterpret_cast<float2*>(dst + 2 + 16 * tq + 8 + n) = make_float2(o[n][2 * h + 1], o[n + 1][2 * h + 1]);
                }
            }
        }
        if (!__any_sync(0xffffffffu, need_count)) continue;
        __threadfence();
        __syncwarp();
        // one arrival per (row, kv head); the last split of a row combines all of its splits in split order
        int ns_row = 0;
        uint32_t old = 0;
        if (c.lane < nq) {
            const int Lr = min(L0 + c.lane, cap);
            ns_row = sp.count(Lr);
            if (ns_row > 1 && Lr > p0) old = atomicAdd(M.split_count + (size_t)(b0 + c.lane) * Hkv + kvh, 1u);
            else ns_row = 0;
        }
        uint32_t last = __ballot_sync(0xffffffffu, ns_row > 1 && old == (uint32_t)(ns_row - 1));
        if (!last) continue;
        __threadfence();
        while (last) {
            const int i = __ffs(last) - 1;
            last &= last - 1;
            const int row = b0 + i, ns = __shfl_sync(0xffffffffu, ns_row, i);
            for (int g = 0; g < G; ++g) {  // lane j holds split j's (m, l); outputs: lane owns dims 2*lane, 2*lane+1
                const int hq = kvh * G + g;
                const float* base = M.partial + ((size_t)row * Hq + hq) * kMaxSplits * kPartialStride;
                const float m_l = c.lane < ns ? ldcg_f32(base + c.lane * kPartialStride) : -INFINITY;
                const float l_l = c.lane < ns ? ldcg_f32(base + c.lane * kPartialStride + 1) : 0.f;
                const float Mg = warp_max(m_l);
                const float sc_l = (m_l == -INFINITY) ? 0.f : ex2(m_l - Mg);
                float Lsum = 0.f, O0 = 0.f, O1 = 0.f;
                for (int si = 0; si < ns; si += 4) {
                    float2 ov[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        ov[u] = si + u < ns ? __ldcg(reinterpret_cast<const float2*>(base + (si + u) * kPartialStride + 2 + 2 * c.lane))
                                            : make_float2(0.f, 0.f);
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        const float scu = __shfl_sync(0xffffffffu, sc_l, (si + u) & 31);
                        const float ll = __shfl_sync(0xffffffffu, l_l, (si + u) & 31);
                        if (si + u < ns) {
                            Lsum = fmaf(ll, scu, Lsum);
                            O0 = fmaf(ov[u].x, scu, O0);
                            O1 = fmaf(ov[u].y, scu, O1);
                        }
                    }
                }
                *reinterpret_cast<uint32_t*>(M.attn + (size_t)row * Hq * kHeadDim + hq * kHeadDim + 2 * c.lane) = pack_bf16(O0 / Lsum, O1 / Lsum);
            }
            if (c.lane == 0) M.split_count[(size_t)row * Hkv + kvh] = 0u;
        }
    }
}

// One weight phase on the tensor cores.  `target` is the grid barrier's running count: most phases start with a
// distributed pre-step (tc_norm_rows, or the depth attention before a fast wo) followed by an extra grid barrier.
__device__ void phase_gemm_tc(const DevModel& M, const CallArgs& A, const Ctx& c, const Phase& ph, umma::Bars* bars,
                              umma::Pipe& pipe, uint32_t& target, bool first_in_launch, bool next_in_launch) {
    const bool fast = ph.fast != 0;
    const int kind = ph.kind;
    const int D = fast ? M.fdim : M.dim, F = fast ? M.finter : M.inter;
    const int Hq = fast ? M.fn_head : M.n_head, Hkv = fast ? M.fn_kv : M.n_kv;
    const DevLayer& L = fast ? M.fast_layers[ph.layer] : M.layers[ph.layer];
    const int q_rows = Hq * kHeadDim, k_end = (Hq + Hkv) * kHeadDim;
    const int n_head_rows = fast ? M.codebook_size : M.vocab;
    const int K = (kind == PH_W2) ? F : D;
    const int n_out = kind == PH_QKV ? (Hq + 2 * Hkv) * kHeadDim : kind == PH_W13 ? F : kind == PH_HEAD ? n_head_rows : D;
    const uint16_t* table = fast ? M.fast_rope : M.rope;
    uint16_t* stream = fast ? M.xf : M.x;
    unsigned char* ring = reinterpret_cast<unsigned char*>(((uintptr_t)c.xs + 1023) & ~(uintptr_t)1023);
    int* pos = reinterpret_cast<int*>(ring + umma::kRingBytes);
    // sub-phase timers of CTA 0 (tools/phase_profile.py): pre-step + barrier | tile setup | ring + MMA | epilogue
    const bool prof = (M.prof != nullptr) && c.cta == 0 && c.tid == 0;
    unsigned long long* seg = M.prof + 2 * kMaxProg + (size_t)(kind + (fast ? 8 : 0)) * 4;
    unsigned long long ts = 0;
    if (prof) ts = globaltimer_ns();

    // ---- distributed pre-step ----
    // (a normed phase that follows a wo / w2 inside one launch finds M.xn written by that phase's post-step)
    // (and the first QKV of a depth step finds its input written by the SAMPLE phase before it: phase_sample, tc_feed)
    const bool fed_by_post = !first_in_launch &&
                             (kind == PH_W13 || kind == PH_HEAD || (kind == PH_QKV && ph.layer > 0) ||
                              (kind == PH_QKV && fast && ph.layer == 0 && !A.fast_from_xf));
    if (tc_has_prestep(ph) && !fed_by_post) {
        if (kind == PH_WO) {
            tc_fast_attention(M, A, c, ph.layer, ph.depth_pos);
        } else {
            int src_kind = 3;
            const uint16_t* base = kind == PH_W13 ? M.h : stream;
            uint16_t* spill = nullptr;
            if (kind == PH_QKV && ph.layer == 0) {
                if (!fast) { src_kind = 0; spill = M.x; }
                else if (!A.fast_from_xf) { src_kind = ph.depth_pos == 0 ? 1 : 2; spill = M.xf; }
            }
            const uint16_t* norm_w = kind == PH_QKV ? L.attention_norm : kind == PH_W13 ? L.ffn_norm : (fast ? M.fast_norm : M.norm);
            tc_norm_rows(M, A, c, ph, src_kind, base, spill, norm_w, D);
        }
        fence_proxy_async_all();
        grid_arrive(M.barrier, target, (uint32_t)c.n_ctas);
        grid_wait(M.barrier, target);
        if (c.tid == umma::kTmaProducerA || c.tid == umma::kTmaProducerB) fence_proxy_async_all();   // the threads that issue TMA loads
    }
    if (prof) { const unsigned long long t = globaltimer_ns(); seg[0] += t - ts; ts = t; }

    // ---- operands: activation tile and weight rows through TMA ----
    const unsigned char* tm = M.tmaps;
    const int box_idx = A.batch <= 32 ? 2 : A.batch <= 64 ? 1 : 0;   // activation box of 32 / 64 / 128 rows
    const int a_rows = kTcRows >> box_idx;
    const void* tm_a = tm + (size_t)kTensorMapBytes * (box_idx * TM_ACT_MAPS +
                                                       (kind == PH_WO ? (fast ? TM_ATTN_F : TM_ATTN_S)
                                                        : kind == PH_W2 ? (fast ? TM_ACT_F : TM_ACT_S) : (fast ? TM_XN_F : TM_XN_S)));
    const int which = kind == PH_QKV ? 0 : kind == PH_WO ? 1 : kind == PH_W13 ? 2 : 4;
    const int w_index0 = kind == PH_HEAD ? (fast ? 1 : 0) : tm_weight_index(M.n_layer, fast ? 1 : 0, ph.layer, which);
    const int w_index1 = kind == PH_W13 ? tm_weight_index(M.n_layer, fast ? 1 : 0, ph.layer, 3) : -1;
    const int w_row_base = (kind == PH_HEAD && fast && M.depthwise_output) ? ph.depth_pos * n_head_rows : 0;

    // the residual phases (wo, w2) also cut K: their fp32 partials meet in the post-step
    const bool has_post = kind == PH_WO || kind == PH_W2;
    const int n_split = !has_post ? 1 : (K % (4 * umma::kBK) == 0) ? 4 : (K % (2 * umma::kBK) == 0) ? 2 : 1;
    const int k_len = K / n_split;
    const int m_tiles = (A.batch + kTcRows - 1) / kTcRows;
    const int blk_cap = kind == PH_W13 ? umma::kMaxN / 2 : umma::kMaxN;
    int blk = 16;
    while (blk < blk_cap && m_tiles * ((n_out + blk - 1) / blk) * n_split > c.n_ctas) blk += 16;
    const int n_blocks = (n_out + blk - 1) / blk;
    const int n_units = m_tiles * n_blocks * n_split;

    for (int u = c.cta; u < n_units; u += c.n_ctas) {
#if SMOL_TC_UNIT_ORDER
        const int mt = u % m_tiles, un = u / m_tiles;       // the row tiles that share a weight block on neighbouring CTAs
        const int ks = un % n_split, nb = un / n_split;
#else
        const int ks = u % n_split, un = u / n_split;
        const int mt = un / n_blocks, nb = un - mt * n_blocks;
#endif
        const int m0 = mt * kTcRows, n0 = nb * blk;
        if (kind == PH_QKV && c.tid < kTcRows) {
            const int bg = min(m0 + c.tid, A.batch - 1);
            pos[c.tid] = fast ? ph.depth_pos : ldcg_i32(A.b.seq_len + row_seq(A, bg)) + row_off(A, bg);
        }
        __syncthreads();
        if (prof) { const unsigned long long t = globaltimer_ns(); seg[1] += t - ts; ts = t; }
        umma::BSrc b0, b1;
        b0.tm = tm + (size_t)kTensorMapBytes * tm_weight_slot(w_index0, blk); b0.row0 = w_row_base + n0; b0.n = blk; b0.box = blk;
        b1.tm = w_index1 >= 0 ? tm + (size_t)kTensorMapBytes * tm_weight_slot(w_index1, blk) : nullptr;
        b1.row0 = n0; b1.n = w_index1 >= 0 ? blk : 0; b1.box = blk;
        // slow weights are read once per frame (evict first), the depth transformer's by every depth step (keep in L2):
        // measured DRAM reads 937 -> 891 MB per frame at bs=256, time unchanged (gpurun_out/l2hint_dram.csv)
        umma::tile_mma_tma<kThreads>(ring, bars, pipe, k_len, tm_a, m0, b0, b1, ks * k_len, a_rows,
                                            fast ? SMOL_TC_FAST_POLICY : SMOL_TC_SLOW_POLICY);
        if (prof) { const unsigned long long t = globaltimer_ns(); seg[2] += t - ts; ts = t; }

        if (kind == PH_W13) {
            umma::tile_epilogue_paired(bars, blk, [&](int row, int c0, const float (&ga)[8], const float (&up)[8]) {
                const int bg = m0 + row, u0 = n0 + c0;
                if (bg >= A.batch || u0 >= n_out) return;
                float o[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const float a = bf16_round(ga[e]), g = bf16_round(up[e]);
                    // F.silu in fp32, bf16 out: a is a bf16 value, so the exactly rounded result is a table look-up (the
                    // exact exp / division made this epilogue issue-bound; a fast-math form moved 0.02 % of the results)
                    const float sg = __uint_as_float((uint32_t)__ldg(M.silu_lut + (__float_as_uint(a) >> 16)) << 16);
                    o[e] = __fmul_rn(sg, g);
                }
                *reinterpret_cast<uint4*>(M.act + (size_t)bg * F + u0) = pack8(o);
            }, b0.n + b1.n);
        } else {
            umma::tile_epilogue(bars, blk, [&](int row, int c0, const float (&acc)[8]) {
                const int bg = m0 + row, u0 = n0 + c0;
                if (bg >= A.batch || u0 >= n_out) return;
                if (kind == PH_HEAD) {
                    float* out = fast ? M.depth_logits + ((size_t)bg * M.depth + ph.depth_pos) * n_head_rows
                                      : M.token_logits + (size_t)bg * n_head_rows;
                    *reinterpret_cast<float4*>(out + u0) = make_float4(bf16_round(acc[0]), bf16_round(acc[1]), bf16_round(acc[2]), bf16_round(acc[3]));
                    *reinterpret_cast<float4*>(out + u0 + 4) = make_float4(bf16_round(acc[4]), bf16_round(acc[5]), bf16_round(acc[6]), bf16_round(acc[7]));
                    return;
                }
                if (kind != PH_QKV) {  // wo, w2: this K slice's partial sums (the post-step adds slices and residual)
                    float* pp = M.kpart + ((size_t)ks * M.ws_rows + bg) * D + u0;
                    *reinterpret_cast<float4*>(pp) = make_float4(acc[0], acc[1], acc[2], acc[3]);
                    *reinterpret_cast<float4*>(pp + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
                    return;
                }
                float v[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) v[e] = bf16_round(acc[e]);
                const int p = pos[row];
                const int tp = fast ? p : min(p, M.max_seq_len - 1);  // never past the RoPE table (host checks bound p)
                if (u0 < k_end) {  // q and k rows: interleaved-pair RoPE with the bf16 table (P:616-640)
#pragma unroll
                    for (int e = 0; e < 8; e += 2) {
                        const int j = ((u0 + e) & (kHeadDim - 1)) >> 1;
                        const uint32_t cs = __ldg(reinterpret_cast<const uint32_t*>(table + ((size_t)tp * (kHeadDim / 2) + j) * 2));
                        const float co = bf_lo(cs), si = bf_hi(cs);
                        const float r0 = bf16_round(__fsub_rn(__fmul_rn(v[e], co), __fmul_rn(v[e + 1], si)));
                        const float r1 = bf16_round(__fadd_rn(__fmul_rn(v[e + 1], co), __fmul_rn(v[e], si)));
                        v[e] = r0; v[e + 1] = r1;
                    }
                }
                const uint4 packed = pack8(v);
                if (u0 < q_rows) {
                    *reinterpret_cast<uint4*>(M.q + (size_t)bg * q_rows + u0) = packed;
                    return;
                }
                const int is_v = u0 >= k_end ? 1 : 0;
                const int n1 = u0 - (is_v ? k_end : q_rows);
                const int kvh = n1 / kHeadDim, d = n1 & (kHeadDim - 1);
                if (fast) {
                    uint16_t* dst = M.fkv + (((size_t)(bg * M.n_flayer + ph.layer) * 2 + is_v) * M.depth + ph.depth_pos) * (Hkv * kHeadDim)
                                    + kvh * kHeadDim + d;
                    *reinterpret_cast<uint4*>(dst) = packed;
                } else {
                    if (!seq_active(M, A, c, bg)) return;
                    const int ps = M.page_size;
                    if (p >= A.b.max_pages * ps) return;
                    const int page = ldcg_i32(A.b.block_table + (size_t)row_seq(A, bg) * A.b.max_pages + p / ps);
                    uint16_t* dst = M.kv_pool + ((((size_t)page * M.n_layer + ph.layer) * 2 + is_v) * Hkv + kvh) * ((size_t)ps * kHeadDim)
                                    + (size_t)(p % ps) * kHeadDim + d;
                    *reinterpret_cast<uint4*>(dst) = packed;
                }
            }, b0.n + b1.n);
        }
        if (prof) { const unsigned long long t = globaltimer_ns(); seg[3] += t - ts; ts = t; }
    }

    // ---- post-step of the residual phases: wo: h = stream + wo(attn) (P:499); w2: stream = h + w2(act) (P:500) ----
    if (has_post) {
        grid_arrive(M.barrier, target, (uint32_t)c.n_ctas);
        grid_wait(M.barrier, target);
        const uint16_t* next_norm = nullptr;
        if (next_in_launch) {
            const int n_net = fast ? M.n_flayer : M.n_layer;
            if (kind == PH_WO) next_norm = L.ffn_norm;
            else if (ph.layer + 1 < n_net) next_norm = (fast ? M.fast_layers[ph.layer + 1] : M.layers[ph.layer + 1]).attention_norm;
            else next_norm = fast ? M.fast_norm : M.norm;
        }
        tc_residual_finish(M, A, c, kind == PH_WO ? stream : M.h, kind == PH_WO ? M.h : stream, D, n_split, next_norm);
        if (prof) { const unsigned long long t = globaltimer_ns(); seg[0] += t - ts; ts = t; }
    }
}

}  // namespace smol
