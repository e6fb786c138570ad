// The DualAR decode step as a DATA-FLOW persistent kernel (sm_100a) -- the latency path (batches 1..8).
//
// A frame at batch 1 is a chain of ~200 dependent matrix-vector products; what bounds it is the hand-off between them
// and the dependent instruction chain inside a CTA, not bytes.  No grid barrier anywhere:
// every phase publishes 8-byte words {payload | epoch}, consumers poll exactly the words they need, weights stream
// through a shared-memory ring fed by a TMA producer warp that never waits for activations.  (The round-1 kernel used the
// same protocol with CUDA-core GEMVs, one warp per two rows; it is in the git history, ll_kernel.cu.)
//
//  * GEMV on the tensor cores.  mma.sync m16n8k16 (bf16 in, fp32 accumulate): the 16 rows of a tile are weight rows,
//    the 8 columns all carry the one activation vector.  Weights are packed once at bind time (smol_pack_kernel) as
//    ready-made A fragments, [tile of 16 rows][K / 32][MMA step 2][lane 32][16 bytes] (gated MLP: a tile = 8 rows of w1
//    over the same 8 rows of w3), so that a warp's A fragment is ONE conflict-free 16-byte shared-memory load per lane and
//    a CTA's tiles of a phase are one contiguous run of 24 KB ring stages (one bulk copy each).  The 7 consumer warps
//    split K; a pass carries up to 4 tiles through one K sweep (the B fragments -- the activation -- are loaded once),
//    partial sums meet in shared memory and are added in warp order by a warp that rotates from pass to pass.
//    A 16 x 768 tile costs a warp ~15 instructions per 96 elements of K instead of ~200 FMA/unpack instructions per
//    row pair on the CUDA cores (the round-1 kernel).
//  * Everybody polls, nobody computes alone: all 224 consumer threads poll the input vector (16-byte loads, two words
//    each), every thread normalises four elements in place (RMSNorm: per-warp sums of squares, added in warp order),
//    so staging + norm are a few instructions per thread instead of one warp's 1 200-cycle chain.
//  * A precise hold-off (clock-based) before the first poll of a phase: a poll issued before the producers' stores can
//    have reached L2 only adds L2 traffic and one wasted round trip.
//  * Slow attention with the reference's softmax semantics (torch CPU SDPA, which the oracle runs): score units
//    (kv head x 64 positions) publish q.k scores, PV units (query head x 8 head dims) poll all scores of their head,
//    take the running maximum over blocks of 512 positions, ROUND P TO bf16 before P.V, keep the denominator in fp32
//    and rescale block by block -- two hand-offs, as many as the split-KV/combiner form they replace, but the
//    probabilities are rounded at the same point and relative to the same maximum as the reference's.
//  * One TEAM of CTAs per sequence: grid = batch x team, every team has its own word regions and runs the same program
//    on its own sequence (batches of 2..8 are independent latency chains side by side, not a wider tile).
//
// Reference map (P = modeling/model/rq_transformer.py, M = mlx lm/rq_transformer.py, G = mlx lm/generate.py):
// embed P:205-221; RMSNorm P:601-613; QKV/RoPE/attention P:535-570,616-640; FeedForward P:573-582; block P:492-501;
// slow step P:223-260 / M:173-192; depth loop P:409-448, M:194-220, G:110-141; sampling G:88-99,118-132; frame
// assembly + stop rule G:143-171.

#include <algorithm>

#include "common.cuh"
#include "dev_model.h"

#define LL2_STR2(x) #x
#define LL2_STR(x) LL2_STR2(x)
#define SMOL_BLOCK_SYNC() asm volatile("bar.sync 1, " LL2_STR(LL2_WARPS) " * 32;" ::: "memory")  // the consumer warps

#include "sampler.cuh"

namespace smol {
namespace ll2 {

constexpr int kNW = kLL2Warps;
constexpr int kCons = kNW * 32;
constexpr int kMaxSlots = 8;
constexpr int kDescWords = 16;
constexpr int kGather = (768 + kCons - 1) / kCons;   // 16-byte polls (2 words) per thread and vector: covers K = 3072 (1536 words)
constexpr int kNormPer = (192 + kCons - 1) / kCons;  // 4-element chunks a thread normalises (K <= 768)
constexpr int kSampPer = (2560 + kCons - 1) / kCons; // logits per thread in the sampler
constexpr int kMaxBlocks = 16;    // softmax blocks of 512 positions a PV unit carries (contexts up to 8192)
constexpr int kMaxSeg = kMaxBlocks * 8;  // 64-position segments of a context
constexpr int kBtabCache = 256;

#define LL2_SPIN_GUARD(n) do { if (++(n) > (1u << 22)) __trap(); } while (0)

// ---- small helpers -------------------------------------------------------------------------------
__device__ __forceinline__ void csync() { SMOL_BLOCK_SYNC(); }
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ int ldcg_i32(const void* p) { return __ldcg(reinterpret_cast<const int*>(p)); }
__device__ __forceinline__ uint4 ldcg_v4(const void* p) { return __ldcg(reinterpret_cast<const uint4*>(p)); }
__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
    f[0] = bf_lo(v.x); f[1] = bf_hi(v.x); f[2] = bf_lo(v.y); f[3] = bf_hi(v.y);
    f[4] = bf_lo(v.z); f[5] = bf_hi(v.z); f[6] = bf_lo(v.w); f[7] = bf_hi(v.w);
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
    uint4 v;
    v.x = pack_bf16(f[0], f[1]); v.y = pack_bf16(f[2], f[3]); v.z = pack_bf16(f[4], f[5]); v.w = pack_bf16(f[6], f[7]);
    return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ long long clock_now() {
    long long c;
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(c) :: "memory");
    return c;
}
__device__ __forceinline__ uint32_t clock32_now() {
    uint32_t c;
    asm volatile("mov.u32 %0, %%clock;" : "=r"(c) :: "memory");
    return c;
}
__device__ __forceinline__ uint4 lds_v4(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ float lds_f32(uint32_t a) { return __uint_as_float(lds_u32(a)); }
__device__ __forceinline__ void sts_v4(uint32_t a, const uint4& v) {
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts_v2(uint32_t a, uint32_t x, uint32_t y) {
    asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(a), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_f32(uint32_t a, float v) { sts_u32(a, __float_as_uint(v)); }

// ---- LL words: {payload, epoch}, one aligned 8-byte access -----------------------------------------------------
__device__ __forceinline__ uint4 ld_relaxed_v4(const void* p) {
    uint4 v;
    asm volatile("ld.relaxed.gpu.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint2 ld_relaxed_v2(const void* p) {
    uint2 v;
    asm volatile("ld.relaxed.gpu.global.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_v2(void* p, uint32_t a, uint32_t b) {
    asm volatile("st.relaxed.gpu.global.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(a), "r"(b) : "memory");
}
// read-only loads the compiler may not move (issued early so that their latency hides behind a wait)
__device__ __forceinline__ uint2 ldnc_v2(const void* p) {
    uint2 v;
    asm volatile("ld.global.nc.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t ldnc_u32(const void* p) {
    uint32_t v;
    asm volatile("ld.global.nc.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t ll_get(const unsigned long long* w, uint32_t epoch) {
    uint2 v = ld_relaxed_v2(w);
    uint32_t spins = 0;
    while (v.y != epoch) { LL2_SPIN_GUARD(spins); v = ld_relaxed_v2(w); }
    return v.x;
}

// ---- mbarrier + TMA bulk copy ----------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_n(uint32_t bar, uint32_t n) {
    asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(n) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok, spins = 0;
    for (;;) {
        asm volatile(
            "{\n\t"
            ".reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t"
            "}\n" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
        if (ok) break;
        LL2_SPIN_GUARD(spins);
    }
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar, uint64_t policy) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(policy) : "memory");
}

// ---- thread-block cluster (the fused gated MLP) ---------------------------------------------------------------
__device__ __forceinline__ uint32_t mapa(uint32_t a, uint32_t rank) {   // the same shared-memory offset in CTA `rank`
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(rank));
    return r;
}
// 16 bytes into a cluster peer's shared memory; the peer's mbarrier `bar` counts them on arrival
__device__ __forceinline__ void st_async_v4(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w, uint32_t bar) {
    asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1,%2,%3,%4}, [%5];"
                 ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w), "r"(bar) : "memory");
}
// 8 bytes, likewise
__device__ __forceinline__ void st_async_v2(uint32_t a, uint32_t x, uint32_t y, uint32_t bar) {
    asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.v2.b32 [%0], {%1,%2}, [%3];"
                 ::"r"(a), "r"(x), "r"(y), "r"(bar) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---- per-CTA shared state ------------------------------------------------------------------------
__shared__ __align__(8) uint64_t s_full[kMaxSlots];
__shared__ __align__(8) uint64_t s_empty[kMaxSlots];
__shared__ __align__(8) uint64_t s_actbar;   // fused MLP: the slice's act values have arrived from the cluster
__shared__ __align__(8) uint64_t s_psumbar;  // fused MLP, split staging: the whole output vector has arrived from the cluster
__shared__ SampleScratch s_sc;
__shared__ float s_ssq[kNW];            // per-warp partial sums of squares (RMSNorm)
__shared__ uint32_t s_best;             // HEAD phases: the CTA's best (logit, index) candidate
__shared__ int s_pos, s_step, s_fin;    // cached positions (seq_len) / frames emitted / stop flag, tracked by every CTA
__shared__ SmolRowSampling s_rs;        // the team's sampling parameters (constant during a launch): every CTA reads the same
__shared__ int s_tok[kMaxRows];         // pending input column
__shared__ int s_nw[kMaxRows];          // ids chosen in the current frame
__shared__ uint32_t s_epoch0;           // phases executed by earlier launches
__shared__ int s_btab[kBtabCache];      // the sequence's block table (constant during a launch)
__shared__ float s_bmax[kMaxSeg];       // PV units: maxima of the 64-position segments

using SmemPlan = LL2SmemPlan;

// Geometry of one CTA inside its team.
struct Team {
    int team, cta, n;  // sequence / team index, CTA index inside the team, CTAs per team
};

// ---- descriptors -----------------------------------------------------------------------------------
//   word  0-1  src      LL source region (this team, this CTA's replica) | fast_embeddings row base
//         2-3  normw    RMSNorm weight
//         4-5  out      LL region this phase publishes to (this team, replica 0)
//         6-7  aux      QKV: RoPE table | HEAD: fp32 logits dump
//         8-9  wptr     packed weights: first 8-row group of this CTA
//        10    e_back | src_kind << 8 | nrep << 12 | res_sel << 20 | gather << 21 | psum << 22 (input = a fused MLP's
//              partial sums: 1 every CTA polls all of them, gather_psum; 2 the cluster splits them, gather_psum_split)
//        11    K | n_items << 16
//        12    kind | fast << 4 | layer << 8 | depth_pos << 16
//        13    first item of this CTA
//        14    fused MLP (W13 and W2 phases): lo | hi << 8 | n_units << 16 -- the K-slice [lo, hi) (k-blocks of w2) of this
//              CTA's cluster and the W2 row tiles this CTA carries (i0, i0 + S, ..); 0 = not fused / no work
//              psum == 2 (the phase after a W2 phase): j0 | n_quads << 16 -- the quads of the input vector this CTA stages
//        15    len_out (words per replica of the output region) | n_src_words << 16
//
// Fused gated MLP (batch 1, A.mlp_cluster = S > 0; grid = clusters of S CTAs).  The 7 consumer warps split a w2 tile's
// K = inter into the ranges [kb w / 7, kb (w + 1) / 7), and a w2 row is the sum, in warp order, of one acc / acd MMA chain
// per range.  Cluster c < 7 owns range c: its CTAs compute the act values of the range (the w13 tiles of it, unchanged),
// hand them to each other through DSMEM, and then run warp c's chain of every w2 row tile, one warp per tile, publishing
// the fp32 partial sums with the W2 phase's epoch.  The consumers of the W2 region add the 7 partials in range order and
// the residual (the bf16 roundings of the unfused epilogue): bit for bit the unfused result, with one L2 exchange per
// MLP instead of two.  The W2 phase itself has no tiles and no input: it stays in the program (epochs, descriptors and the
// producer's stream are those of the unfused program) but the consumer warps never visit it.
__device__ __forceinline__ int phase_rows(const DevModel& M, const Phase& ph) {
    const bool fast = ph.fast != 0;
    switch (ph.kind) {
        case PH_QKV: return ((fast ? M.fn_head : M.n_head) + 2 * (fast ? M.fn_kv : M.n_kv)) * kHeadDim;
        case PH_WO: case PH_W2: return fast ? M.fdim : M.dim;
        case PH_W13: return fast ? M.finter : M.inter;
        case PH_HEAD: return fast ? M.codebook_size : M.vocab;
        default: return 0;
    }
}
__device__ __forceinline__ int phase_k(const DevModel& M, const Phase& ph) {
    const bool fast = ph.fast != 0;
    if (ph.kind == PH_W2) return fast ? M.finter : M.inter;
    return fast ? M.fdim : M.dim;
}
__device__ __forceinline__ const uint16_t* phase_weights(const DevModel& M, const Phase& ph) {
    const bool fast = ph.fast != 0;
    const DevLayer& L = fast ? M.fast_layers[ph.layer] : M.layers[ph.layer];
    switch (ph.kind) {
        case PH_QKV: return L.pk_wqkv;
        case PH_WO: return L.pk_wo;
        case PH_W13: return L.pk_w13;
        case PH_W2: return L.pk_w2;
        case PH_HEAD:
            return fast ? M.pk_fast_output + (M.depthwise_output ? (size_t)ph.depth_pos * M.codebook_size * M.fdim : 0) : M.pk_head;
        default: return nullptr;
    }
}
__device__ __forceinline__ int sample_phase_index(const DevModel& M, int r) {  // program index of row r's SAMPLE phase
    const int n_slow = 5 * M.n_layer;
    if (r == 0) return n_slow + 1;
    return n_slow + 2 + (r - 1) * (4 * M.n_flayer + 2) + 4 * M.n_flayer + 1;
}
__device__ __forceinline__ unsigned long long* ll_region(const DevModel& M, int team, int p, int rep) {
    return M.ll + M.ll_off[p] + (size_t)(team * kLLRep + rep) * M.ll_len[p];
}

// Fused MLP: the W2 phase p's partial-sum words, replica rep (batch 1 only: one sequence)
__device__ __forceinline__ unsigned long long* psum_region(const DevModel& M, int p, int rep) {
    const Phase ph = unpack_phase(M.prog[p]);
    const int w2 = ph.fast ? M.n_layer + ph.depth_pos * M.n_flayer + ph.layer : ph.layer;
    return M.ll2_psum + ((size_t)w2 * kLLRep + rep) * kNW * M.dim;
}

__device__ __forceinline__ void build_desc(const DevModel& M, const Team& tm, int S, int split, int p, uint32_t dsc) {
    const int rep = tm.cta % kLLRep;
    const Phase ph = unpack_phase(M.prog[p]);
    const bool fast = ph.fast != 0;
    const int kind = ph.kind;
    const int n_slow = 5 * M.n_layer;
    uint32_t w[kDescWords];
#pragma unroll
    for (int i = 0; i < kDescWords; ++i) w[i] = 0u;
    int src_kind = 3, nrep = kLLRep, n_items = 0, i0 = 0, K = 0, gather = 0, n_src = 0, e_back = 1, psum = 0;
    if (kind != PH_ATTN && kind != PH_SAMPLE) {
        K = phase_k(M, ph);
        // work item = one MMA tile of 16 row slots: 16 rows of the matrix, or 8 rows of w1 over the same 8 rows of w3
        const int items = phase_rows(M, ph) / (kind == PH_W13 ? 8 : 16);
        i0 = (items * tm.cta) / tm.n;
        n_items = (items * (tm.cta + 1)) / tm.n - i0;
        if (S > 0 && (kind == PH_W13 || kind == PH_W2)) {
            const int slice = tm.cta / S, r = tm.cta - slice * S;
            const int kb2 = (fast ? M.finter : M.inter) / 32, rt = (fast ? M.fdim : M.dim) / 16;
            const int lo = slice < kNW ? (kb2 * slice) / kNW : 0, hi = slice < kNW ? (kb2 * (slice + 1)) / kNW : 0;
            const int nu = slice < kNW ? (rt - r + S - 1) / S : 0;
            if (kind == PH_W13) {   // the w13 tiles of the slice's act values (8 per tile)
                i0 = 4 * lo + (4 * (hi - lo) * r) / S;
                n_items = 4 * lo + (4 * (hi - lo) * (r + 1)) / S - i0;
            } else {
                i0 = r;
                n_items = 0;
            }
            w[14] = nu > 0 ? (uint32_t)lo | ((uint32_t)hi << 8) | ((uint32_t)nu << 16) : 0u;
        }
        int p_src = p - 1;
        unsigned long long src = 0ull;
        if (kind == PH_QKV && ph.layer == 0) {
            if (!fast) src_kind = 0;
            else if (ph.depth_pos == 0) p_src = n_slow - 1;  // the slow transformer's pre-norm hidden state (P:259, M:191)
            else {
                src_kind = 2;  // embedding of the previous depth code (G:136-140)
                const int off = M.depthwise_wte ? (M.dup0 ? ph.depth_pos - 1 : ph.depth_pos) * M.codebook_size : 0;
                src = (unsigned long long)(M.fast_embeddings + (size_t)off * M.fdim);
            }
        }
        if (src_kind == 3) {
            src = (unsigned long long)ll_region(M, tm.team, p_src, rep);
            n_src = (kind == PH_WO && fast) ? (M.fn_head + 2 * M.fn_kv) * kHeadDim / 2 : K / 2;
            if (S > 0 && unpack_phase(M.prog[p_src]).kind == PH_W2) {   // 7 fp32 partials per element
                psum = 1;
                n_src = kNW * K;
                src = (unsigned long long)psum_region(M, p_src, rep);
                // Split staging (gather_psum_split) where its early DSMEM stores are safe: in the phase right after the
                // W2 phase (not the depth-0 QKV, which follows HEAD + SAMPLE) and in a slice cluster (not the idle one)
                const int slice = tm.cta / S, r = tm.cta - slice * S, q = K / 4;
                if (split && p_src == p - 1 && slice < kNW && 2 * ((q + S - 1) / S) <= kCons) {
                    psum = 2;
                    const int j0 = (q * r) / S, j1 = (q * (r + 1)) / S;
                    w[14] = (uint32_t)j0 | ((uint32_t)(j1 - j0) << 16);
                }
            }
        }
        e_back = p - p_src;
        const DevLayer& L = fast ? M.fast_layers[ph.layer] : M.layers[ph.layer];
        const uint16_t* nw = kind == PH_QKV ? L.attention_norm : kind == PH_W13 ? L.ffn_norm : kind == PH_HEAD ? (fast ? M.fast_norm : M.norm) : nullptr;
        const unsigned long long out = (unsigned long long)(S > 0 && kind == PH_W2 ? psum_region(M, p, 0) : ll_region(M, tm.team, p, 0));
        unsigned long long aux = 0ull;
        if (kind == PH_QKV) aux = (unsigned long long)(fast ? M.fast_rope + (size_t)ph.depth_pos * kHeadDim : M.rope);
        if (kind == PH_HEAD) {
            aux = (unsigned long long)(fast ? M.depth_logits + ((size_t)tm.team * M.depth + ph.depth_pos) * M.codebook_size
                                            : M.token_logits + (size_t)tm.team * M.vocab);
            nrep = 1;  // logits words are read by the team's sampler CTA only (greedy rows use the candidate words)
        }
        const unsigned long long wp = (unsigned long long)(phase_weights(M, ph) + (size_t)i0 * 16 * K);   // 16 K elements per tile
        // normed phases stage the residual stream for everybody (the wo / w2 epilogues need their rows of it); a split
        // staging needs every CTA of the cluster, tiles or not
        gather = (kind == PH_QKV || kind == PH_W13 || psum == 2) ? 1 : (n_items > 0 ? 1 : 0);
        w[0] = (uint32_t)src; w[1] = (uint32_t)(src >> 32);
        w[2] = (uint32_t)(unsigned long long)nw; w[3] = (uint32_t)((unsigned long long)nw >> 32);
        w[4] = (uint32_t)out; w[5] = (uint32_t)(out >> 32);
        w[6] = (uint32_t)aux; w[7] = (uint32_t)(aux >> 32);
        w[8] = (uint32_t)wp; w[9] = (uint32_t)(wp >> 32);
    }
    const int res_sel = (kind == PH_QKV || kind == PH_WO) ? 0 : 1;
    w[10] = (uint32_t)e_back | ((uint32_t)src_kind << 8) | ((uint32_t)nrep << 12) | ((uint32_t)res_sel << 20) | ((uint32_t)gather << 21) |
            ((uint32_t)psum << 22);
    w[11] = (uint32_t)K | ((uint32_t)n_items << 16);
    w[12] = (uint32_t)kind | ((uint32_t)(fast ? 1 : 0) << 4) | ((uint32_t)ph.layer << 8) | ((uint32_t)ph.depth_pos << 16);
    w[13] = (uint32_t)i0;
    w[15] = (uint32_t)(S > 0 && kind == PH_W2 ? kNW * M.dim : M.ll_len[p]) | ((uint32_t)n_src << 16);
#pragma unroll
    for (int i = 0; i < kDescWords / 4; ++i) sts_v4(dsc + 16u * i, make_uint4(w[4 * i], w[4 * i + 1], w[4 * i + 2], w[4 * i + 3]));
}
// ring stages of a tile: K in chunks of kLL2ChunkKb k-blocks
__device__ __forceinline__ int phase_chunks(int K) { return (K / 32 + kLL2ChunkKb - 1) / kLL2ChunkKb; }

// ---- TMA producer (one lane of the last warp) -------------------------------------------------------------
__device__ __noinline__ void producer(const CallArgs& A, const SmemPlan& SP, uint32_t sm0) {
    uint64_t pol_stream, pol_keep;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol_stream));
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol_keep));
    const uint32_t full0 = smem_u32(s_full), empty0 = smem_u32(s_empty);
    const uint32_t ring = sm0 + (uint32_t)SP.ring;
    const uint32_t ns = (uint32_t)SP.n_slots;
    uint32_t stage = 0, slot = 0, par = 0;   // stages are produced strictly in order: slot / parity run along
    for (int it = 0; it < A.n_iter; ++it) {
        for (int p = 0; p < A.phase_end; ++p) {
            const uint32_t dsc = sm0 + (uint32_t)SP.desc + (uint32_t)p * (kDescWords * 4u);
            const uint4 d2 = lds_v4(dsc + 32u), d3 = lds_v4(dsc + 48u);
            const int kind = (int)(d3.x & 15u);
            const int n_items = (int)(d2.w >> 16), K = (int)(d2.w & 0xffffu);
            const bool units = kind == PH_W2 && d3.z != 0u;   // fused MLP: the K-slice of each of this CTA's w2 row tiles
            if (kind == PH_ATTN || kind == PH_SAMPLE || (n_items == 0 && !units)) continue;
            const bool fast = (d3.x >> 4) & 1u;
            const unsigned char* wp = reinterpret_cast<const unsigned char*>((unsigned long long)d2.x | ((unsigned long long)d2.y << 32));
            // the slow transformer's weights are read once per frame: evict first; the depth transformer's are re-read
            // by every depth step: keep them in L2
            const uint64_t pol = (fast && kind != PH_HEAD) ? pol_keep : pol_stream;
            const int tiles = n_items, chunks = phase_chunks(K), kb = K / 32;
            const size_t tile_bytes = (size_t)K * 32;
            if (units) {   // one stage per (row tile, slice): k-blocks lo .. hi - 1 of tiles i0, i0 + S, ..
                const int lo = (int)(d3.z & 255u), hi = (int)((d3.z >> 8) & 255u), nu = (int)(d3.z >> 16);
                const uint32_t bytes = (uint32_t)((hi - lo) * 1024);
                for (int u = 0; u < nu; ++u) {
                    if (stage >= ns) mbar_wait(empty0 + 8u * slot, par ^ 1u);
                    const uint32_t bar = full0 + 8u * slot;
                    mbar_expect_tx(bar, bytes);
                    bulk_g2s(ring + slot * (uint32_t)kLL2SlotBytes, wp + (size_t)u * A.mlp_cluster * tile_bytes + (size_t)lo * 1024, bytes, bar, pol);
                    ++stage;
                    if (++slot == ns) { slot = 0u; par ^= 1u; }
                }
                continue;
            }
            for (int t = 0; t < tiles; ++t) {
                for (int kc = 0; kc < chunks; ++kc) {
                    const int kb0 = kc * kLL2ChunkKb, nkb = min(kLL2ChunkKb, kb - kb0);
                    if (stage >= ns) mbar_wait(empty0 + 8u * slot, par ^ 1u);
                    const uint32_t bytes = (uint32_t)(nkb * 1024);
                    const uint32_t bar = full0 + 8u * slot;
                    mbar_expect_tx(bar, bytes);
                    bulk_g2s(ring + slot * (uint32_t)kLL2SlotBytes, wp + (size_t)t * tile_bytes + (size_t)kb0 * 1024, bytes, bar, pol);
                    ++stage;
                    if (++slot == ns) { slot = 0u; par ^= 1u; }
                }
            }
        }
    }
}

// ---- token plumbing --------------------------------------------------------------------------------------
struct Seq {   // this team's slice of the batch state
    int32_t* tokens; int32_t* seq_len; const int32_t* btab; uint8_t* finished; const int32_t* seq_id; int32_t* step; int32_t* out_codes;
    const int32_t* force; int32_t* frame_tokens;
};
__device__ __forceinline__ Seq seq_of(const DevModel& M, const CallArgs& A, int team) {
    Seq s;
    const int R = M.n_rows;
    s.tokens = A.b.tokens + (size_t)team * R;
    s.seq_len = A.b.seq_len + team;
    s.btab = A.b.block_table + (size_t)team * A.b.max_pages;
    s.finished = A.b.finished ? A.b.finished + team : nullptr;
    s.seq_id = A.b.seq_id ? A.b.seq_id + team : nullptr;
    s.step = A.b.step ? A.b.step + team : nullptr;
    s.out_codes = A.b.out_codes ? A.b.out_codes + (size_t)team * A.b.max_frames * R : nullptr;
    s.force = M.force ? M.force + (size_t)team * R : nullptr;
    s.frame_tokens = M.frame_tokens + (size_t)team * R;
    return s;
}
// Greedy rows (temperature 0) and forced ids need no sampler CTA: every CTA works the id out itself.  Greedy or sampled is
// decided per team, from its own sampling parameters.
__device__ __forceinline__ bool row_is_local(const DevModel& M, int r) {
    return M.force != nullptr || (r == 0 ? s_rs.temp : s_rs.fast_temp) == 0.0f;
}
// (logit, index) packed so that unsigned max picks the larger logit and, among equal logits, the smaller index
__device__ __forceinline__ uint32_t cand_pack(float v, int idx) {
    uint32_t b = __float_as_uint(v) >> 16;
    b = (b & 0x8000u) ? (~b & 0xffffu) : (b | 0x8000u);
    return (b << 16) | (uint32_t)(0xffff - idx);
}
__device__ __forceinline__ int cand_index(uint32_t c) { return 0xffff - (int)(c & 0xffffu); }
__device__ __forceinline__ unsigned long long* tok_words(const DevModel& M, const Team& tm, int r) {
    return M.ll2_tok + ((size_t)tm.team * M.n_rows + r) * kLLMaxCtas;
}
__device__ __forceinline__ unsigned long long* cand_words(const DevModel& M, const Team& tm, int r, int rep) {
    return M.ll2_cand + (((size_t)tm.team * M.n_rows + r) * kLLRep + rep) * kLLMaxCtas;
}

// frame boundary: adopt the ids chosen in the previous frame (G:143-166).  e_prev0 = epoch of phase 0 of that frame.
__device__ __noinline__ void frame_boundary(const DevModel& M, const CallArgs& A, const Team tm, uint32_t e_prev0) {
    const int tid = threadIdx.x;
    if (tid < M.n_rows && !row_is_local(M, tid))
        s_nw[tid] = (int)ll_get(tok_words(M, tm, tid) + tm.cta, e_prev0 + (uint32_t)sample_phase_index(M, tid));
    csync();
    if (tid == 0 && s_fin == 0) {
        for (int r = 0; r < M.n_rows; ++r) s_tok[r] = s_nw[r];
        s_pos += 1;
        s_step += 1;
        if (A.b.finished != nullptr && A.s.audio_only && !A.s.ignore_stop && s_nw[0] == M.im_end) s_fin = 1;
    }
    __threadfence();  // acquire side of the once-per-frame fence: KV appended last frame is visible
    csync();
}

// BaseTransformer.embed (P:205-221) for one 8-element chunk (once per frame)
__device__ __noinline__ uint4 embed_chunk(const DevModel& M, int ch) {
    const int D = M.dim;
    const int t0 = s_tok[0];
    bool use_vq;
    if (M.mlx_embed_mask) use_vq = (t0 >= M.semantic_start && t0 <= M.semantic_end);
    else use_vq = s_tok[1] != 0;
    float f[8];
    unpack8(ldcg_v4(M.embeddings + (size_t)t0 * D + ch * 8), f);
    if (use_vq) {
        float s[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) s[e] = 0.f;
        for (int r0 = 1; r0 < M.n_rows; r0 += 8) {  // eight row loads in flight, summed in row order
            uint4 rows[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int r = r0 + i;
                if (r < M.n_rows) {
                    const int row = s_tok[r] + (M.dup0 ? (r - 1) : r) * M.codebook_size;
                    rows[i] = ldcg_v4(M.codebook_embeddings + (size_t)row * D + ch * 8);
                }
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                if (r0 + i < M.n_rows) {
                    float g[8];
                    unpack8(rows[i], g);
#pragma unroll
                    for (int e = 0; e < 8; ++e) s[e] = __fadd_rn(s[e], g[e]);
                }
            }
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) f[e] = bf16_round(__fadd_rn(f[e], bf16_round(s[e])));
    }
    return pack8(f);
}

// ---- staging of a phase's input vector ---------------------------------------------------------------------
// All consumer threads poll two words (one 16-byte load) per round of 512 words; a retry re-reads only what is missing.
// The payloads land in shared memory as bf16 (dst, and dst2 if nonzero); returns the thread's sum of squares.
__device__ __noinline__ float gather_words(const unsigned long long* src, int n_words, uint32_t e_src, uint32_t dst, uint32_t dst2) {
    // (A second, staggered poll of every word -- half a round trip behind the first -- was measured: the extra L2 poll
    //  traffic costs more than the earlier discovery gains, 721 vs 656 us per frame.)
    const int tid = threadIdx.x;
    uint4 v[kGather];
    bool need[kGather];
#pragma unroll
    for (int i = 0; i < kGather; ++i) {
        const int w = 2 * (tid + kCons * i);
        need[i] = w < n_words;
        v[i] = make_uint4(0u, e_src, 0u, e_src);
        if (need[i]) v[i] = ld_relaxed_v4(src + w);
    }
    uint32_t spins = 0;
    for (;;) {
        bool ready = true;
#pragma unroll
        for (int i = 0; i < kGather; ++i) {
            if (v[i].y != e_src || v[i].w != e_src) { ready = false; v[i] = ld_relaxed_v4(src + 2 * (tid + kCons * i)); }
        }
        if (ready) break;
        LL2_SPIN_GUARD(spins);
    }
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < kGather; ++i) {
        if (need[i]) {
            const uint32_t off = (uint32_t)(tid + kCons * i) * 8u;
            sts_v2(dst + off, v[i].x, v[i].z);
            if (dst2) sts_v2(dst2 + off, v[i].x, v[i].z);
            ss = fmaf(bf_lo(v[i].x), bf_lo(v[i].x), ss);
            ss = fmaf(bf_hi(v[i].x), bf_hi(v[i].x), ss);
            ss = fmaf(bf_lo(v[i].z), bf_lo(v[i].z), ss);
            ss = fmaf(bf_hi(v[i].z), bf_hi(v[i].z), ss);
        }
    }
    return ss;
}

// Staging of the output of a FUSED MLP: x = bf16(h + bf16(sum of the 7 fp32 partials, in slice order)) -- the reduction and
// the residual epilogue of the unfused W2 phase, with h from res_h (staged by the W13 phase).  Region: word s * K + e = the
// partial of slice s for element e.  The element -> thread map (and so the sum of squares) is that of gather_words: thread
// t holds elements 4 t .. 4 t + 3 (K <= 768: one quad per thread).
__device__ __noinline__ float gather_psum(const unsigned long long* src, int K, uint32_t e_src, uint32_t dst, uint32_t dst2, uint32_t resh) {
    const int tid = threadIdx.x;
    const bool need = 4 * tid < K;
    uint4 v[kNW][2];
#pragma unroll
    for (int s = 0; s < kNW; ++s) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            v[s][h] = make_uint4(0u, e_src, 0u, e_src);
            if (need) v[s][h] = ld_relaxed_v4(src + s * K + 4 * tid + 2 * h);
        }
    }
    uint32_t spins = 0;
    for (;;) {
        bool ready = true;
#pragma unroll
        for (int s = 0; s < kNW; ++s) {
#pragma unroll
            for (int h = 0; h < 2; ++h)
                if (v[s][h].y != e_src || v[s][h].w != e_src) { ready = false; v[s][h] = ld_relaxed_v4(src + s * K + 4 * tid + 2 * h); }
        }
        if (ready) break;
        LL2_SPIN_GUARD(spins);
    }
    if (!need) return 0.f;
    const uint32_t hw0 = lds_u32(resh + (uint32_t)tid * 8u), hw1 = lds_u32(resh + (uint32_t)tid * 8u + 4u);
    const float hv[4] = {bf_lo(hw0), bf_hi(hw0), bf_lo(hw1), bf_hi(hw1)};
    float x[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        float a = 0.f;
#pragma unroll
        for (int s = 0; s < kNW; ++s) a = __fadd_rn(a, __uint_as_float((e & 1) ? v[s][e >> 1].z : v[s][e >> 1].x));
        x[e] = bf16_round(__fadd_rn(hv[e], bf16_round(a)));
    }
    const uint32_t o0 = pack_bf16(x[0], x[1]), o1 = pack_bf16(x[2], x[3]);
    sts_v2(dst + (uint32_t)tid * 8u, o0, o1);
    if (dst2) sts_v2(dst2 + (uint32_t)tid * 8u, o0, o1);
    float ss = 0.f;
#pragma unroll
    for (int e = 0; e < 4; ++e) ss = fmaf(x[e], x[e], ss);
    return ss;
}

// The same staging shared by the S CTAs of a slice cluster (psum == 2): the CTA of cluster rank r polls only the quads
// [j0, j0 + nq) = [q r / S, q (r + 1) / S) of the vector (q = K / 4; thread 2 j + h: elements 4 (j0 + j) + 2 h, + 1, all 7
// partials in flight together), computes them exactly as gather_psum does and sends each quad (8 bytes, st.async) to its
// place in dst (and dst2) of every CTA of the cluster, itself included.  Everybody then waits on s_psumbar (K * 2 bytes
// per destination buffer) and takes its sum of squares from dst with gather_words's thread -> element map.
//
// The peers' stores may land before this CTA is done with the previous phase.  That is safe:
//  * A peer forwards its quads only once all 7 slice clusters have published their partials.  This CTA's own cluster
//    publishes only after every one of its CTAs has sent its act values, and this CTA sends its last ones after its last
//    W13 tile pass (every CTA of a slice cluster has a w13 tile: ll2_mlp_cluster).  From there on it reads neither xbuf
//    (the w2 chains read act and the ring) nor res_x (read by WO only), and this phase follows the W2 phase directly.
//    The idle cluster has no w13 tile and the depth-0 QKV follows HEAD + SAMPLE, which read xbuf: both use gather_psum.
//  * The bytes of the next split staging cannot reach s_psumbar before this one completes: that staging's input is the
//    next MLP's partials, which need this CTA's act values of that MLP, sent after the wait below.  So one barrier phase
//    per staging, with the parity carried by the caller.
__device__ __noinline__ float gather_psum_split(const unsigned long long* src, int K, uint32_t e_src, uint32_t dst, uint32_t dst2,
                                                uint32_t resh, uint32_t quads, int S, uint32_t parity) {
    const int tid = threadIdx.x, lane = tid & 31;
    const uint32_t bar = smem_u32(&s_psumbar);
    if (tid == 0) mbar_expect_tx(bar, (uint32_t)K * (dst2 ? 4u : 2u));
    const int j0 = (int)(quads & 0xffffu), n2 = 2 * (int)(quads >> 16);
    if ((tid & ~31) < n2) {   // the warps that hold a quad (n2 is even: both halves of a quad are in one warp)
        const bool mine = tid < n2;
        const int e = 4 * j0 + 2 * tid;
        uint4 v[kNW];
#pragma unroll
        for (int s = 0; s < kNW; ++s) {
            v[s] = make_uint4(0u, e_src, 0u, e_src);
            if (mine) v[s] = ld_relaxed_v4(src + s * K + e);
        }
        uint32_t spins = 0;
        for (;;) {
            bool ready = true;
#pragma unroll
            for (int s = 0; s < kNW; ++s)
                if (v[s].y != e_src || v[s].w != e_src) { ready = false; v[s] = ld_relaxed_v4(src + s * K + e); }
            if (ready) break;
            LL2_SPIN_GUARD(spins);
        }
        uint32_t w = 0u;
        if (mine) {
            const uint32_t hw = lds_u32(resh + (uint32_t)e * 2u);
            float a0 = 0.f, a1 = 0.f;
#pragma unroll
            for (int s = 0; s < kNW; ++s) {
                a0 = __fadd_rn(a0, __uint_as_float(v[s].x));
                a1 = __fadd_rn(a1, __uint_as_float(v[s].z));
            }
            w = pack_bf16(bf16_round(__fadd_rn(bf_lo(hw), bf16_round(a0))), bf16_round(__fadd_rn(bf_hi(hw), bf16_round(a1))));
        }
        const uint32_t w_other = __shfl_xor_sync(0xffffffffu, w, 1);
        if (mine) {   // the two threads of a quad share its destinations: ranks h, h + 2, ..
            const uint32_t lo = (lane & 1) ? w_other : w, hi = (lane & 1) ? w : w_other;
            const uint32_t off = (uint32_t)(e & ~3) * 2u;
            for (int d = lane & 1; d < S; d += 2) {
                const uint32_t rb = mapa(bar, (uint32_t)d);
                st_async_v2(mapa(dst + off, (uint32_t)d), lo, hi, rb);
                if (dst2) st_async_v2(mapa(dst2 + off, (uint32_t)d), lo, hi, rb);
            }
        }
    }
    mbar_wait(bar, parity);
    if (4 * tid >= K) return 0.f;
    const uint32_t x01 = lds_u32(dst + (uint32_t)tid * 8u), x23 = lds_u32(dst + (uint32_t)tid * 8u + 4u);
    const float x[4] = {bf_lo(x01), bf_hi(x01), bf_lo(x23), bf_hi(x23)};
    float ss = 0.f;
#pragma unroll
    for (int e = 0; e < 4; ++e) ss = fmaf(x[e], x[e], ss);
    return ss;
}

// The two inputs that are not LL regions: the token embedding of the pending column (slow layer 0, P:205-221; the frame
// boundary is taken here) and the embedding of the previous depth code (G:136-140).  Returns the thread's sum of squares.
__device__ __noinline__ float stage_embedding(const DevModel& M, const CallArgs& A, const Team tm, int src_kind, int it, int p, uint32_t epoch,
                                              int per_iter, int depth_pos, int K, const uint16_t* emb_base, uint32_t xb, uint32_t res) {
    const int tid = threadIdx.x;
    float ss = 0.f;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (src_kind == 0) {   // (the frame boundary was taken by the caller)
        if (tid < K / 8) v = embed_chunk(M, tid);
    } else {
        const int r = depth_pos;  // row of depth code depth_pos - 1
        int code;
        if (row_is_local(M, r)) code = s_nw[r];
        else {
            code = (int)ll_get(tok_words(M, tm, r) + tm.cta, epoch - (uint32_t)(p - sample_phase_index(M, r)));
            if (tid == 0) s_nw[r] = code;
        }
        if (tid < K / 8) v = ldcg_v4(emb_base + (size_t)code * K + tid * 8);
    }
    if (tid < K / 8) {
        sts_v4(xb + (uint32_t)tid * 16u, v);
        sts_v4(res + (uint32_t)tid * 16u, v);
        float f[8];
        unpack8(v, f);
#pragma unroll
        for (int e = 0; e < 8; ++e) ss = fmaf(f[e], f[e], ss);
    }
    return ss;
}

// ---- attention of the depth transformer (<= 8 positions), recomputed by every CTA ---------------------------------
// The q|k|v words of this depth step are parked in shared memory (q row; K/V appended to the CTA's own copy of the frame's
// depth K/V); then one warp per head: 4 lanes per position, two-pass softmax, probabilities rounded to bf16 for PV (the
// arithmetic of decode_kernel.cu: fast_attention_rows).  Output: bf16 row in xbuf.
__device__ __noinline__ void fast_attention(const DevModel& M, int layer, int depth_pos, const unsigned long long* qkv,
                                               uint32_t e_qkv, uint32_t fq, uint32_t fkv, uint32_t xs) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int Hq = M.fn_head, Hkv = M.fn_kv, G = Hq / Hkv;
    const int q_rows = Hq * kHeadDim, kvw = 2 * Hkv * kHeadDim;  // elements
    const uint32_t slot = fkv + (uint32_t)((layer * kLL2Depth + depth_pos) * kvw) * 2u;
    {   // 4 elements = 2 words = one 16-byte load; all of a thread's polls are in flight together
        constexpr int kPer = (1024 / 4 + 512 / 4 + kCons - 1) / kCons;   // up to 16 q heads + 8 kv heads
        const int n_it = (q_rows + kvw) / 4;
        uint4 v[kPer];
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const int i = tid + k * kCons;
            v[k] = make_uint4(0u, e_qkv, 0u, e_qkv);
            if (i < n_it) v[k] = ld_relaxed_v4(qkv + 2 * i);
        }
        uint32_t spins = 0;
        for (;;) {
            bool ready = true;
#pragma unroll
            for (int k = 0; k < kPer; ++k)
                if (v[k].y != e_qkv || v[k].w != e_qkv) { ready = false; v[k] = ld_relaxed_v4(qkv + 2 * (tid + k * kCons)); }
            if (ready) break;
            LL2_SPIN_GUARD(spins);
        }
#pragma unroll
        for (int k = 0; k < kPer; ++k) {
            const int i = tid + k * kCons;
            if (i < n_it) {
                const int e = 4 * i;
                const uint32_t dst = e < q_rows ? fq + (uint32_t)e * 2u : slot + (uint32_t)(e - q_rows) * 2u;
                sts_v2(dst, v[k].x, v[k].z);
            }
        }
    }
    csync();
    const int j = lane >> 2, part = lane & 3;
    const bool ok = j <= depth_pos;
    const uint32_t lay = fkv + (uint32_t)(layer * kLL2Depth * kvw) * 2u;
    // a warp carries up to kHeadsPerWarp heads AT ONCE (their FMA chains and shuffle trees interleave): heads warp, warp + kNW, ..
    constexpr int kHP = 2;
#pragma unroll 1
    for (int h0 = warp; h0 < Hq; h0 += kHP * kNW) {
        float s[kHP], sa[kHP];
        uint32_t vw[kHP][8];
        bool hv[kHP];
#pragma unroll
        for (int u = 0; u < kHP; ++u) {
            const int hq = h0 + u * kNW;
            hv[u] = hq < Hq;
            const int kvh = hv[u] ? hq / G : 0;
            s[u] = 0.f; sa[u] = 0.f;
            if (ok && hv[u]) {
                const uint32_t qa = fq + (uint32_t)(hq * kHeadDim + part * 16) * 2u;
                const uint32_t ka = lay + (uint32_t)(j * kvw + kvh * kHeadDim + part * 16) * 2u;
                float qf[8], kf[8];
                unpack8(lds_v4(qa), qf); unpack8(lds_v4(ka), kf);
#pragma unroll
                for (int e = 0; e < 8; ++e) s[u] = fmaf(qf[e], kf[e], s[u]);
                unpack8(lds_v4(qa + 16u), qf); unpack8(lds_v4(ka + 16u), kf);
#pragma unroll
                for (int e = 0; e < 8; ++e) sa[u] = fmaf(qf[e], kf[e], sa[u]);
            }
#pragma unroll
            for (int jj = 0; jj < 8; ++jj)
                vw[u][jj] = (jj <= depth_pos && hv[u]) ? lds_u32(lay + (uint32_t)(jj * kvw + Hkv * kHeadDim + kvh * kHeadDim + 2 * lane) * 2u) : 0u;
        }
        float sc[kHP], m[kHP], pe[kHP], l[kHP];
#pragma unroll
        for (int u = 0; u < kHP; ++u) s[u] = s[u] + sa[u];   // same order as one 16-term chain? no: two 8-term halves, added once
#pragma unroll
        for (int o = 1; o <= 2; o <<= 1) {
#pragma unroll
            for (int u = 0; u < kHP; ++u) s[u] += __shfl_xor_sync(0xffffffffu, s[u], o);
        }
#pragma unroll
        for (int u = 0; u < kHP; ++u) { sc[u] = ok ? s[u] * 0.125f : -INFINITY; m[u] = sc[u]; }
#pragma unroll
        for (int o = 4; o <= 16; o <<= 1) {
#pragma unroll
            for (int u = 0; u < kHP; ++u) m[u] = fmaxf(m[u], __shfl_xor_sync(0xffffffffu, m[u], o));
        }
#pragma unroll
        for (int u = 0; u < kHP; ++u) { pe[u] = ok ? expf(sc[u] - m[u]) : 0.f; l[u] = pe[u] + 0.f; }
#pragma unroll
        for (int o = 4; o <= 16; o <<= 1) {
#pragma unroll
            for (int u = 0; u < kHP; ++u) l[u] += __shfl_xor_sync(0xffffffffu, l[u], o);
        }
#pragma unroll
        for (int u = 0; u < kHP; ++u) {
            const float pb = bf16_round(pe[u]);
            float o0 = 0.f, o1 = 0.f;
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                const float pj = __shfl_sync(0xffffffffu, pb, jj * 4);
                o0 = fmaf(pj, bf_lo(vw[u][jj]), o0);
                o1 = fmaf(pj, bf_hi(vw[u][jj]), o1);
            }
            const float inv = 1.0f / l[u];
            if (hv[u]) sts_u32(xs + (uint32_t)((h0 + u * kNW) * kHeadDim + 2 * lane) * 2u, pack_bf16(bf16_round(o0 * inv), bf16_round(o1 * inv)));
        }
    }
}

// ---- slow attention: score units + PV units --------------------------------------------------------------------
__device__ __forceinline__ unsigned long long* score_words(const DevModel& M, const Team& tm, int layer, int hq) {
    return M.ll2_score + (((size_t)tm.team * 2 + (layer & 1)) * M.n_head + hq) * (size_t)M.ll2_score_len;
}
__device__ __forceinline__ const uint16_t* kv_row(const DevModel& M, const Seq& sq, int layer, int is_v, int kvh, int pos) {
    const int sh = M.page_size == 32 ? 5 : 4;   // pages of 16 or 32 positions (smol_create): no integer division here
    const int pg = pos >> sh;
    const int page = pg < kBtabCache ? s_btab[pg] : ldcg_i32(sq.btab + pg);
    return M.kv_pool + (((((size_t)page * M.n_layer + layer) * 2 + is_v) * M.n_kv + kvh) << (sh + 6)) + (size_t)(pos & ((1 << sh) - 1)) * kHeadDim;
}

__device__ __noinline__ void phase_attn(const DevModel& M, const CallArgs& A, const Team tm, int layer, int p,
                                        uint32_t epoch, uint32_t scratch, int holdoff) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const Seq sq = seq_of(M, A, tm.team);
    const int rep = tm.cta % kLLRep;
    const int Hq = M.n_head, Hkv = M.n_kv, G = Hq / Hkv;
    const int q_words = Hq * kHeadDim / 2, k_end_words = (Hq + Hkv) * kHeadDim / 2;
    const int pos_new = s_pos;
    int Lb = pos_new + 1;
    const int cap = A.b.max_pages * M.page_size;
    if (Lb > cap) Lb = cap;
    const int nseg = (Lb + kLL2ScoreBlock - 1) / kLL2ScoreBlock;   // 64-position segments: score units and reduction grain
    const int n_su = Hkv * nseg;
    const int n_pv = Hq * (kHeadDim / kLL2PvDims);
    const unsigned long long* qkv = ll_region(M, tm.team, p - 1, rep);
    const uint32_t e_qkv = epoch - 1;

    // ---- score units: (kv head, 64 positions): s[h][j] = (q_h . k_j) / 8 for the G query heads of the group ----
    constexpr int kPosPerRound = kCons / 8;                                  // 28 positions x 8 chunks of 8 head dims
    constexpr int kRounds = (kLL2ScoreBlock + kPosPerRound - 1) / kPosPerRound;  // 3
    for (int u = tm.cta; u < n_su; u += tm.n) {
        const int kvh = u / nseg, blk = u - kvh * nseg;
        const int p0 = blk * kLL2ScoreBlock;
        const int p1 = min(Lb, p0 + kLL2ScoreBlock);
        const int chunk = tid & 7;
        uint4 kk[kRounds];
#pragma unroll
        for (int r = 0; r < kRounds; ++r) {   // cached keys: in flight before q arrives
            const int pos = p0 + (tid >> 3) + kPosPerRound * r;
            kk[r] = make_uint4(0u, 0u, 0u, 0u);
            if (pos < p1 && pos != pos_new) kk[r] = ldcg_v4(kv_row(M, sq, layer, 0, kvh, pos) + chunk * 8);
        }
        // q of the group's heads (G * 32 words): one 16-byte poll per thread; pre-scaled by 1/sqrt(64) (exact)
        if (tid < G * 16) {
            const unsigned long long* qp = qkv + (kvh * G) * 32 + 2 * tid;
            uint4 v = ld_relaxed_v4(qp);
            uint32_t spins = 0;
            while (v.y != e_qkv || v.w != e_qkv) { LL2_SPIN_GUARD(spins); v = ld_relaxed_v4(qp); }
            sts_v4(scratch + (uint32_t)tid * 16u,
                   make_uint4(__float_as_uint(bf_lo(v.x) * 0.125f), __float_as_uint(bf_hi(v.x) * 0.125f),
                              __float_as_uint(bf_lo(v.z) * 0.125f), __float_as_uint(bf_hi(v.z) * 0.125f)));
        }
        {   // the newest position's key comes from the QKV phase's words (at most one round of 8 threads owns it)
            const int rel = pos_new - p0 - (tid >> 3);
            if (pos_new < p1 && rel >= 0 && rel % kPosPerRound == 0 && rel / kPosPerRound < kRounds) {
                const unsigned long long* kp = qkv + q_words + kvh * 32 + chunk * 4;
                uint4 a = ld_relaxed_v4(kp), b = ld_relaxed_v4(kp + 2);
                uint32_t spins = 0;
                while (a.y != e_qkv || a.w != e_qkv || b.y != e_qkv || b.w != e_qkv) {
                    LL2_SPIN_GUARD(spins);
                    a = ld_relaxed_v4(kp); b = ld_relaxed_v4(kp + 2);
                }
                const uint4 kn = make_uint4(a.x, a.z, b.x, b.z);
                const int rn = rel / kPosPerRound;
#pragma unroll
                for (int r = 0; r < kRounds; ++r)
                    if (r == rn) kk[r] = kn;
            }
        }
        csync();
        // all (round, head) dot products are independent: their FMA chains and shuffle trees interleave
        float sc[kRounds][kMaxGroup];
        {
            float kf[kRounds][8];
#pragma unroll
            for (int r = 0; r < kRounds; ++r) unpack8(kk[r], kf[r]);
#pragma unroll
            for (int h = 0; h < kMaxGroup; ++h) {
                if (h < G) {
                    const uint32_t qa = scratch + (uint32_t)(h * kHeadDim + chunk * 8) * 4u;
                    const uint4 q0 = lds_v4(qa), q1 = lds_v4(qa + 16u);
#pragma unroll
                    for (int r = 0; r < kRounds; ++r) {
                        float a = __uint_as_float(q0.x) * kf[r][0];
                        a = fmaf(__uint_as_float(q0.y), kf[r][1], a); a = fmaf(__uint_as_float(q0.z), kf[r][2], a);
                        a = fmaf(__uint_as_float(q0.w), kf[r][3], a); a = fmaf(__uint_as_float(q1.x), kf[r][4], a);
                        a = fmaf(__uint_as_float(q1.y), kf[r][5], a); a = fmaf(__uint_as_float(q1.z), kf[r][6], a);
                        sc[r][h] = fmaf(__uint_as_float(q1.w), kf[r][7], a);
                    }
                } else {
#pragma unroll
                    for (int r = 0; r < kRounds; ++r) sc[r][h] = 0.f;
                }
            }
        }
#pragma unroll
        for (int o = 1; o <= 4; o <<= 1) {
#pragma unroll
            for (int r = 0; r < kRounds; ++r) {
#pragma unroll
                for (int h = 0; h < kMaxGroup; ++h)
                    if (h < G) sc[r][h] += __shfl_xor_sync(0xffffffffu, sc[r][h], o);
            }
        }
        if (chunk == 0) {
#pragma unroll
            for (int r = 0; r < kRounds; ++r) {
                const int pos = p0 + (tid >> 3) + kPosPerRound * r;
#pragma unroll
                for (int h = 0; h < kMaxGroup; ++h)
                    if (h < G && pos < p1) st_relaxed_v2(score_words(M, tm, layer, kvh * G + h) + pos, __float_as_uint(sc[r][h]), epoch);
            }
        }
        csync();
    }

    // ---- PV units: (query head, 8 head dims) over the whole context -------------------------------------------------
    // Softmax blocks of 512 positions as in the reference's CPU SDPA kernel: running maximum m_b = max(m_{b-1}, block
    // maximum); p = exp(s - m_b) in fp32; the denominator sums the fp32 p; P is ROUNDED TO bf16 for P.V; blocks are
    // combined in order with the rescale exp(m_{b-1} - m_b).  Work grain = 64-position segments (8 per block): warp w takes
    // segments w, w + 7, ..; lane l the positions 2 l, 2 l + 1 of the segment; per-segment partial sums meet in shared
    // memory and are added in segment order.
    const int nb = (Lb + kLL2AttnBlock - 1) / kLL2AttnBlock;
    const uint32_t red = scratch + (uint32_t)(nseg * kLL2ScoreBlock) * 4u;   // [segment][8 dims + denominator]
    const int seg_new = pos_new >> 6;
    const bool own_new = pos_new < Lb && (seg_new % kNW) == warp && ((pos_new & 63) >> 1) == lane;
    bool waited = false;
    for (int v = tm.cta - (n_su % tm.n); v < n_pv; v += tm.n) {
        if (v < 0) continue;
        const int hq = v / (kHeadDim / kLL2PvDims), ds = v - hq * (kHeadDim / kLL2PvDims), kvh = hq / G;
        // cached value rows of a segment (the newest position is patched in from the QKV phase's words)
        auto load_v = [&](int sgm, int j) -> uint4 {
            const int pos = sgm * kLL2ScoreBlock + 2 * lane + j;
            if (sgm >= nseg || pos >= Lb || pos == pos_new) return make_uint4(0u, 0u, 0u, 0u);
            return ldcg_v4(kv_row(M, sq, layer, 1, kvh, pos) + ds * kLL2PvDims);
        };
        uint4 va = load_v(warp, 0), vb = load_v(warp, 1);   // first round: in flight before the scores are polled
        uint4 vnew = make_uint4(0u, 0u, 0u, 0u);
        if (own_new) {
            const unsigned long long* vp = qkv + k_end_words + kvh * 32 + ds * 4;
            uint4 a = ld_relaxed_v4(vp), b = ld_relaxed_v4(vp + 2);
            uint32_t spins = 0;
            while (a.y != e_qkv || a.w != e_qkv || b.y != e_qkv || b.w != e_qkv) {
                LL2_SPIN_GUARD(spins);
                a = ld_relaxed_v4(vp); b = ld_relaxed_v4(vp + 2);
            }
            vnew = make_uint4(a.x, a.z, b.x, b.z);
        }
        if (!waited && holdoff > 0) {  // the scores are at least one hand-off away
            const uint32_t t0 = clock32_now();
            while (clock32_now() - t0 < (uint32_t)holdoff) {}
            waited = true;
        }
        // scores of this head -> shared memory (fp32), four rounds of polls in flight at a time
        const unsigned long long* sw = score_words(M, tm, layer, hq);
#pragma unroll 1
        for (int r0 = 0; r0 * kNW < nseg; r0 += 4) {
            uint4 s4[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int sgm = (r0 + i) * kNW + warp, pos = sgm * kLL2ScoreBlock + 2 * lane;
                s4[i] = make_uint4(0xff800000u, epoch, 0xff800000u, epoch);   // -inf: position past the context
                if (sgm < nseg && pos < Lb) s4[i] = ld_relaxed_v4(sw + pos);
            }
            uint32_t spins = 0;
            for (;;) {
                bool ready = true;
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int sgm = (r0 + i) * kNW + warp, pos = sgm * kLL2ScoreBlock + 2 * lane;
                    const bool two = sgm < nseg && pos + 1 < Lb;
                    if (s4[i].y != epoch || (two && s4[i].w != epoch)) { ready = false; s4[i] = ld_relaxed_v4(sw + pos); }
                }
                if (ready) break;
                LL2_SPIN_GUARD(spins);
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int sgm = (r0 + i) * kNW + warp, pos = sgm * kLL2ScoreBlock + 2 * lane;
                if (sgm < nseg) {
                    const float a = pos < Lb ? __uint_as_float(s4[i].x) : -INFINITY;
                    const float b = pos + 1 < Lb ? __uint_as_float(s4[i].z) : -INFINITY;
                    sts_v2(scratch + (uint32_t)pos * 4u, __float_as_uint(a), __float_as_uint(b));
                    const float mx = warp_max(fmaxf(a, b));
                    if (lane == 0) s_bmax[sgm] = mx;
                }
            }
        }
        csync();
        // the warp walks its segments in ascending order and keeps the running maximum of all blocks up to the current one;
        // the next segment's value rows are in flight while the current one is reduced
        float m_run = -INFINITY;
        int seg_seen = 0;
#pragma unroll 1
        for (int sgm = warp; sgm < nseg; sgm += kNW) {
            const uint4 na = load_v(sgm + kNW, 0), nb2 = load_v(sgm + kNW, 1);
            if (own_new && sgm == seg_new) { if (pos_new & 1) vb = vnew; else va = vnew; }
            const int upto = min(nseg, ((sgm >> 3) + 1) * 8);   // segments of the blocks up to this segment's block
#pragma unroll 1
            for (; seg_seen < upto; ++seg_seen) m_run = fmaxf(m_run, s_bmax[seg_seen]);
            const int pos = sgm * kLL2ScoreBlock + 2 * lane;
            const uint2 sp = make_uint2(lds_u32(scratch + (uint32_t)pos * 4u), lds_u32(scratch + (uint32_t)pos * 4u + 4u));
            const float p0 = pos < Lb ? expf(__uint_as_float(sp.x) - m_run) : 0.f;
            const float p1 = pos + 1 < Lb ? expf(__uint_as_float(sp.y) - m_run) : 0.f;
            const float b0 = bf16_round(p0), b1 = bf16_round(p1);
            float fa[8], fb[8], acc[8];
            unpack8(va, fa);
            unpack8(vb, fb);
#pragma unroll
            for (int e = 0; e < 8; ++e) acc[e] = fmaf(b1, fb[e], __fmul_rn(b0, fa[e]));
            float ls = p0 + p1;
            // warp reduction: halve the vector at every step (9 shuffles for 8 values), lane bits 4,3,2 select the dim
            {
                const bool up = lane & 16;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float send = up ? acc[e] : acc[e + 4];
                    const float got = __shfl_xor_sync(0xffffffffu, send, 16);
                    acc[e] = (up ? acc[e + 4] : acc[e]) + got;
                }
            }
            {
                const bool up = lane & 8;
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const float send = up ? acc[e] : acc[e + 2];
                    const float got = __shfl_xor_sync(0xffffffffu, send, 8);
                    acc[e] = (up ? acc[e + 2] : acc[e]) + got;
                }
            }
            {
                const bool up = lane & 4;
                const float send = up ? acc[0] : acc[1];
                const float got = __shfl_xor_sync(0xffffffffu, send, 4);
                acc[0] = (up ? acc[1] : acc[0]) + got;
            }
            acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 2);
            acc[0] += __shfl_xor_sync(0xffffffffu, acc[0], 1);
            ls = warp_sum(ls);
            // lane with bits (16, 8, 4) = (b2, b1, b0) holds dim 4 * b2 + 2 * b1 + b0
            if ((lane & 3) == 0) sts_f32(red + (uint32_t)(sgm * 9 + ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1)) * 4u, acc[0]);
            if (lane == 0) sts_f32(red + (uint32_t)(sgm * 9 + 8) * 4u, ls);
            va = na; vb = nb2;
        }
        csync();
        if (warp == 0) {
            // lanes 0..7: one head dim each; segments added in order inside a block, blocks combined in order
            // (dst = dst * c + PV_b; l = l_b + c * l)
            float dst = 0.f, l = 0.f, m_prev = -INFINITY;
            const int d = lane & 7;
#pragma unroll 1
            for (int b = 0; b < nb; ++b) {
                const int s0 = b * 8, s1 = min(nseg, s0 + 8);
                float bm = -INFINITY, o = 0.f, li = 0.f;
#pragma unroll 1
                for (int sg = s0; sg < s1; ++sg) {
                    bm = fmaxf(bm, s_bmax[sg]);
                    o = __fadd_rn(o, lds_f32(red + (uint32_t)(sg * 9 + d) * 4u));
                    li = __fadd_rn(li, lds_f32(red + (uint32_t)(sg * 9 + 8) * 4u));
                }
                const float m_b = fmaxf(m_prev, bm);
                const float c = (m_prev == -INFINITY) ? 0.f : expf(m_prev - m_b);
                l = __fadd_rn(li, __fmul_rn(c, l));
                dst = __fadd_rn(__fmul_rn(dst, c), o);
                m_prev = m_b;
            }
            const float outv = bf16_round(__fdiv_rn(dst, l));
            const float nxt = __shfl_down_sync(0xffffffffu, outv, 1);
            const uint32_t word = pack_bf16(outv, nxt);   // meaningful on even lanes < 8
            // 4 words x kLLRep replicas: lane = word * 8 + replica
            const uint32_t wv = __shfl_sync(0xffffffffu, word, 2 * (lane >> 3));
            unsigned long long* out = ll_region(M, tm.team, p, 0) + (hq * kHeadDim + ds * kLL2PvDims) / 2 + (lane >> 3);
            st_relaxed_v2(out + (size_t)(lane & 7) * M.ll_len[p], wv, epoch);
        }
        csync();
    }
}

// ---- sampling (G:88-99 slow, G:118-132 depth) + frame assembly and the stop rule (G:143-166) ------------
__device__ __noinline__ void phase_sample(const DevModel& M, const CallArgs& A, const Team tm, int is_fast, int depth_pos,
                                          int p, uint32_t epoch, float* lg) {
    const int tid = threadIdx.x;
    const Seq sq = seq_of(M, A, tm.team);
    const bool fast = is_fast != 0;
    const int N = fast ? M.codebook_size : M.vocab;
    const int r = fast ? 1 + depth_pos : 0;
    const int R = M.n_rows;
    const bool local = row_is_local(M, r);
    if (!local && tm.cta != 0) return;  // sampled rows: CTA 0 of the team samples, the others pick the id up when they need it
    int tok;
    if (sq.force != nullptr) {
        tok = ldcg_i32(sq.force + r);
    } else if (local) {
        // greedy: every CTA published its best (logit, index) with the HEAD phase's epoch; everybody reduces them
        const unsigned long long* src = cand_words(M, tm, r, tm.cta % kLLRep);
        uint32_t best = 0u;
        for (int i = tid; i < tm.n; i += kCons) { const uint32_t cnd = ll_get(src + i, epoch - 1); best = cnd > best ? cnd : best; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const uint32_t ob = __shfl_xor_sync(0xffffffffu, best, o);
            best = ob > best ? ob : best;
        }
        if ((tid & 31) == 0) s_sc.i32[tid >> 5] = (int)best;
        csync();
        uint32_t b2 = 0u;
#pragma unroll
        for (int w = 0; w < kNW; ++w) { const uint32_t c = (uint32_t)s_sc.i32[w]; b2 = c > b2 ? c : b2; }
        tok = cand_index(b2);
    } else {
        const unsigned long long* src = ll_region(M, tm.team, p - 1, 0);  // the HEAD phase's logits (replica 0)
        for (int i = tid; i < N / 4; i += kCons) {
            uint4 v = ld_relaxed_v4(src + 2 * i);
            uint32_t spins = 0;
            while (v.y != epoch - 1 || v.w != epoch - 1) { LL2_SPIN_GUARD(spins); v = ld_relaxed_v4(src + 2 * i); }
            *reinterpret_cast<float4*>(lg + 4 * i) = make_float4(bf_lo(v.x), bf_hi(v.x), bf_lo(v.z), bf_hi(v.z));
        }
        csync();
        const uint32_t seq_id = sq.seq_id ? (uint32_t)ldcg_i32(sq.seq_id) : 0u;
        tok = sample_row<kCons, kSampPer>(lg, N, fast ? s_rs.fast_temp : s_rs.temp, fast ? 0 : s_rs.top_k, fast ? 1.0f : s_rs.top_p,
                                    s_rs.min_p, s_rs.seed, (uint32_t)s_step, seq_id, (uint32_t)r, s_sc);
    }
    const bool last = fast && depth_pos == M.depth - 1;
    if (local) {
        if (tid == 0) s_nw[r] = tok;
    } else {
        if (last) __threadfence();  // frame boundary: keep the release chain cumulative
        for (int i = tid; i < tm.n; i += kCons) st_relaxed_v2(tok_words(M, tm, r) + i, (uint32_t)tok, epoch);
        if (tid == 0) s_nw[r] = tok;
    }
    if (tm.cta == 0 && tid == 0) {
        sq.frame_tokens[r] = tok;
        if (last && s_fin == 0) {
            // frame assembly for the host and the next launch; every CTA applies the same update locally
            const int st = s_step;
            int slow = 0;
            for (int rr = 0; rr < R; ++rr) {
                const int v = rr == r ? tok : s_nw[rr];
                if (rr == 0) slow = v;
                sq.tokens[rr] = v;
                if (sq.out_codes != nullptr && st < A.b.max_frames) sq.out_codes[(size_t)st * R + rr] = v;
            }
            if (sq.step) sq.step[0] = st + 1;
            if (M.frame_ns != nullptr && tm.team == 0 && st < M.frame_ns_cap) M.frame_ns[st] = globaltimer_ns();
            sq.seq_len[0] = s_pos + 1;
            if (sq.finished != nullptr && A.s.audio_only && !A.s.ignore_stop && slow == M.im_end) sq.finished[0] = 1;
        }
    }
    csync();
}

// KV append (K:12-22) of one bf16 pair into the paged pool (slow QKV phases)
__device__ __noinline__ void kv_append(const DevModel& M, const CallArgs& A, int team, int layer, int n0, uint32_t word) {
    const Seq sq = seq_of(M, A, team);
    const int Hq = M.n_head, Hkv = M.n_kv, ps = M.page_size;
    const int q_rows = Hq * kHeadDim, k_end = (Hq + Hkv) * kHeadDim;
    const int pos = s_pos;
    if (pos >= A.b.max_pages * ps || s_fin != 0) return;
    const int is_v = n0 >= k_end ? 1 : 0;
    const int n1 = n0 - (is_v ? k_end : q_rows);
    const int kvh = n1 / kHeadDim, d = n1 & (kHeadDim - 1);
    uint16_t* dst = const_cast<uint16_t*>(kv_row(M, sq, layer, is_v, kvh, pos)) + d;
    *reinterpret_cast<uint32_t*>(dst) = word;
}

// One pass of NT tiles through the tensor cores: for every K chunk (ring stage per tile) the warp carries its k-blocks
// through all NT tiles, then leaves its partial sums (row slots g and g + 8 of every tile) in shared memory.
// A tile's k-block is 1024 bytes: for each of the two MMA steps 32 lanes x 16 bytes = the lane's A fragment (a0..a3)
// exactly as mma.m16n8k16 wants it (smol_pack_kernel); the B fragment (the activation vector, the same in all 8 columns)
// is 16 bytes per lane for both steps.  Two accumulators per tile (one per MMA step): no MMA waits for the one issued
// just before it.  Ring stages are consumed strictly in order: (cslot, cpar) = slot and parity of the next one.
template <int NT>
__device__ __forceinline__ void tile_pass(int kb, int chunks, int warp, int lane, uint32_t full0, uint32_t empty0, uint32_t ringl,
                                          uint32_t ns, uint32_t xbl, uint32_t pw, bool writer, uint32_t& cslot, uint32_t& cpar) {
    float acc[NT][4], acd[NT][4];
#pragma unroll
    for (int i = 0; i < NT; ++i) {
#pragma unroll
        for (int e = 0; e < 4; ++e) { acc[i][e] = 0.f; acd[i][e] = 0.f; }
    }
#pragma unroll 1
    for (int kc = 0; kc < chunks; ++kc) {
        const int kb0 = kc * kLL2ChunkKb, nkb = min(kLL2ChunkKb, kb - kb0);
        const int lo = (nkb * warp) / kNW, hi = (nkb * (warp + 1)) / kNW;
        uint32_t abase[NT];
        uint32_t sl = cslot, pr = cpar;
#pragma unroll
        for (int i = 0; i < NT; ++i) {
            mbar_wait(full0 + 8u * sl, pr);
            abase[i] = ringl + sl * (uint32_t)kLL2SlotBytes;
            if (++sl == ns) { sl = 0u; pr ^= 1u; }
        }
        const uint32_t xb = xbl + (uint32_t)kb0 * 64u;
#pragma unroll 1
        for (int j = lo; j < hi; ++j) {
            const uint4 bx = lds_v4(xb + (uint32_t)j * 64u);
            uint4 a0[NT], a1[NT];
#pragma unroll
            for (int i = 0; i < NT; ++i) {
                a0[i] = lds_v4(abase[i] + (uint32_t)j * 1024u);
                a1[i] = lds_v4(abase[i] + (uint32_t)j * 1024u + 512u);
            }
#pragma unroll
            for (int i = 0; i < NT; ++i) mma_bf16_16816(acc[i], a0[i].x, a0[i].y, a0[i].z, a0[i].w, bx.x, bx.y);
#pragma unroll
            for (int i = 0; i < NT; ++i) mma_bf16_16816(acd[i], a1[i].x, a1[i].y, a1[i].z, a1[i].w, bx.z, bx.w);
        }
        __syncwarp();
        if (lane < NT) {   // lane i hands back the stage of tile i
            uint32_t r = cslot + (uint32_t)lane;
            if (r >= ns) r -= ns;
            mbar_arrive(empty0 + 8u * r);
        }
        cslot = sl; cpar = pr;
    }
    if (writer) {   // lanes with c == 0: row slot g (acc[.][0]) and g + 8 (acc[.][2]); every column carries the same vector
#pragma unroll
        for (int i = 0; i < NT; ++i) {
            sts_f32(pw + (uint32_t)(i * kNW * 16) * 4u, __fadd_rn(acc[i][0], acd[i][0]));
            sts_f32(pw + (uint32_t)(i * kNW * 16 + 8) * 4u, __fadd_rn(acc[i][2], acd[i][2]));
        }
    }
}

// A multi-stage tile (K = 3072: 4 ring stages): the warp takes ONE contiguous range of the tile's k-blocks -- it waits for
// the stage(s) the range touches, runs one loop, and only then hands all stages back (every warp arrives once per stage).
__device__ __forceinline__ void tile_pass_long(int kb, int chunks, int warp, int lane, uint32_t full0, uint32_t empty0, uint32_t ringl,
                                               uint32_t ns, uint32_t xbl, uint32_t pw, bool writer, uint32_t& cslot, uint32_t& cpar) {
    float acc[4] = {0.f, 0.f, 0.f, 0.f}, acd[4] = {0.f, 0.f, 0.f, 0.f};
    const int lo = (kb * warp) / kNW, hi = (kb * (warp + 1)) / kNW;
    int cur = -1;
    uint32_t abase = 0u;
#pragma unroll 1
    for (int j = lo; j < hi; ++j) {
        const int kc = j / kLL2ChunkKb;
        if (kc != cur) {   // first k-block of a stage: slot and parity follow from the running (cslot, cpar)
            uint32_t sl = cslot + (uint32_t)kc, pr = cpar;
            if (sl >= ns) { sl -= ns; pr ^= 1u; }
            mbar_wait(full0 + 8u * sl, pr);
            abase = ringl + sl * (uint32_t)kLL2SlotBytes - (uint32_t)(kc * kLL2ChunkKb) * 1024u;
            cur = kc;
        }
        const uint4 bx = lds_v4(xbl + (uint32_t)j * 64u);
        const uint4 a0 = lds_v4(abase + (uint32_t)j * 1024u), a1 = lds_v4(abase + (uint32_t)j * 1024u + 512u);
        mma_bf16_16816(acc, a0.x, a0.y, a0.z, a0.w, bx.x, bx.y);
        mma_bf16_16816(acd, a1.x, a1.y, a1.z, a1.w, bx.z, bx.w);
    }
    __syncwarp();
    if (lane < chunks) {   // lane i hands back stage i of the tile
        uint32_t r = cslot + (uint32_t)lane;
        if (r >= ns) r -= ns;
        mbar_arrive(empty0 + 8u * r);
    }
    uint32_t sl = cslot + (uint32_t)chunks;
    if (sl >= ns) { sl -= ns; cpar ^= 1u; }
    cslot = sl;
    if (writer) {
        sts_f32(pw, __fadd_rn(acc[0], acd[0]));
        sts_f32(pw + 32u, __fadd_rn(acc[2], acd[2]));
    }
}

template <bool kTrace>
__global__ void __launch_bounds__(kLL2Threads, 1)
smol_ll2_kernel(const __grid_constant__ DevModel M, const __grid_constant__ CallArgs A, const __grid_constant__ SmemPlan SP) {
    extern __shared__ __align__(1024) unsigned char smem_dyn[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t sm0 = smem_u32(smem_dyn);
    const uint32_t full0 = smem_u32(s_full), empty0 = smem_u32(s_empty);
    const int per_iter = A.phase_end;
    Team tm;
    tm.n = A.team_ctas;
    tm.team = blockIdx.x / tm.n;
    tm.cta = blockIdx.x - tm.team * tm.n;
    // shared-memory addresses: one add from the constant bank each, never a live register (a spilled value is an L2 round
    // trip here: the L1 is what 220 KB of shared memory leave)
#define XB (sm0 + (uint32_t)SP.xbuf)
#define RESX (sm0 + (uint32_t)SP.res_x)
#define RESH (sm0 + (uint32_t)SP.res_h)
#define PART (sm0 + (uint32_t)SP.part)
#define DSC0 (sm0 + (uint32_t)SP.desc)
#define FQ (sm0 + (uint32_t)SP.fq)
#define FKV (sm0 + (uint32_t)SP.fkv)
#define SCR (sm0 + (uint32_t)SP.scratch)
#define RING (sm0 + (uint32_t)SP.ring)
#define ACT (sm0 + (uint32_t)SP.act)
#define NSLOTS ((uint32_t)SP.n_slots)

    {
        const Seq sq = seq_of(M, A, tm.team);
        if (tid == 0) {
            for (int i = 0; i < SP.n_slots; ++i) { mbar_init(full0 + 8u * i, 1u); mbar_init(empty0 + 8u * i, (uint32_t)kNW); }
            mbar_init(smem_u32(&s_actbar), 1u);
            mbar_init(smem_u32(&s_psumbar), 1u);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            s_pos = ldcg_i32(sq.seq_len);
            s_step = sq.step ? ldcg_i32(sq.step) : 0;
            s_fin = sq.finished != nullptr ? (int)__ldcg(sq.finished) : 0;
            s_rs = row_sampling(A.s, A.b.row_sampling, tm.team);
            s_best = 0u;
        }
        if (tid < M.n_rows) { s_tok[tid] = ldcg_i32(sq.tokens + tid); s_nw[tid] = 0; }
        for (int p = tid; p < per_iter; p += kLL2Threads) build_desc(M, tm, A.mlp_cluster, A.psum_split, p, DSC0 + (uint32_t)p * (kDescWords * 4u));
        for (int i = tid; i < kBtabCache && i < A.b.max_pages; i += kLL2Threads) s_btab[i] = ldcg_i32(sq.btab + i);
    }
    __syncthreads();
    if (tid == 0) s_epoch0 = (uint32_t)ldcg_i32(M.ll_epoch);
    if (A.mlp_cluster > 0) cluster_sync_all();   // every act / psum barrier of the cluster is initialised before the first DSMEM store
    __syncthreads();

    if (warp == kNW) {  // the TMA producer warp
        if (lane == 0) producer(A, SP, sm0);
        return;
    }

    // cycle trace of the launch's last iteration (kTrace): CTA 0 and CTA n/2 of team 0, thread 0:
    // 0 start, 1 input words arrived, 2 past the staging barrier, 3 B fragments ready, 4 MMAs of the last tile done,
    // 5 past the reduction barrier, 6 end of the phase (warp 0 has published if it was the reducing warp)
    unsigned long long* tr = nullptr;
    if (kTrace && M.prof != nullptr && tid == 0 && tm.team == 0 && (tm.cta == 0 || tm.cta == tm.n / 2))
        tr = M.prof + 2 * kMaxProg + 64 + (tm.cta == 0 ? 0 : 1) * kMaxProg * 8;
#define LL2_TRACE(i) do { if (kTrace && tr) { tr[p * 8 + (i)] = (unsigned long long)clock_now(); } \
                          if (kTrace && trg && ((i) == 1 || (i) == 6)) trg[p * 2 + ((i) == 6 ? 1 : 0)] = globaltimer_ns(); } while (0)
    unsigned long long* trg = nullptr;   // skew trace: every CTA of team 0
    if (kTrace && M.prof != nullptr && tid == 0 && tm.team == 0)
        trg = M.prof + 2 * kMaxProg + 64 + 2 * kMaxProg * 8 + (size_t)tm.cta * (kMaxProg * 2);

    uint32_t tile_ctr = 0;   // tiles reduced so far: the reducing warp rotates with it
    uint32_t pass_ctr = 0;   // passes so far: parity of the partial-sum buffer
    uint32_t cslot = 0, cpar = 0;   // ring slot and parity of the next stage this CTA consumes
    uint32_t mlp_par = 0;           // fused MLP: parity of the act barrier's next phase
    uint32_t psum_par = 0;          // fused MLP, split staging: parity of the psum barrier's next phase
    const int g = lane >> 2, c = lane & 3;
    uint32_t t_end = clock32_now();
    for (int it = 0; it < A.n_iter; ++it) {
        int step = 1;
#pragma unroll 1
        for (int p = 0; p < per_iter; p += step) {
            const uint32_t dsc = DSC0 + (uint32_t)p * (kDescWords * 4u);
            const uint32_t epoch = s_epoch0 + (uint32_t)(it * per_iter + p) + 1u;
            const uint4 d2 = lds_v4(dsc + 32u), d3 = lds_v4(dsc + 48u);
            const int kind = (int)(d3.x & 15u);
            // fused MLP: a W13 phase is always followed by its W2 phase, whose work it does -- the consumer warps skip that
            // phase (no descriptor, no barrier; t_end stays the W13 phase's end)
            step = (A.mlp_cluster > 0 && kind == PH_W13) ? 2 : 1;
            const bool fast = (d3.x >> 4) & 1u;
            const int layer = (int)((d3.x >> 8) & 255u), depth_pos = (int)((d3.x >> 16) & 255u);
            LL2_TRACE(0);
            if (kind == PH_ATTN) {
                phase_attn(M, A, tm, layer, p, epoch, SCR, SP.holdoff);
                t_end = clock32_now();
                LL2_TRACE(6);
                continue;
            }
            if (kind == PH_SAMPLE) {
                phase_sample(M, A, tm, fast ? 1 : 0, depth_pos, p, epoch, reinterpret_cast<float*>(smem_dyn + SP.scratch));
                t_end = clock32_now();
                LL2_TRACE(6);
                continue;
            }
            // ================= a phase that streams weights =================
            const uint4 d0 = lds_v4(dsc), d1 = lds_v4(dsc + 16u);
            const int K = (int)(d2.w & 0xffffu), n_items = (int)(d2.w >> 16);
            const int kb = K >> 5;
            const int src_kind = (int)((d2.z >> 8) & 15u), nrep = (int)((d2.z >> 12) & 63u);
            const bool do_gather = (d2.z >> 21) & 1u;
            const uint32_t psum = (d2.z >> 22) & 3u;   // input: a fused MLP's partial sums (1: gather_psum, 2: gather_psum_split)
            const uint32_t e_src = epoch - (d2.z & 255u);
            const uint32_t res = ((d2.z >> 20) & 1u) ? RESH : RESX;
            const bool normed = kind == PH_QKV || kind == PH_W13 || kind == PH_HEAD;
            const unsigned long long* src = reinterpret_cast<const unsigned long long*>((unsigned long long)d0.x | ((unsigned long long)d0.y << 32));
            const uint16_t* normw = reinterpret_cast<const uint16_t*>((unsigned long long)d0.z | ((unsigned long long)d0.w << 32));
            unsigned long long* out = reinterpret_cast<unsigned long long*>((unsigned long long)d1.x | ((unsigned long long)d1.y << 32));
            const unsigned long long aux = (unsigned long long)d1.z | ((unsigned long long)d1.w << 32);
            const int len_out = (int)(d3.w & 0xffffu), n_src = (int)(d3.w >> 16);
            const int i0 = (int)d3.y;
            const uint32_t mlp = kind == PH_W13 ? d3.z : 0u;   // fused MLP: lo | hi << 8 | n_units << 16 (0: unfused)
            const int mlp_lo = (int)(mlp & 255u), mlp_hi = (int)((mlp >> 8) & 255u);
            if (mlp != 0u && tid == 0) mbar_expect_tx(smem_u32(&s_actbar), (uint32_t)(mlp_hi - mlp_lo) * 64u);  // the slice's act, bf16

            const int Hq = fast ? M.fn_head : M.n_head, Hkv = fast ? M.fn_kv : M.n_kv;
            const int q_rows = Hq * kHeadDim, k_end = (Hq + Hkv) * kHeadDim;
            // slow layer 0 of a later frame: adopt the previous frame's ids and advance the position first (the RoPE row
            // prefetched below is the NEW position's)
            if (src_kind == 0 && it > 0) frame_boundary(M, A, tm, epoch - (uint32_t)per_iter);
            // Operands that do not depend on the input are loaded NOW (volatile: the compiler must not sink them below the
            // wait): the norm weights of the 4 elements this thread will normalise, and -- in the warp that will reduce the
            // phase's first tile -- the RoPE pair of its row.
            uint2 nw2[kNormPer];
#pragma unroll
            for (int q = 0; q < kNormPer; ++q) {
                nw2[q] = make_uint2(0u, 0u);
                if (normed && tid + q * kCons < K / 4) nw2[q] = ldnc_v2(normw + 4 * (tid + q * kCons));
            }
            uint32_t rope0 = 0u;
            if (kind == PH_QKV && n_items > 0 && warp == (int)(tile_ctr % kNW) && lane < 16) {
                const int n = i0 * 16 + lane;
                if (n < k_end) {
                    const uint16_t* table = reinterpret_cast<const uint16_t*>(aux) + (fast ? 0 : (size_t)min(s_pos, M.max_seq_len - 1) * kHeadDim);
                    rope0 = ldnc_u32(table + (n & (kHeadDim - 2)));
                }
            }
            if (kind == PH_HEAD && tid == 0) s_best = 0u;

            // ---- the phase's input vector -> xbuf -----------------------------------------------------------
            float ss = 0.f;
            if (src_kind != 3) {   // token embedding (slow layer 0) / embedding of the previous depth code: once per frame / depth step
                ss = stage_embedding(M, A, tm, src_kind, it, p, epoch, per_iter, depth_pos, K, reinterpret_cast<const uint16_t*>(src), XB, res);
            } else if (do_gather) {
                if (SP.holdoff > 0) { while (clock32_now() - t_end < (uint32_t)SP.holdoff) {} }
                if (kind == PH_WO && fast) fast_attention(M, layer, depth_pos, src, e_src, FQ, FKV, XB);
                else if (psum == 2u) {
                    ss = gather_psum_split(src, K, e_src, XB, (normed && kind != PH_HEAD) ? res : 0u, RESH, d3.z, A.mlp_cluster, psum_par);
                    psum_par ^= 1u;
                } else if (psum == 1u) ss = gather_psum(src, K, e_src, XB, (normed && kind != PH_HEAD) ? res : 0u, RESH);
                else ss = gather_words(src, n_src, e_src, XB, (normed && kind != PH_HEAD) ? res : 0u);
            }
            LL2_TRACE(1);
            if (normed) {
                ss = warp_sum(ss);
                if (lane == 0) s_ssq[warp] = ss;
            }
            csync();
            LL2_TRACE(2);
            if (n_items == 0) {
                if (kind == PH_HEAD && M.force == nullptr && (fast ? s_rs.fast_temp : s_rs.temp) == 0.0f && warp == 0 && lane < kLLRep)
                    st_relaxed_v2(cand_words(M, tm, fast ? 1 + depth_pos : 0, lane) + tm.cta, 0u, epoch);   // no rows here: the empty candidate
                t_end = clock32_now();
                LL2_TRACE(6);
                continue;
            }

            // ---- RMSNorm (P:601-613), in place: every thread normalises four elements of the staged row ------------------
            if (normed) {
                float t = 0.f;
#pragma unroll
                for (int w = 0; w < kNW; ++w) t = __fadd_rn(t, s_ssq[w]);
                const float mean = __fdiv_rn(t, (float)K);
                const float rr = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(mean, M.eps)));
#pragma unroll
                for (int q = 0; q < kNormPer; ++q) {
                    if (tid + q * kCons < K / 4) {
                        const uint32_t a = XB + (uint32_t)(tid + q * kCons) * 8u;
                        const uint32_t x0 = lds_u32(a), x1 = lds_u32(a + 4u);
                        const float o0 = bf16_round(__fmul_rn(bf16_round(__fmul_rn(bf_lo(x0), rr)), bf_lo(nw2[q].x)));
                        const float o1 = bf16_round(__fmul_rn(bf16_round(__fmul_rn(bf_hi(x0), rr)), bf_hi(nw2[q].x)));
                        const float o2 = bf16_round(__fmul_rn(bf16_round(__fmul_rn(bf_lo(x1), rr)), bf_lo(nw2[q].y)));
                        const float o3 = bf16_round(__fmul_rn(bf16_round(__fmul_rn(bf_hi(x1), rr)), bf_hi(nw2[q].y)));
                        sts_v2(a, pack_bf16(o0, o1), pack_bf16(o2, o3));
                    }
                }
                csync();
            }
            LL2_TRACE(3);
            if (fast && kind == PH_HEAD && depth_pos == M.depth - 1) __threadfence();  // release side of the once-per-frame fence

            // ---- tiles: 16 row slots x K on the tensor cores, K split over the warps ---------------------------------
            const int tiles = n_items, chunks = phase_chunks(K);
            // Tiles go through the tensor cores in PASSES of up to 4 (one-stage tiles, K <= 768): every warp carries its K slice
            // through all tiles of the pass (the B fragment is loaded once per k-block), then ONE barrier, then the tiles of the
            // pass are reduced / published by different warps at the same time.  Multi-stage tiles (K = 3072) go one per pass.
            // Ring stages are consumed strictly in order: (cslot, cpar) is the slot and parity of the next one.
#pragma unroll 1
            for (int t0 = 0; t0 < tiles;) {
                const int nt = chunks == 1 ? min(4, tiles - t0) : 1;
                const uint32_t pbuf = PART + (pass_ctr & 1u) * (uint32_t)(4 * kNW * 16 * 4);
                const uint32_t ringl = RING + (uint32_t)lane * 16u, xbl = XB + (uint32_t)c * 16u;
                const uint32_t pw = pbuf + (uint32_t)(warp * 16 + g) * 4u;
                if (chunks > 1) tile_pass_long(kb, chunks, warp, lane, full0, empty0, ringl, NSLOTS, xbl, pw, c == 0, cslot, cpar);
                else switch (nt) {
                    case 1: tile_pass<1>(kb, chunks, warp, lane, full0, empty0, ringl, NSLOTS, xbl, pw, c == 0, cslot, cpar); break;
                    case 2: tile_pass<2>(kb, chunks, warp, lane, full0, empty0, ringl, NSLOTS, xbl, pw, c == 0, cslot, cpar); break;
                    case 3: tile_pass<3>(kb, chunks, warp, lane, full0, empty0, ringl, NSLOTS, xbl, pw, c == 0, cslot, cpar); break;
                    default: tile_pass<4>(kb, chunks, warp, lane, full0, empty0, ringl, NSLOTS, xbl, pw, c == 0, cslot, cpar); break;
                }
                if (t0 + nt == tiles) LL2_TRACE(4);
                csync();
                if (t0 + nt == tiles) LL2_TRACE(5);
                const int ti = (warp + kNW - (int)(tile_ctr % kNW)) % kNW;   // tile of the pass this warp reduces (if < nt)
                if (ti < nt) {
                    const int t = t0 + ti;
                    const uint32_t pb = pbuf + (uint32_t)(ti * kNW * 16) * 4u;
                    // ---- reduction in warp order + epilogue + publish: lanes 0..15 = row slots ----
                    float v = 0.f;
                    if (lane < 16) {
#pragma unroll
                        for (int w = 0; w < kNW; ++w) v = __fadd_rn(v, lds_f32(pb + (uint32_t)(w * 16 + lane) * 4u));
                    }
                    int n = 0;          // output element this lane holds (row of the matrix / index of the act vector)
                    bool valid = false;
                    float val = 0.f;    // bf16-representable result
                    if (kind == PH_W13) {
                        const float up = __shfl_down_sync(0xffffffffu, v, 8);
                        n = (i0 + t) * 8 + lane;
                        valid = lane < 8;
                        const float a = bf16_round(v), gt = bf16_round(up);
                        const float sg = bf16_round(__fdiv_rn(a, __fadd_rn(1.0f, expf(-a))));  // F.silu in fp32, bf16 out (P:581)
                        val = bf16_round(__fmul_rn(sg, gt));
                    } else {
                        n = (i0 + t) * 16 + lane;
                        valid = lane < 16;
                        val = bf16_round(v);
                        if (kind == PH_QKV) {
                            const float other = __shfl_xor_sync(0xffffffffu, val, 1);
                            if (valid && n < k_end) {  // q and k rows: interleaved-pair RoPE with the bf16 table (P:616-640)
                                uint32_t cs = rope0;
                                if (t > 0) {
                                    const uint16_t* table = reinterpret_cast<const uint16_t*>(aux) + (fast ? 0 : (size_t)min(s_pos, M.max_seq_len - 1) * kHeadDim);
                                    cs = ldnc_u32(table + (n & (kHeadDim - 2)));
                                }
                                const float co = bf_lo(cs), si = bf_hi(cs);
                                val = (n & 1) ? bf16_round(__fadd_rn(__fmul_rn(val, co), __fmul_rn(other, si)))
                                              : bf16_round(__fsub_rn(__fmul_rn(val, co), __fmul_rn(other, si)));
                            }
                        } else if (kind == PH_WO || kind == PH_W2) {
                            // wo: h = x + wo(attn)  (P:499)      w2: x' = h + w2(act)  (P:500)
                            if (valid) {
                                const uint32_t pr = lds_u32(res + (uint32_t)(n & ~1) * 2u);
                                val = bf16_round(__fadd_rn((n & 1) ? bf_hi(pr) : bf_lo(pr), val));
                            }
                        } else if (kind == PH_HEAD) {
                            if (valid) {
                                reinterpret_cast<float*>(aux)[n] = val;
                                atomicMax(&s_best, cand_pack(val, n));
                            }
                        }
                    }
                    // words = pairs of adjacent lanes; nrep replicas: (word, replica) pairs spread over the lanes
                    const float nxt = __shfl_down_sync(0xffffffffu, val, 1);
                    const uint32_t word = pack_bf16(val, nxt);
                    if (kind == PH_QKV && !fast && valid && !(lane & 1) && n >= q_rows) kv_append(M, A, tm.team, layer, n, word);
                    if (mlp != 0u) {
                        // fused MLP: the tile's 8 act values (16 bytes) into every CTA of the cluster, lane r -> rank r
                        const uint32_t a0 = __shfl_sync(0xffffffffu, word, 0), a1 = __shfl_sync(0xffffffffu, word, 2);
                        const uint32_t a2 = __shfl_sync(0xffffffffu, word, 4), a3 = __shfl_sync(0xffffffffu, word, 6);
                        if (lane < A.mlp_cluster) {
                            const uint32_t dst = ACT + (uint32_t)(((i0 + t) * 8 - mlp_lo * 32) * 2);
                            st_async_v4(mapa(dst, (uint32_t)lane), a0, a1, a2, a3, mapa(smem_u32(&s_actbar), (uint32_t)lane));
                        }
                    } else {
#pragma unroll
                        for (int rnd = 0; rnd < 2; ++rnd) {
                            const int idx = lane + 32 * rnd;
                            const int wi = nrep == 1 ? idx : idx >> 3, rp = nrep == 1 ? 0 : idx & 7;
                            const int sl = 2 * (wi & 7);
                            const uint32_t wv = __shfl_sync(0xffffffffu, word, sl);
                            const int wn = __shfl_sync(0xffffffffu, n, sl);
                            const int wok = __shfl_sync(0xffffffffu, valid ? 1 : 0, sl);
                            if (wi < 8 && wok && (nrep > 1 || rnd == 0)) st_relaxed_v2(out + (size_t)rp * len_out + (wn >> 1), wv, epoch);
                        }
                    }
                }
                tile_ctr += (uint32_t)nt;
                pass_ctr += 1u;
                t0 += nt;
            }
            if (mlp != 0u) {
                // ---- fused MLP, w2 part: one warp per row tile replays warp `slice`'s MMA chain of the unfused K sweep ------
                const int nu = (int)(mlp >> 16), nkb = mlp_hi - mlp_lo, S = A.mlp_cluster, slice = tm.cta / S;
                const uint32_t dw = dsc + (uint32_t)(kDescWords * 4);   // the W2 phase's descriptor: region, row tile i0
                const uint4 w1 = lds_v4(dw + 16u), w3 = lds_v4(dw + 48u);
                unsigned long long* out2 = reinterpret_cast<unsigned long long*>((unsigned long long)w1.x | ((unsigned long long)w1.y << 32));
                const int len2 = (int)(w3.w & 0xffffu), D = (fast ? M.fdim : M.dim);
                mbar_wait(smem_u32(&s_actbar), mlp_par);   // the slice's act values from every CTA of the cluster
                mlp_par ^= 1u;
#pragma unroll 1
                for (int u = warp; u < nu; u += kNW) {
                    uint32_t sl = cslot + (uint32_t)u, pr = cpar;
                    while (sl >= NSLOTS) { sl -= NSLOTS; pr ^= 1u; }
                    mbar_wait(full0 + 8u * sl, pr);
                    const uint32_t ab = RING + sl * (uint32_t)kLL2SlotBytes + (uint32_t)lane * 16u, xb = ACT + (uint32_t)c * 16u;
                    float acc[4] = {0.f, 0.f, 0.f, 0.f}, acd[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
                    for (int j = 0; j < nkb; ++j) {
                        const uint4 bx = lds_v4(xb + (uint32_t)j * 64u);
                        const uint4 a0 = lds_v4(ab + (uint32_t)j * 1024u), a1 = lds_v4(ab + (uint32_t)j * 1024u + 512u);
                        mma_bf16_16816(acc, a0.x, a0.y, a0.z, a0.w, bx.x, bx.y);
                        mma_bf16_16816(acd, a1.x, a1.y, a1.z, a1.w, bx.z, bx.w);
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive_n(empty0 + 8u * sl, (uint32_t)kNW);   // the stage's only consumer
                    // partials of row slots g (acc[0] + acd[0]) and g + 8 (acc[2] + acd[2]), held by the lanes with c == 0:
                    // lane l publishes row slot l & 15 to replicas l >> 4, + 2, + 4, + 6
                    const float q0 = __fadd_rn(acc[0], acd[0]), q1 = __fadd_rn(acc[2], acd[2]);
                    const int rs = lane & 15;
                    const float qa = __shfl_sync(0xffffffffu, q0, (rs & 7) * 4), qb = __shfl_sync(0xffffffffu, q1, (rs & 7) * 4);
                    const uint32_t pv = __float_as_uint(rs < 8 ? qa : qb);
                    unsigned long long* o = out2 + slice * D + ((int)w3.y + u * S) * 16 + rs;   // w3.y = first row tile
#pragma unroll
                    for (int i = 0; i < kLLRep / 2; ++i) st_relaxed_v2(o + (size_t)((lane >> 4) + 2 * i) * len2, pv, epoch + 1u);
                }
                uint32_t sl = cslot + (uint32_t)nu;
                while (sl >= NSLOTS) { sl -= NSLOTS; cpar ^= 1u; }
                cslot = sl;
            }
            if (kind == PH_HEAD && M.force == nullptr && (fast ? s_rs.fast_temp : s_rs.temp) == 0.0f) {
                // greedy row: the CTA's best (logit, index) goes out as one word per replica
                csync();
                if (warp == 0 && lane < kLLRep)
                    st_relaxed_v2(cand_words(M, tm, fast ? 1 + depth_pos : 0, lane) + tm.cta, s_best, epoch);
            }
            t_end = clock32_now();
            LL2_TRACE(6);
        }
    }
    if (blockIdx.x == 0 && tid == 0) *M.ll_epoch = s_epoch0 + (uint32_t)A.n_iter * (uint32_t)per_iter;
}

// ---- bind-time packing of a weight matrix into the tensor-core GEMV layout ------------------------------------------
// dst [tile][K / 32][step 2][lane 32][16 bytes]: the A fragment of lane (g = lane / 4, c = lane % 4) for MMA step s of the
// k-block = { lo[e], hi[e], lo[e + 2], hi[e + 2] } with e = 8 c + 4 s (element pairs) -- lo = row g of the tile's lower
// half, hi = row g of its upper half.  Plain matrix: tile t = rows 16 t .. 16 t + 15 (lower = first 8).  Gated MLP
// (b != nullptr): tile t = rows 8 t .. 8 t + 7 of w1 (lower) over the same rows of w3 (upper).
__global__ void smol_pack_kernel(uint16_t* dst, const uint16_t* a, const uint16_t* b, int rows, int K) {
    const int kbn = K / 32;
    const size_t tiles = (size_t)(b ? rows / 8 : rows / 16);
    const size_t chunks = tiles * kbn * 64;   // 16-byte pieces
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < chunks; i += (size_t)gridDim.x * blockDim.x) {
        const int lane = (int)(i & 31), step = (int)((i >> 5) & 1);
        const size_t rest = i >> 6;
        const int kbi = (int)(rest % kbn);
        const size_t tile = rest / kbn;
        const int g = lane >> 2, c = lane & 3;
        const uint16_t* lo = b ? a + (tile * 8 + g) * (size_t)K : a + (tile * 16 + g) * (size_t)K;
        const uint16_t* hi = b ? b + (tile * 8 + g) * (size_t)K : a + (tile * 16 + 8 + g) * (size_t)K;
        const int e = kbi * 32 + 8 * c + 4 * step;
        uint4 v;
        v.x = *reinterpret_cast<const uint32_t*>(lo + e);
        v.y = *reinterpret_cast<const uint32_t*>(hi + e);
        v.z = *reinterpret_cast<const uint32_t*>(lo + e + 2);
        v.w = *reinterpret_cast<const uint32_t*>(hi + e + 2);
        *reinterpret_cast<uint4*>(dst + i * 8) = v;
    }
}

}  // namespace ll2

// ---- host-side helpers (called from capi.cu) ------------------------------------------------------------------
cudaError_t ll2_pack_launch(uint16_t* dst, const uint16_t* a, const uint16_t* b, int rows, int K, cudaStream_t stream) {
    ll2::smol_pack_kernel<<<1024, 256, 0, stream>>>(dst, a, b, rows, K);
    return cudaGetLastError();
}

struct LL2Plan {
    ll2::SmemPlan sp;
    size_t smem;
};

// Shared-memory plan; smem == 0: this model does not fit the kernel.
bool ll2_plan(const DevModel& M, int holdoff, int flags, ll2::SmemPlan* sp, size_t* smem) {
    auto up = [](size_t v) { return (v + 127) / 128 * 128; };
    if (M.depth > kLL2Depth || M.n_rows > kMaxRows) return false;
    if (M.dim != M.fdim) return false;
    if (M.dim % 32 || M.inter % 32 || M.finter % 32) return false;
    if (M.dim > 768 || M.inter > 3072 || M.finter > 3072) return false;   // three B fragments per warp, kGather polls per thread
    if (M.vocab % 16 || M.codebook_size % 16 || M.dim % 16 || M.inter % 16 || M.finter % 16) return false;   // 16-row tiles
    if (M.vocab > ll2::kCons * ll2::kSampPer || M.codebook_size > ll2::kCons * ll2::kSampPer) return false;
    if (phases_per_frame(M.n_layer, M.n_flayer, M.depth) > kMaxProg / 2) return false;
    if (M.max_seq_len > ll2::kMaxBlocks * kLL2AttnBlock) return false;
    const int kmax = M.inter > M.finter ? M.inter : M.finter;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off = up(off + bytes); return (int)o; };
    sp->xbuf = take((size_t)(kmax > M.dim ? kmax : M.dim) * 2);
    sp->res_x = take((size_t)M.dim * 2);
    sp->res_h = take((size_t)M.dim * 2);
    sp->part = take((size_t)2 * 4 * ll2::kNW * 16 * 4);
    sp->desc = take((size_t)phases_per_frame(M.n_layer, M.n_flayer, M.depth) * ll2::kDescWords * 4);
    sp->fq = take((size_t)M.fdim * 2);
    sp->fkv = take((size_t)M.n_flayer * kLL2Depth * 2 * M.fn_kv * kHeadDim * 2);
    const int nl = M.vocab > M.codebook_size ? M.vocab : M.codebook_size;
    const int lmax = (M.max_seq_len + kLL2AttnBlock - 1) / kLL2AttnBlock * kLL2AttnBlock;
    size_t sc = (size_t)nl * 4;
    const size_t attn = (size_t)lmax * 4 + (size_t)(lmax / kLL2ScoreBlock) * 9 * 4;
    if (attn > sc) sc = attn;
    sp->scratch = take(sc);
    sp->act = take((size_t)((kmax / 32 + ll2::kNW - 1) / ll2::kNW) * 32 * 2);   // the largest K-slice of act (fused MLP)
    off = (off + 1023) / 1024 * 1024;
    sp->ring = (int)off;
    const size_t budget = 227 * 1024 - 4096;   // static shared memory (barriers, sampler scratch, state) stays below 4 KB
    if (off + 4 * (size_t)kLL2SlotBytes > budget) return false;   // a K = 3072 tile holds four stages at once
    int n_slots = (int)((budget - off) / kLL2SlotBytes);
    if (n_slots > ll2::kMaxSlots) n_slots = ll2::kMaxSlots;
    sp->n_slots = n_slots;
    sp->holdoff = holdoff;
    sp->flags = flags;
    *smem = off + (size_t)n_slots * kLL2SlotBytes;
    return true;
}

static size_t g_ll2_smem_configured = 0;
cudaError_t ll2_configure(size_t smem) {
    if (smem <= g_ll2_smem_configured) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(ll2::smol_ll2_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(ll2::smol_ll2_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) g_ll2_smem_configured = smem;
    return e;
}
cudaError_t ll2_max_ctas(size_t smem, int* per_sm) {
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, ll2::smol_ll2_kernel<true>, kLL2Threads, smem);
}
// Cluster size of the fused gated MLP: the largest S <= 16 with at least 7 co-resident clusters of S CTAs (one per K-slice;
// an 8th is taken when it fits: it idles in the MLP phases but gives the other phases a larger grid).  S is also bounded so
// that every CTA of a slice cluster has a w13 tile and a w2 row tile in every layer: each CTA then both sends act values
// and waits for them, which keeps consecutive layers' DSMEM hand-offs from overlapping (one act buffer, one barrier).
// Returns 0 when no cluster size fits (the kernel then runs the unfused program).
int ll2_mlp_cluster(const DevModel& M, size_t smem, int n_slots, int* n_clusters) {
    *n_clusters = 0;
    int smax = 16;
    smax = std::min(smax, std::min(M.dim, M.fdim) / 16);
    smax = std::min(smax, 4 * ((std::min(M.inter, M.finter) / 32) / ll2::kNW));
    // a CTA's w2 row tiles: one warp and one ring stage each, all stages in the ring at once (a warp waits on stage
    // cslot + u with its parity: safe only while no two of them share a slot)
    const int rt = M.dim / 16, max_units = std::min(ll2::kNW, n_slots);
    int smin = (rt + max_units - 1) / max_units;
    const void* fns[2] = {(const void*)ll2::smol_ll2_kernel<false>, (const void*)ll2::smol_ll2_kernel<true>};
    for (const void* fn : fns)
        if (cudaFuncSetAttribute(fn, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
    for (int S = smax; S >= smin && S >= 1; --S) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(8 * S);
        cfg.blockDim = dim3(kLL2Threads);
        cfg.dynamicSmemBytes = smem;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = S; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, fns[1], &cfg) != cudaSuccess) { (void)cudaGetLastError(); continue; }
        if (n >= ll2::kNW) {
            *n_clusters = std::min(n, ll2::kNW + 1);
            return S;
        }
    }
    return 0;
}

cudaError_t ll2_launch(const DevModel& M, const CallArgs& A, const ll2::SmemPlan& sp, size_t smem, int n_ctas, cudaStream_t stream) {
    void* args[3] = {(void*)&M, (void*)&A, (void*)&sp};
    const void* fn = M.prof != nullptr ? (const void*)ll2::smol_ll2_kernel<true> : (const void*)ll2::smol_ll2_kernel<false>;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(n_ctas);
    cfg.blockDim = dim3(kLL2Threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeCooperative;   // only for the co-residency guarantee: CTAs spin on each other's words
    at[0].val.cooperative = 1;
    cfg.numAttrs = 1;
    if (A.mlp_cluster > 0) {
        at[1].id = cudaLaunchAttributeClusterDimension;
        at[1].val.clusterDim.x = A.mlp_cluster; at[1].val.clusterDim.y = 1; at[1].val.clusterDim.z = 1;
        cfg.numAttrs = 2;
    }
    cfg.attrs = at;
    return cudaLaunchKernelExC(&cfg, fn, args);
}

}  // namespace smol
