// Device-visible description of one bound model: shapes, borrowed weight pointers and the
// activation workspace carved out of the caller's buffer.  Uploaded once (capi.cu) and read by
// every CTA of the decode kernel through a const pointer.
#pragma once

#include <stdint.h>

#include "../../include/smoltts_b200.h"

namespace smol {

constexpr int kThreads = 512;          // 16 warps per CTA, one CTA per SM
constexpr int kWarps = kThreads / 32;
constexpr int kBatchTile = 8;          // sequences whose activations sit in shared memory at once
constexpr int kMaxSplits = 32;         // split-KV partials per (sequence, kv head)
constexpr int kSplitMin = 64;          // minimum positions per split
constexpr int kMaxGroup = 4;           // q heads per kv head
constexpr int kMaxDepth = 16;          // depth positions of the fast transformer
constexpr int kPartialStride = 66;     // (m, l, o[64]) per attention partial
constexpr int kMaxProg = 512;          // phases of one frame's program
constexpr int kMaxRows = kMaxDepth + 1; // rows of one token column

// ---- data-flow ("LL") decode kernel (ll2_kernel.cu): tensor-core GEMV, one team of CTAs per sequence ----
constexpr int kLLRep = 8;              // replicas of every broadcast vector (spreads the polls over L2 slices)
constexpr int kLLMaxCtas = 256;        // token words are published once per CTA
#ifndef LL2_WARPS
#define LL2_WARPS 7
#endif
constexpr int kLL2Warps = LL2_WARPS;     // consumer warps; one more warp streams the weights.  8 warps in all = 2 per scheduler: up to
                                         // 255 registers per thread (a 9th warp caps the kernel at 168 and the main loop spills -- a
                                         // spill is an L2 round trip here, the L1 being what 220 KB of shared memory leave).  Measured
                                         // A/B (build parameter): 4 consumer warps 722 us per frame, 7 consumer warps 660 us
constexpr int kLL2Threads = (kLL2Warps + 1) * 32;
constexpr int kLL2MaxTeams = 8;          // sequences one launch can carry (one team of CTAs each)
constexpr int kLL2ChunkKb = 24;          // k-blocks (of 32 elements) per ring stage
constexpr int kLL2SlotBytes = 2 * kLL2ChunkKb * 512;  // one ring slot: a tile of 2 x 8 rows x 24 k-blocks = 24 KB
constexpr int kLL2ScoreBlock = 64;       // cached positions per attention score unit
constexpr int kLL2AttnBlock = 512;       // positions per softmax block (the reference's CPU SDPA kernel: kvSplitSize)
constexpr int kLL2PvDims = 8;            // head dims per PV unit
constexpr int kLL2Depth = 8;             // depth positions whose K/V the kernel keeps in shared memory

struct LL2SmemPlan {   // second-generation data-flow kernel: byte offsets into dynamic shared memory + launch-time knobs
    int xbuf, res_x, res_h, part, desc, fq, fkv, scratch, act, ring;   // act: the fused MLP's K-slice of act (DSMEM)
    int n_slots;
    int holdoff;       // cycles between the end of a phase and the first poll of the next
};

struct DevLayer {
    const uint16_t* wqkv;
    const uint16_t* wo;
    const uint16_t* w1;
    const uint16_t* w3;
    const uint16_t* w2;
    const uint16_t* attention_norm;
    const uint16_t* ffn_norm;
    // tensor-core GEMV layout of the same matrices (ll2_kernel.cu; packed at bind time into the workspace):
    // [tile of 16 rows][K / 32][MMA step][lane][16 bytes = the lane's A fragment]; a pk_w13 tile is 8 rows of w1 over
    // the same 8 rows of w3
    const uint16_t* pk_wqkv;
    const uint16_t* pk_wo;
    const uint16_t* pk_w13;
    const uint16_t* pk_w2;
};

struct DevModel {
    // shapes (RQTransformerModelArgs)
    int dim, n_layer, n_head, n_kv, inter, vocab;
    int fdim, n_flayer, fn_head, fn_kv, finter;
    int codebook_size, num_codebooks, depth, n_rows;  // depth = max_fast_seqlen, n_rows = 1 + depth
    int dup0, depthwise_wte, depthwise_output;
    int max_seq_len, max_batch, page_size;
    int semantic_start, semantic_end, im_end;
    int mlx_embed_mask;
    float eps;

    // weights (borrowed, bf16 as raw 16-bit)
    const uint16_t* embeddings;
    const uint16_t* codebook_embeddings;
    const uint16_t* norm;
    const uint16_t* head;  // output.weight or the tied embeddings
    const uint16_t* fast_embeddings;
    const uint16_t* fast_norm;
    const uint16_t* fast_output;
    const uint16_t* rope;       // [max_seq_len][32][2]
    const uint16_t* fast_rope;  // [depth][32][2]
    DevLayer layers[SMOL_MAX_LAYERS];
    DevLayer fast_layers[SMOL_MAX_FAST_LAYERS];

    // paged KV pool  [n_pages][n_layer][2][n_kv][page_size][64] bf16
    uint16_t* kv_pool;
    int n_pages;

    // workspace (all [max_batch, ...])
    uint16_t* x;        // slow residual stream            [B][dim]
    uint16_t* h;        // post-attention stream (slow+fast) [B][max(dim,fdim)]
    uint16_t* xf;       // fast residual stream            [B][fdim]
    uint16_t* q;        // rotated queries                 [B][max(n_head,fn_head)*64]
    uint16_t* attn;     // attention output                [B][max(dim,fdim)]
    uint16_t* act;      // silu(w1 x) * w3 x               [B][max(inter,finter)]
    uint16_t* xn;       // tensor-core variant: RMSNorm output feeding the next weight phase  [B][max(dim,fdim)]
    const uint16_t* silu_lut;  // bf16 silu of every bf16 input [65536] (exact expression, filled at bind time)
    const unsigned char* tmaps;  // tensor-core variant: TMA tensor maps (128 B each, TensorMapSlot), in the workspace
    float* kpart;       // tensor-core variant: split-K partial sums of the wo / w2 tiles  [kTcKSplit][ws_rows][max(dim,fdim)] fp32
    int ws_rows;        // rows of every workspace buffer
    uint16_t* fkv;      // fast KV  [B][n_flayer][2][depth][fn_kv*64]
    float* token_logits;  // [B][vocab]           (bf16-rounded values)
    float* depth_logits;  // [B][depth][codebook] (bf16-rounded values)
    int32_t* frame_tokens;  // [B][n_rows] ids chosen in the current frame
    float* partial;       // [B][n_head][kMaxSplits][66]
    uint32_t* split_count;  // [B][n_kv]
    uint32_t* barrier;    // [0] arrivals, [1] base of the next launch
    uint32_t prog[kMaxProg];   // the frame's phase program, packed (pack_phase), built on the host
    unsigned long long* prof;  // optional [2 * phases_per_frame] ns accumulators (CTA 0: work, barrier wait)
    const int32_t* force; // optional [B][n_rows] ids that override the sampled ones (teacher forcing)
    unsigned long long* frame_ns;  // optional [frame_ns_cap]: %globaltimer at the end of every frame of sequence 0
    int frame_ns_cap;

    // data-flow kernel: every phase publishes its output as 8-byte words {payload, epoch} that the
    // consumers poll ("LL" protocol: the flag travels with the data, no barrier, no fence)
    unsigned long long* ll;          // phase p, sequence b, replica r: ll + ll_off[p] + (b * kLLRep + r) * ll_len[p]
    uint32_t* ll_epoch;              // [0] phases executed by earlier launches (epochs never repeat)
    uint32_t ll_off[kMaxProg];
    uint16_t ll_len[kMaxProg];

    const uint16_t* pk_head;         // packed LM head
    const uint16_t* pk_fast_output;  // packed depth heads (row groups in checkpoint order)
    unsigned long long* ll2_score;   // attention scores {fp32 bits, epoch} [teams][2][n_head][ll2_score_len] words
    unsigned long long* ll2_tok;     // sampled ids [teams][n_rows][kLLMaxCtas] words
    unsigned long long* ll2_cand;    // greedy candidates [teams][n_rows][kLLRep][kLLMaxCtas] words
    int ll2_score_len;
    unsigned long long* ll2_psum;    // fused MLP (batch 1): fp32 partial sums of the W2 phases {fp32 bits, epoch}
                                     // [W2 phase][kLLRep][7 K-slices][dim] words (ll2_kernel.cu: psum_region)
};

// Words (8 bytes, two bf16 + epoch) one sequence publishes in a phase; multiples of 16 words (128 B).
__host__ __device__ inline int ll_phase_words(int kind, int dim, int n_head, int n_kv, int inter, int n_out) {
    int n = 0;
    switch (kind) {
        case 0: n = (n_head + 2 * n_kv) * 64 / 2; break;  // PH_QKV
        case 1: n = dim / 2; break;                      // PH_ATTN (attention output)
        case 2: n = dim / 2; break;                      // PH_WO
        case 3: n = inter / 2; break;                    // PH_W13
        case 4: n = dim / 2; break;                      // PH_W2 (the fused MLP's partial sums: ll2_psum)
        case 5: n = n_out / 2; break;                    // PH_HEAD
        default: n = 0; break;
    }
    return (n + 15) / 16 * 16;
}

// Per-launch arguments (passed by value).
struct CallArgs {
    SmolBatch b;
    SmolSampling s;
    int batch;
    int prefill;      // 0 decode frames, 1 prefill steps
    int n_iter;       // frames (decode) or prompt positions (prefill) in this launch
    int iter_base;    // prefill: prompt position of iteration 0
    int finalize;     // prefill: this launch ends the prompt -> publish the last column as pending input
    int phase_begin;  // phases [begin, end) of every iteration
    int phase_end;
    int advance;      // slow-only launches: bump seq_len after the last phase
    int fast_from_xf; // depth-step launches: layer 0 reads the caller-filled xf buffer
    int repeat;       // profiling only: run the body of every weight phase 1 + repeat times
    int tile_t;       // prefill: prompt positions handled per iteration (rows = real_batch * tile_t share the weight pass)
    int real_batch;   // prefill: sequences (rows / tile_t)
    int tc_split;     // tensor-core variant: cached positions per attention split (0 = default)
    int team_ctas;    // second-generation data-flow kernel: CTAs per sequence (one team each); grid = batch * team_ctas
    int mlp_cluster;  // data-flow kernel, batch 1: CTAs per thread-block cluster of the fused gated MLP (0 = unfused)
    const int32_t* prompt;      // prefill: [B][n_rows][s_max]
    const int32_t* prompt_len;  // prefill: [B]
    int s_max;
};

// Phase kinds of one decode frame, in program order.
enum PhaseKind {
    PH_QKV = 0,   // [embed] + RMSNorm + wqkv + RoPE + KV append
    PH_ATTN,      // paged split-KV attention (slow layers only)
    PH_WO,        // [fast: attention over <= depth positions] + wo + residual
    PH_W13,       // RMSNorm + w1/w3 + silu*mul
    PH_W2,        // w2 + residual
    PH_HEAD,      // final norm + LM head / depth head
    PH_SAMPLE     // argmax / sampling (+ frame assembly after the last depth code)
};

struct Phase {
    int kind;
    int fast;   // 0 slow, 1 fast
    int layer;
    int depth_pos;
};

__host__ __device__ inline int phases_per_frame(int n_layer, int n_flayer, int depth) {
    return 5 * n_layer + 2 + depth * (4 * n_flayer + 2);
}
__host__ __device__ inline int phases_per_prefill_step(int n_layer) { return 5 * n_layer; }

__host__ __device__ inline Phase decode_phase(int p, int n_layer, int n_flayer) {
    Phase ph;
    ph.fast = 0; ph.layer = 0; ph.depth_pos = 0; ph.kind = PH_QKV;
    const int n_slow = 5 * n_layer;
    if (p < n_slow) {
        ph.layer = p / 5;
        ph.kind = p % 5;
        return ph;
    }
    if (p == n_slow) { ph.kind = PH_HEAD; return ph; }
    if (p == n_slow + 1) { ph.kind = PH_SAMPLE; return ph; }
    const int q = p - (n_slow + 2);
    const int per = 4 * n_flayer + 2;
    ph.fast = 1;
    ph.depth_pos = q / per;
    const int r = q % per;
    if (r < 4 * n_flayer) {
        ph.layer = r / 4;
        const int k = r % 4;
        ph.kind = (k == 0) ? PH_QKV : (k == 1) ? PH_WO : (k == 2) ? PH_W13 : PH_W2;
    } else if (r == 4 * n_flayer) {
        ph.kind = PH_HEAD;
    } else {
        ph.kind = PH_SAMPLE;
    }
    return ph;
}

// Tensor-core variant: phases that start with a grid-wide pre-step (embedding / input gather + RMSNorm into xn, or the
// depth attention) -- every weight phase except the slow wo and the w2's, whose inputs the previous phase left in place.
__host__ __device__ inline bool tc_has_prestep(const Phase& ph) {
    if (ph.kind == PH_ATTN || ph.kind == PH_SAMPLE) return false;
    return !(ph.kind == PH_W2 || (ph.kind == PH_WO && !ph.fast));
}

// Slots of the tensor-map table (DevModel.tmaps).  Activations: boxes of 128 rows (slots 0-5), 64 rows (6-11: batches of
// at most 64 rows load half a tile) and 32 rows (12-17).  Weights: one map per matrix and box height 16 * (v + 1) rows,
// v = 0..5, so that a tile's weight rows are ONE copy per stage (a TMA instruction costs its issuing thread ~60 ns).
enum TensorMapSlot {
    TM_XN_S = 0, TM_XN_F, TM_ATTN_S, TM_ATTN_F, TM_ACT_S, TM_ACT_F, TM_ACT_MAPS = 6, TM_WEIGHTS = 18
};
constexpr int kTmWeightBoxes = 6;
constexpr int kTmWeightStride = 2 + 5 * (SMOL_MAX_LAYERS + SMOL_MAX_FAST_LAYERS);  // weight matrices a model can have
constexpr int kTmTotal = TM_WEIGHTS + kTmWeightBoxes * kTmWeightStride;
// weight index: 0 LM head, 1 depth heads, then 5 per layer (wqkv, wo, w1, w3, w2): slow layers first, fast layers after them
__host__ __device__ inline int tm_weight_index(int n_layer, int fast, int layer, int which) {
    return 2 + ((fast ? n_layer : 0) + layer) * 5 + which;
}
__host__ __device__ inline int tm_weight_slot(int weight_index, int box_rows) {
    return TM_WEIGHTS + (box_rows / 16 - 1) * kTmWeightStride + weight_index;
}
constexpr int kTensorMapBytes = 128;
constexpr int kTcKSplit = 4;  // K slices of the wo / w2 tiles (their sum + residual + next RMSNorm is the phase's post-step)

__host__ __device__ inline uint32_t pack_phase(const Phase& ph) {
    return (uint32_t)ph.kind | ((uint32_t)ph.fast << 4) | ((uint32_t)ph.layer << 8) | ((uint32_t)ph.depth_pos << 16);
}
__host__ __device__ inline Phase unpack_phase(uint32_t w) {
    Phase ph;
    ph.kind = (int)(w & 15u); ph.fast = (int)((w >> 4) & 1u); ph.layer = (int)((w >> 8) & 255u); ph.depth_pos = (int)((w >> 16) & 255u);
    return ph;
}

}  // namespace smol
