// C ABI of the B200 DualAR decode engine (include/smoltts_b200.h).  Host-side only: shape checks,
// workspace carving, launch geometry and kernel selection (data-flow kernel / persistent cooperative
// barrier kernel).  No torch types, no allocation after create, no device synchronisation: every
// compute entry point only enqueues work on the caller's stream.

#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/smoltts_b200.h"
#include "dev_model.h"
#include "tmap_host.h"

namespace smol {
size_t decode_xs_bytes(const DevModel& M, int bt);
size_t decode_stage_bytes(const DevModel& M, int n_ctas);
int decode_batch_tile(int batch);
cudaError_t decode_configure(int bt, size_t smem);
cudaError_t decode_max_ctas(int bt, size_t smem, int* per_sm);
cudaError_t decode_launch(const DevModel& M, const CallArgs& A, int bt, int n_ctas, size_t smem, int xs_bytes,
                          cudaStream_t stream);
cudaError_t sample_launch(const float* logits, int n, int batch, const SmolSampling& s, const SmolRowSampling* table,
                          int stream_id, const int32_t* seq_id, const int32_t* step, int32_t* out, cudaStream_t stream);
cudaError_t store_codes_launch(int32_t* frame_tokens, const int32_t* codes, int batch, int n_rows, int row,
                               cudaStream_t stream);
cudaError_t silu_lut_launch(uint16_t* lut, cudaStream_t stream);
// data-flow kernel (ll2_kernel.cu)
namespace ll2 { using SmemPlan = LL2SmemPlan; }
bool ll2_plan(const DevModel& M, int holdoff, ll2::SmemPlan* sp, size_t* smem);
cudaError_t ll2_configure(size_t smem);
cudaError_t ll2_max_ctas(size_t smem, int* per_sm);
int ll2_mlp_cluster(const DevModel& M, size_t smem, int n_slots, int* n_clusters);
cudaError_t ll2_launch(const DevModel& M, const CallArgs& A, const ll2::SmemPlan& sp, size_t smem, int n_ctas, cudaStream_t stream);
cudaError_t ll2_pack_launch(uint16_t* dst, const uint16_t* a, const uint16_t* b, int rows, int K, cudaStream_t stream);
}  // namespace smol

using smol::CallArgs;
using smol::DevModel;

static_assert(sizeof(SmolRowSampling) == 32, "SmolRowSampling is 32 bytes (include/smoltts_b200.h)");

struct SmolModel {
    SmolConfig cfg;
    DevModel dm;
    bool weights_bound = false, ws_bound = false, kv_bound = false, configured = false;
    int device = 0, n_sms = 0, n_ctas = 0, n_ctas_override = 0;
    size_t smem[9] = {0}, xs_bytes[9] = {0};  // indexed by batch tile (1, 2, 4, 8)
    bool tile_ready[9] = {false};
    int mode = 2;
    int repeat = 0;
    int prefill_tile = 0;  // option: cap of prompt positions per prefill iteration (0 = as many as fit)
    int tc_attn_split = 0;  // option: cached positions per split of the batch attention (0 = the kernel's default)
    int tc_min_batch = 9;  // rows (sequences, or prompt positions of a prefill tile) from which the tcgen05 variant runs:
                           // measured crossover (150m, us per frame): bs 8: 2276 CUDA-core vs 2566 tensor-core; bs 12: 3642 vs 2577
    // data-flow kernel
    int ll2_state = 0;         // 0 unknown, 1 ready, -1 does not fit this model
    int ll2_holdoff = 400;     // option "ll_holdoff": cycles between the end of a phase and the first poll of the next
    int ll2_max_batch = 8;     // option: sequences (teams of CTAs) the kernel carries per launch; larger batches go to the
                               // barrier kernel / its tcgen05 variant (measured at bs=8: 1.5 ms per frame step against 2.3 ms)
    int ll2_fused_mlp = 1;     // option "ll_fused_mlp": batch 1 runs the gated MLP fused in thread-block clusters when they fit
    int ll2_cluster = 0;       // CTAs per cluster of the fused MLP (0: no cluster size fits this model / GPU)
    int ll2_clusters = 0;      // clusters of the fused grid
    int ll2_last_fused = 0;    // the last data-flow launch ran the fused MLP
    smol::ll2::SmemPlan ll2_sp;
    size_t ll2_smem = 0;
    bool packed_ready = false; // tensor-core GEMV layout of the bound weights (rebuilt after a weight / workspace bind)
    int64_t launches = 0;
    bool tmaps_ready = false;  // tensor maps of the tcgen05 variant (rebuilt after a weight / workspace bind)
};

static thread_local std::string g_err;

static int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
static int cuda_fail(cudaError_t e, const char* what) {
    (void)cudaGetLastError();  // launch-configuration errors are not sticky: do not leave them for the next caller
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return SMOL_ERR_CUDA;
}
namespace smol {
// the same error channel for the other translation units of the library (mimi_kernels.cu)
int capi_fail(int code, const std::string& msg) { return fail(code, msg); }
int capi_cuda_fail(cudaError_t e, const char* what) { return cuda_fail(e, what); }
}  // namespace smol
#define CU(call)                                         \
    do {                                                 \
        cudaError_t e__ = (call);                        \
        if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
    } while (0)

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static int imax(int a, int b) { return a > b ? a : b; }

struct WsLayout {
    size_t x, h, xf, q, attn, act, xn, silu_lut, tmaps, kpart, fkv, token_logits, depth_logits, frame_tokens, partial, split_count, barrier;
    size_t ll, ll_epoch, ll2_score, ll2_tok, ll2_cand, ll2_psum, packed, total;
};

// Word offsets of every phase's LL region for `bl` sequences x kLLRep replicas; returns the total words.
static size_t ll_regions(const SmolConfig& c, int depth, int bl, uint32_t* off, uint16_t* len) {
    const int n_prog = smol::phases_per_frame(c.n_layer, c.n_fast_layer, depth);
    size_t words = 0;
    for (int p = 0; p < n_prog; ++p) {
        const smol::Phase ph = smol::decode_phase(p, c.n_layer, c.n_fast_layer);
        const int n = ph.fast ? smol::ll_phase_words(ph.kind, c.fast_dim, c.fast_n_head, c.fast_n_local_heads,
                                                     c.fast_intermediate_size, c.codebook_size)
                              : smol::ll_phase_words(ph.kind, c.dim, c.n_head, c.n_local_heads, c.intermediate_size,
                                                     c.vocab_size);
        if (off) off[p] = (uint32_t)words;
        if (len) len[p] = (uint16_t)n;
        words += (size_t)n * bl * smol::kLLRep;
    }
    return words;
}

static int ll2_score_len(const SmolConfig& c) { return (c.max_seq_len + 511) / 512 * 512; }
// every GEMV matrix once more, in the tensor-core GEMV layout of the second-generation data-flow kernel
static size_t packed_bytes(const SmolConfig& c, int depth) {
    auto layer = [](size_t qkv_rows, size_t D, size_t F) { return (qkv_rows * D + D * D + 3 * D * F) * 2; };
    const size_t slow = layer((size_t)(c.n_head + 2 * c.n_local_heads) * 64, c.dim, c.intermediate_size);
    const size_t fast = layer((size_t)(c.fast_n_head + 2 * c.fast_n_local_heads) * 64, c.fast_dim, c.fast_intermediate_size);
    const size_t heads = ((size_t)c.vocab_size * c.dim + (size_t)c.codebook_size * (c.depthwise_output ? depth : 1) * c.fast_dim) * 2;
    return c.n_layer * align_up(slow, 256) + c.n_fast_layer * align_up(fast, 256) + align_up(heads, 256) + 4096;
}

// Rows of the activation workspace: a prefill iteration carries up to this many rows (sequences x prompt positions, eight
// 128-row tensor-core tiles).  An iteration costs about the same from 128 to 512 rows and ~1.4x at 1024 (it is bound by
// the per-phase fixed costs, DESIGN.md section 4), so the prompt of a batch of 256 is cached four positions at a time
// instead of one, that of a batch of 32 thirty-two at a time instead of four.  Costs ~0.4 GB of workspace.
constexpr int kPrefillRows = 1024;
static int ws_rows(const SmolConfig& c) { return c.max_batch > kPrefillRows ? c.max_batch : kPrefillRows; }

static WsLayout ws_layout(const SmolConfig& c, int depth) {
    WsLayout L;
    // rows: the batch, or one prefill tile of kPrefillRows prompt positions when the batch is smaller
    const size_t B = (size_t)ws_rows(c);
    size_t off = 0;
    auto take = [&](size_t bytes) {
        size_t o = off;
        off = align_up(off + bytes, 256);
        return o;
    };
    const int dmax = imax(c.dim, c.fast_dim);
    L.x = take(B * c.dim * 2);
    L.h = take(B * dmax * 2);
    L.xf = take(B * c.fast_dim * 2);
    L.q = take(B * imax(c.n_head, c.fast_n_head) * 64 * 2);
    L.attn = take(B * dmax * 2);
    L.act = take(B * imax(c.intermediate_size, c.fast_intermediate_size) * 2);
    L.xn = take(B * dmax * 2);
    L.silu_lut = take(65536 * 2);
    L.tmaps = take((size_t)smol::kTmTotal * smol::kTensorMapBytes);
    L.kpart = take((size_t)smol::kTcKSplit * B * dmax * 4);
    L.fkv = take(B * c.n_fast_layer * 2 * depth * c.fast_n_local_heads * 64 * 2);
    L.token_logits = take(B * c.vocab_size * 4);
    L.depth_logits = take(B * depth * c.codebook_size * 4);
    L.frame_tokens = take(B * (1 + depth) * 4);
    L.partial = take(B * c.n_head * smol::kMaxSplits * smol::kPartialStride * 4);
    L.split_count = take(B * c.n_local_heads * 4);
    L.barrier = take(256);
    const int bl = smol::kLL2MaxTeams;   // word regions for up to 8 teams
    L.ll = take(ll_regions(c, depth, bl, nullptr, nullptr) * 8);
    L.ll_epoch = take(256);
    L.ll2_score = take((size_t)bl * 2 * c.n_head * ll2_score_len(c) * 8);
    L.ll2_tok = take((size_t)bl * (1 + depth) * smol::kLLMaxCtas * 8);
    L.ll2_cand = take((size_t)bl * (1 + depth) * smol::kLLRep * smol::kLLMaxCtas * 8);
    // one sequence only: the fused MLP runs at batch 1
    L.ll2_psum = take((size_t)(c.n_layer + depth * c.n_fast_layer) * smol::kLLRep * smol::kLL2Warps * c.dim * 8);
    L.packed = take(packed_bytes(c, depth));
    L.total = off;
    return L;
}

static int depth_of(const SmolConfig& c) { return c.num_codebooks - (c.duplicate_code_0 ? 0 : 1); }

static int ensure_tmaps(SmolModel* m);
static int ensure_packed(SmolModel* m);

extern "C" {

int smol_abi_version(void) { return SMOL_ABI_VERSION; }
const char* smol_last_error(void) { return g_err.c_str(); }

int smol_create(const SmolConfig* cfg, SmolModel** out) {
    if (!cfg || !out) return fail(SMOL_ERR_INVALID, "smol_create: null argument");
    const SmolConfig& c = *cfg;
    auto bad = [&](const char* m) { return fail(SMOL_ERR_UNSUPPORTED, std::string("smol_create: ") + m); };
    if (c.dim <= 0 || c.n_layer <= 0 || c.n_head <= 0 || c.n_local_heads <= 0) return fail(SMOL_ERR_INVALID, "smol_create: bad shape");
    if (c.n_layer > SMOL_MAX_LAYERS || c.n_fast_layer > SMOL_MAX_FAST_LAYERS) return bad("too many layers");
    if (c.head_dim != 64 || c.fast_head_dim != 64) return bad("head_dim must be 64");
    if (c.dim != c.n_head * 64 || c.fast_dim != c.fast_n_head * 64) return bad("dim must equal n_head * 64");
    if (c.fast_dim != c.dim) return bad("fast_project_in (fast_dim != dim) is not on the built path");
    if (c.n_head % c.n_local_heads || c.fast_n_head % c.fast_n_local_heads) return bad("n_head must be a multiple of n_local_heads");
    if (c.n_head / c.n_local_heads > smol::kMaxGroup) return bad("more than 4 query heads per kv head");
    if (c.dim % 8 || c.intermediate_size % 8 || c.fast_intermediate_size % 8) return bad("dims must be multiples of 8");
    if (imax(imax(c.dim, c.intermediate_size), c.fast_intermediate_size) > 3072) return bad("reduction dims above 3072");
    if (c.dim > 768) return bad("model dim above 768");
    if (c.vocab_size > smol::kThreads * 8 || c.codebook_size > smol::kThreads * 8) return bad("vocab / codebook above 4096 rows");
    const int depth = depth_of(c);
    if (depth < 1 || depth > smol::kMaxDepth) return bad("depth out of range");
    if (c.max_batch <= 0 || c.max_seq_len <= 0) return fail(SMOL_ERR_INVALID, "smol_create: bad capacity");
    // the batch attention walks 16-position groups through a 32-entry page-id window: pages of 16 or 32 positions only
    if (c.page_size != 16 && c.page_size != 32) return fail(SMOL_ERR_INVALID, "smol_create: page_size must be 16 or 32");
    if (!c.tie_word_embeddings) { /* output.weight must be bound */ }

    SmolModel* m = new SmolModel();
    m->cfg = c;
    DevModel& d = m->dm;
    std::memset(&d, 0, sizeof(d));
    d.dim = c.dim; d.n_layer = c.n_layer; d.n_head = c.n_head; d.n_kv = c.n_local_heads; d.inter = c.intermediate_size;
    d.vocab = c.vocab_size;
    d.fdim = c.fast_dim; d.n_flayer = c.n_fast_layer; d.fn_head = c.fast_n_head; d.fn_kv = c.fast_n_local_heads;
    d.finter = c.fast_intermediate_size;
    d.codebook_size = c.codebook_size; d.num_codebooks = c.num_codebooks; d.depth = depth; d.n_rows = 1 + depth;
    d.dup0 = c.duplicate_code_0; d.depthwise_wte = c.depthwise_wte; d.depthwise_output = c.depthwise_output;
    d.max_seq_len = c.max_seq_len; d.max_batch = c.max_batch; d.page_size = c.page_size;
    d.semantic_start = c.semantic_start_id; d.semantic_end = c.semantic_end_id; d.im_end = c.im_end_id;
    d.mlx_embed_mask = c.mlx_embed_mask; d.eps = c.norm_eps;
    const int n_prog = smol::phases_per_frame(d.n_layer, d.n_flayer, d.depth);
    if (n_prog > smol::kMaxProg) { delete m; return bad("frame program longer than 512 phases"); }
    for (int p = 0; p < n_prog; ++p) d.prog[p] = smol::pack_phase(smol::decode_phase(p, d.n_layer, d.n_flayer));
    ll_regions(c, depth, smol::kLL2MaxTeams, d.ll_off, d.ll_len);
    *out = m;
    return SMOL_OK;
}

void smol_destroy(SmolModel* m) { delete m; }

int smol_bind_weights(SmolModel* m, const SmolWeights* w) {
    if (!m || !w) return fail(SMOL_ERR_INVALID, "smol_bind_weights: null argument");
    const SmolConfig& c = m->cfg;
    DevModel& d = m->dm;
    auto need = [&](const void* p, const char* name) {
        if (!p) { g_err = std::string("smol_bind_weights: missing ") + name; return false; }
        if (((uintptr_t)p) & 15) { g_err = std::string("smol_bind_weights: not 16-byte aligned: ") + name; return false; }
        return true;
    };
    if (!need(w->embeddings, "embeddings") || !need(w->codebook_embeddings, "codebook_embeddings") || !need(w->norm, "norm") ||
        !need(w->fast_embeddings, "fast_embeddings") || !need(w->fast_norm, "fast_norm") || !need(w->fast_output, "fast_output") ||
        !need(w->rope, "rope") || !need(w->fast_rope, "fast_rope"))
        return SMOL_ERR_INVALID;
    if (!c.tie_word_embeddings && !need(w->output, "output")) return SMOL_ERR_INVALID;
    auto u16 = [](const void* p) { return reinterpret_cast<const uint16_t*>(p); };
    d.embeddings = u16(w->embeddings); d.codebook_embeddings = u16(w->codebook_embeddings); d.norm = u16(w->norm);
    d.head = c.tie_word_embeddings ? u16(w->embeddings) : u16(w->output);
    d.fast_embeddings = u16(w->fast_embeddings); d.fast_norm = u16(w->fast_norm); d.fast_output = u16(w->fast_output);
    d.rope = u16(w->rope); d.fast_rope = u16(w->fast_rope);
    auto bind_layer = [&](const SmolLayerWeights& s, smol::DevLayer& t, const char* what) {
        if (!need(s.wqkv, what) || !need(s.wo, what) || !need(s.w1, what) || !need(s.w3, what) || !need(s.w2, what) ||
            !need(s.attention_norm, what) || !need(s.ffn_norm, what))
            return false;
        t.wqkv = u16(s.wqkv); t.wo = u16(s.wo); t.w1 = u16(s.w1); t.w3 = u16(s.w3); t.w2 = u16(s.w2);
        t.attention_norm = u16(s.attention_norm); t.ffn_norm = u16(s.ffn_norm);
        return true;
    };
    for (int l = 0; l < c.n_layer; ++l)
        if (!bind_layer(w->layers[l], d.layers[l], "layers[*]")) return SMOL_ERR_INVALID;
    for (int l = 0; l < c.n_fast_layer; ++l)
        if (!bind_layer(w->fast_layers[l], d.fast_layers[l], "fast_layers[*]")) return SMOL_ERR_INVALID;
    m->weights_bound = true;
    m->tmaps_ready = false;
    m->packed_ready = false;
    // tensor maps and the packed GEMV layout are built here, at setup time: compute calls stay asynchronous and capturable
    if (m->ws_bound) {
        const int rc = ensure_tmaps(m);
        return rc ? rc : ensure_packed(m);
    }
    return SMOL_OK;
}

size_t smol_workspace_bytes(const SmolModel* m) {
    if (!m) return 0;
    return ws_layout(m->cfg, m->dm.depth).total;
}

int smol_bind_workspace(SmolModel* m, void* d_workspace, size_t bytes) {
    if (!m || !d_workspace) return fail(SMOL_ERR_INVALID, "smol_bind_workspace: null argument");
    const WsLayout L = ws_layout(m->cfg, m->dm.depth);
    if (bytes < L.total) return fail(SMOL_ERR_CAPACITY, "smol_bind_workspace: buffer smaller than smol_workspace_bytes()");
    if (((uintptr_t)d_workspace) & 255) return fail(SMOL_ERR_INVALID, "smol_bind_workspace: buffer must be 256-byte aligned");
    char* base = reinterpret_cast<char*>(d_workspace);
    DevModel& d = m->dm;
    d.x = (uint16_t*)(base + L.x); d.h = (uint16_t*)(base + L.h); d.xf = (uint16_t*)(base + L.xf);
    d.q = (uint16_t*)(base + L.q); d.attn = (uint16_t*)(base + L.attn); d.act = (uint16_t*)(base + L.act);
    d.fkv = (uint16_t*)(base + L.fkv);
    d.xn = (uint16_t*)(base + L.xn); d.tmaps = (const unsigned char*)(base + L.tmaps);
    d.silu_lut = (const uint16_t*)(base + L.silu_lut);
    CU(smol::silu_lut_launch((uint16_t*)(base + L.silu_lut), nullptr));  // setup-time (synchronous with the memsets below)
    d.kpart = (float*)(base + L.kpart); d.ws_rows = ws_rows(m->cfg);
    m->tmaps_ready = false;
    d.token_logits = (float*)(base + L.token_logits); d.depth_logits = (float*)(base + L.depth_logits);
    d.frame_tokens = (int32_t*)(base + L.frame_tokens);
    d.partial = (float*)(base + L.partial); d.split_count = (uint32_t*)(base + L.split_count);
    d.barrier = (uint32_t*)(base + L.barrier);
    d.ll = (unsigned long long*)(base + L.ll); d.ll_epoch = (uint32_t*)(base + L.ll_epoch);
    d.ll2_score = (unsigned long long*)(base + L.ll2_score); d.ll2_tok = (unsigned long long*)(base + L.ll2_tok);
    d.ll2_cand = (unsigned long long*)(base + L.ll2_cand); d.ll2_score_len = ll2_score_len(m->cfg);
    d.ll2_psum = (unsigned long long*)(base + L.ll2_psum);
    m->packed_ready = false;
    // split counters, barrier words and every LL word (epoch 0 = never written) must start at zero
    // (setup-time, synchronous)
    CU(cudaMemset(base + L.split_count, 0, L.packed - L.split_count));
    CU(cudaMemset(base + L.frame_tokens, 0, L.partial - L.frame_tokens));
    m->ws_bound = true;
    if (m->weights_bound) {
        const int rc = ensure_tmaps(m);
        return rc ? rc : ensure_packed(m);
    }
    return SMOL_OK;
}

size_t smol_kv_page_bytes(const SmolModel* m) {
    if (!m) return 0;
    return (size_t)m->cfg.n_layer * 2 * m->cfg.n_local_heads * m->cfg.page_size * 64 * 2;
}

int smol_kv_bind(SmolModel* m, void* d_kv_pool, int32_t n_pages) {
    if (!m || !d_kv_pool || n_pages <= 0) return fail(SMOL_ERR_INVALID, "smol_kv_bind: bad argument");
    if (((uintptr_t)d_kv_pool) & 15) return fail(SMOL_ERR_INVALID, "smol_kv_bind: pool must be 16-byte aligned");
    m->dm.kv_pool = reinterpret_cast<uint16_t*>(d_kv_pool);
    m->dm.n_pages = n_pages;
    m->kv_bound = true;
    return SMOL_OK;
}

}  // extern "C"

// ---- launch plumbing -------------------------------------------------------------------------------
static int ensure_configured(SmolModel* m) {
    if (!m->weights_bound || !m->ws_bound || !m->kv_bound)
        return fail(SMOL_ERR_UNBOUND, "weights, workspace and KV pool must be bound before compute calls");
    if (m->configured) return SMOL_OK;
    CU(cudaGetDevice(&m->device));
    int coop = 0;
    CU(cudaDeviceGetAttribute(&m->n_sms, cudaDevAttrMultiProcessorCount, m->device));
    CU(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, m->device));
    if (!coop) return fail(SMOL_ERR_UNSUPPORTED, "device does not support cooperative launch");
    m->n_ctas = m->n_sms;
    if (m->n_ctas_override > 0 && m->n_ctas_override < m->n_ctas) m->n_ctas = m->n_ctas_override;
    for (int i = 0; i < 9; ++i) m->tile_ready[i] = false;
    if (m->ll2_state > 0) m->ll2_state = 0;
    m->configured = true;
    return SMOL_OK;
}

// TMA tensor maps of the tcgen05 variant: encoded on the host and copied into the workspace once per bind (setup-time,
// synchronous; compute calls never come here again).
static bool tc_eligible(const SmolConfig& c) {  // the tiles stream K in 64-element stages
    return (c.dim % 64) == 0 && (c.fast_dim % 64) == 0 && (c.intermediate_size % 64) == 0 && (c.fast_intermediate_size % 64) == 0;
}

static int ensure_tmaps(SmolModel* m) {
    if (m->tmaps_ready) return SMOL_OK;
    const SmolConfig& c = m->cfg;
    if (!tc_eligible(c)) { m->tmaps_ready = true; return SMOL_OK; }  // such a model stays on the CUDA-core variants
    const DevModel& d = m->dm;
    const int n_slots = smol::kTmTotal;
    std::vector<CUtensorMap> maps((size_t)n_slots);
    std::memset(maps.data(), 0, maps.size() * sizeof(CUtensorMap));
    static_assert(sizeof(CUtensorMap) == smol::kTensorMapBytes, "tensor map size");
    const uint64_t rows = (uint64_t)ws_rows(c);
    const int dmax = imax(c.dim, c.fast_dim), fmax = imax(c.intermediate_size, c.fast_intermediate_size);
    bool ok = true;
    auto act = [&](int slot, const void* p, int K, int pitch) {
        for (int i = 0; i < 3; ++i)  // 128-, 64- and 32-row boxes
            ok = ok && smol::make_tensor_map_2d(&maps[slot + i * smol::TM_ACT_MAPS], p, rows, K, pitch, 128u >> i);
    };
    auto wgt = [&](int index, const void* p, uint64_t n, int K) {
        for (int box = 16; box <= 16 * smol::kTmWeightBoxes; box += 16)
            ok = ok && smol::make_tensor_map_2d(&maps[smol::tm_weight_slot(index, box)], p, n, K, K, (uint32_t)box);
    };
    act(smol::TM_XN_S, d.xn, c.dim, dmax);
    act(smol::TM_XN_F, d.xn, c.fast_dim, dmax);
    act(smol::TM_ATTN_S, d.attn, c.dim, dmax);
    act(smol::TM_ATTN_F, d.attn, c.fast_dim, dmax);
    act(smol::TM_ACT_S, d.act, c.intermediate_size, fmax);
    act(smol::TM_ACT_F, d.act, c.fast_intermediate_size, fmax);
    wgt(0, d.head, c.vocab_size, c.dim);
    wgt(1, d.fast_output, (uint64_t)c.codebook_size * (c.depthwise_output ? d.depth : 1), c.fast_dim);
    for (int f = 0; f < 2; ++f) {
        const int nl = f ? c.n_fast_layer : c.n_layer, D = f ? c.fast_dim : c.dim, F = f ? c.fast_intermediate_size : c.intermediate_size;
        const int qkv = ((f ? c.fast_n_head : c.n_head) + 2 * (f ? c.fast_n_local_heads : c.n_local_heads)) * 64;
        for (int l = 0; l < nl; ++l) {
            const smol::DevLayer& L = f ? d.fast_layers[l] : d.layers[l];
            wgt(smol::tm_weight_index(c.n_layer, f, l, 0), L.wqkv, qkv, D);
            wgt(smol::tm_weight_index(c.n_layer, f, l, 1), L.wo, D, D);
            wgt(smol::tm_weight_index(c.n_layer, f, l, 2), L.w1, F, D);
            wgt(smol::tm_weight_index(c.n_layer, f, l, 3), L.w3, F, D);
            wgt(smol::tm_weight_index(c.n_layer, f, l, 4), L.w2, D, F);
        }
    }
    if (!ok) return fail(SMOL_ERR_CUDA, "cuTensorMapEncodeTiled failed for the tensor-core variant's operands");
    CU(cudaMemcpy(const_cast<unsigned char*>(d.tmaps), maps.data(), (size_t)n_slots * smol::kTensorMapBytes, cudaMemcpyHostToDevice));
    m->tmaps_ready = true;
    return SMOL_OK;
}

// The bound weights once more in the tensor-core GEMV layout ([16-row tile][K / 32][MMA step][lane][16 B]: ll2_kernel.cu),
// written into the workspace by a device kernel at bind time (setup-time; the borrowed checkpoint tensors stay as they are
// for the other kernels).
static int ensure_packed(SmolModel* m) {
    if (m->packed_ready) return SMOL_OK;
    const SmolConfig& c = m->cfg;
    DevModel& d = m->dm;
    if (c.dim % 32 || c.fast_dim % 32 || c.intermediate_size % 32 || c.fast_intermediate_size % 32 || c.vocab_size % 16 || c.codebook_size % 16) {
        m->packed_ready = true;   // such a model stays on the other kernels (ll2_plan refuses it)
        m->ll2_state = -1;
        return SMOL_OK;
    }
    char* ws = reinterpret_cast<char*>(d.x) - ws_layout(c, d.depth).x;
    char* p = ws + ws_layout(c, d.depth).packed;
    auto put = [&](const uint16_t* a, const uint16_t* b, int rows, int K) -> const uint16_t* {
        uint16_t* dst = reinterpret_cast<uint16_t*>(p);
        p += align_up((size_t)rows * (b ? 2 : 1) * K * 2, 256);
        return smol::ll2_pack_launch(dst, a, b, rows, K, nullptr) == cudaSuccess ? dst : nullptr;
    };
    bool ok = true;
    for (int f = 0; f < 2; ++f) {
        const int nl = f ? c.n_fast_layer : c.n_layer, D = f ? c.fast_dim : c.dim, F = f ? c.fast_intermediate_size : c.intermediate_size;
        const int qkv = ((f ? c.fast_n_head : c.n_head) + 2 * (f ? c.fast_n_local_heads : c.n_local_heads)) * 64;
        for (int l = 0; l < nl; ++l) {
            smol::DevLayer& L = f ? d.fast_layers[l] : d.layers[l];
            L.pk_wqkv = put(L.wqkv, nullptr, qkv, D);
            L.pk_wo = put(L.wo, nullptr, D, D);
            L.pk_w13 = put(L.w1, L.w3, F, D);
            L.pk_w2 = put(L.w2, nullptr, D, F);
            ok = ok && L.pk_wqkv && L.pk_wo && L.pk_w13 && L.pk_w2;
        }
    }
    d.pk_head = put(d.head, nullptr, c.vocab_size, c.dim);
    d.pk_fast_output = put(d.fast_output, nullptr, c.codebook_size * (c.depthwise_output ? d.depth : 1), c.fast_dim);
    ok = ok && d.pk_head && d.pk_fast_output;
    if (!ok) return fail(SMOL_ERR_CUDA, "packing the weights for the data-flow kernel failed");
    CU(cudaDeviceSynchronize());   // setup-time only
    m->packed_ready = true;
    return SMOL_OK;
}

static int ensure_ll2(SmolModel* m) {
    if (m->ll2_state != 0) return SMOL_OK;
    m->ll2_sp = smol::ll2::SmemPlan();
    if (!smol::ll2_plan(m->dm, m->ll2_holdoff, &m->ll2_sp, &m->ll2_smem) || m->n_ctas > smol::kLLMaxCtas) { m->ll2_state = -1; return SMOL_OK; }
    CU(smol::ll2_configure(m->ll2_smem));
    int per_sm = 0;
    CU(smol::ll2_max_ctas(m->ll2_smem, &per_sm));
    m->ll2_state = per_sm >= 1 ? 1 : -1;
    if (m->ll2_state == 1) m->ll2_cluster = smol::ll2_mlp_cluster(m->dm, m->ll2_smem, m->ll2_sp.n_slots, &m->ll2_clusters);
    return SMOL_OK;
}

// Grid of the fused gated MLP for a solo decode (ll2_kernel.cu: build_desc): clusters of ll2_cluster CTAs, one per K-slice
// (+ one idle in the MLP when it fits).  An "n_ctas" override keeps it only when it is such a grid.  The fused and the
// unfused program compute the same bits, so every other case simply runs unfused.  Returns the cluster size, 0 = unfused.
static int ll2_fused_cluster(const SmolModel* m, int* n_ctas) {
    const int S = m->ll2_cluster;
    if (!m->ll2_fused_mlp || S <= 0) return 0;
    if (m->n_ctas_override <= 0) { *n_ctas = m->ll2_clusters * S; return S; }
    const int n = m->n_ctas;
    if (n % S || n / S < smol::kLL2Warps || n / S > m->ll2_clusters) return 0;
    *n_ctas = n;
    return S;
}

// Grid of a SOLO decode on the data-flow kernel.  An exchange has as many participants as the grid has CTAs, a phase takes as
// long as its busiest CTA.  Measured on 150m, 1024 frames (profiles/r2_ll2_grid_size_sweep.txt): 128 CTAs -- the gated-MLP
// phase's 384 tiles are 3 per CTA exactly, the same maximum as on 148 -- 617.5 us per frame, 148 CTAs 626.2, 136: 626.2, 120:
// 630.5; 70m (192 tiles): 148 = 128 = 593.5.  Rule: the largest grid within 15 % of the SM count that divides the gated-MLP
// tile count, else one CTA per SM.  Results do not depend on the grid (bit-identical, tests/test_gpu_ll2.py); the caller's
// "n_ctas" option overrides.
static int ll2_solo_ctas(const SmolModel* m) {
    if (m->n_ctas_override > 0 || m->n_ctas <= 0) return m->n_ctas;
    const int tiles = m->cfg.intermediate_size / 8;
    for (int n = m->n_ctas; n * 100 >= m->n_ctas * 85; --n)
        if (tiles % n == 0) return n;
    return m->n_ctas;
}

// Shared-memory budget and function attributes of the kernel variant for this batch tile.
static int ensure_tile(SmolModel* m, int bt) {
    if (bt == 0) {
        const int rc = ensure_tmaps(m);
        if (rc) return rc;
    }
    if (m->tile_ready[bt]) return SMOL_OK;
    m->xs_bytes[bt] = smol::decode_xs_bytes(m->dm, bt);
    m->smem[bt] = m->xs_bytes[bt] + (bt == 0 ? 0 : smol::decode_stage_bytes(m->dm, m->n_ctas));  // bt 0: tensor-core variant, ring only
    if (m->smem[bt] > 227 * 1024)
        return fail(SMOL_ERR_UNSUPPORTED, "activation tile + weight stage exceed 227 KB of shared memory");
    CU(smol::decode_configure(bt, m->smem[bt]));
    int per_sm = 0;
    CU(smol::decode_max_ctas(bt, m->smem[bt], &per_sm));
    if (per_sm < 1) return fail(SMOL_ERR_UNSUPPORTED, "decode kernel does not fit on an SM");
    m->tile_ready[bt] = true;
    return SMOL_OK;
}

static int check_batch(const SmolModel* m, const SmolBatch* b, int batch) {
    if (!b) return fail(SMOL_ERR_INVALID, "null SmolBatch");
    if (batch <= 0 || batch > m->cfg.max_batch) return fail(SMOL_ERR_CAPACITY, "batch outside [1, max_batch]");
    if (!b->tokens || !b->seq_len || !b->block_table || b->max_pages <= 0)
        return fail(SMOL_ERR_INVALID, "SmolBatch needs tokens, seq_len and block_table");
    return SMOL_OK;
}

static bool use_tc(const SmolModel* m, int rows) {
    return m->tc_min_batch > 0 && rows >= m->tc_min_batch && tc_eligible(m->cfg);
}

// Enqueue `n_iter` iterations of phases [begin, end) as one launch: the data-flow kernel (mode 2, whole frames of at most
// ll_max_batch sequences) or the cooperative barrier kernel.
// whole_iters: the call runs complete frames / complete prefill positions (what the data-flow kernel carries).
static int enqueue(SmolModel* m, CallArgs A, cudaStream_t stream, bool whole_iters = false) {
    const int bt = use_tc(m, A.batch) ? 0 : smol::decode_batch_tile(A.batch);
    int rc;
    A.repeat = m->repeat;
    A.tc_split = m->tc_attn_split;
    if (m->mode == 2 && whole_iters && !A.prefill && A.batch <= m->ll2_max_batch && A.batch <= smol::kLL2MaxTeams &&
        A.batch <= m->n_ctas) {
        if ((rc = ensure_ll2(m))) return rc;
        if (m->ll2_state == 1) {
            if (A.n_iter == 0) return SMOL_OK;
            A.team_ctas = A.batch == 1 ? ll2_solo_ctas(m) : m->n_ctas / A.batch;
            A.mlp_cluster = A.batch == 1 ? ll2_fused_cluster(m, &A.team_ctas) : 0;
            m->ll2_last_fused = A.mlp_cluster > 0 ? 1 : 0;
            m->ll2_sp.holdoff = m->ll2_holdoff;
            CU(smol::ll2_launch(m->dm, A, m->ll2_sp, m->ll2_smem, A.team_ctas * A.batch, stream));
            m->launches += 1;
            return SMOL_OK;
        }
    }
    rc = ensure_tile(m, bt);
    if (rc) return rc;
    CU(smol::decode_launch(m->dm, A, bt, m->n_ctas, m->smem[bt], (int)m->xs_bytes[bt], stream));
    m->launches += 1;
    return SMOL_OK;
}

static CallArgs base_args(const SmolBatch* b, int batch, const SmolSampling* s) {
    CallArgs A;
    std::memset(&A, 0, sizeof(A));
    A.b = *b;
    if (s) A.s = *s;
    else { A.s.temp = 0.f; A.s.fast_temp = 0.f; A.s.top_p = 1.f; A.s.ignore_stop = 1; A.b.row_sampling = nullptr; }
    A.batch = batch;
    A.real_batch = batch;
    A.tile_t = 1;
    A.n_iter = 1;
    return A;
}

extern "C" {

int smol_prefill(SmolModel* m, const SmolBatch* b, int32_t batch, const int32_t* d_prompt,
                 const int32_t* d_prompt_len, int32_t s_max, void* stream) {
    if (!m) return fail(SMOL_ERR_INVALID, "null model");
    int rc = ensure_configured(m);
    if (rc) return rc;
    if ((rc = check_batch(m, b, batch))) return rc;
    if (!d_prompt || !d_prompt_len || s_max < 1) return fail(SMOL_ERR_INVALID, "smol_prefill: bad prompt");
    CallArgs A = base_args(b, batch, nullptr);
    A.prefill = 1;
    // tile_t prompt positions per iteration share one pass over the weights (rows = batch * tile_t fit the workspace)
    // -- up to kPrefillRows rows (128-row tensor-core tiles); 8 positions on the CUDA-core variants
    const int rows_cap = ws_rows(m->cfg);
    int T = rows_cap / batch;
    if (T > kPrefillRows) T = kPrefillRows;
    if (T > s_max - 1) T = s_max - 1;
    if (T < 1) T = 1;
    if (m->prefill_tile > 0 && m->prefill_tile < T) T = m->prefill_tile;
    if (!use_tc(m, batch * T) && T > smol::kBatchTile) T = smol::kBatchTile;
    A.tile_t = T;
    A.real_batch = batch;
    A.batch = batch * T;
    A.n_iter = (s_max - 1 + T - 1) / T;
    A.finalize = 1;
    A.phase_begin = 0;
    A.phase_end = smol::phases_per_prefill_step(m->dm.n_layer);
    A.prompt = d_prompt;
    A.prompt_len = d_prompt_len;
    A.s_max = s_max;
    return enqueue(m, A, (cudaStream_t)stream, T == 1);  // tiled prefill runs on the barrier kernel
}

int smol_slow_step(SmolModel* m, const SmolBatch* b, int32_t batch, int32_t advance, void* stream) {
    if (!m) return fail(SMOL_ERR_INVALID, "null model");
    int rc = ensure_configured(m);
    if (rc) return rc;
    if ((rc = check_batch(m, b, batch))) return rc;
    CallArgs A = base_args(b, batch, nullptr);
    A.phase_begin = 0;
    A.phase_end = 5 * m->dm.n_layer + 1;  // slow layers + LM head
    A.advance = advance ? 1 : 0;
    return enqueue(m, A, (cudaStream_t)stream);
}

int smol_fast_step(SmolModel* m, const SmolBatch* b, int32_t batch, int32_t depth_pos, int32_t from_xf, void* stream) {
    if (!m) return fail(SMOL_ERR_INVALID, "null model");
    int rc = ensure_configured(m);
    if (rc) return rc;
    if ((rc = check_batch(m, b, batch))) return rc;
    if (depth_pos < 0 || depth_pos >= m->dm.depth) return fail(SMOL_ERR_INVALID, "smol_fast_step: depth_pos out of range");
    CallArgs A = base_args(b, batch, nullptr);
    const int per = 4 * m->dm.n_flayer + 2;
    A.phase_begin = 5 * m->dm.n_layer + 2 + depth_pos * per;
    A.phase_end = A.phase_begin + 4 * m->dm.n_flayer + 1;  // fast layers + depth head
    A.fast_from_xf = from_xf ? 1 : 0;
    return enqueue(m, A, (cudaStream_t)stream);
}

int smol_fast_embed(SmolModel* m, int32_t batch, const int32_t* d_codes, int32_t depth_pos, void* stream) {
    if (!m || !d_codes) return fail(SMOL_ERR_INVALID, "smol_fast_embed: null argument");
    if (!m->ws_bound) return fail(SMOL_ERR_UNBOUND, "workspace not bound");
    if (batch <= 0 || batch > m->cfg.max_batch) return fail(SMOL_ERR_CAPACITY, "batch outside [1, max_batch]");
    if (depth_pos < 0 || depth_pos >= m->dm.depth) return fail(SMOL_ERR_INVALID, "smol_fast_embed: depth_pos out of range");
    CU(smol::store_codes_launch(m->dm.frame_tokens, d_codes, batch, m->dm.n_rows, 1 + depth_pos, (cudaStream_t)stream));
    m->launches += 1;
    return SMOL_OK;
}

int smol_sample(SmolModel* m, const SmolBatch* b, int32_t batch, const float* d_logits, int32_t n,
                const SmolSampling* s, int32_t stream_id, int32_t* d_out, void* stream) {
    if (!m || !d_logits || !s || !d_out) return fail(SMOL_ERR_INVALID, "smol_sample: null argument");
    if (n <= 0 || n > smol::kThreads * 8) return fail(SMOL_ERR_UNSUPPORTED, "smol_sample: n outside [1, 4096]");
    if (batch <= 0) return fail(SMOL_ERR_INVALID, "smol_sample: bad batch");
    CU(smol::sample_launch(d_logits, n, batch, *s, b ? b->row_sampling : nullptr, stream_id, b ? b->seq_id : nullptr,
                           b ? b->step : nullptr, d_out, (cudaStream_t)stream));
    m->launches += 1;
    return SMOL_OK;
}

int smol_run_phases(SmolModel* m, const SmolBatch* b, int32_t batch, const SmolSampling* s, int32_t phase_begin,
                    int32_t phase_end, void* stream) {
    if (!m) return fail(SMOL_ERR_INVALID, "null model");
    int rc = ensure_configured(m);
    if (rc) return rc;
    if ((rc = check_batch(m, b, batch))) return rc;
    const int total = smol::phases_per_frame(m->dm.n_layer, m->dm.n_flayer, m->dm.depth);
    if (phase_begin < 0 || phase_end > total || phase_begin >= phase_end) return fail(SMOL_ERR_INVALID, "smol_run_phases: bad range");
    CallArgs A = base_args(b, batch, s);
    A.phase_begin = phase_begin;
    A.phase_end = phase_end;
    return enqueue(m, A, (cudaStream_t)stream);
}

int32_t smol_phase_count(const SmolModel* m) {
    return m ? smol::phases_per_frame(m->dm.n_layer, m->dm.n_flayer, m->dm.depth) : 0;
}

int smol_decode_frames(SmolModel* m, const SmolBatch* b, int32_t batch, const SmolSampling* s, int32_t n_frames,
                       void* stream_v) {
    if (!m || !s) return fail(SMOL_ERR_INVALID, "null argument");
    int rc = ensure_configured(m);
    if (rc) return rc;
    if ((rc = check_batch(m, b, batch))) return rc;
    if (n_frames < 1) return fail(SMOL_ERR_INVALID, "n_frames must be >= 1");
    cudaStream_t stream = (cudaStream_t)stream_v;
    CallArgs A = base_args(b, batch, s);
    A.phase_begin = 0;
    A.phase_end = smol::phases_per_frame(m->dm.n_layer, m->dm.n_flayer, m->dm.depth);
    A.n_iter = n_frames;
    return enqueue(m, A, stream, true);
}

int smol_decode_frame(SmolModel* m, const SmolBatch* b, int32_t batch, const SmolSampling* s, void* stream) {
    return smol_decode_frames(m, b, batch, s, 1, stream);
}

int smol_set_force(SmolModel* m, const int32_t* d_force) {
    if (!m) return fail(SMOL_ERR_INVALID, "null model");
    m->dm.force = d_force;
    return SMOL_OK;
}

int smol_set_profile(SmolModel* m, uint64_t* d_phase_ns) {
    if (!m) return fail(SMOL_ERR_INVALID, "null model");
    m->dm.prof = reinterpret_cast<unsigned long long*>(d_phase_ns);
    return SMOL_OK;
}

int smol_set_frame_clock(SmolModel* m, uint64_t* d_frame_ns, int32_t capacity) {
    if (!m) return fail(SMOL_ERR_INVALID, "null model");
    if (d_frame_ns && capacity <= 0) return fail(SMOL_ERR_INVALID, "smol_set_frame_clock: capacity must be positive");
    m->dm.frame_ns = reinterpret_cast<unsigned long long*>(d_frame_ns);
    m->dm.frame_ns_cap = d_frame_ns ? capacity : 0;
    return SMOL_OK;
}

int smol_set_option(SmolModel* m, const char* name, int64_t value) {
    if (!m || !name) return fail(SMOL_ERR_INVALID, "null argument");
    if (!std::strcmp(name, "mode")) {
        if (value == 1) return fail(SMOL_ERR_INVALID, "mode 1 (one launch per phase) was removed: use 0 or 2");
        if (value != 0 && value != 2) return fail(SMOL_ERR_INVALID, "mode must be 0 or 2");
        m->mode = (int)value;
        return SMOL_OK;
    }
    if (!std::strcmp(name, "repeat")) {
        m->repeat = value > 0 ? (int)value : 0;
        return SMOL_OK;
    }
    if (!std::strcmp(name, "prefill_tile")) {
        m->prefill_tile = value > 0 ? (int)value : 0;
        return SMOL_OK;
    }
    if (!std::strcmp(name, "tc_attn_split")) {
        m->tc_attn_split = value > 0 ? (int)value : 0;
        return SMOL_OK;
    }
    if (!std::strcmp(name, "tc_min_batch")) {  // 0 disables the tensor-core variant
        m->tc_min_batch = value > 0 ? (int)value : 0;
        return SMOL_OK;
    }
    if (!std::strcmp(name, "ll_holdoff")) {
        m->ll2_holdoff = value > 0 ? (int)value : 0;
        return SMOL_OK;
    }
    if (!std::strcmp(name, "ll_fused_mlp")) {
        m->ll2_fused_mlp = value != 0 ? 1 : 0;
        return SMOL_OK;
    }
    if (!std::strcmp(name, "ll_max_batch")) {
        if (value < 0 || value > smol::kLL2MaxTeams) return fail(SMOL_ERR_INVALID, "ll_max_batch must be in [0, 8]");
        m->ll2_max_batch = (int)value;
        return SMOL_OK;
    }
    if (!std::strcmp(name, "n_ctas")) {
        if (value < 0) return fail(SMOL_ERR_INVALID, "n_ctas must be >= 0");
        m->n_ctas_override = (int)value;
        m->configured = false;
        return SMOL_OK;
    }
    return fail(SMOL_ERR_INVALID, std::string("unknown option ") + name);
}

int64_t smol_get_option(const SmolModel* m, const char* name) {
    if (!m || !name) return -1;
    if (!std::strcmp(name, "mode")) return m->mode;
    if (!std::strcmp(name, "n_ctas")) return m->n_ctas;
    if (!std::strcmp(name, "n_ctas_override")) return m->n_ctas_override;
    if (!std::strcmp(name, "n_sms")) return m->n_sms;
    if (!std::strcmp(name, "smem_bytes")) return (int64_t)m->smem[1];
    if (!std::strcmp(name, "tc_min_batch")) return m->tc_min_batch;
    if (!std::strcmp(name, "tc_ready")) return m->tile_ready[0] ? 1 : 0;
    if (!std::strcmp(name, "ll_smem_bytes")) return (int64_t)m->ll2_smem;
    if (!std::strcmp(name, "ll_ready")) return (int64_t)m->ll2_state;
    if (!std::strcmp(name, "ll_max_batch")) return (int64_t)m->ll2_max_batch;
    if (!std::strcmp(name, "ll_holdoff")) return (int64_t)m->ll2_holdoff;
    if (!std::strcmp(name, "ll_slots")) return (int64_t)m->ll2_sp.n_slots;
    if (!std::strcmp(name, "ll_solo_ctas")) return (int64_t)ll2_solo_ctas(m);
    if (!std::strcmp(name, "ll_fused_mlp")) return (int64_t)m->ll2_fused_mlp;
    if (!std::strcmp(name, "ll_mlp_cluster")) return (int64_t)m->ll2_cluster;
    if (!std::strcmp(name, "ll_mlp_clusters")) return (int64_t)m->ll2_clusters;
    if (!std::strcmp(name, "ll_last_fused")) return (int64_t)m->ll2_last_fused;
    return -1;
}

void* smol_debug_buffer(SmolModel* m, const char* name) {
    if (!m || !name || !m->ws_bound) return nullptr;
    const DevModel& d = m->dm;
    if (!std::strcmp(name, "x")) return d.x;
    if (!std::strcmp(name, "h")) return d.h;
    if (!std::strcmp(name, "xf")) return d.xf;
    if (!std::strcmp(name, "q")) return d.q;
    if (!std::strcmp(name, "attn")) return d.attn;
    if (!std::strcmp(name, "act")) return d.act;
    if (!std::strcmp(name, "fkv")) return d.fkv;
    if (!std::strcmp(name, "token_logits")) return d.token_logits;
    if (!std::strcmp(name, "depth_logits")) return d.depth_logits;
    if (!std::strcmp(name, "frame_tokens")) return d.frame_tokens;
    if (!std::strcmp(name, "ll")) return d.ll;
    if (!std::strcmp(name, "ll_epoch")) return d.ll_epoch;
    if (!std::strcmp(name, "ll2_score")) return d.ll2_score;
    if (!std::strcmp(name, "ll2_psum")) return d.ll2_psum;
    return nullptr;
}

int smol_ll_region(const SmolModel* m, int32_t phase, uint32_t* word_offset, uint32_t* words) {
    if (!m || !word_offset || !words) return fail(SMOL_ERR_INVALID, "smol_ll_region: null argument");
    if (phase < 0 || phase >= smol_phase_count(m)) return fail(SMOL_ERR_INVALID, "smol_ll_region: phase outside the frame's program");
    *word_offset = m->dm.ll_off[phase];
    *words = m->dm.ll_len[phase];
    return SMOL_OK;
}

int64_t smol_launch_count(const SmolModel* m) { return m ? m->launches : 0; }

}  // extern "C"
