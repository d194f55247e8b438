// C ABI (include/apples_b200.h): context, device buffers, and the per-batch pipeline
//   H2D -> transpose -> dense representative distances -> selection (+ member distances) -> placement -> D2H
// that replaces pool.starmap(queryworker.runquery, queries) (run_apples.py:94-102).
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "common.cuh"

namespace {

// device memory owned by its holder, freed with it (the holder's device must be current then)
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { if (p) cudaFree(p); }
};

enum Stage { T_H2D = 0, T_TRANSPOSE, T_DENSE, T_SELECT, T_PLACE, T_D2H, T_NSTAGE };

struct TimedSpan {
    int stage;
    cudaEvent_t a, b;
};

// host buffers of the ranked records (apples_set_alternatives); keep 1: none
struct AltOut {
    int keep = 1;
    int32_t* count = nullptr;
    int32_t* edge = nullptr;
    double* error = nullptr;
    double* distal = nullptr;
    double* pendant = nullptr;
    uint8_t* int0 = nullptr;
};

}  // namespace

struct apples_ctx {
    int device = 0;
    int num_sms = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;       // host->device staging of the next sub-batch overlaps compute
    cudaEvent_t ev_ready[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
    // the selection stage of the reruns (few large / exotic queries, thin long kernels) runs here, high priority, beside the
    // main placement pass on the main stream
    cudaStream_t side_stream = nullptr;
    std::string err;

    // tree
    int M = 0;
    DevBuf t_parent, t_elen, t_level, t_first;
    // reference
    int kind = -1, L = 0, W = 0, Wp = 0, Lp = 0, n_ref = 0, n_rep = 0, rep_pad = 0, ref_pad = 0;
    DevBuf refs_rm, reps_rm, reps_wm, refs_wm, reps_nv, refs_nv, q_nv, ref_node, goff, gmem;
    DevBuf aa_tab, reps_aa_tm, reps_aav, refs_aa_tm, refs_aav, q_aa_tm, q_aav, aa_valid;   // amino-acid dense kernel operands
    int aa_rep_pad = 0, aa_ref_pad = 0;
    bool refs_aa_ready = false;
    // byte-compare fallback of the nucleotide path (L > 65535 or symbols outside A,C,G,T,-): padded byte rows [n][Lp]
    bool nuc_slow = false;        // the whole context runs in byte mode
    bool bytes_ready = false;     // ref_bytes_p / rep_bytes_p hold the reference
    DevBuf ref_bytes_p, rep_bytes_p, q_bytes_p, q_rowflag, keys_w;
    double n_slow = 0;            // queries that went through the fallback
    // representative-count kernel: 1 = tensor cores (dense_tc.cu, default): the block-scaled fp4 kernel up to
    // dense_fp4_max_sites() columns, the kind::i8 kernel beyond it; 0 = integer-pipe LOP3/POPC kernel (distance.cu; also
    // taken automatically beyond 33 816 columns)
    int dense_mode = 1;
    double n_tc_launch = 0, n_fp4_launch = 0, n_k2p_launch = 0;
    // substitution model: `model` is the setting for the next apples_set_reference*, `k2p` that of the installed reference
    // (K2P count keys, 128 x 160 count tiles, the SEL_K2P selection)
    int model = APPLES_JC69;
    bool k2p = false;
    bool tc_ready = false;        // reps_img holds the representatives' operand images
    bool tc_fp4 = false;          // ... for the fp4 kernel (else for the kind::i8 kernel)
    int tc_nw = 0, tc_rep_pad = 0;
    DevBuf reps_img, q_img;
    bool refs_wm_ready = false;
    // matrix mode
    int n_cols = 0;
    DevBuf col_node;
    // per-batch work buffers
    DevBuf q_rm, q_wm, keys, self_node, obs_node, obs_dist, obs_len, obs_len2, Kd, Vd, statusd, zero_edge, pair_counter;
    DevBuf q_bytes, q_bytes2, q_rm2, bad_flag, clk_probe, stash_keys, stash_ids, stash_count;
    DevBuf kmin, stash_kmin;   // line minima of keys / stash_keys (nucleotide count keys)
    double dense_mhz = 0.0;  // effective SM clock of the last dense launch (clock64 / globaltimer of CTA 0)
    DevBuf obs_node2, obs_dist2, qlist, pl_lists, bin_counts, bin_lists, rec_off, stack_off, recs, stacks;
    DevBuf o_edge, o_err, o_distal, o_pendant, o_status;
    DevBuf o_alt_count, o_alt_edge, o_alt_err, o_alt_distal, o_alt_pendant, o_alt_int0;
    AltOut alt;   // registered by apples_set_alternatives, taken by the next apples_place_batch* call
    DevBuf dbg_x1, dbg_x2, dbg_err, dbg_valid;
    // resident queries
    DevBuf res_q, res_self;
    int64_t res_nq = 0;
    bool res_has_self = false;
    DevBuf res_edge, res_err, res_distal, res_pendant, res_status;
    // timing
    std::vector<TimedSpan> spans;
    std::vector<cudaEvent_t> ev_pool;
    double t_ms[T_NSTAGE] = {0, 0, 0, 0, 0, 0};
    double n_launch = 0, n_dense_launch = 0, n_pairs = 0, n_lines = 0, n_obs = 0, n_valid = 0, n_over = 0, max_K = 0, max_V = 0;
    size_t scratch_limit = (size_t)6 << 30;  // placement scratch pool upper bound (bytes)
    int64_t max_subbatch = 65536;
    int64_t max_batch = 1 << 20;  // queries per macro-batch (batch-wide observed-list buffers)
    std::vector<int> hK, hV, hS;
    std::vector<char> h_over;      // last macro-batch: query went through the overflow rerun
    std::vector<int> h_first;      // host copy of first[]: node u is a leaf iff first[u] == u
    std::vector<int> h_ref_node, h_col_node;  // re-validated when the tree changes
    std::vector<long long> h_rec_off, h_stack_off;
    std::vector<int> h_pl_lists;
    double n_place_class[PLACE_NCLASS] = {0, 0, 0, 0, 0};
    std::vector<char> h_gather;
    int slot_cap = 256;
};

namespace {

int fail(apples_ctx* c, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf;
    return -1;
}

#define CK(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess) return fail(ctx, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), \
                                           __FILE__, __LINE__);                                       \
    } while (0)

int ensure(apples_ctx* ctx, DevBuf& b, size_t bytes) {
    if (bytes <= b.bytes && b.p) return 0;
    if (b.p) CK(cudaFree(b.p));
    b.p = nullptr;
    b.bytes = 0;
    size_t want = std::max<size_t>(bytes, 256);
    CK(cudaMalloc(&b.p, want));
    b.bytes = want;
    return 0;
}

cudaEvent_t get_event(apples_ctx* ctx) {
    if (!ctx->ev_pool.empty()) {
        cudaEvent_t e = ctx->ev_pool.back();
        ctx->ev_pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

struct Span {
    apples_ctx* ctx;
    TimedSpan s;
    cudaStream_t st;
    Span(apples_ctx* c, int stage, cudaStream_t stream = nullptr) : ctx(c), st(stream ? stream : c->stream) {
        s.stage = stage;
        s.a = get_event(c);
        s.b = get_event(c);
        cudaEventRecord(s.a, st);
    }
    ~Span() {
        cudaEventRecord(s.b, st);
        ctx->spans.push_back(s);
    }
};

// APPLES_B200_TRACE=1: device span timeline and host phase times of every macro-batch on stderr (debugging aid)
bool tracing() {
    static const bool trace = getenv("APPLES_B200_TRACE") != nullptr;
    return trace;
}

void collect_spans(apples_ctx* ctx) {
    const bool trace = tracing();
    static const char* names[] = {"h2d", "transpose", "dense", "select", "place", "d2h"};
    for (auto& s : ctx->spans) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) ctx->t_ms[s.stage] += ms;
        if (trace && !ctx->spans.empty()) {   // device timeline: start of every span relative to the first one
            float off = 0.f;
            cudaEventElapsedTime(&off, ctx->spans.front().a, s.a);
            fprintf(stderr, "[apples_b200]   dev %-9s @%8.3f ms  %7.3f ms\n", names[s.stage], off, ms);
        }
        ctx->ev_pool.push_back(s.a);
        ctx->ev_pool.push_back(s.b);
    }
    ctx->spans.clear();
}

inline int round_up(int x, int m) { return (x + m - 1) / m * m; }
inline int next_pow2(int x) {
    int p = 1;
    while (p < x) p <<= 1;
    return p;
}

// smallest valid-site count v with NOT (v / L < overlap_frac)  (distance.py:735, IEEE double division)
int overlap_vmin(int L, double overlap) {
    int lo = 0, hi = L + 1;  // invariant: lo fails (or is 0), hi passes (or is L+1)
    while (hi - lo > 1) {
        int mid = lo + (hi - lo) / 2;
        if ((double)mid / (double)L < overlap) lo = mid; else hi = mid;
    }
    if (hi > L) return L + 1;
    // v == 0 always fails (`not valid`)
    return std::max(hi, 1);
}

NucGate make_gate(int L, double thr, double overlap) {
    NucGate g;
    g.L = L;
    g.vmin = overlap_vmin(L, overlap);
    g.thr = thr;
    // dist <= thr  <=>  p <= p*, p* = 0.75 (1 - exp(-4 thr / 3)).  Fixed-point (16.16) guard band around p*: below
    // P_lo certainly near, above P_hi certainly far, in between the kernel evaluates the fp64 distance itself.
    if (!(thr >= 0.0)) {          // nothing is near (a zero distance still is not <= a negative threshold)
        g.P_lo = 0;
        g.P_hi = 0;               // lhs >= 0 always: everything valid is far
        return g;
    }
    const double pstar = 0.75 * (1.0 - std::exp(-4.0 * thr / 3.0));
    const double lo = std::floor(pstar * (1.0 - 1e-9) * 65536.0) - 1.0;
    const double hi = std::ceil(pstar * (1.0 + 1e-9) * 65536.0) + 1.0;
    g.P_lo = (uint32_t)std::max(0.0, std::min(lo, 49152.0));
    g.P_hi = (uint32_t)std::max(1.0, std::min(hi, 49153.0));
    if (g.P_lo >= 49151u) g.P_lo = 49152u;  // threshold so large that every valid pair (4 m < 3 v) is near
    return g;
}

// every mapped node id must be -1 (not in the tree) or a LEAF of the current tree (ids index tree arrays in the kernels)
int check_leaf_ids(apples_ctx* ctx, const char* what, const int32_t* ids, int n) {
    if (ctx->M <= 0) return 0;  // no tree yet: validated again by apples_set_tree
    for (int i = 0; i < n; ++i) {
        const int v = ids[i];
        if (v == -1) continue;
        if (v < 0 || v >= ctx->M) return fail(ctx, "%s[%d] = %d is outside [-1, %d)", what, i, v, ctx->M);
        if (ctx->h_first[v] != v) return fail(ctx, "%s[%d] = %d is not a leaf of the tree", what, i, v);
    }
    return 0;
}

const double k_blosum45[441] = {
#include "blosum45.inc"
};

inline int aa_chunks(int Lp) { return (Lp + AA_CH - 1) / AA_CH; }

// amino-acid operands of the dense kernel: limb tables (once) and the tile-major copy + valid planes of the representatives
int aa_prepare_reps(apples_ctx* ctx, cudaStream_t s) {
    if (!ctx->aa_tab.p) {
        uint32_t tab[AA_TAB_WORDS];
        aa_build_tables(k_blosum45, tab);
        if (ensure(ctx, ctx->aa_tab, sizeof tab)) return -1;
        CK(cudaMemcpy(ctx->aa_tab.p, tab, sizeof tab, cudaMemcpyHostToDevice));
    }
    const int nc = aa_chunks(ctx->Lp);
    ctx->aa_rep_pad = round_up(ctx->n_rep, AA_TR);
    ctx->aa_ref_pad = round_up(ctx->n_ref, AA_TR);
    if (ensure(ctx, ctx->reps_aa_tm, (size_t)ctx->aa_rep_pad * nc * AA_CH) ||
        ensure(ctx, ctx->reps_aav, (size_t)ctx->aa_rep_pad * nc * (AA_CH / 32) * 4))
        return -1;
    launch_aa_layout((const uint8_t*)ctx->reps_rm.p, ctx->n_rep, ctx->Lp, AA_TR, ctx->aa_rep_pad, (uint8_t*)ctx->reps_aa_tm.p,
                     (uint32_t*)ctx->reps_aav.p, s);
    CK(cudaGetLastError());
    return 0;
}

// padded byte rows of the references and representatives for the byte-compare fallback; a context in fast mode builds
// them from its bit-planes the first time a query needs the fallback
int ensure_ref_bytes(apples_ctx* ctx, cudaStream_t s) {
    if (ctx->bytes_ready) return 0;
    if (ensure(ctx, ctx->ref_bytes_p, (size_t)ctx->n_ref * ctx->Lp) || ensure(ctx, ctx->rep_bytes_p, (size_t)ctx->n_rep * ctx->Lp))
        return -1;
    CK(launch_unpack_nuc((const uint32_t*)ctx->refs_rm.p, ctx->n_ref, ctx->L, ctx->W, ctx->Lp, (uint8_t*)ctx->ref_bytes_p.p, s));
    CK(launch_unpack_nuc((const uint32_t*)ctx->reps_rm.p, ctx->n_rep, ctx->L, ctx->W, ctx->Lp, (uint8_t*)ctx->rep_bytes_p.p, s));
    ctx->bytes_ready = true;
    return 0;
}

size_t query_row_bytes(const apples_ctx* ctx) {
    return ctx->kind == APPLES_AA ? (size_t)ctx->Lp : (size_t)3 * ctx->W * 4;
}

// what apples_set_reference and apples_set_reference_bytes both validate: the group CSR and the leaf ids (`who` names the
// entry point in the messages)
int check_reference(apples_ctx* ctx, const char* who, int n_ref, const int32_t* ref_node, int n_rep,
                    const int32_t* group_offsets, const int32_t* group_members) {
    for (int i = 0; i < n_rep; ++i)
        if (group_offsets[i + 1] < group_offsets[i]) return fail(ctx, "%s: group_offsets not monotone", who);
    const int n_mem = group_offsets[n_rep];
    for (int i = 0; i < n_mem; ++i)
        if (group_members[i] < 0 || group_members[i] >= n_ref) return fail(ctx, "%s: member out of range", who);
    return check_leaf_ids(ctx, "ref_node", ref_node, n_ref);
}

// geometry of a new reference and its device buffers; ref_node becomes the host copy of the leaf map
int set_geometry(apples_ctx* ctx, int kind, int L, int n_ref, const int32_t* ref_node, int n_rep, int n_mem) {
    ctx->h_ref_node.assign(ref_node, ref_node + n_ref);
    CK(cudaSetDevice(ctx->device));
    ctx->kind = kind;
    ctx->L = L;
    ctx->n_ref = n_ref;
    ctx->n_rep = n_rep;
    ctx->W = apples_words_per_row(L);
    ctx->Wp = round_up(ctx->W, DT_WC);
    ctx->Lp = apples_aa_row_bytes(L);
    // the key row (ldk = rep_pad) covers the representative tiles of the count kernel and stays a multiple of DT_TR
    ctx->k2p = ctx->model == APPLES_K2P;
    if (ctx->dense_mode == 1 && L <= dense_fp4_max_sites())
        ctx->rep_pad = round_up(round_up(n_rep, dense_fp4_tile_rows(1, ctx->k2p)), DT_TR);
    else
        ctx->rep_pad = round_up(n_rep, ctx->dense_mode == 1 ? 256 : DT_TR);
    ctx->ref_pad = round_up(n_ref, DT_TR);
    const size_t row = query_row_bytes(ctx);
    if (ensure(ctx, ctx->refs_rm, (size_t)n_ref * row) || ensure(ctx, ctx->reps_rm, (size_t)n_rep * row) ||
        ensure(ctx, ctx->ref_node, (size_t)n_ref * 4) || ensure(ctx, ctx->goff, (size_t)(n_rep + 1) * 4) ||
        ensure(ctx, ctx->gmem, (size_t)std::max(n_mem, 1) * 4))
        return -1;
    return 0;
}

// what the K2P model needs of a reference (apples_ctx_set_model), checked before it is installed
int check_model(apples_ctx* ctx, const char* who, int kind, int L) {
    if (ctx->model != APPLES_K2P) return 0;
    if (kind != APPLES_NUC) return fail(ctx, "%s: the K2P model needs nucleotide sequences", who);
    if (ctx->dense_mode != 1) return fail(ctx, "%s: the K2P model needs the tensor-core count kernel (dense mode 1)", who);
    if (L > dense_fp4_max_sites())
        return fail(ctx, "%s: the K2P model takes alignments of at most %d columns, this one has %d", who, dense_fp4_max_sites(), L);
    return 0;
}

// operands derived from the installed reference (refs_rm / reps_rm) for its kind and the dense mode; every derived-state
// flag is reset first.  In byte mode (nuc_slow) the byte rows are the operands: the installer builds them
int prepare_operands(apples_ctx* ctx, cudaStream_t s) {
    ctx->tc_ready = ctx->bytes_ready = ctx->refs_wm_ready = ctx->refs_aa_ready = false;
    if (ctx->kind == APPLES_AA) return aa_prepare_reps(ctx, s);
    if (ctx->nuc_slow) return 0;
    const size_t wm = (size_t)3 * ctx->Wp * ctx->rep_pad * 4;
    if (ensure(ctx, ctx->reps_wm, wm) || ensure(ctx, ctx->reps_nv, (size_t)ctx->rep_pad * 4)) return -1;
    CK(cudaMemsetAsync(ctx->reps_wm.p, 0, wm, s));
    launch_transpose_nuc((const uint32_t*)ctx->reps_rm.p, ctx->n_rep, ctx->W, (uint32_t*)ctx->reps_wm.p, ctx->Wp, ctx->rep_pad,
                         DT_TR, s);
    launch_row_valid((const uint32_t*)ctx->reps_rm.p, ctx->n_rep, ctx->W, (uint32_t*)ctx->reps_nv.p, ctx->rep_pad, s);
    CK(cudaGetLastError());
    // operand images of the representatives for the tensor-core kernel
    if (ctx->dense_mode != 1 || ctx->L > dense_tc_max_sites()) return 0;
    ctx->tc_nw = (ctx->L + 31) / 32;
    ctx->tc_fp4 = ctx->L <= dense_fp4_max_sites();
    if (ctx->tc_fp4) {
        const int rows = dense_fp4_tile_rows(1, ctx->k2p);
        ctx->tc_rep_pad = round_up(ctx->n_rep, rows);
        if (ensure(ctx, ctx->reps_img, dense_fp4_image_bytes(ctx->tc_rep_pad, ctx->tc_nw))) return -1;
        launch_fp4_image((const uint32_t*)ctx->reps_rm.p, ctx->n_rep, ctx->W, ctx->tc_nw, ctx->tc_rep_pad, rows, ctx->reps_img.p, s);
    } else {
        ctx->tc_rep_pad = round_up(ctx->n_rep, dense_tc_tile_rows());
        if (ensure(ctx, ctx->reps_img, dense_tc_image_bytes(ctx->tc_rep_pad, ctx->tc_nw))) return -1;
        launch_tc_image((const uint32_t*)ctx->reps_rm.p, ctx->n_rep, ctx->W, ctx->tc_nw, ctx->tc_rep_pad, 127, ctx->reps_img.p, s);
    }
    CK(cudaGetLastError());
    ctx->tc_ready = true;
    return 0;
}

TreeDev tree_dev(apples_ctx* ctx) {
    TreeDev t;
    t.M = ctx->M;
    t.parent = (const int*)ctx->t_parent.p;
    t.elen = (const double*)ctx->t_elen.p;
    t.level = (const int*)ctx->t_level.p;
    t.first = (const int*)ctx->t_first.p;
    return t;
}

struct BatchIO {
    // exactly one of these input sources
    const void* h_queries = nullptr;   // host packed queries
    const void* d_queries = nullptr;   // device packed queries (resident)
    const double* h_rows = nullptr;    // host matrix rows
    const uint8_t* h_bytes = nullptr;  // host alignment bytes (packed on the device, SURVEY 8 f1)
    int64_t byte_stride = 0;
    const int32_t* h_self = nullptr;
    const int32_t* d_self = nullptr;
    // outputs: host pointers or device pointers
    int32_t* edge = nullptr; double* error = nullptr; double* distal = nullptr; double* pendant = nullptr;
    int32_t* status = nullptr;
    bool out_on_device = false;
    // parity exports
    int obs_cap = 0; int32_t* obs_count = nullptr; int32_t* obs_node = nullptr; double* obs_dist = nullptr;
    bool stop_after_select = false;
    // count-keys export: every sub-batch's [nb][n_rep] block of the key matrix is copied to h_keys and the batch stops
    // after the count stage (no selection, no placement)
    void* h_keys = nullptr;
    uint32_t* h_kmin = nullptr;   // optional: their line minima [nq][ceil(n_rep / 32)] (nucleotide count keys only)
    bool stop_after_count = false;
    double* dbg_x1 = nullptr; double* dbg_x2 = nullptr; double* dbg_err = nullptr; uint8_t* dbg_valid = nullptr;
    AltOut alt;   // ranked records [nq][alt.keep] when alt.keep > 1 (host output only)
};

int check_params(apples_ctx* ctx, const apples_params* p) {
    if (!p) return fail(ctx, "params is NULL");
    if (p->method < 0 || p->method > 3) return fail(ctx, "unknown method %d", p->method);
    if (p->criterion < 0 || p->criterion > 2) return fail(ctx, "unknown criterion %d", p->criterion);
    return 0;
}

// observed-list rows: `cap` slots per row.  The selection writes them; a placement launch reads row slot_list[entry], or
// the query's own row when it has no slot list
struct ObsRows {
    int cap;
    int* node;
    double* dist;
    int* len;
};

// launch class of a placeable query with V valid nodes (+ 1: pseudo record of the subtree root)
inline int place_class(int V) {
    const int v = V + 1;
    return v <= 64 ? PLACE_CLASS_64 : v <= 128 ? PLACE_CLASS_128 : v <= 256 ? PLACE_CLASS_256 : v <= 512 ? PLACE_CLASS_512 : PLACE_CLASS_BLOCK;
}

// One macro-batch (at most ctx->max_batch queries) through the pipeline; run() calls the stages in this order:
//   first pass    per sub-batch, no host synchronisation: H2D (copy stream) -> operand images -> count kernel ->
//                 selection; then the class-sorting kernel
//   counts        one synchronise: (K, V, status) and the launch-class sizes on the host
//   main pass     the shared-memory placement launches of the ordinary queries, from the class lists the device built
//   reruns        (rare) the byte-compare fallback for exotic queries, larger slots for overflowing ones: selection on the
//                 side stream beside the main pass, placement on the main stream
//   block class   the ordinary queries with V + 1 > 512, one block per query
//   tail          finalize, results D2H / D2D
struct MacroBatch {
    apples_ctx* const ctx;
    const BatchIO& io;
    const apples_params* const prm;
    const int64_t base0;
    const int n;
    const cudaStream_t s;   // main stream
    std::vector<int>& hK;
    std::vector<int>& hV;
    std::vector<int>& hS;
    bool matrix, nuc, slow_ctx;   // slow_ctx: byte-compare fallback for every query of this context
    int sel_kind, n_units;
    int64_t ldk;
    size_t key_bytes, qrow;
    int QB, cap, cap_max;
    bool use_tc, two_bufs;
    int stash_cap = 0;
    const int* d_self = nullptr;
    SelectArgs sa{};   // selection arguments of the first pass
    PlaceArgs pa{};    // placement arguments without the launch's entries and observed-list rows
    int h_bin[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    unsigned long long h_bin_stats[4] = {0, 0, 0, 0};
    const std::chrono::steady_clock::time_point t_begin = std::chrono::steady_clock::now();

    MacroBatch(apples_ctx* c, int64_t b0, int nq, const BatchIO& bio, const apples_params* p)
        : ctx(c), io(bio), prm(p), base0(b0), n(nq), s(c->stream), hK(c->hK), hV(c->hV), hS(c->hS) {
        matrix = io.h_rows != nullptr;
        nuc = !matrix && ctx->kind == APPLES_NUC;
        slow_ctx = nuc && ctx->nuc_slow;
        sel_kind = matrix ? SEL_MATRIX : (ctx->kind == APPLES_AA ? SEL_AA : (slow_ctx ? SEL_NUCW : (ctx->k2p ? SEL_K2P : SEL_NUC)));
        n_units = matrix ? ctx->n_cols : ctx->n_rep;
        ldk = matrix ? ctx->n_cols : ctx->rep_pad;
        key_bytes = (sel_kind == SEL_NUC) ? 4 : 8;
        // sub-batch size: key matrix <= 2 GiB, multiple of the dense tile
        int64_t qb = ((int64_t)2 << 30) / std::max<int64_t>(1, ldk * (int64_t)key_bytes);
        qb = std::min<int64_t>(std::max<int64_t>(qb, DT_TQ), std::max<int64_t>(ctx->max_subbatch, DT_TQ));
        qb = qb / DT_TQ * DT_TQ;
        qb = std::min<int64_t>(qb, round_up(n, DT_TQ));
        QB = (int)qb;
        cap_max = next_pow2(std::max(4, matrix ? ctx->n_cols : ctx->n_ref));
        cap = std::min(ctx->slot_cap, cap_max);
        qrow = matrix ? (size_t)ctx->n_cols * 8 : query_row_bytes(ctx);
        // K2P runs on the fp4 kernel whatever apples_ctx_set_dense_mode said after its reference was installed
        use_tc = sel_kind == SEL_K2P || (sel_kind == SEL_NUC && ctx->tc_ready);
        two_bufs = n > QB;  // more than one sub-batch: stage the next one while this one computes
    }

    // host wall-clock of the pipeline phases
    void mark(const char* what) const {
        if (!tracing()) return;
        const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
        fprintf(stderr, "[apples_b200] %-28s +%8.3f ms\n", what, ms);
    }
    ObsRows main_rows() const {
        return ObsRows{cap, (int*)ctx->obs_node.p, (double*)ctx->obs_dist.p, (int*)ctx->obs_len.p};
    }
    // placement arguments of one launch: `cnt` entries, entry i places query qlist[i] from row slots[i] of `r`
    PlaceArgs place_args(const ObsRows& r, int cnt, const int* qlist, const int* slots) const {
        PlaceArgs a = pa;
        a.n = cnt;
        a.qlist = qlist;
        a.slot_list = slots;
        a.cap = r.cap;
        a.obs_node = r.node;
        a.obs_dist = r.dist;
        a.obs_len = r.len;
        return a;
    }

    int run() {
        if (allocate()) return -1;
        init_args();
        if (first_pass()) return -1;
        if (io.stop_after_count) {
            CK(cudaStreamSynchronize(s));
            collect_spans(ctx);
            return 0;
        }
        std::vector<int> exotic, over;
        bool use_stash = false;
        if (fetch_classes(exotic) || plan_reruns(exotic, over, use_stash)) return -1;
        if (tracing()) fprintf(stderr, "[apples_b200] classes %d %d %d %d %d\n", h_bin[0], h_bin[1], h_bin[2], h_bin[3], h_bin[4]);
        if (!io.stop_after_select && place_main_pass()) return -1;
        mark("main placement launched");
        if (!exotic.empty() && rerun(exotic, true, cap, false)) return -1;
        if (!over.empty() && rerun(over, slow_ctx, (int)std::min<int64_t>((int64_t)cap * 16, cap_max), use_stash)) return -1;
        if (!io.stop_after_select && place_main_block_class()) return -1;
        mark("reruns done");
        if (io.obs_count && export_observed()) return -1;
        add_stats(exotic, over);
        if (!io.stop_after_select) {
            mark("stats done");
            if (place_tail()) return -1;
        }
        mark("tail launched");
        return finish();
    }

    // work buffers of the batch (grown, never shrunk), the zeroing of its counters and flags, and the self-node upload
    int allocate() {
        if (ensure(ctx, ctx->keys, (size_t)(use_tc ? round_up(QB, 256) : QB) * ldk * key_bytes)) return -1;
        if (sel_kind == SEL_NUC && ensure(ctx, ctx->kmin, (size_t)(use_tc ? round_up(QB, 256) : QB) * (ldk / 32) * 4)) return -1;
        if (use_tc && ensure(ctx, ctx->q_img, ctx->tc_fp4 ? dense_fp4_image_bytes(round_up(QB, dense_fp4_tile_rows(0)), ctx->tc_nw)
                                                          : dense_tc_image_bytes(round_up(QB, 256), ctx->tc_nw)))
            return -1;
        if (io.h_bytes) {
            if (ensure(ctx, ctx->q_bytes, (size_t)QB * io.byte_stride) || ensure(ctx, ctx->bad_flag, 4)) return -1;
            if (two_bufs && ensure(ctx, ctx->q_bytes2, (size_t)QB * io.byte_stride)) return -1;
            CK(cudaMemsetAsync(ctx->bad_flag.p, 0, 4, s));
            if (nuc && !slow_ctx) {
                if (ensure(ctx, ctx->q_rowflag, (size_t)n * 4)) return -1;
                CK(cudaMemsetAsync(ctx->q_rowflag.p, 0, (size_t)n * 4, s));
            }
        }
        if (slow_ctx && ensure(ctx, ctx->q_bytes_p, (size_t)QB * ctx->Lp)) return -1;
        // second packed-query buffer: staged packed queries, or the device packer's output for the sub-batch after this one
        if ((io.h_queries || (io.h_bytes && !slow_ctx)) && two_bufs && ensure(ctx, ctx->q_rm2, (size_t)QB * qrow)) return -1;
        if (!matrix) {
            if (ensure(ctx, ctx->q_rm, (size_t)QB * qrow)) return -1;
            if (sel_kind == SEL_NUC && ensure(ctx, ctx->q_wm, (size_t)3 * ctx->Wp * QB * 4)) return -1;
            if (sel_kind == SEL_NUC && ensure(ctx, ctx->q_nv, (size_t)QB * 4)) return -1;
            if (sel_kind == SEL_NUC && ensure(ctx, ctx->clk_probe, 32)) return -1;
            if (sel_kind == SEL_AA) {
                const size_t qp = (size_t)round_up(QB, AA_TQ), nc = (size_t)aa_chunks(ctx->Lp);
                if (ensure(ctx, ctx->q_aa_tm, qp * nc * AA_CH) || ensure(ctx, ctx->q_aav, qp * nc * (AA_CH / 32) * 4) ||
                    ensure(ctx, ctx->aa_valid, (size_t)QB * ldk * 4))
                    return -1;
            }
        }
        if (ensure(ctx, ctx->self_node, (size_t)n * 4)) return -1;
        if (ensure(ctx, ctx->obs_node, (size_t)n * cap * 4)) return -1;
        if (ensure(ctx, ctx->obs_dist, (size_t)n * cap * 8)) return -1;
        if (ensure(ctx, ctx->obs_len, (size_t)n * cap * 4)) return -1;
        if (ensure(ctx, ctx->Kd, (size_t)n * 4) || ensure(ctx, ctx->Vd, (size_t)n * 4) ||
            ensure(ctx, ctx->statusd, (size_t)n * 4) || ensure(ctx, ctx->zero_edge, (size_t)n * 4))
            return -1;
        if (ensure(ctx, ctx->pair_counter, 16)) return -1;   // member distances, key lines read
        if (ensure(ctx, ctx->o_edge, (size_t)n * 4) || ensure(ctx, ctx->o_err, (size_t)n * 8) ||
            ensure(ctx, ctx->o_distal, (size_t)n * 8) || ensure(ctx, ctx->o_pendant, (size_t)n * 8) ||
            ensure(ctx, ctx->o_status, (size_t)n * 4))
            return -1;
        if (io.alt.keep > 1) {
            const size_t nk = (size_t)n * io.alt.keep;
            if (ensure(ctx, ctx->o_alt_count, (size_t)n * 4) || ensure(ctx, ctx->o_alt_edge, nk * 4) ||
                ensure(ctx, ctx->o_alt_err, nk * 8) || ensure(ctx, ctx->o_alt_distal, nk * 8) ||
                ensure(ctx, ctx->o_alt_pendant, nk * 8) || ensure(ctx, ctx->o_alt_int0, nk))
                return -1;
        }
        if (ensure(ctx, ctx->rec_off, (size_t)(n + 1) * 8) || ensure(ctx, ctx->stack_off, (size_t)(n + 1) * 8) ||
            ensure(ctx, ctx->qlist, (size_t)std::max(n, 1) * 4) || ensure(ctx, ctx->pl_lists, (size_t)std::max(n, 1) * 8))
            return -1;
        CK(cudaMemsetAsync(ctx->pair_counter.p, 0, 16, s));
        if (ensure(ctx, ctx->bin_counts, 64) || ensure(ctx, ctx->bin_lists, (size_t)PLACE_NCLASS * std::max(n, 1) * 4)) return -1;
        CK(cudaMemsetAsync(ctx->bin_counts.p, 0, 64, s));
        if (io.dbg_x1) {
            if (ensure(ctx, ctx->dbg_x1, (size_t)ctx->M * 8) || ensure(ctx, ctx->dbg_x2, (size_t)ctx->M * 8) ||
                ensure(ctx, ctx->dbg_err, (size_t)ctx->M * 8) || ensure(ctx, ctx->dbg_valid, (size_t)ctx->M))
                return -1;
            CK(cudaMemsetAsync(ctx->dbg_x1.p, 0, (size_t)ctx->M * 8, s));
            CK(cudaMemsetAsync(ctx->dbg_x2.p, 0, (size_t)ctx->M * 8, s));
            CK(cudaMemsetAsync(ctx->dbg_err.p, 0, (size_t)ctx->M * 8, s));
            CK(cudaMemsetAsync(ctx->dbg_valid.p, 0, (size_t)ctx->M, s));
        }
        if (io.h_self) {
            for (int i = 0; i < n; ++i) {
                const int v = io.h_self[base0 + i];
                if (v < -1 || v >= ctx->M) return fail(ctx, "self_node[%lld] = %d is outside [-1, %d)", (long long)(base0 + i), v, ctx->M);
            }
            CK(cudaMemcpyAsync(ctx->self_node.p, io.h_self + base0, (size_t)n * 4, cudaMemcpyHostToDevice, s));
            d_self = (const int*)ctx->self_node.p;
        } else if (io.d_self) {
            d_self = io.d_self + base0;
        }
        hK.resize(n); hV.resize(n); hS.resize(n);
        ctx->h_rec_off.resize(n + 1); ctx->h_stack_off.resize(n + 1);
        // key-row stash for the overflow reruns (alignment-mode nucleotides): up to 256 MiB of key rows
        if (sel_kind == SEL_NUC && !matrix) {
            stash_cap = (int)std::min<int64_t>(n, std::max<int64_t>(1, ((int64_t)256 << 20) / (ldk * 4)));
            if (ensure(ctx, ctx->stash_keys, (size_t)stash_cap * ldk * 4) || ensure(ctx, ctx->stash_kmin, (size_t)stash_cap * (ldk / 32) * 4) ||
                ensure(ctx, ctx->stash_ids, (size_t)stash_cap * 4) || ensure(ctx, ctx->stash_count, 4))
                return -1;
            CK(cudaMemsetAsync(ctx->stash_count.p, 0, 4, s));
        }
        return 0;
    }

    void init_args() {
        sa.n_units = n_units;
        sa.ldk = ldk;
        sa.keys_nuc = (const uint32_t*)ctx->keys.p;
        sa.keys_f64 = (const double*)ctx->keys.p;
        sa.kmin = (const uint32_t*)ctx->kmin.p;
        sa.goff = (const int*)ctx->goff.p;
        sa.gmem = (const int*)ctx->gmem.p;
        sa.ref_node = (const int*)ctx->ref_node.p;
        sa.refs_nuc = (const uint32_t*)ctx->refs_rm.p;
        sa.W = ctx->W;
        sa.refs_aa = (const uint8_t*)ctx->refs_rm.p;
        sa.refs_bytes = (const uint8_t*)ctx->ref_bytes_p.p;
        sa.refs_bstride = ctx->Lp;
        sa.q_bstride = ctx->Lp;
        sa.Lp = ctx->Lp;
        sa.L = ctx->L;
        sa.col_node = (const int*)ctx->col_node.p;
        sa.self_node = d_self;
        sa.thr = prm->filt_threshold;
        sa.baseobs = prm->base_observation_threshold;
        sa.overlap = prm->overlap_frac;
        sa.gate = make_gate(ctx->L, prm->filt_threshold, prm->overlap_frac);
        sa.K = (int*)ctx->Kd.p;
        sa.V = (int*)ctx->Vd.p;
        sa.status = (int*)ctx->statusd.p;
        sa.zero_edge = (int*)ctx->zero_edge.p;
        sa.tree = tree_dev(ctx);
        if (stash_cap > 0) {
            sa.stash_keys = (uint32_t*)ctx->stash_keys.p;
            sa.stash_kmin = (uint32_t*)ctx->stash_kmin.p;
            sa.stash_ids = (int*)ctx->stash_ids.p;
            sa.stash_count = (int*)ctx->stash_count.p;
            sa.stash_cap = stash_cap;
        }
        const ObsRows r = main_rows();
        sa.cap = r.cap;
        sa.obs_node = r.node;
        sa.obs_dist = r.dist;
        sa.obs_len = r.len;
        sa.pair_counter = (unsigned long long*)ctx->pair_counter.p;
        sa.line_counter = (unsigned long long*)ctx->pair_counter.p + 1;

        const bool dbg = io.dbg_x1 != nullptr;
        pa.K = (const int*)ctx->Kd.p;
        pa.status = (const int*)ctx->statusd.p;
        pa.zero_edge = (const int*)ctx->zero_edge.p;
        pa.criterion = prm->criterion;
        pa.negative_branch = prm->negative_branch;
        pa.tree = tree_dev(ctx);
        pa.out_edge = (int*)ctx->o_edge.p;
        pa.out_error = (double*)ctx->o_err.p;
        pa.out_distal = (double*)ctx->o_distal.p;
        pa.out_pendant = (double*)ctx->o_pendant.p;
        pa.out_status = (int*)ctx->o_status.p;
        pa.keep = io.alt.keep;
        if (io.alt.keep > 1) {
            pa.alt_count = (int*)ctx->o_alt_count.p;
            pa.alt_edge = (int*)ctx->o_alt_edge.p;
            pa.alt_error = (double*)ctx->o_alt_err.p;
            pa.alt_distal = (double*)ctx->o_alt_distal.p;
            pa.alt_pendant = (double*)ctx->o_alt_pendant.p;
            pa.alt_int0 = (unsigned char*)ctx->o_alt_int0.p;
        }
        pa.dbg_query = dbg ? 0 : -1;
        pa.dbg_x1 = dbg ? (double*)ctx->dbg_x1.p : nullptr;
        pa.dbg_x2 = (double*)ctx->dbg_x2.p;
        pa.dbg_err = (double*)ctx->dbg_err.p;
        pa.dbg_valid = (unsigned char*)ctx->dbg_valid.p;
    }

    // count stage and selection of every sub-batch on the main stream, without host synchronisation
    int first_pass() {
        bool used[2] = {false, false};
        const bool staged = !matrix && (io.h_queries || io.h_bytes);   // host input goes through the copy stream
        // host input: a short first sub-batch, so that the compute stream waits for a small copy only; the copies of all later
        // sub-batches hide behind the one before (2.2 ms of exposed PCIe time per 125k-query batch otherwise).  8192 queries: long
        // enough to cover the copy + packing of the full-size sub-batch that follows (0.36 us of compute against 0.1 us of copy per
        // query at config 5 shapes)
        const int ramp = (staged && n > QB) ? std::min(QB, 8192) : QB;
        for (int sb0 = 0, nb = 0, sbi = 0; sb0 < n; sb0 += nb, ++sbi) {
            nb = std::min(sbi == 0 ? ramp : QB, n - sb0);
            const int buf = two_bufs ? (sbi & 1) : 0;
            const void* d_q = nullptr;
            if (stage(sbi, sb0, nb, buf, used[buf], d_q)) return -1;
            used[buf] = used[buf] || staged;
            if (slow_ctx && !io.h_bytes) {   // packed planes in, byte rows needed
                CK(launch_unpack_nuc((const uint32_t*)d_q, nb, ctx->L, ctx->W, ctx->Lp, (uint8_t*)ctx->q_bytes_p.p, s));
                ctx->n_launch += 1;
            }
            if (count(s, d_q, nb, slow_ctx, (const uint8_t*)ctx->q_bytes_p.p, ctx->keys.p)) return -1;
            if (io.stop_after_count) {
                // count-keys export: the rows of this sub-batch, without the padding columns of the key matrix
                const size_t row = (size_t)n_units * key_bytes;
                CK(cudaMemcpy2DAsync((char*)io.h_keys + (size_t)(base0 + sb0) * row, row, ctx->keys.p, (size_t)ldk * key_bytes,
                                     row, nb, cudaMemcpyDeviceToHost, s));
                if (io.h_kmin && sel_kind == SEL_NUC && !slow_ctx) {
                    const size_t mrow = (size_t)((n_units + 31) / 32) * 4;
                    CK(cudaMemcpy2DAsync((char*)io.h_kmin + (size_t)(base0 + sb0) * mrow, mrow, ctx->kmin.p, (size_t)(ldk / 32) * 4,
                                         mrow, nb, cudaMemcpyDeviceToHost, s));
                }
            } else {
                SelectArgs a = sa;
                a.q_begin = sb0;
                if (select(s, a, d_q, nb, slow_ctx, (const uint8_t*)ctx->q_bytes_p.p, ctx->keys.p)) return -1;
            }
            if (used[buf]) CK(cudaEventRecord(ctx->ev_free[buf], s));
        }
        return 0;
    }

    // sub-batch `sbi` (queries sb0 .. sb0 + nb of the batch) to the device.  Host input is staged on the copy stream into
    // buffer `buf`; `reused`: the buffer holds an earlier sub-batch.  d_q = the packed query rows; it stays nullptr for matrix
    // rows (they go to ctx->keys) and in byte mode (byte rows in ctx->q_bytes_p)
    int stage(int sbi, int sb0, int nb, int buf, bool reused, const void*& d_q) {
        if (matrix) {
            Span sp(ctx, T_H2D);
            CK(cudaMemcpyAsync(ctx->keys.p, io.h_rows + (size_t)(base0 + sb0) * ctx->n_cols, (size_t)nb * qrow,
                               cudaMemcpyHostToDevice, s));
            return 0;
        }
        if (!io.h_queries && !io.h_bytes) {
            d_q = (const char*)io.d_queries + (size_t)(base0 + sb0) * qrow;
            return 0;
        }
        // the compute stream waits for the copy, the copy stream waits until the compute stream has finished with the
        // buffer's previous contents
        cudaStream_t cs = ctx->copy_stream;
        if (reused) CK(cudaStreamWaitEvent(cs, ctx->ev_free[buf], 0));
        else if (sbi == 0) {
            // order after whatever the compute stream did before (buffer (re)allocation is synchronous already)
            CK(cudaEventRecord(ctx->ev_free[buf], s));
            CK(cudaStreamWaitEvent(cs, ctx->ev_free[buf], 0));
        }
        void* staging;
        {
            Span sp(ctx, T_H2D, cs);
            if (io.h_queries) {
                staging = buf ? ctx->q_rm2.p : ctx->q_rm.p;
                CK(cudaMemcpyAsync(staging, (const char*)io.h_queries + (size_t)(base0 + sb0) * qrow, (size_t)nb * qrow,
                                   cudaMemcpyHostToDevice, cs));
            } else {
                staging = buf ? ctx->q_bytes2.p : ctx->q_bytes.p;
                CK(cudaMemcpyAsync(staging, io.h_bytes + (size_t)(base0 + sb0) * io.byte_stride, (size_t)nb * io.byte_stride,
                                   cudaMemcpyHostToDevice, cs));
            }
        }
        if (io.h_bytes && !slow_ctx) {
            // packed on the COPY stream, into the buffer that goes with the staging buffer: the packer of sub-batch b + 1
            // runs beside the count kernel of sub-batch b instead of in front of its own (1.1 ms per 125k-query batch)
            void* pk = buf ? ctx->q_rm2.p : ctx->q_rm.p;
            CK(launch_pack(ctx->kind, (const uint8_t*)staging, io.byte_stride, nb, ctx->L, pk, (int*)ctx->bad_flag.p, cs,
                           nuc ? (int*)ctx->q_rowflag.p + sb0 : nullptr));
            ctx->n_launch += 1;
            d_q = pk;
        }
        CK(cudaEventRecord(ctx->ev_ready[buf], cs));
        CK(cudaStreamWaitEvent(s, ctx->ev_ready[buf], 0));
        if (io.h_bytes && slow_ctx) {
            CK(launch_repitch_bytes((const uint8_t*)staging, io.byte_stride, nb, ctx->L, ctx->Lp, (uint8_t*)ctx->q_bytes_p.p, s));
            ctx->n_launch += 1;
        } else if (!io.h_bytes) {
            d_q = staging;
        }
        return 0;
    }

    // count stage of `nb` queries on stream st: their key rows (row stride ldk) into ctx->keys, and for packed nucleotide
    // keys their line minima into ctx->kmin.  d_q = their packed rows; matrix rows are their own keys.  slow: byte-compare fallback, d_qb = the queries' padded byte rows [nb][Lp], 64-bit keys
    // into kw
    int count(cudaStream_t st, const void* d_q, int nb, bool slow, const uint8_t* d_qb, void* kw) {
        if (slow) {
            Span sp(ctx, T_DENSE, st);
            launch_dense_bytes(d_qb, ctx->Lp, nb, (const uint8_t*)ctx->rep_bytes_p.p, ctx->Lp, ctx->n_rep, ctx->Lp,
                               (unsigned long long*)kw, ldk, st);
            ctx->n_launch += 1;
            ctx->n_dense_launch += 1;
            ctx->n_pairs += (double)nb * ctx->n_rep;
            ctx->n_slow += nb;
        } else if (sel_kind == SEL_K2P) {
            const int q_pad = round_up(nb, dense_fp4_tile_rows(0));
            {
                Span sp(ctx, T_TRANSPOSE, st);
                launch_fp4_image((const uint32_t*)d_q, nb, ctx->W, ctx->tc_nw, q_pad, dense_fp4_tile_rows(0), ctx->q_img.p, st);
                ctx->n_launch += 1;
            }
            {
                Span sp(ctx, T_DENSE, st);
                launch_dense_fp4_k2p(ctx->q_img.p, q_pad, ctx->reps_img.p, ctx->tc_rep_pad, ctx->tc_nw,
                                     (unsigned long long*)ctx->keys.p, ldk, ctx->num_sms, st);
                ctx->n_launch += 1;
                ctx->n_dense_launch += 1;
                ctx->n_tc_launch += 1;
                ctx->n_fp4_launch += 1;
                ctx->n_k2p_launch += 1;
            }
            ctx->n_pairs += (double)nb * ctx->n_rep;
        } else if (sel_kind == SEL_NUC && use_tc && ctx->tc_fp4) {
            const int q_pad = round_up(nb, dense_fp4_tile_rows(0));
            {
                Span sp(ctx, T_TRANSPOSE, st);
                launch_fp4_image((const uint32_t*)d_q, nb, ctx->W, ctx->tc_nw, q_pad, dense_fp4_tile_rows(0), ctx->q_img.p, st);
                ctx->n_launch += 1;
            }
            {
                Span sp(ctx, T_DENSE, st);
                launch_dense_fp4(ctx->q_img.p, q_pad, ctx->reps_img.p, ctx->tc_rep_pad, ctx->tc_nw, (uint32_t*)ctx->keys.p, ldk,
                                 (uint32_t*)ctx->kmin.p, sa.gate.vmin, ctx->num_sms, st);
                ctx->n_launch += 1;
                ctx->n_dense_launch += 1;
                ctx->n_tc_launch += 1;
                ctx->n_fp4_launch += 1;
            }
            ctx->n_pairs += (double)nb * ctx->n_rep;
        } else if (sel_kind == SEL_NUC && use_tc) {
            const int q_pad = round_up(nb, 256);
            {
                Span sp(ctx, T_TRANSPOSE, st);
                launch_tc_image((const uint32_t*)d_q, nb, ctx->W, ctx->tc_nw, q_pad, 125, ctx->q_img.p, st);
                ctx->n_launch += 1;
            }
            {
                Span sp(ctx, T_DENSE, st);
                launch_dense_tc(ctx->q_img.p, q_pad, ctx->reps_img.p, ctx->tc_rep_pad, ctx->tc_nw, (uint32_t*)ctx->keys.p, ldk,
                                (uint32_t*)ctx->kmin.p, sa.gate.vmin, ctx->num_sms, st);
                ctx->n_launch += 1;
                ctx->n_dense_launch += 1;
                ctx->n_tc_launch += 1;
            }
            ctx->n_pairs += (double)nb * ctx->n_rep;
        } else if (sel_kind == SEL_NUC) {
            const int nb_pad = round_up(nb, DT_TQ);
            {
                Span sp(ctx, T_TRANSPOSE, st);
                launch_transpose_nuc((const uint32_t*)d_q, nb, ctx->W, (uint32_t*)ctx->q_wm.p, ctx->Wp, nb_pad, DT_TQ, st);
                launch_row_valid((const uint32_t*)d_q, nb, ctx->W, (uint32_t*)ctx->q_nv.p, nb_pad, st);
                ctx->n_launch += 2;
            }
            {
                Span sp(ctx, T_DENSE, st);
                launch_dense_nuc_keys((const uint32_t*)ctx->q_wm.p, (const uint32_t*)ctx->q_nv.p, nb_pad,
                                      (const uint32_t*)ctx->reps_wm.p, (const uint32_t*)ctx->reps_nv.p, ctx->rep_pad,
                                      ctx->W, ctx->Wp, (uint32_t*)ctx->keys.p, ldk, (unsigned long long*)ctx->clk_probe.p,
                                      ctx->num_sms, st);
                launch_line_minima((const uint32_t*)ctx->keys.p, nb, ldk, sa.gate.vmin, (uint32_t*)ctx->kmin.p, st);
                ctx->n_launch += 2;
                ctx->n_dense_launch += 1;
            }
            ctx->n_pairs += (double)nb * ctx->n_rep;
        } else if (sel_kind == SEL_AA) {
            const int q_pad = round_up(nb, AA_TQ);
            {
                Span sp(ctx, T_TRANSPOSE, st);
                launch_aa_layout((const uint8_t*)d_q, nb, ctx->Lp, AA_TQ, q_pad, (uint8_t*)ctx->q_aa_tm.p, (uint32_t*)ctx->q_aav.p, st);
                ctx->n_launch += 1;
            }
            {
                Span sp(ctx, T_DENSE, st);
                launch_dense_aa((const uint8_t*)ctx->q_aa_tm.p, (const uint32_t*)ctx->q_aav.p, q_pad, nb,
                                (const uint8_t*)ctx->reps_aa_tm.p, (const uint32_t*)ctx->reps_aav.p, ctx->aa_rep_pad, ctx->n_rep,
                                ctx->Lp, ctx->L, prm->overlap_frac, (const uint32_t*)ctx->aa_tab.p, (uint32_t*)ctx->aa_valid.p, ldk,
                                (double*)ctx->keys.p, ldk, st);
                ctx->n_launch += 2;
                ctx->n_dense_launch += 1;
                ctx->n_pairs += (double)nb * ctx->n_rep;
            }
        }
        CK(cudaGetLastError());
        return 0;
    }

    // selection of `nb` queries on stream st from the keys of count(); `a` holds the pass's observed-list rows, output map
    // and key rows
    int select(cudaStream_t st, SelectArgs a, const void* d_q, int nb, bool slow, const uint8_t* d_qb,
                   const void* kw) {
        a.n = nb;
        a.q_nuc = (const uint32_t*)d_q;
        a.q_aa = (const uint8_t*)d_q;
        if (slow) {
            a.q_bytes = d_qb;
            a.refs_bytes = (const uint8_t*)ctx->ref_bytes_p.p;
            a.keys_f64 = (const double*)kw;
            a.stash_keys = nullptr;
        }
        {
            Span sp(ctx, T_SELECT, st);
            launch_select(slow ? SEL_NUCW : sel_kind, a, st);
            ctx->n_launch += 1;
        }
        CK(cudaGetLastError());
        return 0;
    }

    // K, V and status of the whole batch to the host
    int fetch_counts(cudaStream_t st) {
        Span sp(ctx, T_D2H, st);
        CK(cudaMemcpyAsync(hK.data(), ctx->Kd.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(hV.data(), ctx->Vd.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(hS.data(), ctx->statusd.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
        return 0;
    }

    // launch classes of the placeable queries, sorted on the device (counts: 5 ints at offset 0, stats: 4 u64 at offset 32),
    // then the one synchronise of the first pass.  exotic = the queries holding bytes other than A,C,G,T,- (they survive
    // fasta2dic only as non-letters and count as ordinary characters in jc69, distance.py:733-737): the 2-bit planes cannot
    // carry them, so those queries are recomputed by the byte-compare fallback; their first-pass results are discarded
    int fetch_classes(std::vector<int>& exotic) {
        const bool flags = io.h_bytes && nuc && !slow_ctx;
        CK(launch_bin_classes(n, (const int*)ctx->statusd.p, (const int*)ctx->Kd.p, (const int*)ctx->Vd.p,
                              flags ? (const int*)ctx->q_rowflag.p : nullptr, (int*)ctx->bin_counts.p, (int*)ctx->bin_lists.p,
                              (unsigned long long*)((char*)ctx->bin_counts.p + 32), s));
        ctx->n_launch += 1;
        CK(cudaMemcpyAsync(h_bin, ctx->bin_counts.p, 32, cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(h_bin_stats, (char*)ctx->bin_counts.p + 32, 32, cudaMemcpyDeviceToHost, s));
        mark("phase 1 launched");
        if (fetch_counts(s)) return -1;
        CK(cudaStreamSynchronize(s));
        mark("phase 1 done on the device");
        if (flags) {
            int bad = 0;
            CK(cudaMemcpy(&bad, ctx->bad_flag.p, 4, cudaMemcpyDeviceToHost));
            if (bad) {
                std::vector<int> row_flag(n);
                CK(cudaMemcpy(row_flag.data(), ctx->q_rowflag.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
                for (int i = 0; i < n; ++i)
                    if (row_flag[i]) exotic.push_back(i);
            }
            // K2P is defined on A,C,G,T,- only: no byte-compare fallback
            if (sel_kind == SEL_K2P && !exotic.empty())
                return fail(ctx, "query row %lld holds a symbol other than A,C,G,T,-, which the K2P model does not define",
                            (long long)(base0 + exotic[0]));
        }
        return 0;
    }

    // the queries that overflowed their slot (not counting the exotic ones, rerun anyway) and ctx->h_over.  The first-level
    // reruns read their key rows from the stash when every overflowing query got a stash row (use_stash; `over` is then in
    // stash order)
    int plan_reruns(const std::vector<int>& exotic, std::vector<int>& over, bool& use_stash) {
        std::vector<char>& is_over = ctx->h_over;
        is_over.assign(n, 0);
        for (int i : exotic) is_over[i] = 1;
        for (int i = 0; i < n; ++i)
            if (hS[i] == ST_OVERFLOW && !is_over[i]) {
                over.push_back(i);
                is_over[i] = 1;
            }
        ctx->n_over += (double)over.size();
        if (stash_cap > 0 && !over.empty() && exotic.empty()) {
            int cnt = 0;
            CK(cudaMemcpy(&cnt, ctx->stash_count.p, 4, cudaMemcpyDeviceToHost));
            if (cnt == (int)over.size() && cnt <= stash_cap) {
                CK(cudaMemcpy(over.data(), ctx->stash_ids.p, (size_t)cnt * 4, cudaMemcpyDeviceToHost));
                use_stash = true;
            }
        }
        return 0;
    }

    // the four shared-memory launch classes (V + 1 <= 64 / 128 / 256 / 512): class c places the count[c] queries at
    // d_ids[begin[c]..], from the rows at d_slots[begin[c]..] of r (d_slots == nullptr: the queries' own rows)
    int place_smem_classes(const int* d_ids, const int* d_slots, const int* begin, const int* count, const ObsRows& r,
                               cudaStream_t st) {
        // (running the classes side by side on extra streams was measured: 4.51 vs 4.56 ms per step -- the first launch fills
        // the shared memory of every SM, so the kernels serialise anyway; kept sequential)
        for (int c = 0; c < PLACE_CLASS_BLOCK; ++c) {
            if (!count[c]) continue;
            CK(launch_place(prm->method, c, place_args(r, count[c], d_ids + begin[c], d_slots ? d_slots + begin[c] : nullptr), st));
            ctx->n_launch += 1;
            ctx->n_place_class[c] += count[c];
        }
        return 0;
    }

    // the block-per-query class (V + 1 > 512): the cnt queries at d_ids (h_ids: the same ids on the host, whose V and K size
    // the exact scratch regions), from the rows at d_slots of r (nullptr: the queries' own rows).  Chunked so that the node
    // slots stay under ctx->scratch_limit; the scratch pool and the offset arrays are reused by the next chunk, hence a
    // synchronise between chunks, and after the last one if sync_last
    int place_block_class(const int* d_ids, const int* h_ids, const int* d_slots, int cnt, const ObsRows& r,
                              cudaStream_t st, bool sync_last) {
        std::vector<long long>& h_rec_off = ctx->h_rec_off;
        std::vector<long long>& h_stack_off = ctx->h_stack_off;
        ctx->n_place_class[PLACE_CLASS_BLOCK] += cnt;
        for (int i0 = 0; i0 < cnt;) {
            long long recs = 0, stk = 0;
            int i1 = i0;
            while (i1 < cnt) {
                const long long v = hV[h_ids[i1]] + 1, k = hK[h_ids[i1]];
                if (i1 > i0 && (size_t)(recs + v) * PLACE_NODE_SLOT_BYTES > ctx->scratch_limit) break;
                h_rec_off[i1 - i0] = recs;
                h_stack_off[i1 - i0] = stk;
                recs += v;
                stk += k;
                ++i1;
            }
            h_rec_off[i1 - i0] = recs;
            h_stack_off[i1 - i0] = stk;
            if (ensure(ctx, ctx->recs, (size_t)std::max<long long>(recs, 1) * PLACE_NODE_SLOT_BYTES)) return -1;
            if (ensure(ctx, ctx->stacks, (size_t)std::max<long long>(stk, 1) * PLACE_CHAIN_SLOT_BYTES)) return -1;
            CK(cudaMemcpyAsync(ctx->rec_off.p, h_rec_off.data(), (size_t)(i1 - i0 + 1) * 8, cudaMemcpyHostToDevice, st));
            CK(cudaMemcpyAsync(ctx->stack_off.p, h_stack_off.data(), (size_t)(i1 - i0 + 1) * 8, cudaMemcpyHostToDevice, st));
            PlaceArgs a = place_args(r, i1 - i0, d_ids + i0, d_slots ? d_slots + i0 : nullptr);
            a.rec_off = (const long long*)ctx->rec_off.p;
            a.stack_off = (const long long*)ctx->stack_off.p;
            a.recs = ctx->recs.p;
            a.stacks = ctx->stacks.p;
            CK(launch_place(prm->method, PLACE_CLASS_BLOCK, a, st));
            ctx->n_launch += 1;
            i0 = i1;
            if (i0 < cnt || sync_last) CK(cudaStreamSynchronize(st));
        }
        return 0;
    }

    // The ordinary queries are placed first, straight from the class lists the device built: no host pass over the batch
    // stands between the last selection kernel and the placement launches, and the host prepares the reruns meanwhile.
    // (Running this pass on a side stream BESIDE the rerun kernels was measured: the step did not change -- the rerun
    // kernels then run with fewer resident blocks and take as much longer as the overlap saves.)
    int place_main_pass() {
        Span sp(ctx, T_PLACE);
        int begin[PLACE_CLASS_BLOCK];
        for (int c = 0; c < PLACE_CLASS_BLOCK; ++c) begin[c] = c * n;
        return place_smem_classes((const int*)ctx->bin_lists.p, nullptr, begin, h_bin, main_rows(), s);
    }

    // the few ordinary queries with more than 511 valid nodes (long unary paths).  Runs after the reruns, which share the
    // scratch pool and whose selection stage should start at once.
    int place_main_block_class() {
        Span sp(ctx, T_PLACE);
        const int nbk = h_bin[PLACE_CLASS_BLOCK];
        if (!nbk) return 0;
        const int* d_ids = (const int*)ctx->bin_lists.p + (size_t)PLACE_CLASS_BLOCK * n;
        std::vector<int> ids(nbk);
        CK(cudaMemcpy(ids.data(), d_ids, (size_t)nbk * 4, cudaMemcpyDeviceToHost));
        return place_block_class(d_ids, ids.data(), nullptr, nbk, main_rows(), s, true);
    }

    // Reruns `list` with slot capacity cap_first, then 16x larger for whoever still overflows (the selection kernel stops a
    // query as soon as it exceeds its slot: 256 -> 4096 -> 65536 -> all leaves).  slow: byte-compare fallback; stash_first:
    // the first level reads its key rows from the stash.  The selection stage (gather, counts, selection, K/V/status) runs on
    // the high-priority side stream, beside the main pass; the placement of the rerun queries runs on the main stream.
    int rerun(std::vector<int> list, bool slow, int cap_first, bool stash_first) {
        const cudaStream_t ss = ctx->side_stream;
        int cap2 = cap_first;
        bool use_st = stash_first;
        if (slow && !slow_ctx && ensure_ref_bytes(ctx, ss)) return -1;
        while (!list.empty()) {
            // queries per rerun launch: bounded by the sub-batch size and by 2 GiB of slots
            const int GB = (int)std::max<int64_t>(1, std::min<int64_t>(QB, ((int64_t)2 << 30) / ((int64_t)cap2 * 16)));
            std::vector<int> still;
            for (size_t o0 = 0; o0 < list.size(); o0 += GB) {
                const int ng = (int)std::min<size_t>(GB, list.size() - o0);
                const int* ids = list.data() + o0;
                if (ensure(ctx, ctx->obs_node2, (size_t)ng * cap2 * 4)) return -1;
                if (ensure(ctx, ctx->obs_dist2, (size_t)ng * cap2 * 8)) return -1;
                if (ensure(ctx, ctx->obs_len2, (size_t)ng * cap2 * 4)) return -1;
                if (!matrix && ensure(ctx, ctx->q_rm, (size_t)QB * qrow)) return -1;
                if (slow && (ensure(ctx, ctx->q_bytes_p, (size_t)QB * ctx->Lp) ||
                             (!slow_ctx && ensure(ctx, ctx->keys_w, (size_t)ng * ldk * 8))))
                    return -1;
                if (gather_rows(ids, ng, slow, ss)) return -1;
                const ObsRows r{cap2, (int*)ctx->obs_node2.p, (double*)ctx->obs_dist2.p, (int*)ctx->obs_len2.p};
                SelectArgs a = sa;
                a.out_map = (const int*)ctx->qlist.p;
                a.q_begin = 0;
                a.cap = r.cap;
                a.obs_node = r.node;
                a.obs_dist = r.dist;
                a.obs_len = r.len;
                a.pair_counter = nullptr;
                a.line_counter = nullptr;
                a.stash_keys = nullptr;
                const void* d_q = matrix ? nullptr : ctx->q_rm.p;
                const uint8_t* d_qb = (const uint8_t*)ctx->q_bytes_p.p;
                void* kw = slow_ctx ? ctx->keys.p : ctx->keys_w.p;
                if (use_st) {
                    a.keys_nuc = (const uint32_t*)ctx->stash_keys.p + (size_t)o0 * ldk;
                    a.kmin = (const uint32_t*)ctx->stash_kmin.p + (size_t)o0 * (ldk / 32);
                }
                else if (count(ss, d_q, ng, slow, d_qb, kw)) return -1;
                if (select(ss, a, d_q, ng, slow, d_qb, kw)) return -1;
                mark("  rerun select launched");
                if (fetch_counts(ss)) return -1;
                CK(cudaStreamSynchronize(ss));
                mark("  rerun select done");
                if (io.obs_count && export_rerun_rows(ids, ng, r)) return -1;
                if (!io.stop_after_select) {
                    if (place_rerun_group(ids, ng, r)) return -1;
                    CK(cudaStreamSynchronize(s));
                }
                for (int j = 0; j < ng; ++j)
                    if (hS[ids[j]] == ST_OVERFLOW) still.push_back(ids[j]);
            }
            if (cap2 >= cap_max && !still.empty()) return fail(ctx, "internal error: observed set larger than the number of leaves");
            list.swap(still);
            cap2 = (int)std::min<int64_t>((int64_t)cap2 * 16, cap_max);
            use_st = false;  // deeper levels recompute: their rows are no longer contiguous in the stash
        }
        return 0;
    }

    // rows of the ng rerun queries `ids` (batch-relative) to the device on stream ss: the ids to ctx->qlist, packed rows to
    // ctx->q_rm (slow: byte rows to ctx->q_bytes_p), matrix rows to ctx->keys
    int gather_rows(const int* ids, int ng, bool slow, cudaStream_t ss) {
        CK(cudaMemcpyAsync(ctx->qlist.p, ids, (size_t)ng * 4, cudaMemcpyHostToDevice, ss));
        // one kernel for device-resident queries, one host-side gather + one copy otherwise (a memcpy call per row would cost
        // more than the rerun itself)
        if (!matrix && !io.h_queries && !io.h_bytes) {
            // qlist holds batch-relative ids; the resident rows of this macro-batch start at base0
            CK(launch_gather_rows((const char*)io.d_queries + (size_t)base0 * qrow, (const int*)ctx->qlist.p, ctx->q_rm.p, ng,
                                  qrow, ss));
            ctx->n_launch += 1;
        } else {
            const size_t rb = matrix ? qrow : (io.h_queries ? qrow : (size_t)io.byte_stride);
            const char* src = matrix ? (const char*)io.h_rows : (io.h_queries ? (const char*)io.h_queries : (const char*)io.h_bytes);
            ctx->h_gather.resize((size_t)ng * rb);
            for (int j = 0; j < ng; ++j) memcpy(ctx->h_gather.data() + (size_t)j * rb, src + ((size_t)base0 + ids[j]) * rb, rb);
            void* dst = matrix ? ctx->keys.p : (io.h_queries ? ctx->q_rm.p : ctx->q_bytes.p);
            CK(cudaMemcpyAsync(dst, ctx->h_gather.data(), (size_t)ng * rb, cudaMemcpyHostToDevice, ss));
            CK(cudaStreamSynchronize(ss));  // h_gather is reused by the next group
        }
        if (io.h_bytes && slow)
            CK(launch_repitch_bytes((const uint8_t*)ctx->q_bytes.p, io.byte_stride, ng, ctx->L, ctx->Lp, (uint8_t*)ctx->q_bytes_p.p, ss));
        else if (io.h_bytes)
            CK(launch_pack(ctx->kind, (const uint8_t*)ctx->q_bytes.p, io.byte_stride, ng, ctx->L, ctx->q_rm.p, (int*)ctx->bad_flag.p, ss));
        else if (slow)
            CK(launch_unpack_nuc((const uint32_t*)ctx->q_rm.p, ng, ctx->L, ctx->W, ctx->Lp, (uint8_t*)ctx->q_bytes_p.p, ss));
        return 0;
    }

    // placement of the ng rerun queries `ids` (query ids[j] from row j of r) on the main stream, sorted into the launch
    // classes on the host
    int place_rerun_group(const int* ids, int ng, const ObsRows& r) {
        int sizes[PLACE_NCLASS] = {0, 0, 0, 0, 0};
        for (int j = 0; j < ng; ++j)
            if (hS[ids[j]] == ST_PLACE) sizes[place_class(hV[ids[j]])]++;
        int begin[PLACE_NCLASS + 1];
        begin[0] = 0;
        for (int c = 0; c < PLACE_NCLASS; ++c) begin[c + 1] = begin[c] + sizes[c];
        const int total = begin[PLACE_NCLASS];
        if (total == 0) return 0;
        // [query ids by class | their rows in r]
        std::vector<int>& lists = ctx->h_pl_lists;
        lists.resize((size_t)2 * total);
        int fill[PLACE_NCLASS];
        for (int c = 0; c < PLACE_NCLASS; ++c) fill[c] = begin[c];
        for (int j = 0; j < ng; ++j) {
            const int qi = ids[j];
            if (hS[qi] != ST_PLACE) continue;
            const int pos = fill[place_class(hV[qi])]++;
            lists[pos] = qi;
            lists[(size_t)total + pos] = j;
        }
        if (ensure(ctx, ctx->pl_lists, (size_t)2 * total * 4)) return -1;
        CK(cudaMemcpyAsync(ctx->pl_lists.p, lists.data(), (size_t)2 * total * 4, cudaMemcpyHostToDevice, s));
        const int* d_ids = (const int*)ctx->pl_lists.p;
        const int* d_slots = d_ids + total;
        Span sp(ctx, T_PLACE);
        if (place_smem_classes(d_ids, d_slots, begin, sizes, r, s)) return -1;
        const int b = begin[PLACE_CLASS_BLOCK];
        return place_block_class(d_ids + b, lists.data() + b, d_slots + b, sizes[PLACE_CLASS_BLOCK], r, s, false);
    }

    // parity export of the observed sets of the rerun queries that fit their slots now (query ids[j] in row j of r)
    int export_rerun_rows(const int* ids, int ng, const ObsRows& r) {
        std::vector<int> un((size_t)ng * r.cap);
        std::vector<double> ud((size_t)ng * r.cap);
        CK(cudaMemcpy(un.data(), r.node, un.size() * 4, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(ud.data(), r.dist, ud.size() * 8, cudaMemcpyDeviceToHost));
        for (int j = 0; j < ng; ++j) {
            const int i = ids[j];
            if (hS[i] == ST_OVERFLOW) continue;
            const int k = std::min(hK[i], io.obs_cap);
            memcpy(io.obs_node + (size_t)(base0 + i) * io.obs_cap, &un[(size_t)j * r.cap], (size_t)k * 4);
            memcpy(io.obs_dist + (size_t)(base0 + i) * io.obs_cap, &ud[(size_t)j * r.cap], (size_t)k * 8);
        }
        return 0;
    }

    // parity export of the observed sets: the counts of every query, the lists of those the reruns did not export
    int export_observed() {
        const int ocap = io.obs_cap;
        std::vector<int> tn((size_t)n * cap);
        std::vector<double> td((size_t)n * cap);
        CK(cudaMemcpy(tn.data(), ctx->obs_node.p, tn.size() * 4, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(td.data(), ctx->obs_dist.p, td.size() * 8, cudaMemcpyDeviceToHost));
        for (int i = 0; i < n; ++i) {
            io.obs_count[base0 + i] = hK[i];
            if (ctx->h_over[i]) continue;
            const int k = std::min(std::min(hK[i], cap), ocap);
            memcpy(io.obs_node + (size_t)(base0 + i) * ocap, &tn[(size_t)i * cap], (size_t)k * 4);
            memcpy(io.obs_dist + (size_t)(base0 + i) * ocap, &td[(size_t)i * cap], (size_t)k * 8);
        }
        return 0;
    }

    // statistics: the device summed the ordinary queries while sorting them, the rerun ones are few
    void add_stats(const std::vector<int>& exotic, const std::vector<int>& over) {
        ctx->n_obs += (double)h_bin_stats[0];
        ctx->n_valid += (double)h_bin_stats[1];
        ctx->max_K = std::max(ctx->max_K, (double)h_bin_stats[2]);
        ctx->max_V = std::max(ctx->max_V, (double)h_bin_stats[3]);
        for (const std::vector<int>* lst : {&exotic, &over})
            for (int i : *lst)
                if (hS[i] == ST_PLACE) {
                    ctx->n_obs += hK[i];
                    ctx->n_valid += hV[i];
                    ctx->max_K = std::max(ctx->max_K, (double)hK[i]);
                    ctx->max_V = std::max(ctx->max_V, (double)hV[i]);
                }
    }

    // zero-distance shortcut / too-few-distances records of the whole batch, then the results D2H (D2D for resident output)
    int place_tail() {
        {
            Span sp(ctx, T_PLACE);
            PlaceArgs a = pa;
            a.n = n;
            CK(launch_place_finalize(a, s));
            ctx->n_launch += 1;
        }
        Span sp(ctx, T_D2H);
        const cudaMemcpyKind kd = io.out_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
        CK(cudaMemcpyAsync(io.edge + base0, ctx->o_edge.p, (size_t)n * 4, kd, s));
        CK(cudaMemcpyAsync(io.error + base0, ctx->o_err.p, (size_t)n * 8, kd, s));
        CK(cudaMemcpyAsync(io.distal + base0, ctx->o_distal.p, (size_t)n * 8, kd, s));
        CK(cudaMemcpyAsync(io.pendant + base0, ctx->o_pendant.p, (size_t)n * 8, kd, s));
        CK(cudaMemcpyAsync(io.status + base0, ctx->o_status.p, (size_t)n * 4, kd, s));
        const AltOut& al = io.alt;
        if (al.keep > 1) {
            const size_t o = (size_t)base0 * al.keep, nk = (size_t)n * al.keep;
            CK(cudaMemcpyAsync(al.count + base0, ctx->o_alt_count.p, (size_t)n * 4, cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(al.edge + o, ctx->o_alt_edge.p, nk * 4, cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(al.error + o, ctx->o_alt_err.p, nk * 8, cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(al.distal + o, ctx->o_alt_distal.p, nk * 8, cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(al.pendant + o, ctx->o_alt_pendant.p, nk * 8, cudaMemcpyDeviceToHost, s));
            CK(cudaMemcpyAsync(al.int0 + o, ctx->o_alt_int0.p, nk, cudaMemcpyDeviceToHost, s));
        }
        return 0;
    }

    // the batch's one synchronise at the end, then the per-edge export, the pair count, the SM clock and the stage times
    int finish() {
        CK(cudaStreamSynchronize(s));
        mark("batch done");
        if (io.dbg_x1) {
            CK(cudaMemcpy(io.dbg_x1, ctx->dbg_x1.p, (size_t)ctx->M * 8, cudaMemcpyDeviceToHost));
            CK(cudaMemcpy(io.dbg_x2, ctx->dbg_x2.p, (size_t)ctx->M * 8, cudaMemcpyDeviceToHost));
            CK(cudaMemcpy(io.dbg_err, ctx->dbg_err.p, (size_t)ctx->M * 8, cudaMemcpyDeviceToHost));
            CK(cudaMemcpy(io.dbg_valid, ctx->dbg_valid.p, (size_t)ctx->M, cudaMemcpyDeviceToHost));
        }
        unsigned long long pc[2] = {0, 0};
        CK(cudaMemcpy(pc, ctx->pair_counter.p, 16, cudaMemcpyDeviceToHost));
        ctx->n_pairs += (double)pc[0];
        ctx->n_lines += (double)pc[1];
        if (sel_kind == SEL_NUC && !matrix && ctx->clk_probe.p) {
            unsigned long long c[4] = {0, 0, 0, 0};
            CK(cudaMemcpy(c, ctx->clk_probe.p, 32, cudaMemcpyDeviceToHost));
            if (c[3] > c[1]) ctx->dense_mhz = 1e3 * (double)(c[2] - c[0]) / (double)(c[3] - c[1]);
        }
        collect_spans(ctx);
        return 0;
    }
};

// the registration of apples_set_alternatives, cleared: it serves one apples_place_batch* call
AltOut take_alternatives(apples_ctx* ctx) {
    const AltOut a = ctx->alt;
    ctx->alt = AltOut{};
    return a;
}

int run_macro(apples_ctx* ctx, int64_t base0, int n, const BatchIO& io, const apples_params* prm) {
    return MacroBatch(ctx, base0, n, io, prm).run();
}

// the whole pipeline for nq queries
int run_batch(apples_ctx* ctx, int64_t nq, const BatchIO& io, const apples_params* prm) {
    if (check_params(ctx, prm)) return -1;
    if (ctx->M <= 0) return fail(ctx, "apples_set_tree has not been called");
    const bool matrix = io.h_rows != nullptr;
    if (matrix && ctx->n_cols <= 0) return fail(ctx, "apples_set_matrix_columns has not been called");
    if (!matrix && ctx->kind < 0) return fail(ctx, "apples_set_reference has not been called");
    if (nq <= 0) return 0;
    CK(cudaSetDevice(ctx->device));
    for (int64_t b0 = 0; b0 < nq; b0 += ctx->max_batch) {
        const int n = (int)std::min<int64_t>(ctx->max_batch, nq - b0);
        if (run_macro(ctx, b0, n, io, prm)) return -1;
    }
    return 0;
}

}  // namespace

// =================================================================================================================
extern "C" {

void apples_ctx_destroy(apples_ctx* ctx);

int32_t apples_words_per_row(int32_t L) { return ((L + 31) / 32 + 3) / 4 * 4; }
int32_t apples_aa_row_bytes(int32_t L) { return (L + 15) / 16 * 16; }

int apples_device_count(int32_t* count) {
    if (!count) return -1;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        *count = 0;
        return -2;
    }
    *count = n;
    return 0;
}

int apples_ctx_create(int device, apples_ctx** out) {
    if (!out) return -1;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device < 0 || device >= n) return -2;
    if (cudaSetDevice(device) != cudaSuccess) return -3;
    apples_ctx* ctx = new apples_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->num_sms = prop.multiProcessorCount;
    int rc = 0;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) rc = -4;
    if (!rc && cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking) != cudaSuccess) rc = -4;
    for (int i = 0; i < 2 && !rc; ++i)
        if (cudaEventCreateWithFlags(&ctx->ev_ready[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&ctx->ev_free[i], cudaEventDisableTiming) != cudaSuccess)
            rc = -4;
    int prio_lo = 0, prio_hi = 0;   // side stream: the rerun selection beside the main placement pass must not queue behind it
    if (!rc) cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    if (!rc && cudaStreamCreateWithPriority(&ctx->side_stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess) rc = -4;
    if (!rc && dense_nuc_configure() != cudaSuccess) rc = -5;
    if (!rc && dense_tc_configure() != cudaSuccess) rc = -5;
    if (rc) {
        apples_ctx_destroy(ctx);  // releases whatever was created
        return rc;
    }
    *out = ctx;
    return 0;
}

void apples_ctx_destroy(apples_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (auto e : ctx->ev_pool) cudaEventDestroy(e);
    for (auto& sp : ctx->spans) {
        cudaEventDestroy(sp.a);
        cudaEventDestroy(sp.b);
    }
    for (int i = 0; i < 2; ++i) {
        if (ctx->ev_ready[i]) cudaEventDestroy(ctx->ev_ready[i]);
        if (ctx->ev_free[i]) cudaEventDestroy(ctx->ev_free[i]);
    }
    if (ctx->side_stream) {
        cudaStreamSynchronize(ctx->side_stream);
        cudaStreamDestroy(ctx->side_stream);
    }
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;   // frees the device buffers
}

const char* apples_last_error(const apples_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
void* apples_ctx_stream(apples_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

int apples_ctx_set_limits(apples_ctx* ctx, int64_t max_subbatch, int64_t scratch_bytes, int32_t slot_cap) {
    if (!ctx) return -1;
    if (max_subbatch > 0) ctx->max_subbatch = max_subbatch;
    if (scratch_bytes > 0) ctx->scratch_limit = (size_t)scratch_bytes;
    if (slot_cap > 0) ctx->slot_cap = next_pow2(std::max(4, slot_cap));
    return 0;
}

int apples_ctx_set_dense_mode(apples_ctx* ctx, int32_t mode) {
    if (!ctx) return -1;
    if (mode != 0 && mode != 1) return fail(ctx, "apples_ctx_set_dense_mode: mode must be 0 (integer pipes) or 1 (tensor cores)");
    ctx->dense_mode = mode;
    ctx->tc_ready = false;   // takes effect with the next apples_set_reference*
    return 0;
}

int apples_ctx_set_model(apples_ctx* ctx, int32_t model) {
    if (!ctx) return -1;
    if (model != APPLES_JC69 && model != APPLES_K2P)
        return fail(ctx, "apples_ctx_set_model: model must be %d (JC69) or %d (K2P)", APPLES_JC69, APPLES_K2P);
    ctx->model = model;   // takes effect with the next apples_set_reference*
    return 0;
}

int apples_set_tree(apples_ctx* ctx, int32_t M, const int32_t* parent, const double* edge_length, const int32_t* level,
                    const int32_t* first) {
    if (!ctx) return -1;
    if (M < 2 || !parent || !edge_length || !level || !first) return fail(ctx, "apples_set_tree: bad arguments");
    for (int u = 0; u < M - 1; ++u)
        if (parent[u] <= u || parent[u] >= M) return fail(ctx, "apples_set_tree: node ids must be post-order ranks");
    if (parent[M - 1] != -1) return fail(ctx, "apples_set_tree: last node must be the root");
    for (int u = 0; u < M; ++u) {
        if (first[u] < 0 || first[u] > u) return fail(ctx, "apples_set_tree: first[%d] = %d is not the smallest id of the subtree", u, first[u]);
        if (level[u] < 0 || (u < M - 1 && level[u] != level[parent[u]] + 1))
            return fail(ctx, "apples_set_tree: level[%d] = %d is not the depth of the node", u, level[u]);
    }
    CK(cudaSetDevice(ctx->device));
    if (ensure(ctx, ctx->t_parent, (size_t)M * 4) || ensure(ctx, ctx->t_elen, (size_t)M * 8) ||
        ensure(ctx, ctx->t_level, (size_t)M * 4) || ensure(ctx, ctx->t_first, (size_t)M * 4))
        return -1;
    CK(cudaMemcpy(ctx->t_parent.p, parent, (size_t)M * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->t_elen.p, edge_length, (size_t)M * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->t_level.p, level, (size_t)M * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->t_first.p, first, (size_t)M * 4, cudaMemcpyHostToDevice));
    ctx->M = M;
    ctx->h_first.assign(first, first + M);
    if (check_leaf_ids(ctx, "ref_node", ctx->h_ref_node.data(), (int)ctx->h_ref_node.size()) ||
        check_leaf_ids(ctx, "col_node", ctx->h_col_node.data(), (int)ctx->h_col_node.size()))
        return -1;
    return 0;
}

int apples_set_reference(apples_ctx* ctx, int kind, int32_t L, int32_t n_ref, const void* packed_refs,
                         const int32_t* ref_node, int32_t n_rep, const void* packed_reps, const int32_t* group_offsets,
                         const int32_t* group_members) {
    if (!ctx) return -1;
    if ((kind != APPLES_NUC && kind != APPLES_AA) || L <= 0 || n_ref <= 0 || n_rep <= 0 || !packed_refs || !ref_node ||
        !packed_reps || !group_offsets || !group_members)
        return fail(ctx, "apples_set_reference: bad arguments");
    if (check_reference(ctx, "apples_set_reference", n_ref, ref_node, n_rep, group_offsets, group_members) ||
        check_model(ctx, "apples_set_reference", kind, L))
        return -1;
    const int n_mem = group_offsets[n_rep];
    if (set_geometry(ctx, kind, L, n_ref, ref_node, n_rep, n_mem)) return -1;
    const size_t row = query_row_bytes(ctx);
    CK(cudaMemcpy(ctx->refs_rm.p, packed_refs, (size_t)n_ref * row, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->reps_rm.p, packed_reps, (size_t)n_rep * row, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->ref_node.p, ref_node, (size_t)n_ref * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->goff.p, group_offsets, (size_t)(n_rep + 1) * 4, cudaMemcpyHostToDevice));
    if (n_mem) CK(cudaMemcpy(ctx->gmem.p, group_members, (size_t)n_mem * 4, cudaMemcpyHostToDevice));
    // 16-bit counts do not hold beyond 65 535 columns: the whole context runs the byte-compare fallback (32-bit counts,
    // 64-bit keys)
    ctx->nuc_slow = kind == APPLES_NUC && L > 65535;
    if (prepare_operands(ctx, ctx->stream) || (ctx->nuc_slow && ensure_ref_bytes(ctx, ctx->stream))) return -1;
    CK(cudaStreamSynchronize(ctx->stream));
    return 0;
}

int apples_set_matrix_columns(apples_ctx* ctx, int32_t n_cols, const int32_t* col_node) {
    if (!ctx) return -1;
    if (n_cols <= 0 || !col_node) return fail(ctx, "apples_set_matrix_columns: bad arguments");
    if (check_leaf_ids(ctx, "col_node", col_node, n_cols)) return -1;
    ctx->h_col_node.assign(col_node, col_node + n_cols);
    CK(cudaSetDevice(ctx->device));
    if (ensure(ctx, ctx->col_node, (size_t)n_cols * 4)) return -1;
    CK(cudaMemcpy(ctx->col_node.p, col_node, (size_t)n_cols * 4, cudaMemcpyHostToDevice));
    ctx->n_cols = n_cols;
    return 0;
}

int apples_set_alternatives(apples_ctx* ctx, int32_t keep, int32_t* count, int32_t* edge, double* error, double* distal,
                            double* pendant, uint8_t* pendant_int0) {
    if (!ctx) return -1;
    ctx->alt = AltOut{};
    if (keep < 1 || keep > APPLES_MAX_KEEP)
        return fail(ctx, "apples_set_alternatives: keep = %d is outside [1, %d]", keep, APPLES_MAX_KEEP);
    const int given = !!count + !!edge + !!error + !!distal + !!pendant + !!pendant_int0;
    if (keep == 1 || given == 0) return 0;
    if (given != 6) return fail(ctx, "apples_set_alternatives: pass all six buffers or none");
    ctx->alt.keep = keep;
    ctx->alt.count = count;
    ctx->alt.edge = edge;
    ctx->alt.error = error;
    ctx->alt.distal = distal;
    ctx->alt.pendant = pendant;
    ctx->alt.int0 = pendant_int0;
    return 0;
}

int apples_place_batch(apples_ctx* ctx, int64_t nq, const void* packed_queries, const int32_t* self_node,
                       const apples_params* params, int32_t* edge, double* error, double* distal, double* pendant,
                       int32_t* status) {
    if (!ctx) return -1;
    const AltOut alt = take_alternatives(ctx);
    if (nq < 0 || (nq > 0 && (!packed_queries || !edge || !error || !distal || !pendant || !status)))
        return fail(ctx, "apples_place_batch: bad arguments");
    BatchIO io;
    io.h_queries = packed_queries;
    io.h_self = self_node;
    io.edge = edge; io.error = error; io.distal = distal; io.pendant = pendant; io.status = status;
    io.alt = alt;
    return run_batch(ctx, nq, io, params);
}

int apples_place_batch_bytes(apples_ctx* ctx, int64_t nq, const uint8_t* bytes, int64_t row_stride,
                             const int32_t* self_node, const apples_params* params, int32_t* edge, double* error,
                             double* distal, double* pendant, int32_t* status) {
    if (!ctx) return -1;
    const AltOut alt = take_alternatives(ctx);
    if (ctx->kind < 0) return fail(ctx, "apples_set_reference has not been called");
    if (nq < 0 || (nq > 0 && (!bytes || row_stride < ctx->L || !edge || !error || !distal || !pendant || !status)))
        return fail(ctx, "apples_place_batch_bytes: bad arguments");
    BatchIO io;
    io.h_bytes = bytes;
    io.byte_stride = row_stride;
    io.h_self = self_node;
    io.edge = edge; io.error = error; io.distal = distal; io.pendant = pendant; io.status = status;
    io.alt = alt;
    return run_batch(ctx, nq, io, params);
}

int apples_set_reference_bytes(apples_ctx* ctx, int kind, int32_t L, int32_t n_ref, const uint8_t* ref_bytes,
                               int64_t row_stride, const int32_t* ref_node, int32_t n_rep, const int32_t* group_offsets,
                               const int32_t* group_members) {
    if (!ctx) return -1;
    if ((kind != APPLES_NUC && kind != APPLES_AA) || L <= 0 || n_ref <= 0 || n_rep <= 0 || !ref_bytes || row_stride < L ||
        !ref_node || !group_offsets || !group_members)
        return fail(ctx, "apples_set_reference_bytes: bad arguments");
    if (check_reference(ctx, "apples_set_reference_bytes", n_ref, ref_node, n_rep, group_offsets, group_members) ||
        check_model(ctx, "apples_set_reference_bytes", kind, L))
        return -1;
    const int n_mem = group_offsets[n_rep];
    if (set_geometry(ctx, kind, L, n_ref, ref_node, n_rep, n_mem)) return -1;
    cudaStream_t s = ctx->stream;
    DevBuf d_bytes, d_rep_bytes;
    if (ensure(ctx, ctx->bad_flag, 4) || ensure(ctx, d_bytes, (size_t)n_ref * row_stride) ||
        ensure(ctx, d_rep_bytes, (size_t)n_rep * L))
        return -1;
    CK(cudaMemcpyAsync(d_bytes.p, ref_bytes, (size_t)n_ref * row_stride, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(ctx->ref_node.p, ref_node, (size_t)n_ref * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(ctx->goff.p, group_offsets, (size_t)(n_rep + 1) * 4, cudaMemcpyHostToDevice, s));
    if (n_mem) CK(cudaMemcpyAsync(ctx->gmem.p, group_members, (size_t)n_mem * 4, cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(ctx->bad_flag.p, 0, 4, s));
    // (f2) consensus representatives, then (f1) packing of references and representatives
    CK(launch_consensus(kind, (const uint8_t*)d_bytes.p, row_stride, L, n_rep, (const int*)ctx->goff.p, (const int*)ctx->gmem.p,
                        (uint8_t*)d_rep_bytes.p, L, s));
    CK(launch_pack(kind, (const uint8_t*)d_bytes.p, row_stride, n_ref, L, ctx->refs_rm.p, (int*)ctx->bad_flag.p, s));
    CK(launch_pack(kind, (const uint8_t*)d_rep_bytes.p, L, n_rep, L, ctx->reps_rm.p, (int*)ctx->bad_flag.p, s));
    int bad = 0;
    CK(cudaMemcpyAsync(&bad, ctx->bad_flag.p, 4, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    // the reference holds bytes other than A,C,G,T,- (ordinary characters for jc69, distance.py:733-737) or is longer
    // than the 16-bit counts allow: keep the byte rows, every query of this context takes the byte-compare fallback
    ctx->nuc_slow = kind == APPLES_NUC && (bad || L > 65535);
    if (ctx->nuc_slow && ctx->k2p) {
        ctx->kind = -1;   // the half-installed reference is unusable
        return fail(ctx, "apples_set_reference_bytes: the reference holds symbols other than A,C,G,T,-, which the K2P model "
                         "does not define");
    }
    if (prepare_operands(ctx, s)) return -1;
    if (ctx->nuc_slow) {
        if (ensure(ctx, ctx->ref_bytes_p, (size_t)n_ref * ctx->Lp) || ensure(ctx, ctx->rep_bytes_p, (size_t)n_rep * ctx->Lp))
            return -1;
        CK(launch_repitch_bytes((const uint8_t*)d_bytes.p, row_stride, n_ref, L, ctx->Lp, (uint8_t*)ctx->ref_bytes_p.p, s));
        CK(launch_repitch_bytes((const uint8_t*)d_rep_bytes.p, L, n_rep, L, ctx->Lp, (uint8_t*)ctx->rep_bytes_p.p, s));
    }
    CK(cudaStreamSynchronize(s));
    ctx->bytes_ready = ctx->nuc_slow;
    return 0;
}

int apples_place_batch_matrix(apples_ctx* ctx, int64_t nq, const double* rows, const int32_t* self_node,
                              const apples_params* params, int32_t* edge, double* error, double* distal,
                              double* pendant, int32_t* status) {
    if (!ctx) return -1;
    const AltOut alt = take_alternatives(ctx);
    if (nq < 0 || (nq > 0 && (!rows || !edge || !error || !distal || !pendant || !status)))
        return fail(ctx, "apples_place_batch_matrix: bad arguments");
    BatchIO io;
    io.h_rows = rows;
    io.h_self = self_node;
    io.edge = edge; io.error = error; io.distal = distal; io.pendant = pendant; io.status = status;
    io.alt = alt;
    return run_batch(ctx, nq, io, params);
}

int apples_queries_upload(apples_ctx* ctx, int64_t nq, const void* packed_queries, const int32_t* self_node) {
    if (!ctx) return -1;
    if (ctx->kind < 0) return fail(ctx, "apples_set_reference has not been called");
    if (nq <= 0 || !packed_queries) return fail(ctx, "apples_queries_upload: bad arguments");
    CK(cudaSetDevice(ctx->device));
    const size_t row = query_row_bytes(ctx);
    if (ensure(ctx, ctx->res_q, (size_t)nq * row)) return -1;
    CK(cudaMemcpy(ctx->res_q.p, packed_queries, (size_t)nq * row, cudaMemcpyHostToDevice));
    ctx->res_has_self = self_node != nullptr;
    if (self_node) {
        if (ensure(ctx, ctx->res_self, (size_t)nq * 4)) return -1;
        CK(cudaMemcpy(ctx->res_self.p, self_node, (size_t)nq * 4, cudaMemcpyHostToDevice));
    }
    if (ensure(ctx, ctx->res_edge, (size_t)nq * 4) || ensure(ctx, ctx->res_err, (size_t)nq * 8) ||
        ensure(ctx, ctx->res_distal, (size_t)nq * 8) || ensure(ctx, ctx->res_pendant, (size_t)nq * 8) ||
        ensure(ctx, ctx->res_status, (size_t)nq * 4))
        return -1;
    ctx->res_nq = nq;
    return 0;
}

int apples_place_resident(apples_ctx* ctx, const apples_params* params) {
    if (!ctx) return -1;
    if (ctx->res_nq <= 0) return fail(ctx, "apples_queries_upload has not been called");
    BatchIO io;
    io.d_queries = ctx->res_q.p;
    io.d_self = ctx->res_has_self ? (const int32_t*)ctx->res_self.p : nullptr;
    io.edge = (int32_t*)ctx->res_edge.p; io.error = (double*)ctx->res_err.p; io.distal = (double*)ctx->res_distal.p;
    io.pendant = (double*)ctx->res_pendant.p; io.status = (int32_t*)ctx->res_status.p;
    io.out_on_device = true;
    return run_batch(ctx, ctx->res_nq, io, params);
}

int apples_results_download(apples_ctx* ctx, int32_t* edge, double* error, double* distal, double* pendant,
                            int32_t* status) {
    if (!ctx) return -1;
    if (ctx->res_nq <= 0) return fail(ctx, "no resident results");
    const size_t n = (size_t)ctx->res_nq;
    CK(cudaSetDevice(ctx->device));
    if (edge) CK(cudaMemcpy(edge, ctx->res_edge.p, n * 4, cudaMemcpyDeviceToHost));
    if (error) CK(cudaMemcpy(error, ctx->res_err.p, n * 8, cudaMemcpyDeviceToHost));
    if (distal) CK(cudaMemcpy(distal, ctx->res_distal.p, n * 8, cudaMemcpyDeviceToHost));
    if (pendant) CK(cudaMemcpy(pendant, ctx->res_pendant.p, n * 8, cudaMemcpyDeviceToHost));
    if (status) CK(cudaMemcpy(status, ctx->res_status.p, n * 4, cudaMemcpyDeviceToHost));
    return 0;
}

int apples_results_to_device(apples_ctx* ctx, void* edge, void* error, void* distal, void* pendant, void* status) {
    if (!ctx) return -1;
    if (ctx->res_nq <= 0) return fail(ctx, "no resident results");
    const size_t n = (size_t)ctx->res_nq;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    if (edge) CK(cudaMemcpyAsync(edge, ctx->res_edge.p, n * 4, cudaMemcpyDeviceToDevice, s));
    if (error) CK(cudaMemcpyAsync(error, ctx->res_err.p, n * 8, cudaMemcpyDeviceToDevice, s));
    if (distal) CK(cudaMemcpyAsync(distal, ctx->res_distal.p, n * 8, cudaMemcpyDeviceToDevice, s));
    if (pendant) CK(cudaMemcpyAsync(pendant, ctx->res_pendant.p, n * 8, cudaMemcpyDeviceToDevice, s));
    if (status) CK(cudaMemcpyAsync(status, ctx->res_status.p, n * 4, cudaMemcpyDeviceToDevice, s));
    CK(cudaStreamSynchronize(s));
    return 0;
}

int apples_distance_counts(apples_ctx* ctx, int64_t nq, const void* packed_queries, double overlap_frac, uint32_t* mism,
                           uint32_t* valid, double* dist) {
    if (!ctx) return -1;
    if (ctx->kind < 0) return fail(ctx, "apples_set_reference has not been called");
    if (nq <= 0 || !packed_queries || !mism || !valid || !dist) return fail(ctx, "apples_distance_counts: bad arguments");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const size_t row = query_row_bytes(ctx);
    const size_t n_out = (size_t)nq * ctx->n_ref;
    DevBuf dq, dm, dv, dd, qwm, qnv;
    if (ensure(ctx, dq, (size_t)nq * row) || ensure(ctx, dm, n_out * 4) || ensure(ctx, dv, n_out * 4) ||
        ensure(ctx, dd, n_out * 8))
        return -1;
    cudaMemcpyAsync(dq.p, packed_queries, (size_t)nq * row, cudaMemcpyHostToDevice, s);
    cudaMemsetAsync(dm.p, 0, n_out * 4, s);
    if (ctx->kind == APPLES_NUC && ctx->nuc_slow) {
        DevBuf qb, kw;
        if (ensure(ctx, qb, (size_t)nq * ctx->Lp) || ensure(ctx, kw, n_out * 8)) return -1;
        launch_unpack_nuc((const uint32_t*)dq.p, (int)nq, ctx->L, ctx->W, ctx->Lp, (uint8_t*)qb.p, s);
        launch_dense_bytes((const uint8_t*)qb.p, ctx->Lp, (int)nq, (const uint8_t*)ctx->ref_bytes_p.p, ctx->Lp, ctx->n_ref, ctx->Lp,
                           (unsigned long long*)kw.p, ctx->n_ref, s);
        launch_bytes_keys_to_counts((const unsigned long long*)kw.p, (int64_t)n_out, overlap_vmin(ctx->L, overlap_frac), (uint32_t*)dm.p,
                                    (uint32_t*)dv.p, (double*)dd.p, s);
        cudaError_t e2 = cudaGetLastError();
        if (e2 == cudaSuccess) e2 = cudaMemcpyAsync(mism, dm.p, n_out * 4, cudaMemcpyDeviceToHost, s);
        if (e2 == cudaSuccess) e2 = cudaMemcpyAsync(valid, dv.p, n_out * 4, cudaMemcpyDeviceToHost, s);
        if (e2 == cudaSuccess) e2 = cudaMemcpyAsync(dist, dd.p, n_out * 8, cudaMemcpyDeviceToHost, s);
        if (e2 == cudaSuccess) e2 = cudaStreamSynchronize(s);
        if (e2 != cudaSuccess) return fail(ctx, "apples_distance_counts: %s", cudaGetErrorString(e2));
        return 0;
    }
    if (ctx->kind == APPLES_NUC) {
        if (!ctx->refs_wm_ready) {
            const size_t wm = (size_t)3 * ctx->Wp * ctx->ref_pad * 4;
            if (ensure(ctx, ctx->refs_wm, wm)) return -1;
            cudaMemsetAsync(ctx->refs_wm.p, 0, wm, s);
            launch_transpose_nuc((const uint32_t*)ctx->refs_rm.p, ctx->n_ref, ctx->W, (uint32_t*)ctx->refs_wm.p, ctx->Wp,
                                 ctx->ref_pad, DT_TR, s);
            if (ensure(ctx, ctx->refs_nv, (size_t)ctx->ref_pad * 4)) return -1;
            launch_row_valid((const uint32_t*)ctx->refs_rm.p, ctx->n_ref, ctx->W, (uint32_t*)ctx->refs_nv.p, ctx->ref_pad, s);
            ctx->refs_wm_ready = true;
        }
        const int q_pad = round_up((int)nq, DT_TQ);
        if (ensure(ctx, qwm, (size_t)3 * ctx->Wp * q_pad * 4) || ensure(ctx, qnv, (size_t)q_pad * 4)) return -1;
        launch_transpose_nuc((const uint32_t*)dq.p, (int)nq, ctx->W, (uint32_t*)qwm.p, ctx->Wp, q_pad, DT_TQ, s);
        launch_row_valid((const uint32_t*)dq.p, (int)nq, ctx->W, (uint32_t*)qnv.p, q_pad, s);
        launch_dense_nuc_full((const uint32_t*)qwm.p, (const uint32_t*)qnv.p, q_pad, (int)nq,
                              (const uint32_t*)ctx->refs_wm.p, (const uint32_t*)ctx->refs_nv.p, ctx->ref_pad,
                              ctx->n_ref, ctx->W, ctx->Wp, overlap_vmin(ctx->L, overlap_frac), (uint32_t*)dm.p, (uint32_t*)dv.p,
                              (double*)dd.p, ctx->num_sms, s);
    } else {
        const int nc = aa_chunks(ctx->Lp);
        if (!ctx->refs_aa_ready) {
            if (ensure(ctx, ctx->refs_aa_tm, (size_t)ctx->aa_ref_pad * nc * AA_CH) ||
                ensure(ctx, ctx->refs_aav, (size_t)ctx->aa_ref_pad * nc * (AA_CH / 32) * 4))
                return -1;
            launch_aa_layout((const uint8_t*)ctx->refs_rm.p, ctx->n_ref, ctx->Lp, AA_TR, ctx->aa_ref_pad,
                             (uint8_t*)ctx->refs_aa_tm.p, (uint32_t*)ctx->refs_aav.p, s);
            ctx->refs_aa_ready = true;
        }
        const int q_pad = round_up((int)nq, AA_TQ);
        if (ensure(ctx, qwm, (size_t)q_pad * nc * AA_CH) || ensure(ctx, qnv, (size_t)q_pad * nc * (AA_CH / 32) * 4)) return -1;
        launch_aa_layout((const uint8_t*)dq.p, (int)nq, ctx->Lp, AA_TQ, q_pad, (uint8_t*)qwm.p, (uint32_t*)qnv.p, s);
        launch_dense_aa((const uint8_t*)qwm.p, (const uint32_t*)qnv.p, q_pad, (int)nq, (const uint8_t*)ctx->refs_aa_tm.p,
                        (const uint32_t*)ctx->refs_aav.p, ctx->aa_ref_pad, ctx->n_ref, ctx->Lp, ctx->L, overlap_frac,
                        (const uint32_t*)ctx->aa_tab.p, (uint32_t*)dv.p, ctx->n_ref, (double*)dd.p, ctx->n_ref, s);
    }
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(mism, dm.p, n_out * 4, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(valid, dv.p, n_out * 4, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dist, dd.p, n_out * 8, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) return fail(ctx, "apples_distance_counts: %s", cudaGetErrorString(e));
    return 0;
}

int apples_count_keys(apples_ctx* ctx, int64_t nq, const void* packed_queries, const apples_params* params,
                      int32_t* key_kind, void* keys, uint32_t* line_minima) {
    if (!ctx) return -1;
    if (ctx->kind < 0) return fail(ctx, "apples_set_reference has not been called");
    if (nq <= 0 || !packed_queries || !key_kind || !keys) return fail(ctx, "apples_count_keys: bad arguments");
    *key_kind = ctx->kind == APPLES_AA ? 2 : (ctx->nuc_slow ? 1 : (ctx->k2p ? 3 : 0));
    BatchIO io;
    io.h_queries = packed_queries;
    io.h_keys = keys;
    io.h_kmin = *key_kind == 0 ? line_minima : nullptr;
    io.stop_after_count = true;
    return run_batch(ctx, nq, io, params);
}

int apples_observed_sets(apples_ctx* ctx, int64_t nq, const void* packed_queries, const double* rows,
                         const int32_t* self_node, const apples_params* params, int32_t cap, int32_t* count,
                         int32_t* node, double* dist) {
    if (!ctx) return -1;
    if (nq <= 0 || (!packed_queries) == (!rows) || cap <= 0 || !count || !node || !dist)
        return fail(ctx, "apples_observed_sets: bad arguments");
    BatchIO io;
    io.h_queries = packed_queries;
    io.h_rows = rows;
    io.h_self = self_node;
    io.obs_cap = cap;
    io.obs_count = count;
    io.obs_node = node;
    io.obs_dist = dist;
    io.stop_after_select = true;
    return run_batch(ctx, nq, io, params);
}

int apples_edge_solutions(apples_ctx* ctx, const void* packed_query, const double* row, int32_t self_node,
                          const apples_params* params, double* x1, double* x2, double* err, uint8_t* valid) {
    if (!ctx) return -1;
    if ((!packed_query) == (!row) || !x1 || !x2 || !err || !valid) return fail(ctx, "apples_edge_solutions: bad arguments");
    BatchIO io;
    io.h_queries = packed_query;
    io.h_rows = row;
    int32_t selfv = self_node;
    io.h_self = &selfv;
    int32_t e = 0, st = 0;
    double er = 0, di = 0, pe = 0;
    io.edge = &e; io.error = &er; io.distal = &di; io.pendant = &pe; io.status = &st;
    io.dbg_x1 = x1; io.dbg_x2 = x2; io.dbg_err = err; io.dbg_valid = valid;
    return run_batch(ctx, 1, io, params);
}

int apples_last_counts(apples_ctx* ctx, int64_t n, int32_t* K, int32_t* V, int32_t* overflowed) {
    if (!ctx) return -1;
    if (n < 0 || (size_t)n > ctx->hK.size() || (size_t)n > ctx->h_over.size()) return fail(ctx, "apples_last_counts: the last batch had %zu queries", ctx->hK.size());
    for (int64_t i = 0; i < n; ++i) {
        if (K) K[i] = ctx->hK[i];
        if (V) V[i] = ctx->hV[i];
        if (overflowed) overflowed[i] = ctx->h_over[i];
    }
    return 0;
}

int apples_get_timings(apples_ctx* ctx, double* out, int n, int reset) {
    if (!ctx || !out) return -1;
    double v[25] = {ctx->t_ms[T_H2D], ctx->t_ms[T_TRANSPOSE], ctx->t_ms[T_DENSE], ctx->t_ms[T_SELECT], ctx->t_ms[T_PLACE],
                    ctx->t_ms[T_D2H], ctx->n_launch, ctx->n_dense_launch, ctx->n_pairs, ctx->n_obs, ctx->n_valid,
                    ctx->n_over, ctx->max_K, ctx->max_V, ctx->dense_mhz, ctx->n_place_class[0], ctx->n_place_class[1],
                    ctx->n_place_class[2], ctx->n_place_class[3], ctx->n_place_class[4], ctx->n_slow, ctx->n_tc_launch, ctx->n_lines,
                    ctx->n_fp4_launch, ctx->n_k2p_launch};
    for (int i = 0; i < n && i < 25; ++i) out[i] = v[i];
    if (reset) {
        for (int i = 0; i < T_NSTAGE; ++i) ctx->t_ms[i] = 0;
        ctx->n_launch = ctx->n_dense_launch = ctx->n_pairs = ctx->n_lines = ctx->n_obs = ctx->n_valid = ctx->n_over = ctx->max_K = ctx->max_V = 0;
        for (int c = 0; c < PLACE_NCLASS; ++c) ctx->n_place_class[c] = 0;
        ctx->n_slow = 0;
        ctx->n_tc_launch = ctx->n_fp4_launch = ctx->n_k2p_launch = 0;
    }
    return 0;
}

}  // extern "C"
