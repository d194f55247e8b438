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

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
};

enum Stage { T_H2D = 0, T_TRANSPOSE, T_DENSE, T_SELECT, T_PLACE, T_D2H, T_NSTAGE };

struct TimedSpan {
    int stage;
    cudaEvent_t a, b;
};

}  // namespace

struct apples_ctx {
    int device = 0;
    int num_sms = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;       // host->device staging of the next sub-batch overlaps compute
    cudaEvent_t ev_ready[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
    // the placement of the ordinary queries runs here while the reruns of the few large / exotic ones (thin, long kernels)
    // occupy the main stream
    cudaStream_t side_stream = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
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
    // representative-count kernel: 1 = tcgen05 kind::i8 tensor-core kernel (dense_tc.cu, default), 0 = integer-pipe LOP3/POPC
    // kernel (distance.cu; also taken automatically beyond 33 816 columns)
    int dense_mode = 1;
    double n_tc_launch = 0;
    bool tc_ready = false;        // reps_img holds the representatives' operand images
    int tc_nw = 0, tc_rep_pad = 0;
    DevBuf reps_img, q_img;
    bool refs_wm_ready = false;
    // matrix mode
    int n_cols = 0;
    DevBuf col_node;
    // per-batch work buffers
    DevBuf q_rm, q_wm, keys, self_node, obs_node, obs_dist, obs_len, obs_len2, Kd, Vd, statusd, zero_edge, pair_counter;
    DevBuf q_bytes, q_bytes2, q_rm2, bad_flag, clk_probe, stash_keys, stash_ids, stash_count;
    double dense_mhz = 0.0;  // effective SM clock of the last dense launch (clock64 / globaltimer of CTA 0)
    DevBuf obs_node2, obs_dist2, qlist, pl_lists, pl_lists2, bin_counts, bin_lists, rec_off, stack_off, recs, stacks;
    DevBuf o_edge, o_err, o_distal, o_pendant, o_status;
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
    double n_launch = 0, n_dense_launch = 0, n_pairs = 0, n_obs = 0, n_valid = 0, n_over = 0, max_K = 0, max_V = 0;
    size_t scratch_limit = (size_t)6 << 30;  // placement scratch pool upper bound (bytes)
    int64_t max_subbatch = 65536;
    int64_t max_batch = 1 << 20;  // queries per macro-batch (batch-wide observed-list buffers)
    std::vector<int> hK, hV, hS;
    std::vector<char> h_over;      // last macro-batch: query went through the overflow rerun
    std::vector<int> h_first;      // host copy of first[]: node u is a leaf iff first[u] == u
    std::vector<int> h_ref_node, h_col_node;  // re-validated when the tree changes
    std::vector<long long> h_rec_off, h_stack_off;
    std::vector<int> h_pl_lists, h_pl_lists2;
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

void release(DevBuf& b) {
    if (b.p) cudaFree(b.p);
    b.p = nullptr;
    b.bytes = 0;
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

void collect_spans(apples_ctx* ctx) {
    static const bool trace = getenv("APPLES_B200_TRACE") != nullptr;
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
    ctx->refs_aa_ready = false;
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

// operand images of the representatives for the tensor-core kernel (after reps_rm is on the device)
int tc_prepare_reps(apples_ctx* ctx, cudaStream_t s) {
    ctx->tc_ready = false;
    if (ctx->dense_mode != 1 || ctx->kind != APPLES_NUC || ctx->nuc_slow || ctx->L > dense_tc_max_sites()) return 0;
    ctx->tc_nw = (ctx->L + 31) / 32;
    ctx->tc_rep_pad = round_up(ctx->n_rep, dense_tc_tile_rows());
    if (ensure(ctx, ctx->reps_img, dense_tc_image_bytes(ctx->tc_rep_pad, ctx->tc_nw))) return -1;
    launch_tc_image((const uint32_t*)ctx->reps_rm.p, ctx->n_rep, ctx->W, ctx->tc_nw, ctx->tc_rep_pad, 127, ctx->reps_img.p, s);
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

size_t query_row_bytes(const apples_ctx* ctx) {
    return ctx->kind == APPLES_AA ? (size_t)ctx->Lp : (size_t)3 * ctx->W * 4;
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
    bool stop_after_count = false;
    double* dbg_x1 = nullptr; double* dbg_x2 = nullptr; double* dbg_err = nullptr; uint8_t* dbg_valid = nullptr;
};

int check_params(apples_ctx* ctx, const apples_params* p) {
    if (!p) return fail(ctx, "params is NULL");
    if (p->method < 0 || p->method > 3) return fail(ctx, "unknown method %d", p->method);
    if (p->criterion < 0 || p->criterion > 2) return fail(ctx, "unknown criterion %d", p->criterion);
    return 0;
}

// One macro-batch (at most ctx->max_batch queries) through the pipeline:
//   phase 1  per sub-batch, no host synchronisation: H2D -> transpose -> dense distances -> selection
//   phase 2  one D2H of (K, V, status) for the whole batch; overflow reruns (rare)
//   phase 3  placement of the whole batch in as few launches as the scratch pool allows (one thread per query:
//            the kernel hides its dependent-load latency only with >= 100k queries in flight)
//   phase 4  results D2H / D2D
int run_macro(apples_ctx* ctx, int64_t base0, int n, const BatchIO& io, const apples_params* prm) {
    cudaStream_t s = ctx->stream;
    // APPLES_B200_TRACE=1: host wall-clock of the pipeline phases of every macro-batch on stderr (debugging aid)
    static const bool trace = getenv("APPLES_B200_TRACE") != nullptr;
    const auto t_begin = std::chrono::steady_clock::now();
    auto mark = [&](const char* what) {
        if (!trace) return;
        const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
        fprintf(stderr, "[apples_b200] %-28s +%8.3f ms\n", what, ms);
    };
    const bool matrix = io.h_rows != nullptr;
    const bool nuc = !matrix && ctx->kind == APPLES_NUC;
    const bool slow_ctx = nuc && ctx->nuc_slow;   // byte-compare fallback for every query of this context
    const int sel_kind = matrix ? SEL_MATRIX : (ctx->kind == APPLES_AA ? SEL_AA : (slow_ctx ? SEL_NUCW : SEL_NUC));
    const int n_units = matrix ? ctx->n_cols : ctx->n_rep;
    const int64_t ldk = matrix ? ctx->n_cols : ctx->rep_pad;
    const size_t key_bytes = (sel_kind == SEL_NUC) ? 4 : 8;
    const int n_leaf_bound = matrix ? ctx->n_cols : ctx->n_ref;

    // sub-batch size: key matrix <= 2 GiB, multiple of the dense tile
    int64_t qb = ((int64_t)2 << 30) / std::max<int64_t>(1, ldk * (int64_t)key_bytes);
    qb = std::min<int64_t>(std::max<int64_t>(qb, DT_TQ), std::max<int64_t>(ctx->max_subbatch, DT_TQ));
    qb = qb / DT_TQ * DT_TQ;
    qb = std::min<int64_t>(qb, round_up(n, DT_TQ));
    const int QB = (int)qb;
    const int cap = std::min(ctx->slot_cap, next_pow2(std::max(4, n_leaf_bound)));

    const size_t qrow = matrix ? (size_t)ctx->n_cols * 8 : query_row_bytes(ctx);
    const bool use_tc = sel_kind == SEL_NUC && ctx->tc_ready;
    if (ensure(ctx, ctx->keys, (size_t)(use_tc ? round_up(QB, 256) : QB) * ldk * key_bytes)) return -1;
    if (use_tc && ensure(ctx, ctx->q_img, dense_tc_image_bytes(round_up(QB, 256), ctx->tc_nw))) return -1;
    const bool two_bufs = n > QB;  // more than one sub-batch: stage the next one while this one computes
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
    if (ensure(ctx, ctx->pair_counter, 8)) return -1;
    if (ensure(ctx, ctx->o_edge, (size_t)n * 4) || ensure(ctx, ctx->o_err, (size_t)n * 8) ||
        ensure(ctx, ctx->o_distal, (size_t)n * 8) || ensure(ctx, ctx->o_pendant, (size_t)n * 8) ||
        ensure(ctx, ctx->o_status, (size_t)n * 4))
        return -1;
    if (ensure(ctx, ctx->rec_off, (size_t)(n + 1) * 8) || ensure(ctx, ctx->stack_off, (size_t)(n + 1) * 8) ||
        ensure(ctx, ctx->qlist, (size_t)std::max(n, 1) * 4) || ensure(ctx, ctx->pl_lists, (size_t)std::max(n, 1) * 8))
        return -1;
    CK(cudaMemsetAsync(ctx->pair_counter.p, 0, 8, s));
    if (ensure(ctx, ctx->bin_counts, 64) || ensure(ctx, ctx->bin_lists, (size_t)PLACE_NCLASS * std::max(n, 1) * 4)) return -1;
    CK(cudaMemsetAsync(ctx->bin_counts.p, 0, 64, s));
    const bool dbg = io.dbg_x1 != nullptr;
    if (dbg) {
        if (ensure(ctx, ctx->dbg_x1, (size_t)ctx->M * 8) || ensure(ctx, ctx->dbg_x2, (size_t)ctx->M * 8) ||
            ensure(ctx, ctx->dbg_err, (size_t)ctx->M * 8) || ensure(ctx, ctx->dbg_valid, (size_t)ctx->M))
            return -1;
        CK(cudaMemsetAsync(ctx->dbg_x1.p, 0, (size_t)ctx->M * 8, s));
        CK(cudaMemsetAsync(ctx->dbg_x2.p, 0, (size_t)ctx->M * 8, s));
        CK(cudaMemsetAsync(ctx->dbg_err.p, 0, (size_t)ctx->M * 8, s));
        CK(cudaMemsetAsync(ctx->dbg_valid.p, 0, (size_t)ctx->M, s));
    }
    const int* d_self = nullptr;
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

    std::vector<int>& hK = ctx->hK; std::vector<int>& hV = ctx->hV; std::vector<int>& hS = ctx->hS;
    hK.resize(n); hV.resize(n); hS.resize(n);
    std::vector<long long>& h_rec_off = ctx->h_rec_off; std::vector<long long>& h_stack_off = ctx->h_stack_off;
    h_rec_off.resize(n + 1); h_stack_off.resize(n + 1);
    const NucGate gate = make_gate(ctx->L, prm->filt_threshold, prm->overlap_frac);

    SelectArgs sa{};
    sa.n_units = n_units;
    sa.ldk = ldk;
    sa.keys_nuc = (const uint32_t*)ctx->keys.p;
    sa.keys_f64 = (const double*)ctx->keys.p;
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
    sa.gate = gate;
    sa.K = (int*)ctx->Kd.p;
    sa.V = (int*)ctx->Vd.p;
    sa.status = (int*)ctx->statusd.p;
    sa.zero_edge = (int*)ctx->zero_edge.p;
    sa.tree = tree_dev(ctx);
    // key-row stash for the overflow reruns (alignment-mode nucleotides): up to 256 MiB of key rows
    int stash_cap = 0;
    if (sel_kind == SEL_NUC && !matrix) {
        stash_cap = (int)std::min<int64_t>(n, std::max<int64_t>(1, ((int64_t)256 << 20) / (ldk * 4)));
        if (ensure(ctx, ctx->stash_keys, (size_t)stash_cap * ldk * 4) || ensure(ctx, ctx->stash_ids, (size_t)stash_cap * 4) ||
            ensure(ctx, ctx->stash_count, 4))
            return -1;
        CK(cudaMemsetAsync(ctx->stash_count.p, 0, 4, s));
        sa.stash_keys = (uint32_t*)ctx->stash_keys.p;
        sa.stash_ids = (int*)ctx->stash_ids.p;
        sa.stash_count = (int*)ctx->stash_count.p;
        sa.stash_cap = stash_cap;
    }

    // distances + selection of the `nb` queries whose packed rows / matrix rows are at d_q / ctx->keys
    // `slow`: byte-compare fallback; d_qb = the queries' padded byte rows [nb][Lp], keys go to `kw` (64-bit, row stride ldk)
    cudaStream_t cur = s;   // stream of distances_and_select (the first-level reruns run on the side stream)
    auto distances_and_select = [&](const void* d_q, int nb, SelectArgs& a, bool keys_ready = false, bool slow = false,
                                    const uint8_t* d_qb = nullptr, void* kw = nullptr) -> int {
        const int nb_pad = round_up(nb, DT_TQ);
        const int kind_now = slow ? SEL_NUCW : sel_kind;
        if (keys_ready) {
            // the key rows are already in a.keys_nuc (stash of the first pass)
        } else if (slow) {
            Span sp(ctx, T_DENSE, cur);
            launch_dense_bytes(d_qb, ctx->Lp, nb, (const uint8_t*)ctx->rep_bytes_p.p, ctx->Lp, ctx->n_rep, ctx->Lp,
                               (unsigned long long*)kw, ldk, cur);
            ctx->n_launch += 1;
            ctx->n_dense_launch += 1;
            ctx->n_pairs += (double)nb * ctx->n_rep;
            ctx->n_slow += nb;
        } else if (sel_kind == SEL_NUC && use_tc) {
            const int q_pad = round_up(nb, 256);
            {
                Span sp(ctx, T_TRANSPOSE, cur);
                launch_tc_image((const uint32_t*)d_q, nb, ctx->W, ctx->tc_nw, q_pad, 125, ctx->q_img.p, cur);
                ctx->n_launch += 1;
            }
            {
                Span sp(ctx, T_DENSE, cur);
                launch_dense_tc(ctx->q_img.p, q_pad, ctx->reps_img.p, ctx->tc_rep_pad, ctx->tc_nw, (uint32_t*)ctx->keys.p, ldk,
                                ctx->num_sms, cur);
                ctx->n_launch += 1;
                ctx->n_dense_launch += 1;
                ctx->n_tc_launch += 1;
            }
            ctx->n_pairs += (double)nb * ctx->n_rep;
        } else if (sel_kind == SEL_NUC) {
            {
                Span sp(ctx, T_TRANSPOSE, cur);
                launch_transpose_nuc((const uint32_t*)d_q, nb, ctx->W, (uint32_t*)ctx->q_wm.p, ctx->Wp, nb_pad, DT_TQ, cur);
                launch_row_valid((const uint32_t*)d_q, nb, ctx->W, (uint32_t*)ctx->q_nv.p, nb_pad, cur);
                ctx->n_launch += 2;
            }
            {
                Span sp(ctx, T_DENSE, cur);
                launch_dense_nuc_keys((const uint32_t*)ctx->q_wm.p, (const uint32_t*)ctx->q_nv.p, nb_pad,
                                      (const uint32_t*)ctx->reps_wm.p, (const uint32_t*)ctx->reps_nv.p, ctx->rep_pad,
                                      ctx->W, ctx->Wp, (uint32_t*)ctx->keys.p, ldk, (unsigned long long*)ctx->clk_probe.p,
                                      ctx->num_sms, cur);
                ctx->n_launch += 1;
                ctx->n_dense_launch += 1;
            }
            ctx->n_pairs += (double)nb * ctx->n_rep;
        } else if (sel_kind == SEL_AA) {
            const int q_pad = round_up(nb, AA_TQ);
            const int nc = aa_chunks(ctx->Lp);
            {
                Span sp(ctx, T_TRANSPOSE, cur);
                launch_aa_layout((const uint8_t*)d_q, nb, ctx->Lp, AA_TQ, q_pad, (uint8_t*)ctx->q_aa_tm.p, (uint32_t*)ctx->q_aav.p, cur);
                ctx->n_launch += 1;
            }
            (void)nc;
            Span sp(ctx, T_DENSE, cur);
            launch_dense_aa((const uint8_t*)ctx->q_aa_tm.p, (const uint32_t*)ctx->q_aav.p, q_pad, nb,
                            (const uint8_t*)ctx->reps_aa_tm.p, (const uint32_t*)ctx->reps_aav.p, ctx->aa_rep_pad, ctx->n_rep,
                            ctx->Lp, ctx->L, prm->overlap_frac, (const uint32_t*)ctx->aa_tab.p, (uint32_t*)ctx->aa_valid.p, ldk,
                            (double*)ctx->keys.p, ldk, cur);
            ctx->n_launch += 2;
            ctx->n_dense_launch += 1;
            ctx->n_pairs += (double)nb * ctx->n_rep;
        }
        CK(cudaGetLastError());
        if (io.stop_after_count) {
            // the rows of this sub-batch, without the padding columns of the key matrix
            const size_t row = (size_t)n_units * key_bytes;
            CK(cudaMemcpy2DAsync((char*)io.h_keys + (size_t)(base0 + a.q_begin) * row, row, slow ? kw : ctx->keys.p,
                                 (size_t)ldk * key_bytes, row, nb, cudaMemcpyDeviceToHost, cur));
            return 0;
        }
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
            Span sp(ctx, T_SELECT, cur);
            launch_select(kind_now, a, cur);
            ctx->n_launch += 1;
        }
        CK(cudaGetLastError());
        return 0;
    };

    // ---------------- phase 1 ----------------
    sa.out_map = nullptr;
    sa.cap = cap;
    sa.obs_node = (int*)ctx->obs_node.p;
    sa.obs_dist = (double*)ctx->obs_dist.p;
    sa.obs_len = (int*)ctx->obs_len.p;
    sa.pair_counter = (unsigned long long*)ctx->pair_counter.p;
    bool used[2] = {false, false};
    int sbi = 0;
    // host input: a short first sub-batch, so that the compute stream waits for a small copy only; the copies of all later
    // sub-batches hide behind the one before (2.2 ms of exposed PCIe time per 125k-query batch otherwise).  8192 queries: long
    // enough to cover the copy + packing of the full-size sub-batch that follows (0.36 us of compute against 0.1 us of copy per
    // query at config 5 shapes)
    const int ramp = (!matrix && (io.h_queries || io.h_bytes) && n > QB) ? std::min(QB, 8192) : QB;
    for (int sb0 = 0, nb = 0; sb0 < n; sb0 += nb, ++sbi) {
        nb = std::min(sbi == 0 ? ramp : QB, n - sb0);
        const void* d_q = nullptr;
        const int buf = two_bufs ? (sbi & 1) : 0;
        if (matrix) {
            Span sp(ctx, T_H2D);
            CK(cudaMemcpyAsync(ctx->keys.p, io.h_rows + (size_t)(base0 + sb0) * ctx->n_cols, (size_t)nb * qrow,
                               cudaMemcpyHostToDevice, s));
        } else if (io.h_queries || io.h_bytes) {
            // staged on the copy stream into one of two buffers; the compute stream waits for the copy, the copy
            // stream waits until the compute stream has finished with the buffer's previous contents
            cudaStream_t cs = ctx->copy_stream;
            if (used[buf]) CK(cudaStreamWaitEvent(cs, ctx->ev_free[buf], 0));
            else if (sbi == 0) {
                // order after whatever the compute stream did before (buffer (re)allocation is synchronous already)
                CK(cudaEventRecord(ctx->ev_free[buf], s));
                CK(cudaStreamWaitEvent(cs, ctx->ev_free[buf], 0));
            }
            void* stage;
            {
                Span sp(ctx, T_H2D, cs);
                if (io.h_queries) {
                    stage = buf ? ctx->q_rm2.p : ctx->q_rm.p;
                    CK(cudaMemcpyAsync(stage, (const char*)io.h_queries + (size_t)(base0 + sb0) * qrow, (size_t)nb * qrow,
                                       cudaMemcpyHostToDevice, cs));
                } else {
                    stage = buf ? ctx->q_bytes2.p : ctx->q_bytes.p;
                    CK(cudaMemcpyAsync(stage, io.h_bytes + (size_t)(base0 + sb0) * io.byte_stride,
                                       (size_t)nb * io.byte_stride, cudaMemcpyHostToDevice, cs));
                }
            }
            if (io.h_bytes && !slow_ctx) {
                // packed on the COPY stream, into the buffer that goes with the staging buffer: the packer of sub-batch b + 1
                // runs beside the count kernel of sub-batch b instead of in front of its own (1.1 ms per 125k-query batch)
                void* pk = buf ? ctx->q_rm2.p : ctx->q_rm.p;
                CK(launch_pack(ctx->kind, (const uint8_t*)stage, io.byte_stride, nb, ctx->L, pk, (int*)ctx->bad_flag.p, cs,
                               nuc ? (int*)ctx->q_rowflag.p + sb0 : nullptr));
                ctx->n_launch += 1;
                d_q = pk;
            }
            CK(cudaEventRecord(ctx->ev_ready[buf], cs));
            CK(cudaStreamWaitEvent(s, ctx->ev_ready[buf], 0));
            if (io.h_bytes && slow_ctx) {
                CK(launch_repitch_bytes((const uint8_t*)stage, io.byte_stride, nb, ctx->L, ctx->Lp, (uint8_t*)ctx->q_bytes_p.p, s));
                ctx->n_launch += 1;
            } else if (!io.h_bytes) {
                d_q = stage;
            }
            used[buf] = true;
        } else {
            d_q = (const char*)io.d_queries + (size_t)(base0 + sb0) * qrow;
        }
        if (slow_ctx && !io.h_bytes) {   // packed planes in, byte rows needed
            CK(launch_unpack_nuc((const uint32_t*)d_q, nb, ctx->L, ctx->W, ctx->Lp, (uint8_t*)ctx->q_bytes_p.p, s));
            ctx->n_launch += 1;
        }
        sa.q_begin = sb0;
        if (distances_and_select(d_q, nb, sa, false, slow_ctx, (const uint8_t*)ctx->q_bytes_p.p, ctx->keys.p)) return -1;
        if (used[buf]) CK(cudaEventRecord(ctx->ev_free[buf], s));
    }
    if (io.stop_after_count) {
        CK(cudaStreamSynchronize(s));
        collect_spans(ctx);
        return 0;
    }

    // launch classes of the placeable queries, sorted on the device (counts: 5 ints at offset 0, stats: 4 u64 at offset 32)
    CK(launch_bin_classes(n, (const int*)ctx->statusd.p, (const int*)ctx->Kd.p, (const int*)ctx->Vd.p,
                          (io.h_bytes && nuc && !slow_ctx) ? (const int*)ctx->q_rowflag.p : nullptr, (int*)ctx->bin_counts.p,
                          (int*)ctx->bin_lists.p, (unsigned long long*)((char*)ctx->bin_counts.p + 32), s));
    ctx->n_launch += 1;
    int h_bin[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    unsigned long long h_bin_stats[4] = {0, 0, 0, 0};
    CK(cudaMemcpyAsync(h_bin, ctx->bin_counts.p, 32, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(h_bin_stats, (char*)ctx->bin_counts.p + 32, 32, cudaMemcpyDeviceToHost, s));
    mark("phase 1 launched");
    // ---------------- phase 2 ----------------
    auto fetch_counts = [&](cudaStream_t fs) -> int {
        Span sp(ctx, T_D2H, fs);
        CK(cudaMemcpyAsync(hK.data(), ctx->Kd.p, (size_t)n * 4, cudaMemcpyDeviceToHost, fs));
        CK(cudaMemcpyAsync(hV.data(), ctx->Vd.p, (size_t)n * 4, cudaMemcpyDeviceToHost, fs));
        CK(cudaMemcpyAsync(hS.data(), ctx->statusd.p, (size_t)n * 4, cudaMemcpyDeviceToHost, fs));
        return 0;
    };
    if (fetch_counts(s)) return -1;
    CK(cudaStreamSynchronize(s));
    mark("phase 1 done on the device");
    // queries holding bytes other than A,C,G,T,- (they survive fasta2dic only as non-letters and count as ordinary
    // characters in jc69, distance.py:733-737): the 2-bit planes cannot carry them, so those queries are recomputed by the
    // byte-compare fallback below; their first-pass results are discarded
    std::vector<int> exotic;
    if (io.h_bytes && nuc && !slow_ctx) {
        int bad = 0;
        CK(cudaMemcpy(&bad, ctx->bad_flag.p, 4, cudaMemcpyDeviceToHost));
        if (bad) {
            std::vector<int> flags(n);
            CK(cudaMemcpy(flags.data(), ctx->q_rowflag.p, (size_t)n * 4, cudaMemcpyDeviceToHost));
            for (int i = 0; i < n; ++i)
                if (flags[i]) exotic.push_back(i);
        }
    }

    PlaceArgs pa{};
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
    pa.dbg_query = dbg ? 0 : -1;
    pa.dbg_x1 = dbg ? (double*)ctx->dbg_x1.p : nullptr;
    pa.dbg_x2 = (double*)ctx->dbg_x2.p;
    pa.dbg_err = (double*)ctx->dbg_err.p;
    pa.dbg_valid = (unsigned char*)ctx->dbg_valid.p;

    // placement of `cnt` candidate entries (entry i -> query id(i), observed lists in row slot(i) of the given buffers;
    // slot == nullptr: row = query id).  The PLACE-status queries are sorted into launch classes by their node count:
    // four shared-memory launches (V + 1 <= 64 / 128 / 256 / 512) and one block-per-query launch with global scratch, chunked
    // if the scratch pool would be exceeded.
    auto place_entries = [&](int cnt, auto id, auto active, bool entry_slots, int capx, const int* on, const double* od,
                             const int* ol, cudaStream_t st, DevBuf& dl, std::vector<int>& L) -> int {
        L.clear();
        int begin[PLACE_NCLASS + 1];
        // pass 1: class sizes; pass 2: fill (query ids first, then the slot rows in the second half of the buffer)
        int sizes[PLACE_NCLASS] = {0, 0, 0, 0, 0};
        auto cls_of = [&](int qi) {
            const int v = hV[qi] + 1;  // + 1: pseudo record of the subtree root
            return v <= 64 ? PLACE_CLASS_64 : v <= 128 ? PLACE_CLASS_128 : v <= 256 ? PLACE_CLASS_256 : v <= 512 ? PLACE_CLASS_512 : PLACE_CLASS_BLOCK;
        };
        for (int i = 0; i < cnt; ++i) {
            const int qi = id(i);
            if (hS[qi] == ST_PLACE && active(qi)) sizes[cls_of(qi)]++;
        }
        begin[0] = 0;
        for (int c = 0; c < PLACE_NCLASS; ++c) begin[c + 1] = begin[c] + sizes[c];
        const int total = begin[PLACE_NCLASS];
        if (total == 0) return 0;
        L.resize((size_t)2 * total);
        int fill[PLACE_NCLASS];
        for (int c = 0; c < PLACE_NCLASS; ++c) fill[c] = begin[c];
        for (int i = 0; i < cnt; ++i) {
            const int qi = id(i);
            if (hS[qi] != ST_PLACE || !active(qi)) continue;
            const int pos = fill[cls_of(qi)]++;
            L[pos] = qi;
            L[(size_t)total + pos] = i;
        }
        if (ensure(ctx, dl, (size_t)2 * total * 4)) return -1;
        CK(cudaMemcpyAsync(dl.p, L.data(), (size_t)(entry_slots ? 2 : 1) * total * 4, cudaMemcpyHostToDevice, st));
        const int* d_q = (const int*)dl.p;
        const int* d_slot = entry_slots ? d_q + total : nullptr;
        pa.cap = capx;
        pa.obs_node = on;
        pa.obs_dist = od;
        pa.obs_len = ol;
        // (running the classes side by side on extra streams was measured: 4.51 vs 4.56 ms per step -- the first launch fills
        // the shared memory of every SM, so the kernels serialise anyway; kept sequential)
        Span sp_all(ctx, T_PLACE, st);
        for (int c = 0; c < PLACE_CLASS_BLOCK; ++c) {
            if (!sizes[c]) continue;
            pa.n = sizes[c];
            pa.qlist = d_q + begin[c];
            pa.slot_list = d_slot ? d_slot + begin[c] : nullptr;
            CK(launch_place(prm->method, c, pa, st));
            ctx->n_launch += 1;
            ctx->n_place_class[c] += sizes[c];
        }
        // block-per-query class: exact scratch regions, chunked by the pool limit
        int i0 = begin[PLACE_CLASS_BLOCK];
        const int iend = begin[PLACE_NCLASS];
        ctx->n_place_class[PLACE_CLASS_BLOCK] += iend - i0;
        while (i0 < iend) {
            long long recs = 0, stk = 0;
            int i1 = i0;
            while (i1 < iend) {
                const int qi = L[i1];
                const long long v = hV[qi] + 1, k = hK[qi];
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
            pa.n = i1 - i0;
            pa.qlist = d_q + i0;
            pa.slot_list = d_slot ? d_slot + i0 : nullptr;
            pa.rec_off = (const long long*)ctx->rec_off.p;
            pa.stack_off = (const long long*)ctx->stack_off.p;
            pa.recs = ctx->recs.p;
            pa.stacks = ctx->stacks.p;
            CK(launch_place(prm->method, PLACE_CLASS_BLOCK, pa, st));
            ctx->n_launch += 1;
            i0 = i1;
            if (i0 < iend) CK(cudaStreamSynchronize(st));  // the scratch pool and the offset arrays are reused by the next chunk
        }
        return 0;
    };

    // ---------------- reruns (rare): byte-compare fallback for exotic queries; larger slots for overflowing ones ----------------
    // the selection kernel stops a query as soon as it exceeds its slot; it is rerun with a 16x larger slot (256 ->
    // 4096 -> 65536 -> all leaves) until it fits
    std::vector<char>& is_over = ctx->h_over;
    is_over.assign(n, 0);
    for (int i : exotic) is_over[i] = 1;
    std::vector<int> over;
    for (int i = 0; i < n; ++i)
        if (hS[i] == ST_OVERFLOW && !is_over[i]) {
            over.push_back(i);
            is_over[i] = 1;
        }
    ctx->n_over += (double)over.size();
    // first-level reruns read their key rows from the stash when every overflowing query got a stash row
    bool use_stash = false;
    if (stash_cap > 0 && !over.empty() && exotic.empty()) {
        int cnt = 0;
        CK(cudaMemcpy(&cnt, ctx->stash_count.p, 4, cudaMemcpyDeviceToHost));
        if (cnt == (int)over.size() && cnt <= stash_cap) {
            CK(cudaMemcpy(over.data(), ctx->stash_ids.p, (size_t)cnt * 4, cudaMemcpyDeviceToHost));  // stash order
            use_stash = true;
        }
    }
    const int cap_max = next_pow2(std::max(4, n_leaf_bound));
    // reruns `list` with slot capacity cap_first, then 16x larger for whoever still overflows
    // `ss`: stream of the selection stage (gather, distances, selection, counts); the placement of the rerun queries stays on `s`
    auto rerun = [&](std::vector<int> list, bool slow, int cap_first, bool stash_first, cudaStream_t ss) -> int {
        int cap2 = cap_first;
        bool use_st = stash_first;
        if (slow && !slow_ctx && ensure_ref_bytes(ctx, ss)) return -1;
        while (!list.empty()) {
            // queries per rerun launch: bounded by the sub-batch size and by 2 GiB of slots
            const int GB = (int)std::max<int64_t>(1, std::min<int64_t>(QB, ((int64_t)2 << 30) / ((int64_t)cap2 * 16)));
            std::vector<int> still;
            for (size_t o0 = 0; o0 < list.size(); o0 += GB) {
                const int ng = (int)std::min<size_t>(GB, list.size() - o0);
                if (ensure(ctx, ctx->obs_node2, (size_t)ng * cap2 * 4)) return -1;
                if (ensure(ctx, ctx->obs_dist2, (size_t)ng * cap2 * 8)) return -1;
                if (ensure(ctx, ctx->obs_len2, (size_t)ng * cap2 * 4)) return -1;
                if (!matrix && ensure(ctx, ctx->q_rm, (size_t)QB * qrow)) return -1;
                if (slow && (ensure(ctx, ctx->q_bytes_p, (size_t)QB * ctx->Lp) ||
                             (!slow_ctx && ensure(ctx, ctx->keys_w, (size_t)ng * ldk * 8))))
                    return -1;
                CK(cudaMemcpyAsync(ctx->qlist.p, list.data() + o0, (size_t)ng * 4, cudaMemcpyHostToDevice, ss));
                // gather the rows of the queries: one kernel for device-resident queries, one host-side gather + one copy
                // otherwise (a memcpy call per row would cost more than the rerun itself)
                if (!matrix && !io.h_queries && !io.h_bytes) {
                    // qlist holds batch-relative ids; the resident rows of this macro-batch start at base0
                    CK(launch_gather_rows((const char*)io.d_queries + (size_t)base0 * qrow, (const int*)ctx->qlist.p, ctx->q_rm.p,
                                          ng, qrow, ss));
                    ctx->n_launch += 1;
                } else {
                    const size_t rb = matrix ? qrow : (io.h_queries ? qrow : (size_t)io.byte_stride);
                    const char* src = matrix ? (const char*)io.h_rows : (io.h_queries ? (const char*)io.h_queries : (const char*)io.h_bytes);
                    ctx->h_gather.resize((size_t)ng * rb);
                    for (int j = 0; j < ng; ++j)
                        memcpy(ctx->h_gather.data() + (size_t)j * rb, src + ((size_t)base0 + list[o0 + j]) * rb, rb);
                    void* dst = matrix ? ctx->keys.p : (io.h_queries ? ctx->q_rm.p : ctx->q_bytes.p);
                    CK(cudaMemcpyAsync(dst, ctx->h_gather.data(), (size_t)ng * rb, cudaMemcpyHostToDevice, ss));
                    CK(cudaStreamSynchronize(ss));  // h_gather is reused by the next group
                }
                if (io.h_bytes && slow)
                    CK(launch_repitch_bytes((const uint8_t*)ctx->q_bytes.p, io.byte_stride, ng, ctx->L, ctx->Lp,
                                            (uint8_t*)ctx->q_bytes_p.p, ss));
                else if (io.h_bytes)
                    CK(launch_pack(ctx->kind, (const uint8_t*)ctx->q_bytes.p, io.byte_stride, ng, ctx->L, ctx->q_rm.p,
                                   (int*)ctx->bad_flag.p, ss));
                else if (slow)
                    CK(launch_unpack_nuc((const uint32_t*)ctx->q_rm.p, ng, ctx->L, ctx->W, ctx->Lp, (uint8_t*)ctx->q_bytes_p.p, ss));
                SelectArgs sb = sa;
                sb.out_map = (const int*)ctx->qlist.p;
                sb.q_begin = 0;
                sb.cap = cap2;
                sb.obs_node = (int*)ctx->obs_node2.p;
                sb.obs_dist = (double*)ctx->obs_dist2.p;
                sb.obs_len = (int*)ctx->obs_len2.p;
                sb.pair_counter = nullptr;
                sb.stash_keys = nullptr;
                if (use_st) sb.keys_nuc = (const uint32_t*)ctx->stash_keys.p + (size_t)o0 * ldk;
                cur = ss;
                const int drc = distances_and_select(matrix ? nullptr : ctx->q_rm.p, ng, sb, use_st, slow, (const uint8_t*)ctx->q_bytes_p.p,
                                                     slow_ctx ? ctx->keys.p : ctx->keys_w.p);
                cur = s;
                if (drc) return -1;
                mark("  rerun select launched");
                if (fetch_counts(ss)) return -1;
                CK(cudaStreamSynchronize(ss));
                mark("  rerun select done");
                if (io.obs_count) {
                    std::vector<int> un((size_t)ng * cap2);
                    std::vector<double> ud((size_t)ng * cap2);
                    CK(cudaMemcpy(un.data(), ctx->obs_node2.p, un.size() * 4, cudaMemcpyDeviceToHost));
                    CK(cudaMemcpy(ud.data(), ctx->obs_dist2.p, ud.size() * 8, cudaMemcpyDeviceToHost));
                    for (int j = 0; j < ng; ++j) {
                        const int i = list[o0 + j];
                        if (hS[i] == ST_OVERFLOW) continue;
                        const int k = std::min(hK[i], io.obs_cap);
                        memcpy(io.obs_node + (size_t)(base0 + i) * io.obs_cap, &un[(size_t)j * cap2], (size_t)k * 4);
                        memcpy(io.obs_dist + (size_t)(base0 + i) * io.obs_cap, &ud[(size_t)j * cap2], (size_t)k * 8);
                    }
                }
                if (!io.stop_after_select) {
                    const int* ov = list.data() + o0;
                    if (place_entries(ng, [&](int i) { return ov[i]; }, [&](int) { return true; }, true, cap2,
                                      (const int*)ctx->obs_node2.p, (const double*)ctx->obs_dist2.p, (const int*)ctx->obs_len2.p, s,
                                      ctx->pl_lists, ctx->h_pl_lists))
                        return -1;
                    CK(cudaStreamSynchronize(s));
                }
                for (int j = 0; j < ng; ++j)
                    if (hS[list[o0 + j]] == ST_OVERFLOW) still.push_back(list[o0 + j]);
            }
            if (cap2 >= cap_max && !still.empty()) return fail(ctx, "internal error: observed set larger than the number of leaves");
            list.swap(still);
            cap2 = (int)std::min<int64_t>((int64_t)cap2 * 16, cap_max);
            use_st = false;  // deeper levels recompute: their rows are no longer contiguous in the stash
        }
        return 0;
    };
    // the few ordinary queries with more than 511 valid nodes (long unary paths): block-per-query kernel, scratch sized on the
    // host from their counts.  Runs after the reruns, which share the scratch pool and whose selection stage should start at once.
    auto main_block_class = [&]() -> int {
        Span sp(ctx, T_PLACE);
        const int nbk = h_bin[PLACE_CLASS_BLOCK];
        if (nbk) {
            pa.cap = cap;   // the reruns pointed the arguments at their own slots
            pa.obs_node = (const int*)ctx->obs_node.p;
            pa.obs_dist = (const double*)ctx->obs_dist.p;
            pa.obs_len = (const int*)ctx->obs_len.p;
            pa.slot_list = nullptr;
            const int* d_list = (const int*)ctx->bin_lists.p + (size_t)PLACE_CLASS_BLOCK * n;
            std::vector<int> ids(nbk);
            CK(cudaMemcpy(ids.data(), d_list, (size_t)nbk * 4, cudaMemcpyDeviceToHost));
            ctx->n_place_class[PLACE_CLASS_BLOCK] += nbk;
            int i0 = 0;
            while (i0 < nbk) {
                long long recs = 0, stk = 0;
                int i1 = i0;
                while (i1 < nbk) {
                    const long long v = hV[ids[i1]] + 1, k = hK[ids[i1]];
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
                CK(cudaMemcpyAsync(ctx->rec_off.p, h_rec_off.data(), (size_t)(i1 - i0 + 1) * 8, cudaMemcpyHostToDevice, s));
                CK(cudaMemcpyAsync(ctx->stack_off.p, h_stack_off.data(), (size_t)(i1 - i0 + 1) * 8, cudaMemcpyHostToDevice, s));
                pa.n = i1 - i0;
                pa.qlist = d_list + i0;
                pa.rec_off = (const long long*)ctx->rec_off.p;
                pa.stack_off = (const long long*)ctx->stack_off.p;
                pa.recs = ctx->recs.p;
                pa.stacks = ctx->stacks.p;
                CK(launch_place(prm->method, PLACE_CLASS_BLOCK, pa, s));
                ctx->n_launch += 1;
                i0 = i1;
                CK(cudaStreamSynchronize(s));  // the scratch pool and the offset arrays are reused (next chunk, reruns)
            }
        }
        return 0;
    };
    // The ordinary queries are placed first, straight from the class lists the device built: no host pass over the batch
    // stands between the last selection kernel and the placement launches, and the host prepares the reruns meanwhile.
    // (Running this pass on a side stream BESIDE the rerun kernels was measured: the step did not change -- the rerun
    // kernels then run with fewer resident blocks and take as much longer as the overlap saves.)
    bool main_placed = false;
    if (trace) fprintf(stderr, "[apples_b200] classes %d %d %d %d %d\n", h_bin[0], h_bin[1], h_bin[2], h_bin[3], h_bin[4]);
    if (!io.stop_after_select) {
        pa.cap = cap;
        pa.obs_node = (const int*)ctx->obs_node.p;
        pa.obs_dist = (const double*)ctx->obs_dist.p;
        pa.obs_len = (const int*)ctx->obs_len.p;
        pa.slot_list = nullptr;
        Span sp(ctx, T_PLACE);
        for (int c = 0; c < PLACE_CLASS_BLOCK; ++c) {
            if (!h_bin[c]) continue;
            pa.n = h_bin[c];
            pa.qlist = (const int*)ctx->bin_lists.p + (size_t)c * n;
            CK(launch_place(prm->method, c, pa, s));
            ctx->n_launch += 1;
            ctx->n_place_class[c] += h_bin[c];
        }
        main_placed = true;
    }
    mark("main placement launched");
    // selection stage of the reruns on the high-priority side stream, beside the shared-memory placement launches above
    cudaStream_t rs = ctx->side_stream;
    if (!exotic.empty() && rerun(exotic, true, cap, false, rs)) return -1;
    if (!over.empty() && rerun(over, slow_ctx, (int)std::min<int64_t>((int64_t)cap * 16, cap_max), use_stash, rs)) return -1;
    if (main_placed && main_block_class()) return -1;

    mark("reruns done");
    // ---------------- parity export of the observed sets ----------------
    if (io.obs_count) {
        const int ocap = io.obs_cap;
        std::vector<int> tn((size_t)n * cap);
        std::vector<double> td((size_t)n * cap);
        CK(cudaMemcpy(tn.data(), ctx->obs_node.p, tn.size() * 4, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(td.data(), ctx->obs_dist.p, td.size() * 8, cudaMemcpyDeviceToHost));
        for (int i = 0; i < n; ++i) {
            io.obs_count[base0 + i] = hK[i];
            if (is_over[i]) continue;
            const int k = std::min(std::min(hK[i], cap), ocap);
            memcpy(io.obs_node + (size_t)(base0 + i) * ocap, &tn[(size_t)i * cap], (size_t)k * 4);
            memcpy(io.obs_dist + (size_t)(base0 + i) * ocap, &td[(size_t)i * cap], (size_t)k * 8);
        }
    }
    // statistics: the device summed the ordinary queries while sorting them, the rerun ones are few
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
    if (!io.stop_after_select) {
        // ---------------- phase 3 ----------------
        if (main_placed) {
            // launched before the reruns
        } else if (place_entries(n, [](int i) { return i; }, [&](int qi) { return !is_over[qi]; }, false, cap,
                                 (const int*)ctx->obs_node.p, (const double*)ctx->obs_dist.p, (const int*)ctx->obs_len.p, s,
                                 ctx->pl_lists, ctx->h_pl_lists)) {
            return -1;
        }
        mark("stats done");
        {   // zero-distance shortcut / too-few-distances records of the whole batch
            Span sp(ctx, T_PLACE);
            pa.n = n;
            CK(launch_place_finalize(pa, s));
            ctx->n_launch += 1;
        }
        // ---------------- phase 4 ----------------
        {
            Span sp(ctx, T_D2H);
            const cudaMemcpyKind kd = io.out_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
            CK(cudaMemcpyAsync(io.edge + base0, ctx->o_edge.p, (size_t)n * 4, kd, s));
            CK(cudaMemcpyAsync(io.error + base0, ctx->o_err.p, (size_t)n * 8, kd, s));
            CK(cudaMemcpyAsync(io.distal + base0, ctx->o_distal.p, (size_t)n * 8, kd, s));
            CK(cudaMemcpyAsync(io.pendant + base0, ctx->o_pendant.p, (size_t)n * 8, kd, s));
            CK(cudaMemcpyAsync(io.status + base0, ctx->o_status.p, (size_t)n * 4, kd, s));
        }
    }
    mark("tail launched");
    CK(cudaStreamSynchronize(s));
    mark("batch done");
    if (dbg) {
        CK(cudaMemcpy(io.dbg_x1, ctx->dbg_x1.p, (size_t)ctx->M * 8, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(io.dbg_x2, ctx->dbg_x2.p, (size_t)ctx->M * 8, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(io.dbg_err, ctx->dbg_err.p, (size_t)ctx->M * 8, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(io.dbg_valid, ctx->dbg_valid.p, (size_t)ctx->M, cudaMemcpyDeviceToHost));
    }
    {
        unsigned long long pc = 0;
        CK(cudaMemcpy(&pc, ctx->pair_counter.p, 8, cudaMemcpyDeviceToHost));
        ctx->n_pairs += (double)pc;
    }
    if (sel_kind == SEL_NUC && !matrix && ctx->clk_probe.p) {
        unsigned long long c[4] = {0, 0, 0, 0};
        CK(cudaMemcpy(c, ctx->clk_probe.p, 32, cudaMemcpyDeviceToHost));
        if (c[3] > c[1]) ctx->dense_mhz = 1e3 * (double)(c[2] - c[0]) / (double)(c[3] - c[1]);
    }
    collect_spans(ctx);
    return 0;
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
    if (!rc && (cudaStreamCreateWithPriority(&ctx->side_stream, cudaStreamNonBlocking, prio_hi) != cudaSuccess ||
                cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
                cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming) != cudaSuccess))
        rc = -4;
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
    DevBuf* all[] = {&ctx->t_parent, &ctx->t_elen, &ctx->t_level, &ctx->t_first, &ctx->refs_rm, &ctx->reps_rm,
                     &ctx->reps_wm, &ctx->refs_wm, &ctx->reps_nv, &ctx->refs_nv, &ctx->q_nv, &ctx->aa_tab, &ctx->reps_aa_tm, &ctx->reps_aav,
                     &ctx->refs_aa_tm, &ctx->refs_aav, &ctx->q_aa_tm, &ctx->q_aav, &ctx->aa_valid, &ctx->ref_bytes_p, &ctx->rep_bytes_p,
                     &ctx->q_bytes_p, &ctx->q_rowflag, &ctx->keys_w, &ctx->reps_img, &ctx->q_img, &ctx->ref_node, &ctx->goff, &ctx->gmem, &ctx->col_node, &ctx->q_rm,
                     &ctx->q_wm, &ctx->keys, &ctx->self_node, &ctx->obs_node, &ctx->obs_dist, &ctx->obs_len, &ctx->obs_len2, &ctx->Kd, &ctx->Vd,
                     &ctx->statusd, &ctx->zero_edge, &ctx->pair_counter, &ctx->q_bytes, &ctx->q_bytes2, &ctx->q_rm2, &ctx->bad_flag, &ctx->clk_probe, &ctx->stash_keys, &ctx->stash_ids, &ctx->stash_count, &ctx->obs_node2, &ctx->obs_dist2, &ctx->qlist, &ctx->pl_lists, &ctx->pl_lists2, &ctx->bin_counts, &ctx->bin_lists,
                     &ctx->rec_off, &ctx->stack_off, &ctx->recs, &ctx->stacks, &ctx->o_edge, &ctx->o_err,
                     &ctx->o_distal, &ctx->o_pendant, &ctx->o_status, &ctx->dbg_x1, &ctx->dbg_x2, &ctx->dbg_err,
                     &ctx->dbg_valid, &ctx->res_q, &ctx->res_self, &ctx->res_edge, &ctx->res_err, &ctx->res_distal,
                     &ctx->res_pendant, &ctx->res_status};
    for (DevBuf* b : all) release(*b);
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
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->ev_join) cudaEventDestroy(ctx->ev_join);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
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
    for (int i = 0; i < n_rep; ++i)
        if (group_offsets[i + 1] < group_offsets[i]) return fail(ctx, "apples_set_reference: group_offsets not monotone");
    const int n_mem = group_offsets[n_rep];
    for (int i = 0; i < n_mem; ++i)
        if (group_members[i] < 0 || group_members[i] >= n_ref) return fail(ctx, "apples_set_reference: member out of range");
    if (check_leaf_ids(ctx, "ref_node", ref_node, n_ref)) return -1;
    ctx->h_ref_node.assign(ref_node, ref_node + n_ref);
    CK(cudaSetDevice(ctx->device));
    ctx->kind = kind;
    ctx->L = L;
    ctx->n_ref = n_ref;
    ctx->n_rep = n_rep;
    ctx->W = apples_words_per_row(L);
    ctx->Wp = round_up(ctx->W, DT_WC);
    ctx->Lp = apples_aa_row_bytes(L);
    ctx->rep_pad = round_up(n_rep, ctx->dense_mode == 1 ? 256 : DT_TR);
    ctx->ref_pad = round_up(n_ref, DT_TR);
    ctx->refs_wm_ready = false;
    const size_t row = query_row_bytes(ctx);
    if (ensure(ctx, ctx->refs_rm, (size_t)n_ref * row) || ensure(ctx, ctx->reps_rm, (size_t)n_rep * row) ||
        ensure(ctx, ctx->ref_node, (size_t)n_ref * 4) || ensure(ctx, ctx->goff, (size_t)(n_rep + 1) * 4) ||
        ensure(ctx, ctx->gmem, (size_t)std::max(n_mem, 1) * 4))
        return -1;
    CK(cudaMemcpy(ctx->refs_rm.p, packed_refs, (size_t)n_ref * row, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->reps_rm.p, packed_reps, (size_t)n_rep * row, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->ref_node.p, ref_node, (size_t)n_ref * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->goff.p, group_offsets, (size_t)(n_rep + 1) * 4, cudaMemcpyHostToDevice));
    if (n_mem) CK(cudaMemcpy(ctx->gmem.p, group_members, (size_t)n_mem * 4, cudaMemcpyHostToDevice));
    ctx->nuc_slow = false;
    ctx->bytes_ready = false;
    if (kind == APPLES_NUC && L > 65535) {
        // 16-bit counts do not hold: the whole context runs the byte-compare fallback (32-bit counts, 64-bit keys)
        ctx->nuc_slow = true;
        if (ensure_ref_bytes(ctx, ctx->stream)) return -1;
        CK(cudaStreamSynchronize(ctx->stream));
        return 0;
    }
    if (kind == APPLES_AA) {
        if (aa_prepare_reps(ctx, ctx->stream)) return -1;
        CK(cudaStreamSynchronize(ctx->stream));
    }
    if (kind == APPLES_NUC) {
        const size_t wm = (size_t)3 * ctx->Wp * ctx->rep_pad * 4;
        if (ensure(ctx, ctx->reps_wm, wm)) return -1;
        CK(cudaMemsetAsync(ctx->reps_wm.p, 0, wm, ctx->stream));
        launch_transpose_nuc((const uint32_t*)ctx->reps_rm.p, n_rep, ctx->W, (uint32_t*)ctx->reps_wm.p, ctx->Wp,
                             ctx->rep_pad, DT_TR, ctx->stream);
        if (ensure(ctx, ctx->reps_nv, (size_t)ctx->rep_pad * 4)) return -1;
        launch_row_valid((const uint32_t*)ctx->reps_rm.p, n_rep, ctx->W, (uint32_t*)ctx->reps_nv.p, ctx->rep_pad, ctx->stream);
        CK(cudaGetLastError());
        if (tc_prepare_reps(ctx, ctx->stream)) return -1;
        CK(cudaStreamSynchronize(ctx->stream));
    }
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

int apples_place_batch(apples_ctx* ctx, int64_t nq, const void* packed_queries, const int32_t* self_node,
                       const apples_params* params, int32_t* edge, double* error, double* distal, double* pendant,
                       int32_t* status) {
    if (!ctx) return -1;
    if (nq < 0 || (nq > 0 && (!packed_queries || !edge || !error || !distal || !pendant || !status)))
        return fail(ctx, "apples_place_batch: bad arguments");
    BatchIO io;
    io.h_queries = packed_queries;
    io.h_self = self_node;
    io.edge = edge; io.error = error; io.distal = distal; io.pendant = pendant; io.status = status;
    return run_batch(ctx, nq, io, params);
}

int apples_place_batch_bytes(apples_ctx* ctx, int64_t nq, const uint8_t* bytes, int64_t row_stride,
                             const int32_t* self_node, const apples_params* params, int32_t* edge, double* error,
                             double* distal, double* pendant, int32_t* status) {
    if (!ctx) return -1;
    if (ctx->kind < 0) return fail(ctx, "apples_set_reference has not been called");
    if (nq < 0 || (nq > 0 && (!bytes || row_stride < ctx->L || !edge || !error || !distal || !pendant || !status)))
        return fail(ctx, "apples_place_batch_bytes: bad arguments");
    BatchIO io;
    io.h_bytes = bytes;
    io.byte_stride = row_stride;
    io.h_self = self_node;
    io.edge = edge; io.error = error; io.distal = distal; io.pendant = pendant; io.status = status;
    return run_batch(ctx, nq, io, params);
}

int apples_set_reference_bytes(apples_ctx* ctx, int kind, int32_t L, int32_t n_ref, const uint8_t* ref_bytes,
                               int64_t row_stride, const int32_t* ref_node, int32_t n_rep, const int32_t* group_offsets,
                               const int32_t* group_members) {
    if (!ctx) return -1;
    if ((kind != APPLES_NUC && kind != APPLES_AA) || L <= 0 || n_ref <= 0 || n_rep <= 0 || !ref_bytes || row_stride < L ||
        !ref_node || !group_offsets || !group_members)
        return fail(ctx, "apples_set_reference_bytes: bad arguments");
    for (int i = 0; i < n_rep; ++i)
        if (group_offsets[i + 1] < group_offsets[i]) return fail(ctx, "apples_set_reference_bytes: group_offsets not monotone");
    const int n_mem = group_offsets[n_rep];
    for (int i = 0; i < n_mem; ++i)
        if (group_members[i] < 0 || group_members[i] >= n_ref) return fail(ctx, "apples_set_reference_bytes: member out of range");
    if (check_leaf_ids(ctx, "ref_node", ref_node, n_ref)) return -1;
    ctx->h_ref_node.assign(ref_node, ref_node + n_ref);
    CK(cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    ctx->kind = kind;
    ctx->L = L;
    ctx->n_ref = n_ref;
    ctx->n_rep = n_rep;
    ctx->W = apples_words_per_row(L);
    ctx->Wp = round_up(ctx->W, DT_WC);
    ctx->Lp = apples_aa_row_bytes(L);
    ctx->rep_pad = round_up(n_rep, ctx->dense_mode == 1 ? 256 : DT_TR);
    ctx->ref_pad = round_up(n_ref, DT_TR);
    ctx->refs_wm_ready = false;
    const size_t row = query_row_bytes(ctx);
    DevBuf d_bytes, d_rep_bytes;
    auto cleanup = [&]() { release(d_bytes); release(d_rep_bytes); };
    if (ensure(ctx, ctx->refs_rm, (size_t)n_ref * row) || ensure(ctx, ctx->reps_rm, (size_t)n_rep * row) ||
        ensure(ctx, ctx->ref_node, (size_t)n_ref * 4) || ensure(ctx, ctx->goff, (size_t)(n_rep + 1) * 4) ||
        ensure(ctx, ctx->gmem, (size_t)std::max(n_mem, 1) * 4) || ensure(ctx, ctx->bad_flag, 4) ||
        ensure(ctx, d_bytes, (size_t)n_ref * row_stride) || ensure(ctx, d_rep_bytes, (size_t)n_rep * L)) {
        cleanup();
        return -1;
    }
    cudaError_t e = cudaMemcpyAsync(d_bytes.p, ref_bytes, (size_t)n_ref * row_stride, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->ref_node.p, ref_node, (size_t)n_ref * 4, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->goff.p, group_offsets, (size_t)(n_rep + 1) * 4, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess && n_mem) e = cudaMemcpyAsync(ctx->gmem.p, group_members, (size_t)n_mem * 4, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemsetAsync(ctx->bad_flag.p, 0, 4, s);
    // (f2) consensus representatives, then (f1) packing of references and representatives
    if (e == cudaSuccess) e = launch_consensus(kind, (const uint8_t*)d_bytes.p, row_stride, L, n_rep, (const int*)ctx->goff.p,
                                               (const int*)ctx->gmem.p, (uint8_t*)d_rep_bytes.p, L, s);
    if (e == cudaSuccess) e = launch_pack(kind, (const uint8_t*)d_bytes.p, row_stride, n_ref, L, ctx->refs_rm.p, (int*)ctx->bad_flag.p, s);
    if (e == cudaSuccess) e = launch_pack(kind, (const uint8_t*)d_rep_bytes.p, L, n_rep, L, ctx->reps_rm.p, (int*)ctx->bad_flag.p, s);
    int bad = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&bad, ctx->bad_flag.p, 4, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    ctx->nuc_slow = false;
    ctx->bytes_ready = false;
    if (e == cudaSuccess && kind == APPLES_NUC && (bad || L > 65535)) {
        // the reference holds bytes other than A,C,G,T,- (ordinary characters for jc69, distance.py:733-737) or is longer
        // than the 16-bit counts allow: keep the byte rows, every query of this context takes the byte-compare fallback
        ctx->nuc_slow = true;
        if (ensure(ctx, ctx->ref_bytes_p, (size_t)n_ref * ctx->Lp) || ensure(ctx, ctx->rep_bytes_p, (size_t)n_rep * ctx->Lp)) {
            cleanup();
            return -1;
        }
        e = launch_repitch_bytes((const uint8_t*)d_bytes.p, row_stride, n_ref, L, ctx->Lp, (uint8_t*)ctx->ref_bytes_p.p, s);
        if (e == cudaSuccess) e = launch_repitch_bytes((const uint8_t*)d_rep_bytes.p, L, n_rep, L, ctx->Lp, (uint8_t*)ctx->rep_bytes_p.p, s);
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);
        ctx->bytes_ready = e == cudaSuccess;
    }
    cleanup();
    if (e != cudaSuccess) return fail(ctx, "apples_set_reference_bytes: %s", cudaGetErrorString(e));
    if (ctx->nuc_slow) return 0;
    if (kind == APPLES_AA) {
        if (aa_prepare_reps(ctx, s)) return -1;
        CK(cudaStreamSynchronize(s));
    }
    if (kind == APPLES_NUC) {
        const size_t wm = (size_t)3 * ctx->Wp * ctx->rep_pad * 4;
        if (ensure(ctx, ctx->reps_wm, wm)) return -1;
        CK(cudaMemsetAsync(ctx->reps_wm.p, 0, wm, s));
        launch_transpose_nuc((const uint32_t*)ctx->reps_rm.p, n_rep, ctx->W, (uint32_t*)ctx->reps_wm.p, ctx->Wp,
                             ctx->rep_pad, DT_TR, s);
        if (ensure(ctx, ctx->reps_nv, (size_t)ctx->rep_pad * 4)) return -1;
        launch_row_valid((const uint32_t*)ctx->reps_rm.p, n_rep, ctx->W, (uint32_t*)ctx->reps_nv.p, ctx->rep_pad, s);
        CK(cudaGetLastError());
        if (tc_prepare_reps(ctx, s)) return -1;
        CK(cudaStreamSynchronize(s));
    }
    return 0;
}

int apples_place_batch_matrix(apples_ctx* ctx, int64_t nq, const double* rows, const int32_t* self_node,
                              const apples_params* params, int32_t* edge, double* error, double* distal,
                              double* pendant, int32_t* status) {
    if (!ctx) return -1;
    if (nq < 0 || (nq > 0 && (!rows || !edge || !error || !distal || !pendant || !status)))
        return fail(ctx, "apples_place_batch_matrix: bad arguments");
    BatchIO io;
    io.h_rows = rows;
    io.h_self = self_node;
    io.edge = edge; io.error = error; io.distal = distal; io.pendant = pendant; io.status = status;
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
    int rc = 0;
    auto cleanup = [&]() { release(dq); release(dm); release(dv); release(dd); release(qwm); release(qnv); };
    if (ensure(ctx, dq, (size_t)nq * row) || ensure(ctx, dm, n_out * 4) || ensure(ctx, dv, n_out * 4) ||
        ensure(ctx, dd, n_out * 8)) { cleanup(); return -1; }
    cudaMemcpyAsync(dq.p, packed_queries, (size_t)nq * row, cudaMemcpyHostToDevice, s);
    cudaMemsetAsync(dm.p, 0, n_out * 4, s);
    if (ctx->kind == APPLES_NUC && ctx->nuc_slow) {
        DevBuf qb, kw;
        auto cleanup2 = [&]() { release(qb); release(kw); cleanup(); };
        if (ensure(ctx, qb, (size_t)nq * ctx->Lp) || ensure(ctx, kw, n_out * 8)) { cleanup2(); return -1; }
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
        if (e2 != cudaSuccess) rc = fail(ctx, "apples_distance_counts: %s", cudaGetErrorString(e2));
        cleanup2();
        return rc;
    }
    if (ctx->kind == APPLES_NUC) {
        if (!ctx->refs_wm_ready) {
            const size_t wm = (size_t)3 * ctx->Wp * ctx->ref_pad * 4;
            if (ensure(ctx, ctx->refs_wm, wm)) { cleanup(); return -1; }
            cudaMemsetAsync(ctx->refs_wm.p, 0, wm, s);
            launch_transpose_nuc((const uint32_t*)ctx->refs_rm.p, ctx->n_ref, ctx->W, (uint32_t*)ctx->refs_wm.p, ctx->Wp,
                                 ctx->ref_pad, DT_TR, s);
            if (ensure(ctx, ctx->refs_nv, (size_t)ctx->ref_pad * 4)) { cleanup(); return -1; }
            launch_row_valid((const uint32_t*)ctx->refs_rm.p, ctx->n_ref, ctx->W, (uint32_t*)ctx->refs_nv.p, ctx->ref_pad, s);
            ctx->refs_wm_ready = true;
        }
        const int q_pad = round_up((int)nq, DT_TQ);
        if (ensure(ctx, qwm, (size_t)3 * ctx->Wp * q_pad * 4)) { cleanup(); return -1; }
        if (ensure(ctx, qnv, (size_t)q_pad * 4)) { cleanup(); return -1; }
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
                ensure(ctx, ctx->refs_aav, (size_t)ctx->aa_ref_pad * nc * (AA_CH / 32) * 4)) { cleanup(); return -1; }
            launch_aa_layout((const uint8_t*)ctx->refs_rm.p, ctx->n_ref, ctx->Lp, AA_TR, ctx->aa_ref_pad,
                             (uint8_t*)ctx->refs_aa_tm.p, (uint32_t*)ctx->refs_aav.p, s);
            ctx->refs_aa_ready = true;
        }
        const int q_pad = round_up((int)nq, AA_TQ);
        if (ensure(ctx, qwm, (size_t)q_pad * nc * AA_CH) || ensure(ctx, qnv, (size_t)q_pad * nc * (AA_CH / 32) * 4)) { cleanup(); return -1; }
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
    if (e != cudaSuccess) rc = fail(ctx, "apples_distance_counts: %s", cudaGetErrorString(e));
    cleanup();
    return rc;
}

int apples_count_keys(apples_ctx* ctx, int64_t nq, const void* packed_queries, const apples_params* params,
                      int32_t* key_kind, void* keys) {
    if (!ctx) return -1;
    if (ctx->kind < 0) return fail(ctx, "apples_set_reference has not been called");
    if (nq <= 0 || !packed_queries || !key_kind || !keys) return fail(ctx, "apples_count_keys: bad arguments");
    *key_kind = ctx->kind == APPLES_AA ? 2 : (ctx->nuc_slow ? 1 : 0);
    BatchIO io;
    io.h_queries = packed_queries;
    io.h_keys = keys;
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
    double v[22] = {ctx->t_ms[T_H2D], ctx->t_ms[T_TRANSPOSE], ctx->t_ms[T_DENSE], ctx->t_ms[T_SELECT], ctx->t_ms[T_PLACE],
                    ctx->t_ms[T_D2H], ctx->n_launch, ctx->n_dense_launch, ctx->n_pairs, ctx->n_obs, ctx->n_valid,
                    ctx->n_over, ctx->max_K, ctx->max_V, ctx->dense_mhz, ctx->n_place_class[0], ctx->n_place_class[1],
                    ctx->n_place_class[2], ctx->n_place_class[3], ctx->n_place_class[4], ctx->n_slow, ctx->n_tc_launch};
    for (int i = 0; i < n && i < 22; ++i) out[i] = v[i];
    if (reset) {
        for (int i = 0; i < T_NSTAGE; ++i) ctx->t_ms[i] = 0;
        ctx->n_launch = ctx->n_dense_launch = ctx->n_pairs = ctx->n_obs = ctx->n_valid = ctx->n_over = ctx->max_K = ctx->max_V = 0;
        for (int c = 0; c < PLACE_NCLASS; ++c) ctx->n_place_class[c] = 0;
        ctx->n_slow = 0;
        ctx->n_tc_launch = 0;
    }
    return 0;
}

}  // extern "C"
