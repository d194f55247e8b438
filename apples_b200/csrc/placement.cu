// Kernel (b): least-squares placement over every edge of the query's restricted backbone.
//
// Replaces, per query: Subtree (apples/Subtree.py:23-70), Algorithm.dp_frag (apples/Algorithm.py:16-21) with
// FM/OLS/BME/BE all_S_values + all_R_values (FM.py:6-76, OLS.py:12-80, BME.py:6-60, BE.py:6-57),
// placement_per_edge + util.solve2_2 (FM.py:79-93, util.py:6-54), error_per_edge (FM.py:97-124) and
// Algorithm.placement (Algorithm.py:62-101).
//
// Layout: node id = post-order (DFS) rank = edge_index.  The observed leaves arrive sorted by id, i.e. left to
// right.  "Chain i" = leaf i and its ancestors up to (excluding) the first ancestor that also contains leaf i+1
// (the last chain stops below the MRCA).  Concatenating the chains enumerates the valid nodes of the restricted
// subtree (Subtree.py:23-43) in post-order, so a prefix sum over the chain lengths gives every valid node a compact
// index, and the attach level of a chain (level of the node above its top) describes the whole topology:
//   * the node a chain hangs from lives on the next chain to the right with a strictly smaller attach level,
//   * chains hanging from the same node are consecutive "next smaller-or-equal" neighbours, in child order.
// A cooperating group of threads works on chains / nodes in parallel: chain discovery and linking, then the S moments
// bucket by bucket from the deepest attach level up, the R moments from the shallowest down, then every edge is solved
// in closed form and the criterion argmin is a reduction (first minimum in post-order wins, like Python's min()).
//
// Two instantiations of the same code:
//   * WARP + SHARED MEMORY (queries with V + 1 <= 64 / 128 / 256 / 512 node slots, 99 % of a batch): one warp per query, the
//     per-node records (S[6], R[6], edge length, links) and the chain table live in SHARED memory as structure-of-arrays,
//     sized by the class of the launch -- nothing but the observed list is read from and nothing but the 32-byte
//     result is written to global memory (round 1 kept 128-byte records in a global scratch pool: 12x the algorithmic
//     traffic and a DRAM round trip on every dependent step);
//   * BLOCK + GLOBAL MEMORY (the few queries with hundreds to thousands of observed leaves): one 256-thread block per
//     query, records in a global scratch region sized exactly from the counts the selection kernel returned.
//
// One template for the four weightings: moment vector m[6] = sums over leaves of
//   [w, w d, w d^2, w D, w D d, w D^2]      d = path length, D = observed distance,
//   w = 1 (OLS, BME), 1/D^2 (FM), 1/D (BE); BME averages over valid children (BME.py:19,36-37).
// Children are always summed in child order and fp64 operations are written in the reference's order; the file is
// compiled with -fmad=false, so S/R moments, x_1, x_2 are bit-identical to the reference's for identical observed
// distances (the error differs only through Python's pow(x, 2), see DESIGN.md "parity").
#include "common.cuh"

#define FULLMASK 0xffffffffu
constexpr int PL_HIST = 256;          // attach-level buckets per query in shared memory (deeper: level-sweep fallback)
constexpr int PL_BLOCK_THREADS = 256; // threads per query of the global-memory instantiation

__device__ __forceinline__ void leaf_moments(int method, double D, double* m) {
    m[1] = 0.0; m[2] = 0.0; m[4] = 0.0;
    if (method == APPLES_FM) {          // FM.py:21-26
        m[0] = 1.0 / (D * D); m[3] = 1.0 / D; m[5] = 1.0;
    } else if (method == APPLES_BE) {   // BE.py:10-15
        m[0] = 1.0 / D; m[3] = 1.0; m[5] = D;
    } else {                            // OLS.py:25-30, BME.py:10-15
        m[0] = 1.0; m[3] = D; m[5] = D * D;
    }
}

// moments of a child's leaf set seen from the parent end of the child's edge (FM.py:30-40, OLS.py:34-44, ...)
__device__ __forceinline__ void shifted(const double* m, double ln, double* o) {
    o[0] = m[0];
    o[1] = ln * m[0] + m[1];
    o[2] = m[0] * ln * ln + m[2] + 2.0 * ln * m[1];
    o[3] = m[3];
    o[4] = ln * m[3] + m[4];
    o[5] = m[5];
}

template <bool BME>
__device__ __forceinline__ void accumulate(double* acc, const double* m, double ln, double coef) {
    double sh[6];
    shifted(m, ln, sh);
#pragma unroll
    for (int t = 0; t < 6; ++t) acc[t] = acc[t] + (BME ? coef * sh[t] : sh[t]);
}

struct EdgeSol {
    double x1, x2, err;
    bool int0;
    bool deg;   // the reference raises here: 1 / 0.0 (ZeroDivisionError) or det == 0 (assert), util.py:26-27
};

// placement_per_edge + solve2_2 + error_per_edge for one node
__device__ __forceinline__ EdgeSol solve_edge(const double* S, const double* R, double ln, int negative_branch) {
    const double a11 = R[0] + S[0];
    const double a12 = R[0] - S[0];
    const double a21 = a12, a22 = a11;
    const double c1 = R[3] + S[3] - ln * S[0] - R[1] - S[1];
    const double c2 = R[3] - S[3] + ln * S[0] - R[1] + S[1];
    const double den = a11 * a22 - a12 * a21;
    const double det = 1.0 / den;
    const double x1n = (a22 * c1 - a12 * c2) * det;
    const double x2n = (-a21 * c1 + a11 * c2) * det;
    EdgeSol e;
    e.x1 = x1n;
    e.x2 = x2n;
    e.int0 = false;
    e.deg = den == 0.0 || det == 0.0;
    if (!negative_branch) {  // util.py:32-49, same case order and strict inequalities
        if (x1n < 0.0 && x2n < 0.0) {
            e.x1 = 0.0; e.x2 = 0.0; e.int0 = true;
        } else if (x1n > 0.0 && x2n < 0.0) {
            const double t = c1 / a11;
            if (0.0 > t) { e.x1 = 0.0; e.int0 = true; } else { e.x1 = t; }
            e.x2 = 0.0;
        } else if (x1n < 0.0 && 0.0 <= x2n && x2n <= ln) {
            e.x1 = 0.0; e.int0 = true;
            double t = c2 / a22;
            if (0.0 > t) t = 0.0;
            e.x2 = (ln < t) ? ln : t;
        } else if (x1n < 0.0 && x2n > ln) {
            e.x1 = 0.0; e.int0 = true; e.x2 = ln;
        } else if (x1n > 0.0 && x2n > ln) {
            const double t = (c1 - a12 * ln) / a11;
            if (0.0 > t) { e.x1 = 0.0; e.int0 = true; } else { e.x1 = t; }
            e.x2 = ln;
        }
    }
    const double u = e.x1 + e.x2;        // path growth on the R side
    const double v = ln + e.x1 - e.x2;   // path growth on the S side
    const double A = R[5] + S[5];
    const double B = 2.0 * u * R[1] + 2.0 * v * S[1];
    const double C = u * u * R[0] + v * v * S[0];   // (..)**2 in the reference: pow(x, 2), may differ by 1 ulp
    const double D = -2.0 * u * R[3] - 2.0 * v * S[3];
    const double E = -2.0 * R[4] - 2.0 * S[4];
    const double F = R[2] + S[2];
    e.err = A + B + C + D + E + F;
    return e;
}

// ---------------------------------------------------------------------------------------------------------------
// cooperation policies: a warp (shuffles) or a whole block (shared-memory scratch + __syncthreads)
// ---------------------------------------------------------------------------------------------------------------
struct WarpCoop {
    static constexpr int G = 32;
    __device__ static int lane() { return threadIdx.x & 31; }
    __device__ static void sync() { __syncwarp(); }
    // inclusive prefix sum over the group; `total` = sum over the group
    __device__ static int scan(int v, int& total) {
        const int l = lane();
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(FULLMASK, incl, o);
            if (l >= o) incl += t;
        }
        total = __shfl_sync(FULLMASK, incl, 31);
        return incl;
    }
    __device__ static int max_all(int v) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(FULLMASK, v, o));
        return v;
    }
    __device__ static bool any(bool p) { return __any_sync(FULLMASK, p) != 0; }
    // lexicographic (value, index) minimum; members without a candidate pass idx = INT_MAX
    __device__ static void argmin(double& val, int& idx) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double ov = __shfl_xor_sync(FULLMASK, val, o);
            const int oi = __shfl_xor_sync(FULLMASK, idx, o);
            const bool take = (oi != 0x7fffffff) && (idx == 0x7fffffff || ov < val || (ov == val && oi < idx));
            if (take) { val = ov; idx = oi; }
        }
    }
};

struct BlockCoop {
    static constexpr int G = PL_BLOCK_THREADS;
    __device__ static int lane() { return threadIdx.x; }
    __device__ static void sync() { __syncthreads(); }
    __device__ static int* scratch_i() { __shared__ int s[PL_BLOCK_THREADS / 32 + 1]; return s; }
    __device__ static double* scratch_d() { __shared__ double s[PL_BLOCK_THREADS / 32]; return s; }
    __device__ static int scan(int v, int& total) {
        int* s = scratch_i();
        const int l = threadIdx.x & 31, w = threadIdx.x >> 5;
        int wt;
        const int incl = WarpCoop::scan(v, wt);
        __syncthreads();
        if (l == 31) s[w] = wt;
        __syncthreads();
        int before = 0, tot = 0;
#pragma unroll
        for (int i = 0; i < PL_BLOCK_THREADS / 32; ++i) {
            const int x = s[i];
            if (i < w) before += x;
            tot += x;
        }
        total = tot;
        return incl + before;
    }
    __device__ static int max_all(int v) {
        int* s = scratch_i();
        v = WarpCoop::max_all(v);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = v;
        __syncthreads();
        int m = s[0];
#pragma unroll
        for (int i = 1; i < PL_BLOCK_THREADS / 32; ++i) m = max(m, s[i]);
        return m;
    }
    __device__ static bool any(bool p) { return __syncthreads_or(p ? 1 : 0) != 0; }
    __device__ static void argmin(double& val, int& idx) {
        int* si = scratch_i();
        double* sd = scratch_d();
        WarpCoop::argmin(val, idx);
        __syncthreads();
        if ((threadIdx.x & 31) == 0) { si[threadIdx.x >> 5] = idx; sd[threadIdx.x >> 5] = val; }
        __syncthreads();
        val = sd[0];
        idx = si[0];
#pragma unroll
        for (int i = 1; i < PL_BLOCK_THREADS / 32; ++i) {
            const double ov = sd[i];
            const int oi = si[i];
            const bool take = (oi != 0x7fffffff) && (idx == 0x7fffffff || ov < val || (ov == val && oi < idx));
            if (take) { val = ov; idx = oi; }
        }
    }
};

// per-query working set as structure-of-arrays over `cap` node slots (V valid nodes + 1 pseudo record for the subtree
// root, the MRCA) and `kcap` chain slots; lives in shared memory (warp instantiation) or in a global scratch region
struct Work {
    double* S;      // [6][cap]
    double* R;      // [6][cap]
    double* len;    // [cap]
    int* orig;      // [cap] tree node id
    int* fchild;    // [cap] compact index of the first valid child (-1: none)
    int* rsib;      // [cap] next valid child of the same parent (-1: none)
    int* nchild;    // [cap] valid children
    int* par;       // [cap] compact index of the parent (V = the subtree root)
    int* cA;        // [kcap] chain: attach level (level of the node above the chain's top)
    int* cfirst;    // [kcap] compact index of the chain's leaf
    int* clast;     // [kcap] level of the chain's leaf
    int* corder;    // [kcap] chains sorted by attach level
    int cap;
};

__host__ __device__ constexpr size_t work_bytes(int cap, int kcap) {
    return (size_t)cap * (13 * 8 + 5 * 4) + (size_t)kcap * 16;
}

__device__ __forceinline__ Work carve(unsigned char* base, int cap, int kcap) {
    Work w;
    w.cap = cap;
    w.S = reinterpret_cast<double*>(base);
    w.R = w.S + 6 * (size_t)cap;
    w.len = w.R + 6 * (size_t)cap;
    w.orig = reinterpret_cast<int*>(w.len + cap);
    w.fchild = w.orig + cap;
    w.rsib = w.fchild + cap;
    w.nchild = w.rsib + cap;
    w.par = w.nchild + cap;
    w.cA = w.par + cap;
    w.cfirst = w.cA + kcap;
    w.clast = w.cfirst + kcap;
    w.corder = w.clast + kcap;
    return w;
}

// `cnt` ranked records of query q are written: the count, and edge -1 / zeros in the unused slots
__device__ __forceinline__ void close_records(const PlaceArgs& a, int q, int cnt) {
    a.alt_count[q] = cnt;
    for (int j = cnt; j < a.keep; ++j) {
        const size_t o = (size_t)q * a.keep + j;
        a.alt_edge[o] = -1;
        a.alt_error[o] = 0.0;
        a.alt_distal[o] = 0.0;
        a.alt_pendant[o] = 0.0;
        a.alt_int0[o] = 0;
    }
}

// The ranked records of one query (keep > 1), in the order of a stable sort by the criterion's key:
//   MLSE / ME  the valid edges by (key, post-order index); record 0 is the argmin `first` of place_query.  keep - 1
//              rounds of "next smallest (key, p) after the last one", each a solve of every edge and one group argmin;
//   HYBRID     the nc candidates of place_query (hist[0 .. nc), in (error, index) order) by (x_1, candidate rank); one
//              candidate per member of the group, keep rounds of the group argmin.  Record 0 is the first minimum of x_1.
// S / R / len / orig are the query's working set over `cap` node slots (see Work).  (An out-of-line version raised the
// registers of every kernel: 76 instead of 68.)
template <class Coop>
__device__ __forceinline__ void rank_records(const PlaceArgs& a, const int q, const double* S, const double* R,
                                             const double* len, const int* orig, const int cap, const int* hist,
                                             const int V, const int nc, const int first) {
    constexpr int G = Coop::G;
    const int lane = Coop::lane();
    auto solve_at = [&](int p) {
        double s[6], r[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            s[k] = S[k * cap + p];
            r[k] = R[k * cap + p];
        }
        return solve_edge(s, r, len[p], a.negative_branch);
    };
    auto put = [&](int j, int p) {   // record j = edge p
        const EdgeSol e = solve_at(p);
        const size_t o = (size_t)q * a.keep + j;
        a.alt_edge[o] = orig[p];
        a.alt_error[o] = e.err;
        a.alt_distal[o] = len[p] - e.x2;
        a.alt_pendant[o] = e.x1;
        a.alt_int0[o] = e.int0 ? 1 : 0;
    };
    int cnt = 0;
    if (a.criterion == APPLES_HYBRID) {
        Coop::sync();   // hist was written by member 0
        double cx = 0.0;
        if (lane < nc) cx = solve_at(hist[lane]).x1;
        double last_x = 0.0;
        int last_r = -1;
        for (; cnt < a.keep; ++cnt) {
            double v = 0.0;
            int ix = 0x7fffffff;
            if (lane < nc && (last_r < 0 || cx > last_x || (cx == last_x && lane > last_r))) { v = cx; ix = lane; }
            Coop::argmin(v, ix);
            if (ix == 0x7fffffff) break;
            if (lane == 0) put(cnt, hist[ix]);
            last_x = v;
            last_r = ix;
        }
    } else {
        const bool me = a.criterion == APPLES_ME;
        if (lane == 0) put(0, first);
        const EdgeSol e0 = solve_at(first);
        double last_k = me ? e0.x1 : e0.err;
        int last_p = first;
        for (cnt = 1; cnt < a.keep; ++cnt) {
            double v = 0.0;
            int ix = 0x7fffffff;
            for (int p = lane; p < V; p += G) {
                const EdgeSol e = solve_at(p);
                const double key = me ? e.x1 : e.err;
                const bool after = key > last_k || (key == last_k && p > last_p);
                if (after && (ix == 0x7fffffff || key < v)) { v = key; ix = p; }
            }
            Coop::argmin(v, ix);
            if (ix == 0x7fffffff) break;
            if (lane == 0) put(cnt, ix);
            last_k = v;
            last_p = ix;
        }
    }
    if (lane == 0) close_records(a, q, cnt);
}

template <int METHOD, class Coop>
__device__ __forceinline__ void place_query(const PlaceArgs& a, const int q, const int slot, const Work w, int* hist) {
    constexpr bool BME = METHOD == APPLES_BME;
    constexpr int G = Coop::G;
    const int lane = Coop::lane();
    const int K = a.K[q];
    const int cap = w.cap;
    const int* __restrict__ onode = a.obs_node + (size_t)slot * a.cap;
    const double* __restrict__ odist = a.obs_dist + (size_t)slot * a.cap;
    const int* __restrict__ olen = a.obs_len + (size_t)slot * a.cap;
    const int* __restrict__ parent = a.tree.parent;
    const int* __restrict__ level = a.tree.level;
    const double* __restrict__ elen = a.tree.elen;

    // ---------------- chains: attach level, leaf level, compact offsets (prefix sum over chain lengths) ----------------
    int carry = 0, maxlev = 0;
    for (int i0 = 0; i0 < K; i0 += G) {
        const int i = i0 + lane;
        int len = 0, ll = 0;
        if (i < K) {
            len = olen[i];
            ll = level[onode[i]];
        }
        int tot;
        const int incl = Coop::scan(len, tot);
        if (i < K) {
            w.cA[i] = ll - len;
            w.cfirst[i] = carry + incl - len;
            w.clast[i] = ll;
        }
        carry += tot;
        maxlev = max(maxlev, ll);
    }
    maxlev = Coop::max_all(maxlev);
    const int V = carry;
    Coop::sync();
    const int rootlev = w.cA[K - 1];  // the last chain stops below the MRCA

    // ---------------- node records: one thread walks one chain ----------------
    for (int i = lane; i < K; i += G) {
        int u = onode[i];
        const int off = w.cfirst[i], len = w.clast[i] - w.cA[i];
        for (int s = 0; s < len; ++s) {
            const int p = off + s;
            w.len[p] = elen[u];
            w.orig[p] = u;
            w.fchild[p] = s ? p - 1 : -1;
            w.rsib[p] = -1;
            w.nchild[p] = s ? 1 : 0;
            w.par[p] = p + 1;  // the top of the chain is re-linked below
            if (s == 0) {
                double m[6];
                leaf_moments(METHOD, odist[i], m);
#pragma unroll
                for (int k = 0; k < 6; ++k) w.S[k * cap + p] = m[k];
            }
            u = parent[u];
        }
    }
    if (lane == 0) {
        w.fchild[V] = -1;
        w.nchild[V] = 0;
    }
    Coop::sync();

    // ---------------- link every chain top to the node it hangs from ----------------
    for (int j = lane; j < K; j += G) {
        const int alj = w.cA[j];
        const int top = w.cfirst[j] + (w.clast[j] - alj) - 1;
        // next chain to the right with attach level <= mine (next sibling or my owner), then < mine (my owner)
        int nse = j + 1;
        while (nse < K && w.cA[nse] > alj) ++nse;
        int own = nse;
        while (own < K && w.cA[own] >= alj) ++own;
        const int P = (own < K) ? w.cfirst[own] + (w.clast[own] - alj) : V;   // compact index of the node I hang from
        w.par[top] = P;
        if (nse < K && w.cA[nse] == alj)
            w.rsib[top] = w.cfirst[nse] + (w.clast[nse] - alj) - 1;          // next attached chain of the same node
        else if (own < K)
            w.rsib[top] = P - 1;                                            // the owner chain's own child comes last
        // am I the first child?  (no chain to the left hangs from the same node)
        int pse = j - 1;
        while (pse >= 0 && w.cA[pse] > alj) --pse;
        if (pse < 0 || w.cA[pse] < alj) w.fchild[P] = top;
        atomicAdd(&w.nchild[P], 1);
    }
    Coop::sync();

    // ---------------- S and R moments ----------------
    // A chain only depends on chains with a DEEPER attach level (the chains hanging from its nodes) for S, and on the
    // one chain with a shallower attach level that owns the node it hangs from for R.  So chains are bucketed by attach
    // level (counting sort); S walks the buckets from the deepest level up, R from the shallowest down, and inside a
    // bucket every thread owns whole chains (sequential along the chain, which is what the recursion is anyway).
    // Work is O(V + K) instead of O(levels x K).  Trees deeper than PL_HIST levels below the MRCA fall back to a
    // level-by-level sweep.
    auto s_node = [&](int p) {
        const double coef = BME ? 1.0 / (double)w.nchild[p] : 1.0;   // BME.py:19
        double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        for (int c = w.fchild[p]; c >= 0; c = w.rsib[c]) {
            double m[6];
#pragma unroll
            for (int k = 0; k < 6; ++k) m[k] = w.S[k * cap + c];
            accumulate<BME>(acc, m, w.len[c], coef);
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) w.S[k * cap + p] = acc[k];
    };
    // all_R_values: siblings in child order, then the parent's R shifted by the parent's edge unless the parent is
    // the subtree root (FM.py:53-76); BME: coefficient 1 / (nonroot + #valid siblings) (BME.py:36-37)
    auto r_node = [&](int p) {
        const int P = w.par[p];
        const bool nonroot = P < V;
        const double coef = BME ? 1.0 / (double)((nonroot ? 1 : 0) + w.nchild[P] - 1) : 1.0;
        double acc[6] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
        for (int sb = w.fchild[P]; sb >= 0; sb = w.rsib[sb])
            if (sb != p) {
                double m[6];
#pragma unroll
                for (int k = 0; k < 6; ++k) m[k] = w.S[k * cap + sb];
                accumulate<BME>(acc, m, w.len[sb], coef);
            }
        if (nonroot) {
            double m[6];
#pragma unroll
            for (int k = 0; k < 6; ++k) m[k] = w.R[k * cap + P];
            accumulate<BME>(acc, m, w.len[P], coef);
        }
#pragma unroll
        for (int k = 0; k < 6; ++k) w.R[k * cap + p] = acc[k];
    };
    const int range = maxlev - rootlev;  // attach levels lie in [rootlev, maxlev - 1]
    if (range <= PL_HIST) {
        int* h = hist;
        for (int x = lane; x <= range; x += G) h[x] = 0;
        Coop::sync();
        for (int i = lane; i < K; i += G) atomicAdd(&h[w.cA[i] - rootlev], 1);
        Coop::sync();
        // exclusive prefix sum over h[0 .. range): at most PL_HIST entries, one pass of the group's scan per G entries
        {
            int run = 0;
            for (int x0 = 0; x0 < range; x0 += G) {
                const int x = x0 + lane;
                const int c = x < range ? h[x] : 0;
                int tot;
                const int incl = Coop::scan(c, tot);
                if (x < range) h[x] = run + incl - c;
                run += tot;
            }
        }
        Coop::sync();
        for (int i = lane; i < K; i += G) w.corder[atomicAdd(&h[w.cA[i] - rootlev], 1)] = i;  // h[x] becomes the bucket END
        Coop::sync();
        for (int x = range - 1; x >= 0; --x) {          // S: deepest attach level first
            const int b = x ? h[x - 1] : 0, e = h[x];
            for (int k = b + lane; k < e; k += G) {
                const int i = w.corder[k];
                const int off = w.cfirst[i], len = w.clast[i] - w.cA[i];
                for (int sdx = 1; sdx < len; ++sdx) s_node(off + sdx);
            }
            if (b != e) Coop::sync();
        }
        for (int x = 0; x < range; ++x) {               // R: shallowest attach level first, each chain top-down
            const int b = x ? h[x - 1] : 0, e = h[x];
            for (int k = b + lane; k < e; k += G) {
                const int i = w.corder[k];
                const int off = w.cfirst[i], len = w.clast[i] - w.cA[i];
                for (int sdx = len - 1; sdx >= 0; --sdx) r_node(off + sdx);
            }
            if (b != e) Coop::sync();
        }
    } else {
        for (int lv = maxlev - 1; lv > rootlev; --lv) {  // S: level by level upwards
            for (int i = lane; i < K; i += G) {
                const int al = w.cA[i], ll = w.clast[i];
                if (al < lv && lv < ll) s_node(w.cfirst[i] + (ll - lv));
            }
            Coop::sync();
        }
        for (int lv = rootlev + 1; lv <= maxlev; ++lv) {  // R: level by level downwards
            for (int i = lane; i < K; i += G) {
                const int al = w.cA[i], ll = w.clast[i];
                if (al < lv && lv <= ll) r_node(w.cfirst[i] + (ll - lv));
            }
            Coop::sync();
        }
    }

    // ---------------- per-edge closed-form solve + criterion selection (first minimum in post-order) ----------------
    auto solve_at = [&](int p) {
        double S[6], R[6];
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            S[k] = w.S[k * cap + p];
            R[k] = w.R[k * cap + p];
        }
        return solve_edge(S, R, w.len[p], a.negative_branch);
    };
    const bool dbg = a.dbg_x1 != nullptr && q == a.dbg_query;
    double bval = 0.0;
    int bidx = 0x7fffffff;
    bool degenerate = false;
    for (int p = lane; p < V; p += G) {
        const EdgeSol e = solve_at(p);
        degenerate |= e.deg;
        if (dbg) {
            const int u = w.orig[p];
            a.dbg_x1[u] = e.x1;
            a.dbg_x2[u] = e.x2;
            a.dbg_err[u] = e.err;
            a.dbg_valid[u] = 1;
        }
        const double key = (a.criterion == APPLES_ME) ? e.x1 : e.err;
        if (bidx == 0x7fffffff || key < bval) { bval = key; bidx = p; }  // ascending p per thread: first minimum kept
    }
    Coop::argmin(bval, bidx);
    degenerate = Coop::any(degenerate);
    int best = bidx;
    int nc = 0;   // HYBRID: candidates found
    if (a.criterion == APPLES_HYBRID) {
        // heapq.nsmallest(floor(log2 V), key=error) in (error, order) order, then the first minimum of x_1 among
        // them (Algorithm.py:77-82): floor(log2 V) rounds of "next smallest (error, index)"
        const int rounds = 31 - __clz(V);
        double last_e = 0.0, best_x1 = 0.0;
        int last_p = -1;
        best = -1;
        for (int rd = 0; rd < rounds; ++rd) {
            double v = 0.0;
            int ix = 0x7fffffff;
            for (int p = lane; p < V; p += G) {
                const double e = solve_at(p).err;
                const bool after = last_p < 0 || e > last_e || (e == last_e && p > last_p);
                if (after && (ix == 0x7fffffff || e < v)) { v = e; ix = p; }
            }
            Coop::argmin(v, ix);
            if (ix == 0x7fffffff) break;
            // rank_records re-sorts the candidates by x_1; the bucket table is free once the moments are done
            if (a.keep > 1 && lane == 0) hist[nc] = ix;
            ++nc;
            const double x1 = solve_at(ix).x1;
            if (best < 0 || x1 < best_x1) { best = ix; best_x1 = x1; }
            last_e = v;
            last_p = ix;
        }
    }
    if (a.keep > 1) rank_records<Coop>(a, q, w.S, w.R, w.len, w.orig, cap, hist, V, nc, bidx);
    if (lane == 0) {
        const EdgeSol bs = solve_at(best);
        const double blen = w.len[best];
        // Algorithm.py:93-99
        const bool flag = bs.x1 == 0.0 && bs.err > 0.0 && (bs.x2 == 0.0 || bs.x2 == blen);
        a.out_edge[q] = w.orig[best];
        a.out_error[q] = bs.err;
        a.out_distal[q] = blen - bs.x2;
        a.out_pendant[q] = bs.x1;
        a.out_status[q] = (flag ? APPLES_PLACED_MISPLACEMENT_FLAG : APPLES_PLACED) | (bs.int0 ? APPLES_FLAG_PENDANT_INT0 : 0) |
                          (degenerate ? APPLES_FLAG_DEGENERATE : 0);
    }
}

// one warp per query, working set in shared memory (VCAP node slots per query), WARPS queries per block
template <int VCAP>
struct SmemClass {
    static constexpr int WARPS = 1;   // 10 / 19 / 37 / 73 KB per block: 22 / 11 / 6 / 3 queries in flight per SM
    static constexpr size_t PER_WARP = work_bytes(VCAP, VCAP) + (PL_HIST + 1) * 4 + 12;   // multiple of 16
    static constexpr size_t BYTES = WARPS * PER_WARP;
};

template <int METHOD, int VCAP>
__global__ void __launch_bounds__(SmemClass<VCAP>::WARPS * 32) place_smem_kernel(const PlaceArgs a) {
    extern __shared__ __align__(16) unsigned char pl_smem[];
    using C = SmemClass<VCAP>;
    static_assert(C::PER_WARP % 16 == 0, "per-warp region must keep the doubles aligned");
    const int wib = threadIdx.x >> 5;
    const int t = blockIdx.x * C::WARPS + wib;
    if (t >= a.n) return;
    unsigned char* base = pl_smem + (size_t)wib * C::PER_WARP;
    const Work w = carve(base, VCAP, VCAP);
    int* hist = reinterpret_cast<int*>(base + work_bytes(VCAP, VCAP));
    const int q = a.qlist[t];
    place_query<METHOD, WarpCoop>(a, q, a.slot_list ? a.slot_list[t] : q, w, hist);
}

// one block per query, working set in a global scratch region (rec_off / stack_off in node / chain slots).  Three blocks
// per SM (80 registers): without the bound the code of the ranked records would raise the register count of some methods
// past it, or their spills
template <int METHOD>
__global__ void __launch_bounds__(PL_BLOCK_THREADS, 3) place_block_kernel(const PlaceArgs a) {
    __shared__ int hist[PL_HIST + 1];
    const int t = blockIdx.x;
    const int q = a.qlist[t];
    const int K = a.K[q];
    // the host sized the region: rec_off[t] .. rec_off[t + 1] node slots of 128 bytes, stack_off likewise in 16-byte slots
    const int cap = (int)(a.rec_off[t + 1] - a.rec_off[t]);
    unsigned char* nodes = reinterpret_cast<unsigned char*>(a.recs) + (size_t)a.rec_off[t] * 128;
    Work w = carve(nodes, cap, 0);
    int* chains = reinterpret_cast<int*>(reinterpret_cast<unsigned char*>(a.stacks) + (size_t)a.stack_off[t] * 16);
    w.cA = chains;
    w.cfirst = chains + K;
    w.clast = chains + 2 * (size_t)K;
    w.corder = chains + 3 * (size_t)K;
    place_query<METHOD, BlockCoop>(a, q, a.slot_list ? a.slot_list[t] : q, w, hist);
}

// queries that are not placed by least squares: zero-distance shortcut and "<= 2 observed distances"
// (PoolQueryWorker.py:72-75, 97-98); one thread per query of the batch
__global__ void finalize_kernel(const PlaceArgs a) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= a.n) return;
    const int st = a.status[q];
    if (st != ST_ZERO && st != ST_TOO_FEW) return;
    a.out_edge[q] = (st == ST_ZERO) ? a.zero_edge[q] : -1;
    a.out_error[q] = 0.0;
    a.out_distal[q] = 0.0;
    a.out_pendant[q] = 0.0;
    a.out_status[q] = (st == ST_ZERO) ? APPLES_ZERO_DIST_LEAF : APPLES_TOO_FEW_DISTANCES;
    if (a.keep > 1) {   // one record, the one above
        const size_t o = (size_t)q * a.keep;
        a.alt_edge[o] = a.out_edge[q];
        a.alt_error[o] = 0.0;
        a.alt_distal[o] = 0.0;
        a.alt_pendant[o] = 0.0;
        a.alt_int0[o] = 0;
        close_records(a, q, 1);
    }
}

// Sorts the batch's placeable queries into the launch classes on the device (the host would need two passes over the
// batch between two kernel launches, with the GPU idle): lists[c * n ..] = query ids of class c in arbitrary order (the
// results do not depend on it), counts[c] = how many.  Queries whose observed set overflowed (status) or that wait for the
// byte-compare fallback (row_flag) are left to the reruns.  stats = {sum K, sum V, max K, max V} over the binned queries.
__global__ void bin_classes_kernel(int n, const int* __restrict__ status, const int* __restrict__ K, const int* __restrict__ V,
                                   const int* __restrict__ row_flag, int* __restrict__ counts, int* __restrict__ lists,
                                   unsigned long long* __restrict__ stats) {
    // ranks inside the block through shared-memory counters, one global atomic per class and block (a global atomic per
    // query serialised on nine addresses: 0.37 ms per 125k queries)
    __shared__ int s_cnt[PLACE_NCLASS], s_base[PLACE_NCLASS];
    __shared__ unsigned long long s_stat[4];
    if (threadIdx.x < PLACE_NCLASS) s_cnt[threadIdx.x] = 0;
    if (threadIdx.x < 4) s_stat[threadIdx.x] = 0ull;
    __syncthreads();
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    const bool on = q < n && status[q] == ST_PLACE && !(row_flag && row_flag[q]);
    int c = 0, rank = 0;
    if (on) {
        const int v = V[q] + 1, k = K[q];
        c = v <= 64 ? PLACE_CLASS_64 : v <= 128 ? PLACE_CLASS_128 : v <= 256 ? PLACE_CLASS_256 : v <= 512 ? PLACE_CLASS_512 : PLACE_CLASS_BLOCK;
        rank = atomicAdd(&s_cnt[c], 1);
        atomicAdd(&s_stat[0], (unsigned long long)k);
        atomicAdd(&s_stat[1], (unsigned long long)(v - 1));
        atomicMax(&s_stat[2], (unsigned long long)k);
        atomicMax(&s_stat[3], (unsigned long long)(v - 1));
    }
    __syncthreads();
    if (threadIdx.x < PLACE_NCLASS && s_cnt[threadIdx.x]) s_base[threadIdx.x] = atomicAdd(&counts[threadIdx.x], s_cnt[threadIdx.x]);
    if (threadIdx.x < 2 && s_stat[threadIdx.x]) atomicAdd(&stats[threadIdx.x], s_stat[threadIdx.x]);
    if (threadIdx.x >= 2 && threadIdx.x < 4 && s_stat[threadIdx.x]) atomicMax(&stats[threadIdx.x], s_stat[threadIdx.x]);
    __syncthreads();
    if (on) lists[(size_t)c * n + s_base[c] + rank] = q;
}

cudaError_t launch_bin_classes(int n, const int* status, const int* K, const int* V, const int* row_flag, int* counts, int* lists,
                               unsigned long long* stats, cudaStream_t s) {
    if (n <= 0) return cudaSuccess;
    bin_classes_kernel<<<(n + 255) / 256, 256, 0, s>>>(n, status, K, V, row_flag, counts, lists, stats);
    return cudaGetLastError();
}

cudaError_t launch_place_finalize(const PlaceArgs& a, cudaStream_t s) {
    if (a.n <= 0) return cudaSuccess;
    finalize_kernel<<<(a.n + 255) / 256, 256, 0, s>>>(a);
    return cudaGetLastError();
}

template <int METHOD, int VCAP>
static cudaError_t launch_smem(const PlaceArgs& a, cudaStream_t s) {
    using C = SmemClass<VCAP>;
    const dim3 grid((a.n + C::WARPS - 1) / C::WARPS), block(C::WARPS * 32);
    cudaError_t e = cudaFuncSetAttribute(place_smem_kernel<METHOD, VCAP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::BYTES);
    if (e != cudaSuccess) return e;
    place_smem_kernel<METHOD, VCAP><<<grid, block, C::BYTES, s>>>(a);
    return cudaGetLastError();
}

template <int METHOD>
static cudaError_t launch_place_method(int vclass, const PlaceArgs& a, cudaStream_t s) {
    switch (vclass) {
        case PLACE_CLASS_64: return launch_smem<METHOD, 64>(a, s);
        case PLACE_CLASS_128: return launch_smem<METHOD, 128>(a, s);
        case PLACE_CLASS_256: return launch_smem<METHOD, 256>(a, s);
        case PLACE_CLASS_512: return launch_smem<METHOD, 512>(a, s);
        default:
            place_block_kernel<METHOD><<<a.n, PL_BLOCK_THREADS, 0, s>>>(a);
            return cudaGetLastError();
    }
}

cudaError_t launch_place(int method, int vclass, const PlaceArgs& a, cudaStream_t s) {
    if (a.n <= 0) return cudaSuccess;
    switch (method) {
        case APPLES_FM: return launch_place_method<APPLES_FM>(vclass, a, s);
        case APPLES_BME: return launch_place_method<APPLES_BME>(vclass, a, s);
        case APPLES_BE: return launch_place_method<APPLES_BE>(vclass, a, s);
        default: return launch_place_method<APPLES_OLS>(vclass, a, s);
    }
}
