// Kernel (c): APPLES-2 query-specific observed-set selection, one warp per query.
//
// Alignment mode replaces ReducedReference.get_obs_dist (apples/Reference.py:117-157): the reference pops
// representatives in ascending (distance, index) order and expands a cluster while
// `dist <= threshold or obs_num < baseobs`.  Because pops are ascending and obs_num only grows, that is
//   taken = { clusters with dist <= threshold }  U  { the next clusters in (dist, index) order while obs_num < baseobs }
// (SURVEY.md section 8 a3).  The warp scans the query's key row once, expands near clusters (at once in select_kernel,
// batched through a queue in select_nuc_kernel) and keeps, per lane, the two smallest far keys of its residue class;
// afterwards the far clusters are extracted in ascending order (warp-wide minimum of the lane minima; a lane that has
// used both keys re-scans its residue class for the next two) until obs_num reaches baseobs.  The scan is branch-free
// per key (two multiplies, one compare); the exact classification runs only for the few keys that can matter.  A query
// whose observed set outgrows its slot stashes its key row and is rerun with a larger slot (HEAVY instantiation).
// select_nuc_kernel reaches the same set without the full scan: it reads only the key lines that the count stage's
// line minima call for (see the kernel).
// Two kernels: select_nuc_kernel for the packed nucleotide counts of the dense kernels (the hot path), select_kernel for
// the byte-compare fallback (SEL_NUCW), protein (SEL_AA) and distance-matrix (SEL_MATRIX) inputs.
// Nucleotide keys are the exact integer pairs (mismatch, valid) from the dense kernel: ordering by the rational
// mismatch/valid is ordering by jc69 distance (equal rationals give the identical double), so no fp64 is needed
// for the ~R representatives per query; the corrected fp64 distance is evaluated only for the selected members.
//
// Distance-matrix mode replaces valid_dists (apples/PoolQueryWorker.py:44-59): stable ascending order by
// (value, column), keep while `tx <= baseobs or v <= threshold` -- the same rule with one member per unit.
//
// Then, as PoolQueryWorker.runquery:63-98 does: drop the query's own backbone entry, take the zero-distance
// shortcut (first zero in the reference's dict order), flag `<= 2` observed distances; otherwise sort the observed
// leaves by node id (= left-to-right order in the DFS layout) and count the valid nodes of the restricted subtree
// (Subtree.py:23-43) so the host can size the placement scratch.
#include "common.cuh"

#define FULLMASK 0xffffffffu

// software prefetch into L2: the key rows come straight from DRAM (the dense kernel wrote 11 GB since), the member rows
// are random rows of a 384 MB array; the scan and the member loop wait on exactly these loads (ncu: 46 % of the stall
// samples of round 1's kernel)
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

template <int KIND>
struct Key;

template <>
struct Key<SEL_NUC> {
    uint32_t m, v;
    int idx;
};
// SEL_NUCW: nucleotide counts of the byte-compare fallback (alignments longer than 65 535 columns, or symbols other than
// A,C,G,T,- that survive fasta2dic and count as ordinary characters in jc69, distance.py:733-737): 32-bit counts in
// 64-bit keys, 64-bit products
template <>
struct Key<SEL_NUCW> {
    uint32_t m, v;
    int idx;
};
template <>
struct Key<SEL_AA> {
    double d;
    int idx;
};
template <>
struct Key<SEL_MATRIX> {
    double d;
    int idx;
};
// SEL_K2P: 64-bit count keys (ts | tv << 16 | valid << 32) of the K2P count kernel, ordered and classified by their K2P
// distance as SEL_AA is by its fp64 keys
template <>
struct Key<SEL_K2P> {
    double d;
    int idx;
};

__device__ __forceinline__ bool key_less(const Key<SEL_NUC>& a, const Key<SEL_NUC>& b) {
    const uint32_t x = a.m * b.v, y = b.m * a.v;  // counts <= 65535: products fit 32 bits
    return x < y || (x == y && a.idx < b.idx);
}
__device__ __forceinline__ bool key_less(const Key<SEL_NUCW>& a, const Key<SEL_NUCW>& b) {
    const uint64_t x = (uint64_t)a.m * b.v, y = (uint64_t)b.m * a.v;
    return x < y || (x == y && a.idx < b.idx);
}
__device__ __forceinline__ bool key_less(const Key<SEL_AA>& a, const Key<SEL_AA>& b) {
    return a.d < b.d || (a.d == b.d && a.idx < b.idx);
}
__device__ __forceinline__ bool key_less(const Key<SEL_MATRIX>& a, const Key<SEL_MATRIX>& b) {
    return a.d < b.d || (a.d == b.d && a.idx < b.idx);
}
__device__ __forceinline__ bool key_less(const Key<SEL_K2P>& a, const Key<SEL_K2P>& b) {
    return a.d < b.d || (a.d == b.d && a.idx < b.idx);
}

// "no key": compares greater than every real key (ratio 1 / 0 for counts, +inf for distances)
constexpr int KEY_NONE_IDX = 0x7fffffff;
template <int KIND>
__device__ __forceinline__ Key<KIND> key_none() {
    Key<KIND> k;
    if constexpr (KIND == SEL_NUC || KIND == SEL_NUCW) {
        k.m = 1u;
        k.v = 0u;
    } else {
        k.d = __longlong_as_double(0x7ff0000000000000ll);
    }
    k.idx = KEY_NONE_IDX;
    return k;
}
template <int KIND>
__device__ __forceinline__ bool key_is_none(const Key<KIND>& k) {
    return k.idx == KEY_NONE_IDX;
}

__device__ __forceinline__ Key<SEL_NUC> key_shfl(const Key<SEL_NUC>& k, int src) {
    Key<SEL_NUC> o;
    o.m = __shfl_sync(FULLMASK, k.m, src);
    o.v = __shfl_sync(FULLMASK, k.v, src);
    o.idx = __shfl_sync(FULLMASK, k.idx, src);
    return o;
}
__device__ __forceinline__ Key<SEL_NUCW> key_shfl(const Key<SEL_NUCW>& k, int src) {
    Key<SEL_NUCW> o;
    o.m = __shfl_sync(FULLMASK, k.m, src);
    o.v = __shfl_sync(FULLMASK, k.v, src);
    o.idx = __shfl_sync(FULLMASK, k.idx, src);
    return o;
}
template <int KIND>
__device__ __forceinline__ Key<KIND> key_shfl(const Key<KIND>& k, int src) {
    Key<KIND> o;
    o.d = __shfl_sync(FULLMASK, k.d, src);
    o.idx = __shfl_sync(FULLMASK, k.idx, src);
    return o;
}
__device__ __forceinline__ Key<SEL_NUC> key_shfl_xor(const Key<SEL_NUC>& k, int o) {
    Key<SEL_NUC> r;
    r.m = __shfl_xor_sync(FULLMASK, k.m, o);
    r.v = __shfl_xor_sync(FULLMASK, k.v, o);
    r.idx = __shfl_xor_sync(FULLMASK, k.idx, o);
    return r;
}
__device__ __forceinline__ Key<SEL_NUCW> key_shfl_xor(const Key<SEL_NUCW>& k, int o) {
    Key<SEL_NUCW> r;
    r.m = __shfl_xor_sync(FULLMASK, k.m, o);
    r.v = __shfl_xor_sync(FULLMASK, k.v, o);
    r.idx = __shfl_xor_sync(FULLMASK, k.idx, o);
    return r;
}
template <int KIND>
__device__ __forceinline__ Key<KIND> key_shfl_xor(const Key<KIND>& k, int o) {
    Key<KIND> r;
    r.d = __shfl_xor_sync(FULLMASK, k.d, o);
    r.idx = __shfl_xor_sync(FULLMASK, k.idx, o);
    return r;
}

// raw key of one unit as stored in the key matrix (kept in registers during the scan; the Key is rebuilt on demand)
template <int KIND>
struct RawT {
    using T = double;
};
template <>
struct RawT<SEL_NUC> {
    using T = uint32_t;
};
template <>
struct RawT<SEL_NUCW> {
    using T = unsigned long long;   // mismatch | valid << 32
};
template <>
struct RawT<SEL_K2P> {
    using T = unsigned long long;   // ts | tv << 16 | valid << 32
};
__device__ __forceinline__ double k2p_key_dist(unsigned long long raw, int vmin) {
    return k2p_from_counts((uint32_t)(raw & 0xffffu), (uint32_t)((raw >> 16) & 0xffffu), (uint32_t)(raw >> 32), vmin);
}
__device__ __forceinline__ Key<SEL_NUC> make_key_nuc(uint32_t raw, int idx) {
    Key<SEL_NUC> k;
    k.m = raw & 0xffffu;
    k.v = raw >> 16;
    k.idx = idx;
    return k;
}
template <int KIND>
__device__ __forceinline__ Key<KIND> make_key(typename RawT<KIND>::T raw, int idx) {
    if constexpr (KIND == SEL_NUC) {
        return make_key_nuc(raw, idx);
    } else if constexpr (KIND == SEL_NUCW) {
        Key<SEL_NUCW> k;
        k.m = (uint32_t)(raw & 0xffffffffull);
        k.v = (uint32_t)(raw >> 32);
        k.idx = idx;
        return k;
    } else {
        Key<KIND> k;
        k.d = raw;
        k.idx = idx;
        return k;
    }
}
// the generic kernel's keys: K2P keys become their distance (the overlap gate comes from the launch)
template <int KIND>
__device__ __forceinline__ Key<KIND> make_key_sel(const SelectArgs& a, typename RawT<KIND>::T raw, int idx) {
    if constexpr (KIND == SEL_K2P) {
        Key<SEL_K2P> k;
        k.d = k2p_key_dist(raw, a.gate.vmin);
        k.idx = idx;
        return k;
    } else {
        return make_key<KIND>(raw, idx);
    }
}
template <int KIND>
__device__ __forceinline__ typename RawT<KIND>::T load_raw(const SelectArgs& a, int row, int u) {
    if constexpr (KIND == SEL_NUC)
        return a.keys_nuc[(size_t)row * a.ldk + u];
    else if constexpr (KIND == SEL_NUCW || KIND == SEL_K2P)
        return reinterpret_cast<const unsigned long long*>(a.keys_f64)[(size_t)row * a.ldk + u];
    else
        return a.keys_f64[(size_t)row * a.ldk + u];
}

// VEC consecutive raw keys starting at unit u (u a multiple of VEC; count-key rows are 16-byte aligned and padded)
template <int KIND, int VEC>
__device__ __forceinline__ void load_raw_vec(const SelectArgs& a, int row, int u, typename RawT<KIND>::T* out) {
    if constexpr (KIND == SEL_NUC && VEC == 4) {
        const uint4 v = *reinterpret_cast<const uint4*>(a.keys_nuc + (size_t)row * a.ldk + u);
        out[0] = v.x; out[1] = v.y; out[2] = v.z; out[3] = v.w;
    } else {
        static_assert(VEC == 1, "fp64 keys are read one at a time");
        out[0] = load_raw<KIND>(a, row, u);
    }
}

// inside the guard band the fp64 distance decides.  Not inlined: the scan loop is unrolled eight times and this path
// is taken by a handful of keys per million
__device__ __noinline__ bool band_is_near(uint32_t m, uint32_t v, int vmin, double thr) {
    return jc69_from_counts(m, v, vmin) <= thr;
}

// classify one unit.  returns 0 = invalid, 1 = near (dist <= threshold), 2 = far
__device__ __forceinline__ int classify(const SelectArgs& a, const Key<SEL_NUC>& k) {
    // distance.py:735 (no overlap), :741-743 (1 - 4p/3 <= 0  <=>  4 m >= 3 v)
    if (k.v == 0u || (int)k.v < a.gate.vmin || 4u * k.m >= 3u * k.v) return 0;
    // dist <= threshold  <=>  m / v <= p*: decided in 16.16 fixed point with a guard band (counts <= 65535 and
    // P < 49154, so every product fits 32 bits); only the sliver inside the band evaluates the fp64 distance
    const uint32_t lhs = k.m << 16;
    if (a.gate.P_hi == 0u) return 2;  // negative threshold: nothing is near
    if (lhs <= a.gate.P_lo * k.v) return 1;
    if (lhs >= a.gate.P_hi * k.v) return 2;
    return band_is_near(k.m, k.v, a.gate.vmin, a.thr) ? 1 : 2;
}
__device__ __forceinline__ int classify(const SelectArgs& a, const Key<SEL_NUCW>& k) {
    if (k.v == 0u || (long long)k.v < (long long)a.gate.vmin || 4ull * k.m >= 3ull * k.v) return 0;
    const uint64_t lhs = (uint64_t)k.m << 16;
    if (a.gate.P_hi == 0u) return 2;
    if (lhs <= (uint64_t)a.gate.P_lo * k.v) return 1;
    if (lhs >= (uint64_t)a.gate.P_hi * k.v) return 2;
    return band_is_near(k.m, k.v, a.gate.vmin, a.thr) ? 1 : 2;
}
__device__ __forceinline__ int classify(const SelectArgs& a, const Key<SEL_AA>& k) {
    if (!(k.d >= 0.0)) return 0;  // Reference.py:141
    return k.d <= a.thr ? 1 : 2;
}
__device__ __forceinline__ int classify(const SelectArgs& a, const Key<SEL_K2P>& k) {
    if (!(k.d >= 0.0)) return 0;
    return k.d <= a.thr ? 1 : 2;
}
__device__ __forceinline__ int classify(const SelectArgs& a, const Key<SEL_MATRIX>& k) {
    if (!(k.d >= 0.0) || a.col_node[k.idx] < 0) return 0;  // PoolQueryWorker.py:52
    return k.d <= a.thr ? 1 : 2;
}

// ---- member distances (warp-cooperative) ----------------------------------------------------------------------
// packed (mismatch | valid << 16) counts of the query against NR reference rows at once (independent loads in
// flight: the member loop is latency-bound); every lane returns the same totals
template <int NR>
__device__ __forceinline__ void member_counts_nuc(const SelectArgs& a, const uint32_t* __restrict__ qrow, const int* rows,
                                                  int lane, uint32_t* out) {
    uint32_t acc[NR];
#pragma unroll
    for (int k = 0; k < NR; ++k) acc[k] = 0;
    for (int w = 4 * lane; w < a.W; w += 128) {
        const uint4 ql = *reinterpret_cast<const uint4*>(qrow + w);
        const uint4 qh = *reinterpret_cast<const uint4*>(qrow + a.W + w);
        const uint4 qv = *reinterpret_cast<const uint4*>(qrow + 2 * a.W + w);
        uint4 rl[NR], rh[NR], rv[NR];
#pragma unroll
        for (int k = 0; k < NR; ++k) {
            const uint32_t* __restrict__ r = a.refs_nuc + (size_t)rows[k] * 3 * a.W;
            rl[k] = *reinterpret_cast<const uint4*>(r + w);
            rh[k] = *reinterpret_cast<const uint4*>(r + a.W + w);
            rv[k] = *reinterpret_cast<const uint4*>(r + 2 * a.W + w);
        }
#pragma unroll
        for (int k = 0; k < NR; ++k) {
            uint32_t v, m;
#define APPLES_ACC(c)                                                                   \
            v = qv.c & rv[k].c; m = ((ql.c ^ rl[k].c) | (qh.c ^ rh[k].c)) & v; acc[k] += __popc(m) + (__popc(v) << 16);
            APPLES_ACC(x) APPLES_ACC(y) APPLES_ACC(z) APPLES_ACC(w)
#undef APPLES_ACC
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int k = 0; k < NR; ++k) acc[k] += __shfl_xor_sync(FULLMASK, acc[k], o);
#pragma unroll
    for (int k = 0; k < NR; ++k) out[k] = acc[k];
}

// K2P twin: (mismatch | valid << 16) as above and the transversions apart (lo differs: purine against pyrimidine)
template <int NR>
__device__ __forceinline__ void member_counts_k2p(const SelectArgs& a, const uint32_t* __restrict__ qrow, const int* rows,
                                                  int lane, uint32_t* out, uint32_t* out_tv) {
    uint32_t acc[NR], atv[NR];
#pragma unroll
    for (int k = 0; k < NR; ++k) acc[k] = atv[k] = 0;
    for (int w = 4 * lane; w < a.W; w += 128) {
        const uint4 ql = *reinterpret_cast<const uint4*>(qrow + w);
        const uint4 qh = *reinterpret_cast<const uint4*>(qrow + a.W + w);
        const uint4 qv = *reinterpret_cast<const uint4*>(qrow + 2 * a.W + w);
        uint4 rl[NR], rh[NR], rv[NR];
#pragma unroll
        for (int k = 0; k < NR; ++k) {
            const uint32_t* __restrict__ r = a.refs_nuc + (size_t)rows[k] * 3 * a.W;
            rl[k] = *reinterpret_cast<const uint4*>(r + w);
            rh[k] = *reinterpret_cast<const uint4*>(r + a.W + w);
            rv[k] = *reinterpret_cast<const uint4*>(r + 2 * a.W + w);
        }
#pragma unroll
        for (int k = 0; k < NR; ++k) {
            uint32_t v, m, d;
#define APPLES_ACC(c)                                                                                        \
            v = qv.c & rv[k].c; d = ql.c ^ rl[k].c; m = (d | (qh.c ^ rh[k].c)) & v;                          \
            acc[k] += __popc(m) + (__popc(v) << 16); atv[k] += __popc(d & v);
            APPLES_ACC(x) APPLES_ACC(y) APPLES_ACC(z) APPLES_ACC(w)
#undef APPLES_ACC
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int k = 0; k < NR; ++k) {
            acc[k] += __shfl_xor_sync(FULLMASK, acc[k], o);
            atv[k] += __shfl_xor_sync(FULLMASK, atv[k], o);
        }
#pragma unroll
    for (int k = 0; k < NR; ++k) {
        out[k] = acc[k];
        out_tv[k] = atv[k];
    }
}

// byte-compare twin for the fallback: the reference's own definition on raw bytes (distance.py:733-737): a site counts
// when neither byte is '-', and mismatches when the bytes differ.  4 sites per 32-bit word, SWAR.
__device__ __forceinline__ void bytes_counts_word(uint32_t a, uint32_t b, uint32_t& m, uint32_t& v) {
    // per byte: high bit set iff the byte is non-zero (bytes are < 0x80 after fasta2dic's ASCII input; the general form
    // below is exact for any byte value)
    auto nz = [](uint32_t x) { return (((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u; };
    const uint32_t da = nz(a ^ 0x2d2d2d2du), db = nz(b ^ 0x2d2d2d2du);   // 0x2d = '-'
    const uint32_t both = da & db;
    v += __popc(both);
    m += __popc(nz(a ^ b) & both);
}

template <int NR>
__device__ __forceinline__ void member_counts_bytes(const SelectArgs& a, const uint8_t* __restrict__ qrow, const int* rows, int lane,
                                                    uint32_t* om, uint32_t* ov) {
    uint32_t m[NR], v[NR];
#pragma unroll
    for (int k = 0; k < NR; ++k) m[k] = v[k] = 0;
    // rows are padded with '-' to a.Lp (a multiple of 16) bytes by the caller: whole words, no tail
    const int nw = a.Lp / 4;
    for (int w = lane; w < nw; w += 32) {
        const uint32_t q = *reinterpret_cast<const uint32_t*>(qrow + 4 * w);
#pragma unroll
        for (int k = 0; k < NR; ++k) {
            const uint32_t r = *reinterpret_cast<const uint32_t*>(a.refs_bytes + (size_t)rows[k] * a.refs_bstride + 4 * w);
            bytes_counts_word(q, r, m[k], v[k]);
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int k = 0; k < NR; ++k) {
            m[k] += __shfl_xor_sync(FULLMASK, m[k], o);
            v[k] += __shfl_xor_sync(FULLMASK, v[k], o);
        }
#pragma unroll
    for (int k = 0; k < NR; ++k) { om[k] = m[k]; ov[k] = v[k]; }
}

__constant__ double c_blosum45_sel[441] = {
#include "blosum45.inc"
};

// `tab` is the 21x21 table in SHARED memory: lanes index it with different (query, reference) code pairs, which the
// constant cache would serialise
__device__ __forceinline__ double member_dist_aa(const SelectArgs& a, const double* tab, const uint8_t* qrow, int ref_row,
                                                 int lane) {
    const uint8_t* r = a.refs_aa + (size_t)ref_row * a.Lp;
    double sum = 0.0;
    uint32_t val = 0;
    for (int x = 4 * lane; x < a.Lp; x += 128) {
        const uint32_t qw = *reinterpret_cast<const uint32_t*>(qrow + x);
        const uint32_t rw = *reinterpret_cast<const uint32_t*>(r + x);
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const uint32_t qc = (qw >> (8 * b)) & 0xffu, rc = (rw >> (8 * b)) & 0xffu;
            sum += tab[qc * 21 + rc];
            val += (qc < 20u && rc < 20u) ? 1u : 0u;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sum += __shfl_xor_sync(FULLMASK, sum, o);
        val += __shfl_xor_sync(FULLMASK, val, o);
    }
    // every lane must hold the identical double: take lane 0's (the xor-butterfly sums are order-dependent per lane)
    sum = __shfl_sync(FULLMASK, sum, 0);
    return scoredist_from_sum(sum, val, a.L, a.overlap);
}

// ---- per-warp selection state ------------------------------------------------------------------------------------
template <int KIND>
struct WarpSel {
    int obs_num;    // valid member distances so far, own entry included (Reference.py:150-152 / PoolQueryWorker.py:54)
    int kcount;     // entries of the observed dict after removal of the query's own entry
    bool has_zero;  // a zero distance has been seen
    Key<KIND> zkey; // unit key of the best zero so far (dict order = unit order, then position in the group)
    int zpos;
    int znode;
};

template <int KIND>
__device__ __forceinline__ void observe(const SelectArgs& a, WarpSel<KIND>& st, int slot, int self, int node, double d,
                                        bool is_zero, const Key<KIND>& ukey, int pos, int lane) {
    // called by all lanes with identical arguments
    st.obs_num++;
    if (node < 0 || node == self) return;  // own backbone entry is deleted afterwards (PoolQueryWorker.py:63-66)
    if (is_zero) {                           // PoolQueryWorker.py:72-75: first zero in dict order wins
        bool better = !st.has_zero || key_less(ukey, st.zkey) || (!key_less(st.zkey, ukey) && pos < st.zpos);
        if (better) {
            st.has_zero = true;
            st.zkey = ukey;
            st.zpos = pos;
            st.znode = node;
        }
    }
    if (st.kcount < a.cap && lane == 0) {
        a.obs_node[(size_t)slot * a.cap + st.kcount] = node;
        // nucleotide members arrive as their packed integer counts: parked in the (still unused) chain-length row until
        // the tail of the kernel sorts the leaves and writes the corrected fp64 distances
        if constexpr (KIND == SEL_NUC) a.obs_len[(size_t)slot * a.cap + st.kcount] = (int)__double_as_longlong(d);
        else a.obs_dist[(size_t)slot * a.cap + st.kcount] = d;
    }
    st.kcount++;
}

// nucleotide members are stored as their integer counts first (bit pattern in the double slot); the fp64 jc69
// correction is applied afterwards for all observed leaves in parallel (finish_distances)
__device__ __forceinline__ void observe_nuc_counts(const SelectArgs& a, WarpSel<SEL_NUC>& st, int slot, int self, int node,
                                                   uint32_t c, const Key<SEL_NUC>& ukey, int pos, int lane) {
    const uint32_t m = c & 0xffffu, v = c >> 16;
    if (v == 0u || (int)v < a.gate.vmin || 4u * m >= 3u * v) return;  // distance < 0: not stored (Reference.py:150)
    observe<SEL_NUC>(a, st, slot, self, node, __longlong_as_double((long long)c), m == 0u, ukey, pos, lane);
}

__device__ __forceinline__ void observe_nucw_counts(const SelectArgs& a, WarpSel<SEL_NUCW>& st, int slot, int self, int node,
                                                    uint32_t m, uint32_t v, const Key<SEL_NUCW>& ukey, int pos, int lane) {
    if (v == 0u || (long long)v < (long long)a.gate.vmin || 4ull * m >= 3ull * v) return;   // distance < 0: not stored
    const unsigned long long c = (unsigned long long)m | ((unsigned long long)v << 32);
    observe<SEL_NUCW>(a, st, slot, self, node, __longlong_as_double((long long)c), m == 0u, ukey, pos, lane);
}

template <int KIND, int NR = 2>
__device__ __forceinline__ void expand_unit(const SelectArgs& a, WarpSel<KIND>& st, int slot, int q, int self,
                                            const Key<KIND>& ukey, int lane, const double* aa_tab) {
    if constexpr (KIND == SEL_MATRIX) {
        observe<KIND>(a, st, slot, self, a.col_node[ukey.idx], ukey.d, ukey.d == 0.0, ukey, 0, lane);
    } else {
        const int b = a.goff[ukey.idx], e = a.goff[ukey.idx + 1];
        if constexpr (KIND == SEL_NUCW) {
            const uint8_t* qrow = a.q_bytes + (size_t)q * a.q_bstride;
            for (int x = b; x < e && st.kcount <= a.cap; x += NR) {
                int rows[NR], nodes[NR];
                uint32_t cm[NR], cv[NR];
#pragma unroll
                for (int k = 0; k < NR; ++k) rows[k] = a.gmem[min(x + k, e - 1)];
                // node ids with the rows, not inside observe(): there each load would wait behind the previous entry's
                // store (possible alias) -- a serial L2 round trip per observed leaf
#pragma unroll
                for (int k = 0; k < NR; ++k) nodes[k] = a.ref_node[rows[k]];
                member_counts_bytes<NR>(a, qrow, rows, lane, cm, cv);
#pragma unroll
                for (int k = 0; k < NR; ++k)
                    if (x + k < e) observe_nucw_counts(a, st, slot, self, nodes[k], cm[k], cv[k], ukey, x + k - b, lane);
            }
        } else if constexpr (KIND == SEL_K2P) {
            const uint32_t* qrow = a.q_nuc + (size_t)q * 3 * a.W;
            for (int x = b; x < e && st.kcount <= a.cap; x += NR) {
                int rows[NR], nodes[NR];
                uint32_t c[NR], ctv[NR];
#pragma unroll
                for (int k = 0; k < NR; ++k) rows[k] = a.gmem[min(x + k, e - 1)];
#pragma unroll
                for (int k = 0; k < NR; ++k) nodes[k] = a.ref_node[rows[k]];
                member_counts_k2p<NR>(a, qrow, rows, lane, c, ctv);
#pragma unroll
                for (int k = 0; k < NR; ++k)
                    if (x + k < e) {
                        const double d = k2p_from_counts((c[k] & 0xffffu) - ctv[k], ctv[k], c[k] >> 16, a.gate.vmin);
                        if (!(d < 0.0)) observe<KIND>(a, st, slot, self, nodes[k], d, d == 0.0, ukey, x + k - b, lane);
                    }
            }
        } else {
            for (int x = b; x < e && st.kcount <= a.cap; ++x) {
                const int row = a.gmem[x];
                const double d = member_dist_aa(a, aa_tab, a.q_aa + (size_t)q * a.Lp, row, lane);
                if (!(d < 0.0)) observe<KIND>(a, st, slot, self, a.ref_node[row], d, d == 0.0, ukey, x - b, lane);  // Reference.py:150
            }
        }
        if (lane == 0 && a.pair_counter) atomicAdd(a.pair_counter, (unsigned long long)(e - b));
    }
}

// warp bitonic sort of the slot's (node, dist) entries by node id; n2 = power of two >= kcount, padding pre-filled
__device__ void sort_slot(int* node, double* dist, int n2, int lane) {
    for (int k = 2; k <= n2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = lane; i < n2; i += 32) {
                const int l = i ^ j;
                if (l > i) {
                    const int ni = node[i], nl = node[l];
                    const bool up = (i & k) == 0;
                    if ((ni > nl) == up) {
                        node[i] = nl;
                        node[l] = ni;
                        const double t = dist[i];
                        dist[i] = dist[l];
                        dist[l] = t;
                    }
                }
            }
            __syncwarp();
        }
    }
}

// the same order through shared memory: keys (node id << log2(n2) | position), one compare-exchange per lane and step.
// The in-place version above walks global memory with a possible alias between every store and the next load, i.e. one
// L2 round trip per compare-exchange: 1.5 ms for the 4096-entry slot of the largest rerun query.
__device__ void sort_keys_smem(uint32_t* key, int n2, int lane) {
    for (int k = 2; k <= n2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = lane; t < (n2 >> 1); t += 32) {
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));  // t with a zero inserted at bit log2(j)
                const int l = i | j;
                const uint32_t x = key[i], y = key[l];
                if ((x > y) == ((i & k) == 0)) {
                    key[i] = y;
                    key[l] = x;
                }
            }
            __syncwarp();
        }
    }
}

// valid nodes = union of leaf -> MRCA paths, MRCA excluded (Subtree.py:23-43).  With leaves sorted by id the chain owned
// by leaf i runs up to (excluding) the first ancestor that also contains leaf i+1; the last leaf's chain stops below the
// first ancestor that contains leaf 0 (the MRCA).  Writes the chain lengths, returns their sum (every lane).
__device__ __forceinline__ int chain_lengths(const SelectArgs& a, const int* node, int* len_out, int K, int lane) {
    const int leaf0 = node[0];
    int c = 0;
    for (int i = lane; i < K; i += 32) {
        int u = node[i];
        const int nxt = (i + 1 < K) ? node[i + 1] : -1;
        int len = 1;
        while (true) {
            const int p = a.tree.parent[u];
            const bool top = (i + 1 < K) ? (p >= nxt) : (a.tree.first[p] <= leaf0);
            if (top) break;
            len++;
            u = p;
        }
        len_out[i] = len;
        c += len;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(FULLMASK, c, o);
    return c;
}

// nucleotide mode: 8 blocks of 4 warps per SM (64 registers, some spills) measured faster than 4 (128 registers): 12.1
// vs 12.9 ms per 125k queries -- the kernel is latency-bound and wants warps, not registers
#ifndef SEL_MINBLOCKS
#define SEL_MINBLOCKS 8
#endif
#ifndef SEL_NR
#define SEL_NR 2
#endif
#ifndef SEL_GEN_WARPS
#define SEL_GEN_WARPS 1   // warps (queries) per block of the generic kernel (protein bench: 11.6 / 11.1 / 10.85 ms at 4 / 2 / 1)
#endif
template <int KIND>
__global__ void __launch_bounds__(32 * SEL_GEN_WARPS, 16 / SEL_GEN_WARPS) select_kernel(const SelectArgs a) {
    static_assert(KIND != SEL_NUC, "packed nucleotide counts go through select_nuc_kernel");
    constexpr int NR = SEL_NR;
    const int lane = threadIdx.x & 31;
    const int slot = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);  // row of this launch's key / query matrices
    __shared__ double s_aa_tab[KIND == SEL_AA ? 441 : 1];
    const double* aa_tab = s_aa_tab;
    if constexpr (KIND == SEL_AA) {
        for (int i = threadIdx.x; i < 441; i += blockDim.x) s_aa_tab[i] = c_blosum45_sel[i];
        __syncthreads();
    }
    if (slot >= a.n) return;
    const int gid = a.out_map ? a.out_map[slot] : a.q_begin + slot;       // query index inside the batch
    const int oslot = a.out_map ? slot : gid;                             // row of the observed-list buffers
    const int self = a.self_node ? a.self_node[gid] : -1;

    WarpSel<KIND> st;
    st.obs_num = 0;
    st.kcount = 0;
    st.has_zero = false;
    st.zpos = 0;
    st.znode = -1;
    st.zkey.idx = 0;

    // ---- one scan of the key row.  Near units (dist <= threshold) are expanded as they are met (rare: a handful per
    // query, handled after a warp vote).  Far units only update the lane's two smallest far keys -- registers only, no
    // warp traffic -- because the far set is needed only while obs_num < baseobs, and then only its few smallest
    // members: they are extracted afterwards, one at a time, as the warp-wide minimum of the 32 lane minima; a lane
    // that has used both of its keys gets the next two by a cooperative re-scan of just its class (R / 32 keys).
    // Lane l owns the units u with u % 32 == l.  16-byte loads of four packed count keys per lane measured slower on
    // B200 (15.9 vs 14.0 ms per 125k queries), as did 16 scalar loads in flight: the scan is bound by its instructions,
    // not by bytes in flight. ----
    using Raw = typename RawT<KIND>::T;
    constexpr int VEC = 1;
    constexpr int U = 8;  // independent loads in flight per lane
    Key<KIND> l1 = key_none<KIND>(), l2 = key_none<KIND>();
    uint32_t bm = 1u, bv = 0u;  // count keys: event bound as a ratio; starts at l2 = none (1 / 0: every key with v > 0)
    for (int u0 = 0; u0 < a.n_units && st.kcount <= a.cap; u0 += 32 * U) {
        {   // the 128-byte lines of the chunk after next (32 * U keys = 8 or 16 lines per chunk)
            constexpr int PER_LINE = 128 / (int)sizeof(Raw);
            const int u = u0 + 2 * 32 * U + lane * PER_LINE;
            if (lane < 32 * U / PER_LINE && u < a.n_units) {
                prefetch_l2(a.keys_f64 + (size_t)slot * a.ldk + u);
            }
        }
        Raw raw[U];
#pragma unroll
        for (int j = 0; j < U; ++j) {
            const int u = u0 + j * 32 + lane;
            raw[j] = 0;
            if (u < a.n_units) raw[j] = load_raw<KIND>(a, slot, u);
        }
        // Per key, branch-free: is it an EVENT for this lane -- a far key smaller than the lane's second-smallest, or a
        // key that needs the exact classification (near, or inside the guard band)?  Both are "ratio m / v below a bound":
        // the bound (bm / bv) is the larger of the band's upper edge P_hi / 65536 and the ratio of l2, so one key costs two
        // multiplies and one compare (the scan used to be 70 %, then 35 % of this kernel's instructions).  Almost every
        // key is above the bound.  Keys past the end of the row were loaded as 0 (0 < 0 fails); a key under the overlap
        // gate that passes is rejected by the exact classification.
        unsigned ev = 0u;
#pragma unroll
        for (int j = 0; j < U; ++j) {
            if constexpr (KIND == SEL_NUCW) {
                const uint32_t m = (uint32_t)(raw[j] & 0xffffffffull), v = (uint32_t)(raw[j] >> 32);
                if ((uint64_t)m * bv < (uint64_t)bm * v) ev |= 1u << j;
            } else if constexpr (KIND == SEL_K2P) {
                const int u = u0 + j * 32 + lane;
                if (u < a.n_units && !(k2p_key_dist(raw[j], a.gate.vmin) > l2.d)) ev |= 1u << j;   // near and missing keys included
            } else {
                const int u = u0 + j * 32 + lane;
                if (u < a.n_units && !(raw[j] > l2.d)) ev |= 1u << j;  // NaN and near keys included
            }
        }
        unsigned nearb = 0u;  // bit j: raw[j] is a near unit
        if (__any_sync(FULLMASK, ev != 0u)) {
            // events, one per round (a lane rarely has two among its eight keys)
            while (ev) {
                const int j = __ffs(ev) - 1;
                ev &= ev - 1;
                Raw rj = raw[0];
#pragma unroll
                for (int t = 1; t < U; ++t)
                    if (j == t) rj = raw[t];
                const Key<KIND> kj = make_key_sel<KIND>(a, rj, u0 + j * 32 + lane);
                const int c = classify(a, kj);
                if (c == 1) nearb |= 1u << j;
                if (c == 2 && key_less(kj, l2)) {
                    if (key_less(kj, l1)) {
                        l2 = l1;
                        l1 = kj;
                    } else {
                        l2 = kj;
                    }
                }
            }
            if constexpr (KIND == SEL_NUCW) {
                const bool far_rules = ((uint64_t)l2.m << 16) > (uint64_t)a.gate.P_hi * l2.v;
                bm = far_rules ? l2.m : a.gate.P_hi;
                bv = far_rules ? l2.v : 65536u;
            }
        }
        if (__any_sync(FULLMASK, nearb != 0u)) {
            // queued (lane t holds the t-th pending key) and expanded from ONE loop so that the member-distance code
            // is instantiated once
            unsigned nearm[U];
            bool any = false;
#pragma unroll
            for (int j = 0; j < U; ++j) {
                nearm[j] = __ballot_sync(FULLMASK, (nearb >> j) & 1u);
                any |= nearm[j] != 0u;
            }
            while (any) {
                int qn = 0;
                Key<KIND> qkey;
                qkey.idx = -1;
                any = false;
#pragma unroll
                for (int j = 0; j < U; ++j) {
                    while (nearm[j] && qn < 32) {
                        const int src = __ffs(nearm[j]) - 1;
                        nearm[j] &= nearm[j] - 1;
                        const Key<KIND> uk = make_key_sel<KIND>(a, __shfl_sync(FULLMASK, raw[j], src), u0 + j * 32 + src);
                        if (lane == qn) qkey = uk;
                        ++qn;
                    }
                    any |= nearm[j] != 0u;
                }
                for (int t = 0; t < qn && st.kcount <= a.cap; ++t) {
                    const Key<KIND> uk = key_shfl(qkey, t);
                    expand_unit<KIND, NR>(a, st, oslot, slot, self, uk, lane, aa_tab);
                }
            }
        }
    }
    // ---- far units in ascending (distance, index) order while obs_num < baseobs (Reference.py:146) ----
    bool more = !key_is_none(l2);  // the class may hold far keys beyond the two kept
    while (st.obs_num < a.baseobs && st.kcount <= a.cap) {
        // warp-wide minimum of the lane minima
        Key<KIND> g = l1;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const Key<KIND> og = key_shfl_xor(g, o);
            if (key_less(og, g)) g = og;
        }
        if (key_is_none(g)) break;  // no far unit left
        expand_unit<KIND, NR>(a, st, oslot, slot, self, g, lane, aa_tab);
        const bool mine = l1.idx == g.idx;
        if (mine) {
            l1 = l2;
            l2 = key_none<KIND>();
        }
        const unsigned refill = __ballot_sync(FULLMASK, mine && more && key_is_none(l1));
        if (refill) {
            // the owner has used both of its keys: the two next-smallest keys of its class (loads (k * 32 + owner),
            // k split over the lanes, four in flight per lane)
            const int owner = __ffs(refill) - 1;
            Key<KIND> n1 = key_none<KIND>(), n2 = key_none<KIND>();
            constexpr int RU = 4;
            for (int k0 = lane; k0 * 32 * VEC < a.n_units; k0 += 32 * RU) {
                Raw rr[RU * VEC];
#pragma unroll
                for (int j = 0; j < RU; ++j) {
                    const int u = ((k0 + 32 * j) * 32 + owner) * VEC;
#pragma unroll
                    for (int c = 0; c < VEC; ++c) rr[j * VEC + c] = 0;
                    if (u < a.n_units) load_raw_vec<KIND, VEC>(a, slot, u, &rr[j * VEC]);
                }
#pragma unroll
                for (int j = 0; j < RU * VEC; ++j) {
                    const int u = ((k0 + 32 * (j / VEC)) * 32 + owner) * VEC + j % VEC;
                    const Key<KIND> kj = make_key_sel<KIND>(a, rr[j], u);
                    if (u < a.n_units && classify(a, kj) == 2 && key_less(g, kj) && key_less(kj, n2)) {
                        if (key_less(kj, n1)) {
                            n2 = n1;
                            n1 = kj;
                        } else {
                            n2 = kj;
                        }
                    }
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {  // merge the sorted pairs
                const Key<KIND> b1 = key_shfl_xor(n1, o), b2 = key_shfl_xor(n2, o);
                if (key_less(b1, n1)) {
                    n2 = key_less(n1, b2) ? n1 : b2;
                    n1 = b1;
                } else if (key_less(b1, n2)) {
                    n2 = b1;
                }
            }
            if (lane == owner) {
                l1 = n1;
                l2 = n2;
                more = !key_is_none(n2);
            }
        }
    }

    // ---- PoolQueryWorker.runquery:72-98 ----
    int status = ST_PLACE;
    int V = 0;
    if (st.kcount > a.cap) {
        status = ST_OVERFLOW;  // the scan was cut short: rerun with a larger slot (the host escalates the capacity)
    } else if (st.has_zero) {
        status = ST_ZERO;
    } else if (st.kcount <= 2) {
        status = ST_TOO_FEW;
    } else {
        int* node = a.obs_node + (size_t)oslot * a.cap;
        double* dist = a.obs_dist + (size_t)oslot * a.cap;
        const int K = st.kcount;
        int n2 = 1;
        while (n2 < K) n2 <<= 1;
        __syncwarp();
        if constexpr (KIND == SEL_NUCW) {
            for (int i = lane; i < K; i += 32) {
                const unsigned long long c = (unsigned long long)__double_as_longlong(dist[i]);
                dist[i] = jc69_from_counts((uint32_t)(c & 0xffffffffull), (uint32_t)(c >> 32), a.gate.vmin);
            }
        }
        for (int i = K + lane; i < n2; i += 32) {
            node[i] = 0x7fffffff;
            dist[i] = 0.0;
        }
        __syncwarp();
        sort_slot(node, dist, n2, lane);
        __syncwarp();
        V = chain_lengths(a, node, a.obs_len + (size_t)oslot * a.cap, K, lane);
    }
    if (lane == 0) {
        a.K[gid] = st.kcount;
        a.V[gid] = V;
        a.status[gid] = status;
        a.zero_edge[gid] = st.znode;
    }
}

// ---- nucleotide alignment mode: the same selection with the member distances batched ------------------------------
// The generic kernel above expands a cluster the moment it meets it: cluster offsets -> member rows -> reference rows is
// a chain of three dependent round trips to L2 / DRAM per cluster, 12k clocks for a 9-member cluster on B200 -- 80 % of
// the time of the rerun launch and the main stall of the first pass.  Here near units are only QUEUED during the scan
// (shared memory, per warp); once 32 are pending, lane t takes unit t: one parallel load of the 32 cluster extents, a warp
// prefix sum, and the members of all 32 clusters land in one flat list (row, owner lane, position in the cluster).  The
// list is then walked NR rows at a time with the rows PF entries ahead prefetched into L2 -- their addresses are known
// from the list, so nothing waits on a dependent chain any more.  The far units (needed while obs_num < baseobs,
// Reference.py:146) go through the same queue one at a time, in ascending order.  The observed SET, the counts and the
// zero tie-break (by unit key and position) do not depend on the order of expansion, so the results are those of the
// generic kernel bit for bit.
// one warp (query) per block: a block's registers and shared memory stay allocated until its slowest query is done, and
// the queries of a block differ by 10x in work.  Measured 4 / 2 / 1 warps per block: 45.3 / 44.7 / 44.6 ms per step for the
// first pass, 43.8-44.2 with the rerun launch at 1 as well (tools/ab_variants.sh, same box)
#ifndef SEL_NUC_WARPS
#define SEL_NUC_WARPS 1
#endif
#ifndef SEL_HEAVY_WARPS
#define SEL_HEAVY_WARPS 1
#endif
// shared 32-bit words per warp: `words` for the queue, the member list and the sort, then one byte per key line
__host__ __device__ inline int sel_nuc_warp_words(int words, int n_units) { return words + (n_units + 127) / 128; }

template <bool HEAVY>
__global__ void __launch_bounds__(32 * (HEAVY ? SEL_HEAVY_WARPS : SEL_NUC_WARPS), (HEAVY ? 16 : 32) / (HEAVY ? SEL_HEAVY_WARPS : SEL_NUC_WARPS))
select_nuc_kernel(const SelectArgs a) {
    constexpr int KIND = SEL_NUC;
    constexpr int NR = HEAVY ? 8 : SEL_NR;
    constexpr int WORDS = HEAVY ? 4096 : 1024;  // shared 32-bit words per warp (also the sort buffer of the tail)
    constexpr int QCAP = 320;                   // pending units: fewer than 32 left over + one chunk of 256 keys
    constexpr int LCAP = (WORDS - QCAP) / 2;    // member list entries
#ifndef SEL_PF
#define SEL_PF 8
#endif
    constexpr int PF = HEAVY ? 16 : SEL_PF;     // rows prefetched ahead of the one being counted
    constexpr int POS_BITS = 27;
    extern __shared__ uint32_t s_sortbuf[];
    uint32_t* wbuf = s_sortbuf + (threadIdx.x >> 5) * sel_nuc_warp_words(WORDS, a.n_units);
    int* queue = reinterpret_cast<int*>(wbuf);
    int* lrow = reinterpret_cast<int*>(wbuf + QCAP);
    uint32_t* lmeta = wbuf + QCAP + LCAP;
    const int lane = threadIdx.x & 31;
    const int slot = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (slot >= a.n) return;
    const int gid = a.out_map ? a.out_map[slot] : a.q_begin + slot;
    const int oslot = a.out_map ? slot : gid;
    const int self = a.self_node ? a.self_node[gid] : -1;
    const uint32_t* __restrict__ krow = a.keys_nuc + (size_t)slot * a.ldk;
    const uint32_t* __restrict__ qrow = a.q_nuc + (size_t)slot * 3 * a.W;
    const int lines = (3 * a.W * 4 + 127) / 128;   // 128-byte lines of a packed reference row

    WarpSel<KIND> st;
    st.obs_num = 0;
    st.kcount = 0;
    st.has_zero = false;
    st.zpos = 0;
    st.znode = -1;
    st.zkey.idx = 0;

    // ---- the key row is read line by line (32 keys, one 128-byte load), driven by the line minima of the count stage
    // (common.cuh).  Near phase: the minima row is read 32 lines at a time and only the lines whose minimum could be near
    // (ratio below the guard band's upper edge P_hi / 65536; the LINE_NONE minimum never is, and nothing is when P_hi =
    // 0) are opened: their near keys go to the queue, their smallest far key becomes the line's entry.  A line that is
    // not opened holds no near key (its usable keys all have a ratio >= its minimum's).  Far phase: an exact lazy merge
    // over the lines, in (ratio, index) order.  The entry of a line not opened is its minimum with index 32 l, a lower
    // bound of every key of the line under key_less; the entry of an opened line is its smallest far key after the last
    // one taken.  The warp-wide smallest entry is either a bound (the line is opened, its entry replaced) or the next far
    // unit (queued and expanded as before; its line's entry becomes the line's next far key).  Lane o keeps the smallest
    // entry of the lines l with l % 32 == o; after a line of lane o changes, the warp recomputes that minimum (one
    // entry per lane).  The per-line state lives in shared memory, one byte per line after the WORDS of the queue:
    // LS_UNOPENED, the position (0..31) of the line's current far key, or LS_DONE. ----
    constexpr uint8_t LS_UNOPENED = 0xff, LS_DONE = 32;
    uint8_t* lst = reinterpret_cast<uint8_t*>(wbuf + WORDS);
    const int n_kl = (a.n_units + 31) >> 5;
    const uint32_t* __restrict__ mrow = a.kmin + (size_t)slot * (size_t)(a.ldk >> 5);
    // entry of line l (every lane may ask for a different line)
    auto line_entry = [&](int l) -> Key<KIND> {
        const uint32_t ls = lst[l];
        if (ls == LS_UNOPENED) {
            const uint32_t mk = mrow[l];
            return mk == LINE_NONE ? key_none<KIND>() : make_key<KIND>(mk, 32 * l);
        }
        return ls < 32u ? make_key<KIND>(krow[32 * l + ls], 32 * l + (int)ls) : key_none<KIND>();
    };
    // the smallest far key of line l after g (after nothing: all = true), the same on every lane; lane 0 records its position
    auto load_line = [&](int l, const Key<KIND>& g, bool all, int& cls) -> Key<KIND> {
        const int u = 32 * l + lane;
        const Key<KIND> k = make_key<KIND>(u < a.n_units ? krow[u] : 0u, u);
        cls = classify(a, k);
        Key<KIND> f = (cls == 2 && (all || key_less(g, k))) ? k : key_none<KIND>();
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const Key<KIND> of = key_shfl_xor(f, o);
            if (key_less(of, f)) f = of;
        }
        if (lane == 0) lst[l] = key_is_none(f) ? LS_DONE : (uint8_t)(f.idx & 31);
        __syncwarp();
        return f;
    };
    // the smallest entry of the lines of lane `owner`, computed by the warp
    auto class_min = [&](int owner) -> Key<KIND> {
        Key<KIND> b = key_none<KIND>();
        for (int l = owner + 32 * lane; l < n_kl; l += 32 * 32) {
            const Key<KIND> e = line_entry(l);
            if (key_less(e, b)) b = e;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const Key<KIND> ob = key_shfl_xor(b, o);
            if (key_less(ob, b)) b = ob;
        }
        return b;
    };

    Key<KIND> best = key_none<KIND>();   // far phase: the smallest entry of this lane's lines
    int l0 = 0, cl0 = 0, np = 0, qhead = 0;
    unsigned cand = 0u;                   // lines cl0 + t of the current chunk of minima still to be opened
    bool scan_done = n_kl <= 0, far_init = false;
    unsigned long long pairs = 0ull, lines_read = 0ull;

    for (;;) {
        if (np < 32 && !scan_done) {
            // leftovers to the front of the queue
            int keep = 0;
            if (lane < np) keep = queue[qhead + lane];
            __syncwarp();
            if (lane < np) queue[lane] = keep;
            qhead = 0;
            do {
                if (cand == 0u) {
                    // ---- the next 32 line minima ----
                    const int l = l0 + lane;
                    if (lane == 0 && l0 + 64 < n_kl) prefetch_l2(mrow + l0 + 64);
                    const uint32_t mk = l < n_kl ? mrow[l] : LINE_NONE;
                    if (l < n_kl) lst[l] = LS_UNOPENED;
                    cand = __ballot_sync(FULLMASK, ((mk & 0xffffu) << 16) < a.gate.P_hi * (mk >> 16));
                    cl0 = l0;
                    l0 += 32;
                    __syncwarp();
                } else {
                    // ---- open one line: near keys to the queue (at most 32 on top of fewer than 32 left over) ----
                    const int l = cl0 + __ffs(cand) - 1;
                    cand &= cand - 1;
                    int cls;
                    load_line(l, key_none<KIND>(), true, cls);
                    const unsigned bal = __ballot_sync(FULLMASK, cls == 1);
                    if (cls == 1) queue[np + __popc(bal & ((1u << lane) - 1u))] = 32 * l + lane;
                    np += __popc(bal);
                    ++lines_read;
                }
                scan_done = l0 >= n_kl && cand == 0u;
            } while (np < 32 && !scan_done);
            __syncwarp();
        }
        if (np == 0) {
            // ---- the scan is over and every near unit is expanded: far units, ascending, while obs_num < baseobs ----
            if (!(st.obs_num < a.baseobs && st.kcount <= a.cap)) break;
            if (!far_init) {
                for (int l = lane; l < n_kl; l += 32) {
                    const Key<KIND> e = line_entry(l);
                    if (key_less(e, best)) best = e;
                }
                far_init = true;
            }
            for (;;) {
                Key<KIND> g = best;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const Key<KIND> og = key_shfl_xor(g, o);
                    if (key_less(og, g)) g = og;
                }
                if (key_is_none(g)) break;  // no far unit left
                const int l = g.idx >> 5;
                const bool bound = lst[l] == LS_UNOPENED;
                int cls;
                load_line(l, g, bound, cls);   // opens the line, or moves its entry past g
                lines_read += bound ? 1ull : 0ull;
                const Key<KIND> nb = class_min(l & 31);
                if (lane == (l & 31)) best = nb;
                if (!bound) {
                    if (lane == 0) queue[0] = g.idx;
                    qhead = 0;
                    np = 1;
                    break;
                }
            }
            if (np == 0) break;
            __syncwarp();
        }
        // ---- expand up to 32 pending units: lane t owns unit t ----
        const int take = min(np, 32);
        Key<KIND> ukey = key_none<KIND>();
        int b = 0, e = 0;
        if (lane < take) {
            const int idx = queue[qhead + lane];
            ukey = make_key<KIND>(krow[idx], idx);
            b = a.goff[idx];
            e = a.goff[idx + 1];
        }
        qhead += take;
        np -= take;
        int cur = b;
        for (;;) {
            const int rem = e - cur;
            int incl = rem;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(FULLMASK, incl, o);
                if (lane >= o) incl += t;
            }
            const int total = __shfl_sync(FULLMASK, incl, 31);
            if (total == 0) break;
            const int excl = incl - rem;
            const int tk = max(0, min(rem, LCAP - excl));
            for (int x = 0; x < tk; ++x) {
                lrow[excl + x] = a.gmem[cur + x];
                lmeta[excl + x] = ((uint32_t)lane << POS_BITS) | (uint32_t)(cur + x - b);
            }
            cur += tk;
            const int nl = min(total, LCAP);
            __syncwarp();
            for (int i = lane; i < min(PF, nl) * lines; i += 32)
                prefetch_l2(reinterpret_cast<const char*>(a.refs_nuc + (size_t)lrow[i / lines] * 3 * a.W) + (i % lines) * 128);
            for (int x0 = 0; x0 < nl && st.kcount <= a.cap; x0 += NR) {
                int rows[NR], nodes[NR];
                uint32_t meta[NR], c[NR];
#pragma unroll
                for (int k = 0; k < NR; ++k) {
                    const int x = min(x0 + k, nl - 1);
                    rows[k] = lrow[x];
                    meta[k] = lmeta[x];
                }
#pragma unroll
                for (int k = 0; k < NR; ++k) nodes[k] = a.ref_node[rows[k]];
                for (int i = lane; i < NR * lines; i += 32) {
                    const int x = x0 + PF + i / lines;
                    if (x < nl) prefetch_l2(reinterpret_cast<const char*>(a.refs_nuc + (size_t)lrow[x] * 3 * a.W) + (i % lines) * 128);
                }
                member_counts_nuc<NR>(a, qrow, rows, lane, c);
#pragma unroll
                for (int k = 0; k < NR; ++k)
                    if (x0 + k < nl) {
                        const Key<KIND> uk = key_shfl(ukey, (int)(meta[k] >> POS_BITS));
                        observe_nuc_counts(a, st, oslot, self, nodes[k], c[k], uk, (int)(meta[k] & ((1u << POS_BITS) - 1u)), lane);
                    }
                pairs += (unsigned long long)min(NR, nl - x0);
            }
            __syncwarp();
            if (st.kcount > a.cap) break;
        }
        if (st.kcount > a.cap) break;
    }
    if (lane == 0 && a.pair_counter && pairs) atomicAdd(a.pair_counter, pairs);
    if (lane == 0 && a.line_counter && lines_read) atomicAdd(a.line_counter, lines_read);

    // ---- PoolQueryWorker.runquery:72-98 (as in select_kernel) ----
    int status = ST_PLACE;
    int V = 0;
    if (st.kcount > a.cap) {
        status = ST_OVERFLOW;
        if (a.stash_keys != nullptr) {
            int pos = 0;
            if (lane == 0) pos = atomicAdd(a.stash_count, 1);
            pos = __shfl_sync(FULLMASK, pos, 0);
            if (pos < a.stash_cap) {
                const uint4* src = reinterpret_cast<const uint4*>(krow);
                uint4* dst = reinterpret_cast<uint4*>(a.stash_keys + (size_t)pos * a.ldk);
                for (int64_t x = lane; x < a.ldk / 4; x += 32) dst[x] = src[x];
                uint32_t* mdst = a.stash_kmin + (size_t)pos * (size_t)(a.ldk >> 5);
                for (int64_t x = lane; x < (a.ldk >> 5); x += 32) mdst[x] = mrow[x];
                if (lane == 0) a.stash_ids[pos] = gid;
            }
        }
    } else if (st.has_zero) {
        status = ST_ZERO;
    } else if (st.kcount <= 2) {
        status = ST_TOO_FEW;
    } else {
        int* node = a.obs_node + (size_t)oslot * a.cap;
        double* dist = a.obs_dist + (size_t)oslot * a.cap;
        int* cnt = a.obs_len + (size_t)oslot * a.cap;   // packed counts parked by observe()
        const int K = st.kcount;
        int n2 = 1, sh = 0;
        while (n2 < K) {
            n2 <<= 1;
            ++sh;
        }
        __syncwarp();
        if (n2 <= WORDS && ((unsigned long long)a.tree.M << sh) <= (1ull << 32)) {
            uint32_t* skey = wbuf;   // the queue and the member list are dead by now
            for (int i = lane; i < n2; i += 32) skey[i] = i < K ? (((uint32_t)node[i] << sh) | (uint32_t)i) : 0xffffffffu;
            __syncwarp();
            sort_keys_smem(skey, n2, lane);
            for (int i = lane; i < K; i += 32) {   // gather: jc69 correction of the observed leaves in sorted order
                const uint32_t key = skey[i];
                const uint32_t c = (uint32_t)cnt[key & (uint32_t)(n2 - 1)];
                dist[i] = jc69_from_counts(c & 0xffffu, c >> 16, a.gate.vmin);
                node[i] = (int)(key >> sh);
            }
        } else {   // slots beyond the buffer (second-level reruns) or node ids too wide for the packed key
            for (int i = lane; i < K; i += 32) {
                const uint32_t c = (uint32_t)cnt[i];
                dist[i] = jc69_from_counts(c & 0xffffu, c >> 16, a.gate.vmin);
            }
            for (int i = K + lane; i < n2; i += 32) {
                node[i] = 0x7fffffff;
                dist[i] = 0.0;
            }
            __syncwarp();
            sort_slot(node, dist, n2, lane);
        }
        __syncwarp();   // the chain lengths below overwrite the parked counts
        V = chain_lengths(a, node, a.obs_len + (size_t)oslot * a.cap, K, lane);
    }
    if (lane == 0) {
        a.K[gid] = st.kcount;
        a.V[gid] = V;
        a.status[gid] = status;
        a.zero_edge[gid] = st.znode;
    }
}

void launch_select(int kind, const SelectArgs& a, cudaStream_t s) {
    if (a.n <= 0) return;
    if (kind == SEL_NUC && a.out_map) {  // overflow rerun
        const int w = SEL_HEAVY_WARPS;
        const size_t sm = (size_t)w * sel_nuc_warp_words(4096, a.n_units) * 4;   // select_nuc_kernel<true>: WORDS = 4096
        cudaFuncSetAttribute(select_nuc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        select_nuc_kernel<true><<<(a.n + w - 1) / w, w * 32, sm, s>>>(a);
    } else if (kind == SEL_NUC) {
        const int w = SEL_NUC_WARPS;
        const size_t sm = (size_t)w * sel_nuc_warp_words(1024, a.n_units) * 4;
        cudaFuncSetAttribute(select_nuc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm);
        select_nuc_kernel<false><<<(a.n + w - 1) / w, w * 32, sm, s>>>(a);
    } else {
        const int w = SEL_GEN_WARPS;
        const dim3 g((a.n + w - 1) / w), b(w * 32);
        if (kind == SEL_NUCW) select_kernel<SEL_NUCW><<<g, b, 0, s>>>(a);
        else if (kind == SEL_AA) select_kernel<SEL_AA><<<g, b, 0, s>>>(a);
        else if (kind == SEL_K2P) select_kernel<SEL_K2P><<<g, b, 0, s>>>(a);
        else select_kernel<SEL_MATRIX><<<g, b, 0, s>>>(a);
    }
}
