// Shared declarations for the sm_100a kernels behind include/apples_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/apples_b200.h"

// ---------------------------------------------------------------------------------------------------------------
// tile shape of the dense query x representative distance kernel (distance.cu)
// ---------------------------------------------------------------------------------------------------------------
#ifndef DT_TQ_V
#define DT_TQ_V 128
#endif
constexpr int DT_TQ = DT_TQ_V;  // queries per CTA tile
#ifndef DT_TR_V
#define DT_TR_V 64
#endif
constexpr int DT_TR = DT_TR_V;  // representatives per CTA tile
#ifndef DT_WC_V
#define DT_WC_V 32
#endif
constexpr int DT_WC = DT_WC_V;  // 32-site words per pipeline stage
#ifndef DT_STAGES_V
#define DT_STAGES_V 2
#endif
#ifndef DT_MINBLOCKS
#define DT_MINBLOCKS 1
#endif
constexpr int DT_STAGES = DT_STAGES_V;    // TMA pipeline depth
constexpr int DT_CONSUMERS = (DT_TQ / 4) * (DT_TR / 4);  // one thread per 4x4 block of pairs
#ifndef DT_SELF_PRODUCE
#define DT_SELF_PRODUCE 1  // 1: no producer warp, thread 0 keeps the ring full (128 registers per thread); 0: 17th warp
#endif
constexpr int DT_THREADS = DT_CONSUMERS + (DT_SELF_PRODUCE ? 0 : 32);  // + one producer warp unless warp 0 produces
constexpr int DT_STAGE_WORDS = 3 * DT_WC * (DT_TQ + DT_TR);
constexpr int DT_STAGE_BYTES = DT_STAGE_WORDS * 4;
constexpr int DT_SMEM_BYTES = DT_STAGES * DT_STAGE_BYTES + 2 * DT_STAGES * 8 + 16;

// tile shape of the dense amino-acid kernel (distance.cu)
constexpr int AA_CH = 64;        // sites per pipeline stage
constexpr int AA_TR = 256;       // references per CTA tile (2 per thread)
constexpr int AA_TQ = 8;         // queries per CTA tile
constexpr int AA_THREADS = 128;
constexpr int AA_TABW = 32;      // table row pitch in words
constexpr int AA_LIMB = 22;      // bits of the low limb
constexpr int AA_FRAC = 43;      // fixed-point fraction bits
constexpr int AA_TAB_WORDS = 2 * 21 * AA_TABW;

// internal per-query status used between the selection and the placement kernel
constexpr int ST_PLACE = 0;      // observed set ready, go on to placement
constexpr int ST_ZERO = 1;       // zero-distance shortcut, zero_edge holds the leaf
constexpr int ST_TOO_FEW = 2;    // <= 2 observed distances
constexpr int ST_OVERFLOW = 100; // more observed leaves than the slot capacity: rerun with a larger one

struct TreeDev {
    int M;
    const int* parent;
    const double* elen;
    const int* level;
    const int* first;
};

// gates of jc69 (distance.py:735-745) in the integer domain plus the fast near/far classification
struct NucGate {
    int L;
    int vmin;     // smallest valid-site count that passes `valid / L < overlap_frac` (distance.py:735)
    uint32_t P_lo;  // (mism << 16) <= P_lo * valid  =>  certainly dist <= threshold
    uint32_t P_hi;  // (mism << 16) >= P_hi * valid  =>  certainly dist >  threshold
    double thr;
};

// jc69 from the integer counts: the fp64 operations of distance.py:737-745 in the same order
__device__ __forceinline__ double jc69_from_counts(uint32_t m, uint32_t v, int vmin) {
    if (v == 0u || (int)v < vmin) return -1.0;
    if (m == 0u) return 0.0;  // p - eps < 0  <=>  p == 0 for p = m/v with v <= 65535
    double p = (double)m / (double)v;
    double loc = 1.0 - (4.0 * p) / 3.0;
    if (0.0 >= loc) return -1.0;
    return -0.75 * log(loc);
}

// Kimura two-parameter distance from the integer counts: transitions ts, transversions tv, valid sites v (the gate of
// jc69_from_counts), the fp64 operations of tests/k2p_oracle.py in the same order.  Only for the -fmad=false units: the
// 0 >= w1 / 0 >= w2 decisions must be the oracle's bit for bit
__device__ __forceinline__ double k2p_from_counts(uint32_t ts, uint32_t tv, uint32_t v, int vmin) {
    if (v == 0u || (int)v < vmin) return -1.0;
    if (ts + tv == 0u) return 0.0;
    const double P = (double)ts / (double)v;
    const double Q = (double)tv / (double)v;
    const double w1 = 1.0 - 2.0 * P - Q;
    const double w2 = 1.0 - 2.0 * Q;
    if (0.0 >= w1 || 0.0 >= w2) return -1.0;
    return -0.5 * log(w1) - 0.25 * log(w2);
}

// ---- per-line key minima (count stage -> selection).  A line is the 32 keys [32 l, 32 l + 32) of a key row; its minimum
// is the key of smallest ratio m / v among the keys the selection can use (v >= max(vmin, 1) and 4 m < 3 v, the gate of
// classify() in select.cu), the smallest column on equal ratios, or LINE_NONE when no key of the line is usable.  A pure
// function of the keys: both count kernels fold it with these two helpers.
constexpr uint32_t LINE_NONE = 1u;   // m = 1, v = 0: compares greater than every usable key

// the key itself when the selection can use it, LINE_NONE otherwise (vmin1 = max(vmin, 1))
__device__ __forceinline__ uint32_t line_usable(uint32_t k, uint32_t vmin1) {
    const uint32_t m = k & 0xffffu, v = k >> 16;
    return (v >= vmin1 && 4u * m < 3u * v) ? k : LINE_NONE;
}
// the smaller ratio of two usable-or-LINE_NONE keys, exactly (counts <= 65535: products fit 32 bits); a = the smaller column
__device__ __forceinline__ uint32_t line_min2(uint32_t a, uint32_t b) {
    return (b & 0xffffu) * (a >> 16) < (a & 0xffffu) * (b >> 16) ? b : a;
}
// minimum of 32 consecutive keys (k[j] = column 32 l + j, already passed through line_usable): a pairwise tree, left wins ties
__device__ __forceinline__ uint32_t line_min32(uint32_t* k) {
#pragma unroll
    for (int s = 1; s < 32; s <<= 1)
#pragma unroll
        for (int j = 0; j < 32; j += 2 * s) k[j] = line_min2(k[j], k[j + s]);
    return k[0];
}

// scoredist from the BLOSUM45 sum and the valid count (distance.py:699-712)
__device__ __forceinline__ double scoredist_from_sum(double tot, uint32_t v, int L, double overlap) {
    if (v == 0u || (double)v / (double)L < overlap) return -1.0;
    double x = 1.0 - tot / (double)v;
    if (0.0 >= x) return -1.0;
    double cd = -log(x);
    return cd * 1.3;
}

// ---------------------------------------------------------------------------------------------------------------
// selection (select.cu) and placement (placement.cu) launch arguments
// ---------------------------------------------------------------------------------------------------------------
enum { SEL_NUC = 0, SEL_AA = 1, SEL_MATRIX = 2, SEL_NUCW = 3, SEL_K2P = 4 };

struct SelectArgs {
    int n;                 // queries in this launch; their key / query rows are rows 0..n-1 of keys_* / q_*
    const int* out_map;    // optional: row -> query index inside the batch (NULL: q_begin + row).  With a map the
                           // observed lists go to row `row` of obs_*, otherwise to row `query index`
    int q_begin;
    int n_units;           // representatives (alignment) or matrix columns
    int64_t ldk;           // row stride of the key matrix
    const uint32_t* keys_nuc;  // [nq][ldk] packed (mismatch | valid << 16)
    const uint32_t* kmin;      // SEL_NUC: [nq][ldk / 32] line minima of keys_nuc (LINE_NONE etc., see above)
    const double* keys_f64;    // [nq][ldk] distances (protein representatives / matrix rows); SEL_NUCW, SEL_K2P: 64-bit count keys
    const int* goff;       // cluster CSR
    const int* gmem;
    const int* ref_node;
    const uint32_t* refs_nuc;  // row-major [n_ref][3][W]
    const uint32_t* q_nuc;     // row-major [n][3][W]
    int W;
    const uint8_t* refs_bytes; // SEL_NUCW: raw alignment bytes [n_ref][refs_bstride]
    int64_t refs_bstride;
    const uint8_t* q_bytes;    // SEL_NUCW: [n][q_bstride]
    int64_t q_bstride;
    const uint8_t* refs_aa;    // [n_ref][Lp]
    const uint8_t* q_aa;       // [n][Lp]
    int Lp;
    int L;
    const int* col_node;
    const int* self_node;  // [batch] or NULL
    double thr;
    int baseobs;
    double overlap;
    NucGate gate;
    int cap;               // slot capacity (power of two)
    int* obs_node;         // [slots][cap] observed leaves, sorted by node id
    double* obs_dist;      // [slots][cap]
    int* obs_len;          // [slots][cap] length of the chain each observed leaf owns (placement.cu)
    int* K;                // [nq] observed leaves (may exceed cap)
    int* V;                // [nq] valid nodes of the restricted subtree
    int* status;           // [nq] ST_*
    int* zero_edge;        // [nq]
    unsigned long long* pair_counter;  // number of member distances evaluated (statistics)
    unsigned long long* line_counter;  // SEL_NUC: number of key lines loaded (statistics)
    // key-row stash (nucleotide alignment mode, first pass only): a query that overflows its slot copies its key row
    // aside so that its rerun needs no second distance pass.  stash_count is bumped for every overflowing query; only
    // the first stash_cap of them are stored (the host falls back to recomputing when there are more)
    uint32_t* stash_keys;  // [stash_cap][ldk] or NULL
    uint32_t* stash_kmin;  // [stash_cap][ldk / 32] their line minima
    int* stash_ids;        // [stash_cap] query index inside the batch
    int* stash_count;
    int stash_cap;
    TreeDev tree;
};

// placement launch classes: working set in shared memory for up to 64 / 128 / 256 / 512 node slots (V + 1), else one
// block per query with the working set in the global scratch pool
enum { PLACE_CLASS_64 = 0, PLACE_CLASS_128 = 1, PLACE_CLASS_256 = 2, PLACE_CLASS_512 = 3, PLACE_CLASS_BLOCK = 4, PLACE_NCLASS = 5 };
constexpr int PLACE_NODE_SLOT_BYTES = 128;   // global scratch per node slot (13 doubles + 5 ints = 124 bytes used)
constexpr int PLACE_CHAIN_SLOT_BYTES = 16;   // global scratch per chain (4 ints)

struct PlaceArgs {
    int n;                 // entries in this launch (finalize: queries of the batch)
    const int* qlist;      // launch entry -> query index inside the batch
    const int* slot_list;  // launch entry -> row of the observed-list buffers (NULL: the query index)
    int cap;               // slots per row of the observed-list buffers
    const int* obs_node;
    const double* obs_dist;
    const int* obs_len;
    const int* K;
    const int* status;
    const int* zero_edge;
    const long long* rec_off;    // PLACE_CLASS_BLOCK: n + 1 offsets into the node-slot pool
    const long long* stack_off;  // PLACE_CLASS_BLOCK: n + 1 offsets into the chain-slot pool
    void* recs;
    void* stacks;
    int criterion;
    int negative_branch;
    TreeDev tree;
    int* out_edge;
    double* out_error;
    double* out_distal;
    double* out_pendant;
    int* out_status;
    // ranked records (keep > 1, apples_set_alternatives): record j of query q at [q * keep + j], records 0 .. count[q] - 1
    // in criterion order (record 0 = the placement above), unused slots edge -1 and zeros
    int keep;
    int* alt_count;
    int* alt_edge;
    double* alt_error;
    double* alt_distal;
    double* alt_pendant;
    unsigned char* alt_int0;
    // optional per-edge export for one query (index inside the batch), arrays of M
    int dbg_query;
    double* dbg_x1;
    double* dbg_x2;
    double* dbg_err;
    unsigned char* dbg_valid;
};

// kernels / launchers implemented in the .cu files
void launch_transpose_nuc(const uint32_t* rm, int rows, int W, uint32_t* wm, int Wp, int rows_pad, int tile_rows,
                          cudaStream_t s);
void launch_row_valid(const uint32_t* rm, int rows, int W, uint32_t* nv, int rows_pad, cudaStream_t s);
void launch_dense_nuc_keys(const uint32_t* q_wm, const uint32_t* q_nv, int q_pad, const uint32_t* r_wm,
                           const uint32_t* r_nv, int r_pad, int W, int Wp, uint32_t* keys, int64_t ldk,
                           unsigned long long* clk, int num_sms, cudaStream_t s);
void launch_line_minima(const uint32_t* keys, int rows, int64_t ldk, int vmin, uint32_t* kmin, cudaStream_t s);
void launch_dense_nuc_full(const uint32_t* q_wm, const uint32_t* q_nv, int q_pad, int nq, const uint32_t* r_wm,
                           const uint32_t* r_nv, int r_pad, int n_ref, int W, int Wp, int vmin, uint32_t* mism, uint32_t* valid,
                           double* dist, int num_sms, cudaStream_t s);
void launch_aa_layout(const uint8_t* codes, int rows, int Lp, int T, int rows_pad, uint8_t* tm, uint32_t* vm, cudaStream_t s);
void launch_dense_aa(const uint8_t* q_tm, const uint32_t* q_vm, int q_pad, int nq, const uint8_t* r_tm, const uint32_t* r_vm,
                     int r_pad, int n_r, int Lp, int L, double overlap, const uint32_t* tab, uint32_t* valid, int64_t ldv,
                     double* dist, int64_t ldd, cudaStream_t s);
void aa_build_tables(const double* blosum441, uint32_t* out);
void launch_select(int kind, const SelectArgs& a, cudaStream_t s);
cudaError_t launch_place(int method, int vclass, const PlaceArgs& a, cudaStream_t s);
cudaError_t launch_place_finalize(const PlaceArgs& a, cudaStream_t s);
cudaError_t launch_bin_classes(int n, const int* status, const int* K, const int* V, const int* row_flag, int* counts, int* lists,
                               unsigned long long* stats, cudaStream_t s);
cudaError_t dense_nuc_configure();
// tensor-core experiment (dense_tc.cu)
cudaError_t dense_tc_configure();
int dense_tc_max_sites();
int dense_tc_tile_rows();
size_t dense_tc_image_bytes(int rows_pad, int n_w);
void launch_tc_image(const uint32_t* planes, int rows, int W, int n_w, int rows_pad, int vw, void* out, cudaStream_t s);
void launch_dense_tc(const void* a_img, int q_pad, const void* b_img, int r_pad, int n_w, uint32_t* keys, int64_t ldk,
                     uint32_t* kmin, int vmin, int num_sms, cudaStream_t s);
// block-scaled fp4 count kernel (dense_tc.cu): tiles of 128 queries (side 0) x 224 representatives (side 1), or x 160
// representatives for the K2P keys (k2p)
int dense_fp4_max_sites();
int dense_fp4_tile_rows(int side, bool k2p = false);
size_t dense_fp4_image_bytes(int rows_pad, int n_w);
void launch_fp4_image(const uint32_t* planes, int rows, int W, int n_w, int rows_pad, int tile_rows, void* out, cudaStream_t s);
void launch_dense_fp4(const void* a_img, int q_pad, const void* b_img, int r_pad, int n_w, uint32_t* keys, int64_t ldk,
                      uint32_t* kmin, int vmin, int num_sms, cudaStream_t s);
// K2P keys (ts | tv << 16 | valid << 32) [q_pad][ldk]; b_img built with dense_fp4_tile_rows(1, true) rows per tile
void launch_dense_fp4_k2p(const void* a_img, int q_pad, const void* b_img, int r_pad, int n_w, unsigned long long* keys,
                          int64_t ldk, int num_sms, cudaStream_t s);
cudaError_t launch_pack(int kind, const uint8_t* bytes, int64_t row_stride, int n, int L, void* out, int* bad, cudaStream_t s,
                        int* row_flag = nullptr);
cudaError_t launch_repitch_bytes(const uint8_t* src, int64_t src_stride, int n, int L, int Lp, uint8_t* dst, cudaStream_t s);
cudaError_t launch_unpack_nuc(const uint32_t* planes, int n, int L, int W, int Lp, uint8_t* dst, cudaStream_t s);
void launch_dense_bytes(const uint8_t* q, int64_t q_stride, int nq, const uint8_t* r, int64_t r_stride, int n_r, int Lp,
                        unsigned long long* keys, int64_t ldk, cudaStream_t s);
void launch_bytes_keys_to_counts(const unsigned long long* keys, int64_t n, int vmin, uint32_t* mism, uint32_t* valid, double* dist,
                                 cudaStream_t s);
cudaError_t launch_gather_rows(const void* src, const int* idx, void* dst, int n, size_t row_bytes, cudaStream_t s);
cudaError_t launch_consensus(int kind, const uint8_t* bytes, int64_t row_stride, int L, int n_rep, const int* goff,
                             const int* gmem, uint8_t* out, int64_t out_stride, cudaStream_t s);
