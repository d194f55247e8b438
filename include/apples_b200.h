/* apples_b200.h -- C ABI of the B200 placement hot path (libapples_b200.so).
 *
 * The reference (balabanmetin/apples v2.0.11) is pure Python and has no FFI; the seam this library sits behind is
 * the one call that fans queries out to worker processes,
 *     results = pool.starmap(queryworker.runquery, queries)                     run_apples.py:94-102
 * i.e. per query: PoolQueryWorker.runquery (apples/PoolQueryWorker.py:28-141)
 *     -> ReducedReference.get_obs_dist (apples/Reference.py:117-157) / valid_dists (PoolQueryWorker.py:44-59)
 *     -> jc69 / scoredist (apples/distance.py:718-745, 681-715)
 *     -> Subtree (apples/Subtree.py:23-43) -> FM/OLS/BME/BE moments (apples/FM.py, OLS.py, BME.py, BE.py)
 *     -> util.solve2_2 (apples/util.py:6-54) -> Algorithm.placement (apples/Algorithm.py:62-101).
 * INTEGRATION.md shows the ctypes binding a maintainer of the reference would add at that call site.
 *
 * Conventions: every function returns 0 on success and a negative code on error (text via apples_last_error).
 * No exceptions cross the boundary.  The caller owns every host buffer, the context owns every device buffer.
 * One context per GPU; a context is not thread-safe (one host thread per context); contexts on different devices
 * are independent.  All pointers are plain host pointers unless a function says "device".
 *
 * Node ids everywhere are the reference's `edge_index` (post-order rank of the node, root last; util.py:57-69).
 */
#ifndef APPLES_B200_H
#define APPLES_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct apples_ctx apples_ctx;

/* sequence kinds (fasta2dic.py:56-61 alphabets) */
#define APPLES_NUC 0 /* 3 bit-planes (lo, hi, valid) of uint32 words per row: uint32[rows][3][W], W = apples_words_per_row(L) */
#define APPLES_AA 1  /* one uint8 code per site (0..19 in a2i order, 20 = gap): uint8[rows][apples_aa_row_bytes(L)] */

/* weighting methods (PoolQueryWorker.py:104-111) and selection criteria (Algorithm.py:76-91) */
#define APPLES_FM 0
#define APPLES_OLS 1
#define APPLES_BME 2
#define APPLES_BE 3
#define APPLES_MLSE 0
#define APPLES_ME 1
#define APPLES_HYBRID 2

/* per-query status = code | flags; carries the control flow of PoolQueryWorker.runquery:62-130 */
#define APPLES_STATUS_CODE_MASK 0xff
#define APPLES_PLACED 0                   /* p = [edge, error, 1, distal, pendant]                      (:114-120) */
#define APPLES_ZERO_DIST_LEAF 1           /* an observed distance is 0: edge = that leaf, rest 0,1,0,0  (:72-75)   */
#define APPLES_TOO_FEW_DISTANCES 2        /* <= 2 observed distances: edge = -1                         (:97-98)   */
#define APPLES_PLACED_MISPLACEMENT_FLAG 3 /* placed, potential_misplacement_flag == 1                   (:121-130) */
#define APPLES_FLAG_PENDANT_INT0 0x100    /* pendant is the Python int 0 (clipped), prints as 0 not 0.0 (util.py:34-47) */
#define APPLES_FLAG_DEGENERATE 0x200      /* the 2x2 system of at least one edge of this query is singular in fp64
                                           * (a_11 a_22 - a_12 a_21 == 0 or its reciprocal == 0): the reference raises
                                           * ZeroDivisionError / AssertionError in util.solve2_2 (util.py:26-27) and the
                                           * whole run dies; the other outputs of the query are then inf/nan arithmetic
                                           * and carry no meaning.  apples_b200.placer.place_batch raises likewise. */

typedef struct apples_params {
    int32_t method;                     /* -m  APPLES_FM|OLS|BME|BE                 (OptionsRun.py:26-33) */
    int32_t criterion;                  /* -c  APPLES_MLSE|ME|HYBRID                (OptionsRun.py:34-41) */
    int32_t negative_branch;            /* -n                                       (OptionsRun.py:42-48) */
    int32_t base_observation_threshold; /* -b  default 25                           (OptionsRun.py:49-57) */
    double filt_threshold;              /* -f  default 0.2                          (OptionsBasic.py:45-54) */
    double overlap_frac;                /* -V  default 0.001                        (OptionsRun.py:58-66) */
} apples_params;

int32_t apples_words_per_row(int32_t L); /* uint32 words per bit-plane row (multiple of 4) */
int32_t apples_aa_row_bytes(int32_t L);  /* bytes per amino-acid code row (multiple of 16) */

/* number of CUDA devices visible to the process (run_apples.py --gpus 0 = all of them, like -T 0 = all cores) */
int apples_device_count(int32_t* count);
int apples_ctx_create(int device, apples_ctx** out);
void apples_ctx_destroy(apples_ctx* ctx);
const char* apples_last_error(const apples_ctx* ctx);
/* the CUDA stream (cudaStream_t) all work of this context is issued on */
void* apples_ctx_stream(apples_ctx* ctx);

/* Tuning knobs (0 keeps the current value): max_subbatch = queries per pipeline pass (rounded to the dense tile),
 * scratch_bytes = upper bound of the placement scratch pool; slot_cap = observed-leaf slots per query before the
 * overflow rerun (power of two). */
int apples_ctx_set_limits(apples_ctx* ctx, int64_t max_subbatch, int64_t scratch_bytes, int32_t slot_cap);

/* Which kernel computes the query x representative mismatch / overlap counts of nucleotide alignments.
 * 1 (default) = the tcgen05 tensor-core kernels (dense_tc.cu): the block-scaled fp4 kernel (kind::mxf4; simplex embedding
 * of A,C,G,T into one fp32 accumulator, validity into a second, both exact) up to its length limit, the kind::i8 kernel
 * (the two counts of distance.py:733-737 as ONE int8 dot product per pair, exact s32 accumulation in TMEM) beyond it;
 * 0 = the integer-pipe LOP3/POPC kernel of the north star (distance.cu).  All give bit-identical 32-bit keys.  Call before
 * apples_set_reference*.  Alignments the tensor-core kernels do not cover (more than 33 816 columns) use the
 * integer-pipe kernel automatically. */
int apples_ctx_set_dense_mode(apples_ctx* ctx, int32_t mode);

/* Substitution model of the nucleotide distances of alignment input.  APPLES_JC69 (default) is upstream's Jukes-Cantor
 * distance.  APPLES_K2P is the Kimura two-parameter distance: with P and Q the fractions of transitions (A<->G, C<->T) and
 * transversions among the valid sites (overlap gate as for JC69),
 *     d = -0.5 ln(1 - 2P - Q) - 0.25 ln(1 - 2Q),   missing when 1 - 2P - Q <= 0 or 1 - 2Q <= 0,   0 without differences.
 * The representatives, the two-phase selection and the placement are upstream's, with K2P in place of JC69.  Call before
 * apples_set_reference*: the model fixes the representative image and the key width.  apples_set_reference* fail for a
 * K2P context with APPLES_AA, with dense mode 0, with more than 33 816 columns, or with reference bytes other than
 * A,C,G,T,-; a place call fails on the first query row holding such bytes.  Distance-matrix calls ignore the model. */
#define APPLES_JC69 0
#define APPLES_K2P 1
int apples_ctx_set_model(apples_ctx* ctx, int32_t model);

/* Backbone tree as flat arrays over the M nodes (replaces the treeswift node graph prepared by
 * prepareTree.py:24-34 + util.py:57-88).  parent[root] = -1; edge_length of a node is the length of the edge above
 * it; level = BFS depth (root 0); first[u] = smallest id in the subtree of u. */
int apples_set_tree(apples_ctx* ctx, int32_t M, const int32_t* parent, const double* edge_length,
                    const int32_t* level, const int32_t* first);

/* Reduced reference (replaces the ReducedReference object, Reference.py:64-112): n_ref packed reference rows with
 * the tree node of each (-1 = not in the tree), n_rep packed representative (consensus) rows in
 * `representatives` list order, and the members of each representative's cluster as reference row indices, in
 * group order: members of representative i are group_members[group_offsets[i] .. group_offsets[i+1]). */
int apples_set_reference(apples_ctx* ctx, int kind, int32_t L, int32_t n_ref, const void* packed_refs,
                         const int32_t* ref_node, int32_t n_rep, const void* packed_reps,
                         const int32_t* group_offsets, const int32_t* group_members);

/* Distance-matrix mode (run_apples.py:39-58): tree node of each matrix column (-1 = tag not in the tree). */
int apples_set_matrix_columns(apples_ctx* ctx, int32_t n_cols, const int32_t* col_node);

/* The hot path, alignment input: replaces pool.starmap(queryworker.runquery, queries) for nq aligned queries.
 * self_node[q] = tree node carrying the query's own name, or -1 (PoolQueryWorker.py:63-70); may be NULL.
 * Outputs (host, nq each): edge (-1 = not placeable), error, distal, pendant, status. */
int apples_place_batch(apples_ctx* ctx, int64_t nq, const void* packed_queries, const int32_t* self_node,
                       const apples_params* params, int32_t* edge, double* error, double* distal, double* pendant,
                       int32_t* status);

/* SURVEY.md section 8 (f1)/(f2): the same two calls fed with ALIGNMENT BYTES as fasta2dic leaves them
 * (fasta2dic.py:42-72: upper-case letters, '-' for gaps and for letters outside the alphabet), uint8[rows][row_stride]
 * with the first L bytes of every row used.  Packing into the device layout and the per-cluster consensus
 * representatives (PoolRepresentativeWorker.py:30-85: column-wise majority in alphabet order, first maximum wins) are
 * computed on the device.  Nucleotide bytes other than A,C,G,T,- (non-letters: fasta2dic maps every other letter to '-')
 * are ordinary characters for jc69 (distance.py:733-737); rows that hold them, and alignments longer than 65 535
 * columns, are computed by a byte-compare fallback with 32-bit counts (exact, about 30x slower than the bit-plane path). */
int apples_set_reference_bytes(apples_ctx* ctx, int kind, int32_t L, int32_t n_ref, const uint8_t* ref_bytes,
                               int64_t row_stride, const int32_t* ref_node, int32_t n_rep, const int32_t* group_offsets,
                               const int32_t* group_members);
int apples_place_batch_bytes(apples_ctx* ctx, int64_t nq, const uint8_t* bytes, int64_t row_stride,
                             const int32_t* self_node, const apples_params* params, int32_t* edge, double* error,
                             double* distal, double* pendant, int32_t* status);

/* Ranked records (pplacer's --keep-at-most): the best `keep` placements of every query, ranked on the device by the
 * criterion -- a stable sort of the valid edges by the criterion's key in edge_index order, truncated to keep (MLSE: error,
 * ME: x_1; HYBRID: the floor(log2 V) candidates of the smallest error sorted by x_1, so at most that many records).
 * Registers caller-owned host buffers that the NEXT apples_place_batch / _bytes / _matrix call fills, beside its usual
 * outputs; that call takes the registration (also when it fails), so it serves one call.  count[nq]; edge, error,
 * distal, pendant and pendant_int0 (1 where the pendant is the Python int 0, as APPLES_FLAG_PENDANT_INT0) are
 * [nq][keep]: record j of query q at q * keep + j for j < count[q].  Record 0 is the placement the call returns in its
 * own outputs.  Queries that are not placed by least squares (APPLES_ZERO_DIST_LEAF, APPLES_TOO_FEW_DISTANCES) have
 * count 1.  Unused slots hold edge -1 and zeros.  1 <= keep <= APPLES_MAX_KEEP; keep = 1 or six NULL buffers clear the
 * registration.  One call beside the three place calls instead of three twins of them: their signatures stay. */
#define APPLES_MAX_KEEP 16
int apples_set_alternatives(apples_ctx* ctx, int32_t keep, int32_t* count, int32_t* edge, double* error, double* distal,
                            double* pendant, uint8_t* pendant_int0);

/* The hot path, distance-matrix input: rows is double[nq][n_cols] (run_apples.py:43-54). */
int apples_place_batch_matrix(apples_ctx* ctx, int64_t nq, const double* rows, const int32_t* self_node,
                              const apples_params* params, int32_t* edge, double* error, double* distal,
                              double* pendant, int32_t* status);

/* Device-resident variant used by bench.py's kernel-only timing: upload once, place many times.  Results stay on
 * the device until apples_results_download. */
int apples_queries_upload(apples_ctx* ctx, int64_t nq, const void* packed_queries, const int32_t* self_node);
int apples_place_resident(apples_ctx* ctx, const apples_params* params);
int apples_results_download(apples_ctx* ctx, int32_t* edge, double* error, double* distal, double* pendant,
                            int32_t* status);
/* same, into DEVICE buffers of the caller (e.g. the send buffers of the final NCCL gather of placements) */
int apples_results_to_device(apples_ctx* ctx, void* edge, void* error, void* distal, void* pendant, void* status);

/* ---- parity exports (test-only seams named in SURVEY.md section 8b) ---- */

/* kernel (a): mismatch / valid-overlap site counts and corrected distance of every query x reference pair
 * (distance.py:733-745, 698-712).  Arrays are [nq][n_ref].  For APPLES_AA `mism` is not defined and left 0. */
int apples_distance_counts(apples_ctx* ctx, int64_t nq, const void* packed_queries, double overlap_frac,
                           uint32_t* mism, uint32_t* valid, double* dist);

/* kernel (a) as the hot path runs it: the query x REPRESENTATIVE keys of nq packed queries, straight from the count stage
 * of apples_place_batch (same kernels, kernel choice, sub-batches and key-matrix layout; the batch stops before the
 * selection).  keys is [nq][n_rep] (padding columns dropped); *key_kind tells what it holds:
 *   0  uint32  mismatch | valid << 16   (tensor-core or integer-pipe kernel)
 *   1  uint64  mismatch | valid << 32   (byte-compare fallback: L > 65 535 or bytes other than A,C,G,T,- in the reference)
 *   2  double  scoredist with params->overlap_frac (APPLES_AA)
 *   3  uint64  transitions | transversions << 16 | valid << 32   (APPLES_K2P contexts)
 * The caller sizes keys for 8 bytes per entry unless it knows the context's kind.
 * line_minima (optional, NULL = not wanted; written for kind 0 only) is [nq][ceil(n_rep / 32)]: per line of 32 keys
 * [32 l, 32 l + 32), the key of smallest ratio mismatch / valid among the keys with valid >= max(vmin, 1) and
 * 4 mismatch < 3 valid (vmin: the smallest valid count that passes params->overlap_frac), the smallest column on equal
 * ratios, or 0x00000001 when no key of the line qualifies.  The selection reads only the lines these minima call for. */
int apples_count_keys(apples_ctx* ctx, int64_t nq, const void* packed_queries, const apples_params* params,
                      int32_t* key_kind, void* keys, uint32_t* line_minima);

/* kernel (c): the observed set of each query as the reference would hold it after PoolQueryWorker.py:40-70 (self
 * entry removed), sorted by node id; count[q] may exceed cap (then only cap entries are written).
 * Exactly one of packed_queries / rows is non-NULL. */
int apples_observed_sets(apples_ctx* ctx, int64_t nq, const void* packed_queries, const double* rows,
                         const int32_t* self_node, const apples_params* params, int32_t cap, int32_t* count,
                         int32_t* node, double* dist);

/* kernel (b): per-edge solution of ONE query: x_1, x_2 (util.py:50-53) and error_per_edge for every node of the
 * tree (arrays of M), valid[u] = 1 where the node is in the query's restricted subtree (Subtree.py:23-43). */
int apples_edge_solutions(apples_ctx* ctx, const void* packed_query, const double* row, int32_t self_node,
                          const apples_params* params, double* x1, double* x2, double* err, uint8_t* valid);

/* test seam: per-query counts of the LAST macro-batch placed through this context (at most 2^20 queries): K = observed
 * leaves, V = valid nodes of the restricted subtree (Subtree.num_nodes, Subtree.py:42), overflowed = 1 where the query
 * went through a rerun (observed set larger than the slot capacity, or the byte-compare fallback).  Any pointer may be NULL. */
int apples_last_counts(apples_ctx* ctx, int64_t n, int32_t* K, int32_t* V, int32_t* overflowed);

/* accumulated device time per stage since the last call with reset != 0, in milliseconds (CUDA events):
 * [0] h2d  [1] transpose  [2] rep distance  [3] selection  [4] placement  [5] d2h  [6] launches (count)
 * [7] rep-distance launches (count) [8] query-representative pairs evaluated [9] observed leaves [10] valid nodes
 * [11] overflow reruns (queries) [12] largest observed set [13] largest restricted subtree
 * [14] effective SM clock in MHz during the last representative-distance launch (clock64 / globaltimer, in-kernel)
 * [15..19] queries placed by the shared-memory placement launches of 64 / 128 / 256 / 512 node slots and by the
 * block-per-query launch (global scratch)  [20] queries that went through the byte-compare fallback
 * [21] representative-distance launches that ran on the tensor cores
 * [22] key lines (32 keys) the nucleotide selection opened, first pass
 * [23] representative-distance launches that ran the block-scaled fp4 tensor-core kernel (counted in [21] too)
 * [24] representative-distance launches that ran its K2P instantiation (counted in [21] and [23] too) */
int apples_get_timings(apples_ctx* ctx, double* out, int n, int reset);

/* ---- host side of SURVEY.md section 8 (f1) / (f3) in native code (no CUDA kernel involved) ---- */

/* FASTA / FASTQ file -> byte matrix, replacing apples/fasta2dic.py:4-72 (readfq + fasta2dic): records in file order,
 * name = header up to the first blank, sequences upper-cased (mask_flag: lower case -> '-'), letters outside the
 * alphabet (nucleotide: everything but A,C,G,T; protein: B,J,O,U,X,Z) -> '-', every other byte kept.  The matrix is
 * uint8[n][stride], stride = max length rounded up to 16, rows padded with '-'; it is pinned host memory when
 * want_pinned != 0 and a CUDA device is usable, so apples_place_batch_bytes can DMA straight from it.
 * n_threads <= 0: all cores.  err (may be NULL) receives a message on failure. */
typedef struct apples_fasta apples_fasta;
int apples_fasta_open(const char* path, int prot_flag, int mask_flag, int n_threads, int want_pinned, apples_fasta** out,
                      char* err, int errlen);
void apples_fasta_close(apples_fasta* f);
int64_t apples_fasta_count(const apples_fasta* f);
int64_t apples_fasta_max_len(const apples_fasta* f);
int64_t apples_fasta_stride(const apples_fasta* f);
int apples_fasta_uniform(const apples_fasta* f);            /* 1 when every sequence has the same length (an alignment) */
int apples_fasta_pinned(const apples_fasta* f);
const uint8_t* apples_fasta_matrix(const apples_fasta* f);
const int64_t* apples_fasta_lengths(const apples_fasta* f); /* n */
const char* apples_fasta_names(const apples_fasta* f);      /* NUL-terminated names, concatenated */
const int64_t* apples_fasta_name_offsets(const apples_fasta* f); /* n + 1 */

/* Result arrays -> jplace file, replacing join_jplace + json.dumps(result, sort_keys=True, indent=4) for the
 * "placements" list (jutil.py:1-19, run_apples.py:106-118): writes `prefix`, the list, `suffix`.  prefix / suffix are
 * the JSON text before / after the list (the caller renders the small rest of the document).  Records are the ones
 * PoolQueryWorker.runquery returns for the given status codes (names of queries found in the backbone get "-query");
 * numbers are written as Python's float repr, names as json.dumps' ASCII escapes.  n_written = records kept. */
int apples_jplace_write(const char* path, const char* prefix, const char* suffix, int64_t n, const char* names,
                        const int64_t* name_off, const uint8_t* in_backbone, const int32_t* edge, const double* error,
                        const double* distal, const double* pendant, const int32_t* status, int exclude_intplace,
                        int n_threads, int64_t* n_written, char* err, int errlen);
/* The same with the ranked records of apples_set_alternatives: a query placed by least squares (status APPLES_PLACED, or
 * APPLES_PLACED_MISPLACEMENT_FLAG without exclude_intplace) gets alt_count[i] records in "p", record 0 from the five
 * arrays as above, records 1.. from alt_*[i * keep + j] with like_weight_ratio 0.  Every other query keeps its single
 * record.  keep = 1 (alt_* may be NULL) writes exactly what apples_jplace_write writes. */
int apples_jplace_write_k(const char* path, const char* prefix, const char* suffix, int64_t n, const char* names,
                          const int64_t* name_off, const uint8_t* in_backbone, const int32_t* edge, const double* error,
                          const double* distal, const double* pendant, const int32_t* status, int exclude_intplace,
                          int32_t keep, const int32_t* alt_count, const int32_t* alt_edge, const double* alt_error,
                          const double* alt_distal, const double* alt_pendant, const uint8_t* alt_int0, int n_threads,
                          int64_t* n_written, char* err, int errlen);

/* Newick text -> flat post-order arrays, replacing treeswift.read_tree_newick + index_edges + set_levels
 * (apples/prepareTree.py:24, apples/util.py:57-88): node id = edge_index = post-order rank (children left to right, root
 * last); parent (-1 for the root), edge_length (0 where the text has none) + has_length, level (root 0), first (smallest
 * id of the subtree), labels (bytes of the text, concatenated; label_offsets n + 1; has_label tells "" from none).
 * Returns 0, a negative value on bad arguments, or APPLES_NEWICK_UNSUPPORTED for text this parser does not take
 * (unbalanced brackets or quotes, branch lengths that are not plain decimals, exotic blanks): the caller then uses its
 * own parser (apples_b200/tree.py, the definition of the accepted language). */
#define APPLES_NEWICK_UNSUPPORTED 1
typedef struct apples_newick apples_newick;
int apples_newick_parse(const char* text, int64_t len, apples_newick** out, char* err, int errlen);
void apples_newick_free(apples_newick* t);
int64_t apples_newick_nodes(const apples_newick* t);
int apples_newick_rooted(const apples_newick* t);             /* text starts with [&R] */
const int32_t* apples_newick_parent(const apples_newick* t);
const int32_t* apples_newick_level(const apples_newick* t);
const int32_t* apples_newick_first(const apples_newick* t);
const double* apples_newick_edge_length(const apples_newick* t);
const uint8_t* apples_newick_has_length(const apples_newick* t);
const uint8_t* apples_newick_has_label(const apples_newick* t);
const char* apples_newick_labels(const apples_newick* t);
const int64_t* apples_newick_label_offsets(const apples_newick* t);

/* Flat arrays -> the newick string with `{edge_index}` after every non-root node, replacing jutil.extended_newick
 * (apples/jutil.py:22-96): lengths as str(int(x)) when integral, else Python's float repr; "[&R] " in front when rooted.
 * *out_text is malloc'ed (apples_free_text).  APPLES_NEWICK_UNSUPPORTED: an integral length beyond 9e18. */
int apples_newick_extended(int64_t n, const int32_t* parent, const double* edge_length, const uint8_t* has_length,
                           const char* labels, const int64_t* label_offsets, const uint8_t* has_label, int rooted,
                           char** out_text, int64_t* out_len, char* err, int errlen);
void apples_free_text(char* p);

#ifdef __cplusplus
}
#endif
#endif
