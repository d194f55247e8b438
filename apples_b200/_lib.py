"""ctypes binding of libapples_b200.so (include/apples_b200.h).  There is no CPU fallback: if the library has
not been built (`python -c "import __graft_entry__ as g; g.build()"` or `make -C apples_b200/csrc`) importing the
hot path raises."""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('APPLES_B200_LIB') or os.path.join(_HERE, 'libapples_b200.so')  # env: tuning experiments only

NUC, AA = 0, 1
FM, OLS, BME, BE = 0, 1, 2, 3
MLSE, ME, HYBRID = 0, 1, 2
METHODS = {'FM': FM, 'OLS': OLS, 'BME': BME, 'BE': BE}
CRITERIA = {'MLSE': MLSE, 'ME': ME, 'HYBRID': HYBRID}
STATUS_CODE_MASK = 0xff
PLACED, ZERO_DIST_LEAF, TOO_FEW_DISTANCES, PLACED_MISPLACEMENT_FLAG = 0, 1, 2, 3
FLAG_PENDANT_INT0 = 0x100
FLAG_DEGENERATE = 0x200
MAX_KEEP = 16            # APPLES_MAX_KEEP: ranked records per query (apples_set_alternatives)
NEWICK_UNSUPPORTED = 1   # apples_newick_*: text outside the native parser's language, use the Python twin

# every symbol the header declares (tests/test_cabi.py checks the library exports exactly these)
SYMBOLS = [
    'apples_words_per_row', 'apples_aa_row_bytes', 'apples_device_count', 'apples_ctx_create', 'apples_ctx_destroy', 'apples_last_error',
    'apples_ctx_stream', 'apples_ctx_set_limits', 'apples_ctx_set_dense_mode', 'apples_set_tree', 'apples_set_reference', 'apples_set_matrix_columns', 'apples_place_batch',
    'apples_place_batch_matrix', 'apples_set_reference_bytes', 'apples_place_batch_bytes', 'apples_queries_upload', 'apples_place_resident', 'apples_results_download', 'apples_results_to_device',
    'apples_set_alternatives', 'apples_distance_counts', 'apples_count_keys', 'apples_observed_sets', 'apples_edge_solutions', 'apples_get_timings', 'apples_last_counts',
    'apples_fasta_open', 'apples_fasta_close', 'apples_fasta_count', 'apples_fasta_max_len', 'apples_fasta_stride',
    'apples_fasta_uniform', 'apples_fasta_pinned', 'apples_fasta_matrix', 'apples_fasta_lengths', 'apples_fasta_names',
    'apples_fasta_name_offsets', 'apples_jplace_write', 'apples_jplace_write_k',
    'apples_newick_parse', 'apples_newick_free', 'apples_newick_nodes', 'apples_newick_rooted', 'apples_newick_parent',
    'apples_newick_level', 'apples_newick_first', 'apples_newick_edge_length', 'apples_newick_has_length',
    'apples_newick_has_label', 'apples_newick_labels', 'apples_newick_label_offsets', 'apples_newick_extended',
    'apples_free_text',
]


class Params(C.Structure):
    _fields_ = [('method', C.c_int32), ('criterion', C.c_int32), ('negative_branch', C.c_int32),
                ('base_observation_threshold', C.c_int32), ('filt_threshold', C.c_double),
                ('overlap_frac', C.c_double)]


_lib = None


def load():
    """Load the shared library (once).  Raises RuntimeError when it is missing -- the product has no other path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise RuntimeError('%s is missing: build it with `make -C apples_b200/csrc` (nvcc, sm_100a). '
                           'apples_b200 has no CPU fallback.' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    lib.apples_words_per_row.argtypes = [i32]
    lib.apples_words_per_row.restype = i32
    lib.apples_aa_row_bytes.argtypes = [i32]
    lib.apples_aa_row_bytes.restype = i32
    lib.apples_device_count.argtypes = [C.POINTER(i32)]
    lib.apples_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.apples_ctx_destroy.argtypes = [vp]
    lib.apples_ctx_destroy.restype = None
    lib.apples_last_error.argtypes = [vp]
    lib.apples_last_error.restype = C.c_char_p
    lib.apples_ctx_stream.argtypes = [vp]
    lib.apples_ctx_stream.restype = vp
    lib.apples_ctx_set_limits.argtypes = [vp, i64, i64, i32]
    lib.apples_ctx_set_dense_mode.argtypes = [vp, i32]
    lib.apples_set_tree.argtypes = [vp, i32, vp, vp, vp, vp]
    lib.apples_set_reference.argtypes = [vp, C.c_int, i32, i32, vp, vp, i32, vp, vp, vp]
    lib.apples_set_matrix_columns.argtypes = [vp, i32, vp]
    lib.apples_place_batch.argtypes = [vp, i64, vp, vp, C.POINTER(Params), vp, vp, vp, vp, vp]
    lib.apples_place_batch_matrix.argtypes = [vp, i64, vp, vp, C.POINTER(Params), vp, vp, vp, vp, vp]
    lib.apples_set_reference_bytes.argtypes = [vp, C.c_int, i32, i32, vp, i64, vp, i32, vp, vp]
    lib.apples_place_batch_bytes.argtypes = [vp, i64, vp, i64, vp, C.POINTER(Params), vp, vp, vp, vp, vp]
    lib.apples_queries_upload.argtypes = [vp, i64, vp, vp]
    lib.apples_place_resident.argtypes = [vp, C.POINTER(Params)]
    lib.apples_set_alternatives.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp]
    lib.apples_results_download.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.apples_results_to_device.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.apples_distance_counts.argtypes = [vp, i64, vp, dbl, vp, vp, vp]
    lib.apples_count_keys.argtypes = [vp, i64, vp, C.POINTER(Params), C.POINTER(i32), vp]
    lib.apples_observed_sets.argtypes = [vp, i64, vp, vp, vp, C.POINTER(Params), i32, vp, vp, vp]
    lib.apples_edge_solutions.argtypes = [vp, vp, vp, i32, C.POINTER(Params), vp, vp, vp, vp]
    lib.apples_get_timings.argtypes = [vp, vp, C.c_int, C.c_int]
    lib.apples_last_counts.argtypes = [vp, i64, vp, vp, vp]
    lib.apples_fasta_open.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp), C.c_char_p, C.c_int]
    lib.apples_fasta_close.argtypes = [vp]
    lib.apples_fasta_close.restype = None
    for fn in ('count', 'max_len', 'stride'):
        getattr(lib, 'apples_fasta_' + fn).argtypes = [vp]
        getattr(lib, 'apples_fasta_' + fn).restype = i64
    for fn in ('uniform', 'pinned'):
        getattr(lib, 'apples_fasta_' + fn).argtypes = [vp]
        getattr(lib, 'apples_fasta_' + fn).restype = C.c_int
    for fn in ('matrix', 'lengths', 'names', 'name_offsets'):
        getattr(lib, 'apples_fasta_' + fn).argtypes = [vp]
        getattr(lib, 'apples_fasta_' + fn).restype = vp
    lib.apples_jplace_write.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, i64, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int,
                                        C.c_int, C.POINTER(i64), C.c_char_p, C.c_int]
    lib.apples_jplace_write_k.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p, i64, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int,
                                          i32, vp, vp, vp, vp, vp, vp, C.c_int, C.POINTER(i64), C.c_char_p, C.c_int]
    lib.apples_newick_parse.argtypes = [vp, i64, C.POINTER(vp), C.c_char_p, C.c_int]
    lib.apples_newick_free.argtypes = [vp]
    lib.apples_newick_free.restype = None
    lib.apples_newick_nodes.argtypes = [vp]
    lib.apples_newick_nodes.restype = i64
    lib.apples_newick_rooted.argtypes = [vp]
    for fn in ('parent', 'level', 'first', 'edge_length', 'has_length', 'has_label', 'labels', 'label_offsets'):
        getattr(lib, 'apples_newick_' + fn).argtypes = [vp]
        getattr(lib, 'apples_newick_' + fn).restype = vp
    lib.apples_newick_extended.argtypes = [i64, vp, vp, vp, vp, vp, vp, C.c_int, C.POINTER(vp), C.POINTER(i64), C.c_char_p, C.c_int]
    lib.apples_free_text.argtypes = [vp]
    lib.apples_free_text.restype = None
    _lib = lib
    return lib


def device_count():
    """CUDA devices visible to the process (0 when there is no usable driver / device)."""
    n = C.c_int32(0)
    load().apples_device_count(C.byref(n))
    return int(n.value)


def ptr(a):
    """host pointer of a C-contiguous numpy array (or a torch CPU tensor) or None"""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        assert a.flags['C_CONTIGUOUS']
        return a.ctypes.data
    return a.data_ptr()  # torch tensor (pinned host memory in bench.py)


def make_params(method='FM', criterion='MLSE', negative_branch=False, base_observation_threshold=25,
                filt_threshold=0.2, overlap_frac=0.001):
    m = METHODS.get(method, OLS) if isinstance(method, str) else int(method)  # PoolQueryWorker.py:104-111: else -> OLS
    c = CRITERIA.get(criterion, MLSE) if isinstance(criterion, str) else int(criterion)  # Algorithm.py:88: else -> MLSE
    return Params(m, c, 1 if negative_branch else 0, int(base_observation_threshold), float(filt_threshold),
                  float(overlap_frac))
