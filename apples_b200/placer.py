"""Host side of the hot path: `place_batch` replaces the one call that fans queries out to CPU workers,

    results = pool.starmap(queryworker.runquery, queries)            run_apples.py:94-102

and returns the same list of per-query jplace dicts (PoolQueryWorker.runquery, apples/PoolQueryWorker.py:28-141),
in the same order, with the same warnings / stderr messages.  All per-query work (distances, observed-set
selection, restricted subtree, least-squares moments, per-edge solve, criterion selection) runs in CUDA behind
the C ABI of include/apples_b200.h.  There is no CPU path here.
"""
import gc
import logging
import sys

import numpy as np

from . import _lib
from . import fasta as _fasta


def _edge_index_of(v):
    return int(v.edge_index) if hasattr(v, 'edge_index') else int(v)


class GpuPlacer:
    """One GPU context holding the replicated read-only state (tree, packed reference, clusters) -- the analogue of
    PoolQueryWorker's fork-inherited class attributes (PoolQueryWorker.py:11-25)."""

    def __init__(self, tree, reference=None, name_to_node_map=None, device=0, matrix_tags=None):
        self.lib = _lib.load()
        self.tree = tree
        self.name_to_node = {k: _edge_index_of(v) for k, v in
                             (name_to_node_map if name_to_node_map is not None else tree.name_to_node).items()}
        h = _lib.C.c_void_p()
        rc = self.lib.apples_ctx_create(int(device), _lib.C.byref(h))
        if rc != 0:
            raise RuntimeError('apples_ctx_create(device=%d) failed with code %d (no usable CUDA device?)' % (device, rc))
        self.h = h
        self.device = int(device)
        # A/B switch for measurements: APPLES_B200_DENSE=intpipe selects the integer-pipe LOP3/POPC kernel for the
        # representative counts instead of the default tensor-core kernel (identical results)
        import os as _os
        if _os.environ.get('APPLES_B200_DENSE', '') == 'intpipe':
            self._check(self.lib.apples_ctx_set_dense_mode(self.h, 0))
        self._check(self.lib.apples_set_tree(self.h, tree.num_nodes, _lib.ptr(tree.parent), _lib.ptr(tree.edge_length),
                                             _lib.ptr(tree.level), _lib.ptr(tree.first)))
        self.reference = None
        self.kind = None
        self.L = None
        self.n_rep = None
        self.ref_names = None
        self.matrix_tags = None
        if reference is not None:
            self.set_reference(reference)
        if matrix_tags is not None:
            self.set_matrix_tags(matrix_tags)

    # ------------------------------------------------------------------------------------------------ plumbing
    def _check(self, rc):
        if rc != 0:
            raise RuntimeError('libapples_b200: ' + self.lib.apples_last_error(self.h).decode())

    def close(self):
        if getattr(self, 'h', None) is not None and self.h:
            self.lib.apples_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_dense_mode(self, mode):
        """1 = tensor-core kernel (default), 0 = integer-pipe kernel; identical results; call before set_reference."""
        self._check(self.lib.apples_ctx_set_dense_mode(self.h, int(mode)))

    def set_limits(self, max_subbatch=0, scratch_bytes=0, slot_cap=0):
        self._check(self.lib.apples_ctx_set_limits(self.h, int(max_subbatch), int(scratch_bytes), int(slot_cap)))

    @property
    def stream(self):
        return self.lib.apples_ctx_stream(self.h)

    def set_reference(self, reference, on_device=True):
        """on_device: ship the raw alignment bytes and let the device pack them and build the consensus
        representatives (SURVEY.md section 8 f1/f2); otherwise pack / build on the host with numpy."""
        if on_device and hasattr(reference, 'device_arrays_bytes'):
            self.set_reference_bytes(**reference.device_arrays_bytes(self.name_to_node))
        else:
            self.set_reference_arrays(**reference.device_arrays(self.name_to_node))
        self.reference = reference

    def set_reference_bytes(self, kind, L, ref_names, ref_bytes, ref_node, group_offsets, group_members):
        """Alignment bytes of the references; the device packs them and builds the consensus representatives."""
        self.kind, self.L, self.ref_names, self.n_rep = kind, int(L), ref_names, len(group_offsets) - 1
        rb = ref_bytes
        if not (rb.dtype == np.uint8 and rb.ndim == 2 and rb.strides[1] == 1 and rb.strides[0] >= rb.shape[1]):
            rb = np.ascontiguousarray(rb, dtype=np.uint8)
        go = np.ascontiguousarray(group_offsets, dtype=np.int32)
        gm = np.ascontiguousarray(group_members, dtype=np.int32)
        rn = np.ascontiguousarray(ref_node, dtype=np.int32)
        # rows may be padded (the native reader's matrix): the stride is passed on, no gigabyte-sized copy
        self._check(self.lib.apples_set_reference_bytes(self.h, kind, self.L, rb.shape[0], rb.ctypes.data,
                                                        rb.strides[0] if rb.shape[0] else self.L, _lib.ptr(rn),
                                                        self.n_rep, _lib.ptr(go), _lib.ptr(gm)))

    def set_reference_arrays(self, kind, L, ref_names, packed_refs, ref_node, packed_reps, group_offsets, group_members):
        self.kind, self.L, self.ref_names = kind, int(L), ref_names
        self._keep = (np.ascontiguousarray(packed_refs), np.ascontiguousarray(ref_node, dtype=np.int32),
                      np.ascontiguousarray(packed_reps), np.ascontiguousarray(group_offsets, dtype=np.int32),
                      np.ascontiguousarray(group_members, dtype=np.int32))
        pr, rn, pp, go, gm = self._keep
        self.n_rep = pp.shape[0]
        self._check(self.lib.apples_set_reference(self.h, kind, int(L), pr.shape[0], _lib.ptr(pr), _lib.ptr(rn),
                                                  pp.shape[0], _lib.ptr(pp), _lib.ptr(go), _lib.ptr(gm)))
        self._keep = None

    def set_matrix_tags(self, tags):
        self.matrix_tags = list(tags)
        col = np.array([self.name_to_node.get(t, -1) for t in self.matrix_tags], dtype=np.int32)
        self._check(self.lib.apples_set_matrix_columns(self.h, len(col), _lib.ptr(col)))

    def pack_queries(self, seqs):
        """'S1' rows (or a uint8 [n, L] matrix) -> packed device-layout rows."""
        mat = _fasta.as_byte_matrix(seqs, self.L)
        if mat.shape[1] != self.L:
            raise ValueError('query alignment has %d columns, reference has %d' % (mat.shape[1], self.L))
        return _fasta.pack(mat, self.kind)

    def self_nodes(self, names):
        return np.array([self.name_to_node.get(n, -1) for n in names], dtype=np.int32)

    @staticmethod
    def params_from_options(options, reference=None):
        """Alignment mode takes the cluster-expansion threshold from the REFERENCE object, as upstream does
        (Reference.py:146 `head.dist <= self.threshold`; with `-a database` that is the build-time -f, whatever -f the
        run was given); distance-matrix mode uses the run's -f (PoolQueryWorker.py:55)."""
        thr = options.filt_threshold
        if reference is not None and getattr(reference, 'threshold', None) is not None:
            thr = reference.threshold
        return _lib.make_params(options.method_name, options.criterion_name, bool(options.negative_branch),
                                options.base_observation_threshold, thr,
                                getattr(options, 'minimum_alignment_overlap', 0.001))

    # ------------------------------------------------------------------------------------------------ hot path
    def _outputs(self, nq):
        return (np.empty(nq, np.int32), np.empty(nq, np.float64), np.empty(nq, np.float64), np.empty(nq, np.float64),
                np.empty(nq, np.int32))

    @staticmethod
    def _alt_outputs(nq, keep):
        """ranked-record arrays: (count [nq], edge, error, distal, pendant, pendant_int0 [nq, keep])"""
        return (np.empty(nq, np.int32), np.empty((nq, keep), np.int32), np.empty((nq, keep), np.float64),
                np.empty((nq, keep), np.float64), np.empty((nq, keep), np.float64), np.empty((nq, keep), np.uint8))

    def _register_alternatives(self, nq, keep, alt):
        """keep > 1: the ranked-record arrays the next place call fills (apples_set_alternatives); None for keep 1"""
        keep = check_keep(keep)
        if keep == 1:
            return None
        alt = alt if alt is not None else self._alt_outputs(nq, keep)
        self._check(self.lib.apples_set_alternatives(self.h, keep, *[_lib.ptr(a) for a in alt]))
        return alt

    def place_packed(self, packed, self_node, params, out=None, keep=1, alt=None):
        """packed queries (host) -> (edge, error, distal, pendant, status) arrays.  keep > 1: returns (those arrays,
        ranked records) with the records as _alt_outputs lays them out (record 0 = the placement of the five arrays)."""
        nq = int(packed.shape[0])
        out = out if out is not None else self._outputs(nq)
        packed = np.ascontiguousarray(packed)
        alt = self._register_alternatives(nq, keep, alt)
        self._check(self.lib.apples_place_batch(self.h, nq, _lib.ptr(packed), _lib.ptr(self_node), _lib.C.byref(params),
                                                *[_lib.ptr(o) for o in out]))
        return out if alt is None else (out, alt)

    def place_bytes(self, mat, self_node, params, out=None, keep=1, alt=None):
        """alignment bytes uint8 [nq, L] (host) -> result arrays; packing happens on the device.  keep: as place_packed."""
        if mat.shape[1] != self.L:
            raise ValueError('query alignment has %d columns, reference has %d' % (mat.shape[1], self.L))
        if not (mat.dtype == np.uint8 and mat.ndim == 2 and mat.strides[1] == 1 and mat.strides[0] >= mat.shape[1]):
            mat = np.ascontiguousarray(mat, dtype=np.uint8)
        nq = int(mat.shape[0])
        out = out if out is not None else self._outputs(nq)
        alt = self._register_alternatives(nq, keep, alt)
        # rows may be padded (the native reader's matrix: row stride = L rounded up to 16): the stride is passed on
        self._check(self.lib.apples_place_batch_bytes(self.h, nq, mat.ctypes.data, mat.strides[0] if nq else self.L,
                                                      _lib.ptr(self_node), _lib.C.byref(params), *[_lib.ptr(o) for o in out]))
        return out if alt is None else (out, alt)

    def place_rows(self, rows, self_node, params, out=None, keep=1, alt=None):
        """distance-matrix rows float64 [nq, n_cols] -> result arrays.  keep: as place_packed."""
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        nq = int(rows.shape[0])
        out = out if out is not None else self._outputs(nq)
        alt = self._register_alternatives(nq, keep, alt)
        self._check(self.lib.apples_place_batch_matrix(self.h, nq, _lib.ptr(rows), _lib.ptr(self_node),
                                                       _lib.C.byref(params), *[_lib.ptr(o) for o in out]))
        return out if alt is None else (out, alt)

    def upload_queries(self, packed, self_node=None):
        packed = np.ascontiguousarray(packed) if isinstance(packed, np.ndarray) else packed
        self._res_n = int(packed.shape[0])
        self._check(self.lib.apples_queries_upload(self.h, self._res_n, _lib.ptr(packed), _lib.ptr(self_node)))

    def place_resident(self, params):
        self._check(self.lib.apples_place_resident(self.h, _lib.C.byref(params)))

    def download_results(self):
        out = self._outputs(self._res_n)
        self._check(self.lib.apples_results_download(self.h, *[_lib.ptr(o) for o in out]))
        return out

    def results_to_device(self, edge, error, distal, pendant, status):
        """copy the resident results into caller-owned device tensors (objects with .data_ptr())"""
        self._check(self.lib.apples_results_to_device(self.h, *[t.data_ptr() for t in (edge, error, distal, pendant, status)]))

    def last_counts(self, n):
        """(K observed leaves, V valid nodes, overflowed flag) per query of the last macro-batch (test seam)."""
        K, V, ov = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int32)
        self._check(self.lib.apples_last_counts(self.h, int(n), _lib.ptr(K), _lib.ptr(V), _lib.ptr(ov)))
        return K, V, ov

    def timings(self, reset=False):
        v = np.zeros(22, np.float64)
        self.lib.apples_get_timings(self.h, _lib.ptr(v), 22, 1 if reset else 0)
        keys = ['h2d_ms', 'transpose_ms', 'rep_distance_ms', 'selection_ms', 'placement_ms', 'd2h_ms', 'launches',
                'rep_distance_launches', 'pairs', 'observed', 'valid_nodes', 'overflow_queries', 'max_observed',
                'max_valid_nodes', 'rep_distance_sm_mhz', 'placed_smem64', 'placed_smem128', 'placed_smem256',
                'placed_smem512', 'placed_block', 'fallback_queries', 'tensor_core_launches']
        return dict(zip(keys, v.tolist()))

    # ------------------------------------------------------------------------------------------------ parity exports
    def distance_counts(self, packed, overlap_frac=0.001):
        packed = np.ascontiguousarray(packed)
        nq, nr = int(packed.shape[0]), len(self.ref_names)
        mism = np.zeros((nq, nr), np.uint32)
        valid = np.zeros((nq, nr), np.uint32)
        dist = np.zeros((nq, nr), np.float64)
        self._check(self.lib.apples_distance_counts(self.h, nq, _lib.ptr(packed), float(overlap_frac), _lib.ptr(mism),
                                                    _lib.ptr(valid), _lib.ptr(dist)))
        return mism, valid, dist

    def count_keys(self, packed, params):
        """Query x representative keys of the hot path's count stage (apples_count_keys): ([nq, n_rep] array, kind) with
        kind 0 = uint32 mismatch | valid << 16, 1 = uint64 mismatch | valid << 32 (byte mode), 2 = float64 scoredist."""
        packed = np.ascontiguousarray(packed)
        nq = int(packed.shape[0])
        raw = np.zeros(nq * self.n_rep, np.uint64)
        kind = _lib.C.c_int32(-1)
        self._check(self.lib.apples_count_keys(self.h, nq, _lib.ptr(packed), _lib.C.byref(params), _lib.C.byref(kind),
                                               _lib.ptr(raw)))
        dtype = {0: np.uint32, 1: np.uint64, 2: np.float64}[kind.value]
        return raw.view(dtype)[:nq * self.n_rep].reshape(nq, self.n_rep), kind.value

    def observed_sets(self, params, packed=None, rows=None, self_node=None, cap=4096):
        src = packed if packed is not None else rows
        src = np.ascontiguousarray(src)
        nq = int(src.shape[0])
        count = np.zeros(nq, np.int32)
        node = np.full((nq, cap), -1, np.int32)
        dist = np.zeros((nq, cap), np.float64)
        self._check(self.lib.apples_observed_sets(self.h, nq, _lib.ptr(src) if packed is not None else None,
                                                  _lib.ptr(src) if packed is None else None, _lib.ptr(self_node),
                                                  _lib.C.byref(params), cap, _lib.ptr(count), _lib.ptr(node),
                                                  _lib.ptr(dist)))
        return count, node, dist

    def edge_solutions(self, params, packed_row=None, row=None, self_node=-1):
        M = self.tree.num_nodes
        x1, x2, err = np.zeros(M), np.zeros(M), np.zeros(M)
        valid = np.zeros(M, np.uint8)
        src = np.ascontiguousarray(packed_row if packed_row is not None else row)
        self._check(self.lib.apples_edge_solutions(self.h, _lib.ptr(src) if packed_row is not None else None,
                                                   _lib.ptr(src) if packed_row is None else None, int(self_node),
                                                   _lib.C.byref(params), _lib.ptr(x1), _lib.ptr(x2), _lib.ptr(err),
                                                   _lib.ptr(valid)))
        return x1, x2, err, valid


def results_to_jplace(names, in_backbone, out, exclude_intplace=False, log=True, degenerate='raise', alt=None):
    """Device result arrays -> the per-query dicts PoolQueryWorker.runquery returns, with its messages.

    alt: the ranked records of place_*(keep > 1).  A query placed by least squares (PLACED, or PLACED_MISPLACEMENT_FLAG
    without exclude_intplace) then carries its count records in 'p', records 1.. with like_weight_ratio 0.

    degenerate='raise' (default): a query whose status carries APPLES_FLAG_DEGENERATE raises ZeroDivisionError, as the
    reference does in util.solve2_2 (util.py:26-27: `1 / (a_11 * a_22 - a_12 * a_21)`, `assert det != 0`), where the
    exception ends the whole run.  degenerate='keep' returns the record with whatever inf/nan arithmetic produced."""
    # the common record (placed, no flag, name not in the backbone) is built in one comprehension; the per-record
    # control flow below only runs for the others (6.5 -> 1.4 s per million queries)
    st_arr = np.asarray(out[4])
    if degenerate == 'raise':
        bad = np.flatnonzero(st_arr & _lib.FLAG_DEGENERATE)
        if bad.size:
            raise ZeroDivisionError('float division by zero: the least-squares system of query %s is singular on at least '
                                    'one edge (the reference raises in util.solve2_2 as well)' % names[int(bad[0])])
    special = np.flatnonzero((st_arr != _lib.PLACED) | np.asarray(in_backbone, dtype=bool)).tolist()
    edge, error, distal, pendant, status = [o.tolist() for o in out]
    # five container objects per record: the cyclic GC would walk the growing list again and again (5x slower)
    gc_was_on = gc.isenabled()
    gc.disable()
    try:
        results = [{'placements': [{'p': [[e, r, 1, d, q]], 'n': [nm]}]}
                   for e, r, d, q, nm in zip(edge, error, distal, pendant, names)]
    finally:
        if gc_was_on:
            gc.enable()
    for i in special:
        name = names[i]
        if in_backbone[i]:  # PoolQueryWorker.py:63-70
            if log:
                logging.warning('The query named %s exists in the backbone. Changing its name to %s-query.' % (name, name))
            name = name + '-query'
        code = status[i] & _lib.STATUS_CODE_MASK
        if code == _lib.ZERO_DIST_LEAF:  # :72-75
            p = [edge[i], 0, 1, 0, 0]
        elif code == _lib.TOO_FEW_DISTANCES:  # :77-98
            if log:
                sys.stderr.write('Taxon {} cannot be placed. At least three non-infinity distances '
                                 'should be observed to place a taxon. '
                                 'Consequently, this taxon is ignored (no output).\n'.format(name))
            p = [-1, 0, 1, 0, 0]
        else:
            pend = 0 if (status[i] & _lib.FLAG_PENDANT_INT0) else pendant[i]
            p = [edge[i], error[i], 1, distal[i], pend]
            if code == _lib.PLACED_MISPLACEMENT_FLAG:  # :121-130
                ignored = ''
                if exclude_intplace:
                    p[0] = -1
                    ignored = ' Consequently, this sequence is ignored (no output).'
                if log:
                    logging.warning('Best placement for query sequence %s has zero pendant edge length and placed at '
                                    'an internal node with a non-zero least squares error. This is a potential '
                                    'misplacement.%s' % (name, ignored))
        results[i] = {'placements': [{'p': [p], 'n': [name]}]}
    if alt is not None:
        cnt, a_edge, a_err, a_distal, a_pend, a_int0 = alt
        code = st_arr & _lib.STATUS_CODE_MASK
        ls = (code == _lib.PLACED) | ((code == _lib.PLACED_MISPLACEMENT_FLAG) & (not exclude_intplace))
        for i in np.flatnonzero(ls & (np.asarray(cnt) > 1)).tolist():
            p = results[i]['placements'][0]['p']
            for j in range(1, int(cnt[i])):
                p.append([int(a_edge[i, j]), float(a_err[i, j]), 0, float(a_distal[i, j]),
                          0 if a_int0[i, j] else float(a_pend[i, j])])
    return results


def check_keep(keep):
    """--keep-at-most K: 1 <= K <= 16 (APPLES_MAX_KEEP)"""
    if isinstance(keep, bool) or int(keep) != keep or not 1 <= keep <= _lib.MAX_KEEP:
        raise ValueError('--keep-at-most must be an integer from 1 to %d, got %r' % (_lib.MAX_KEEP, keep))
    return int(keep)


class MultiGpuPlacer:
    """Queries sharded over several GPUs of one box: one GpuPlacer (context) per device with the tree and the packed
    reference replicated, one host thread per context (the C ABI's threading rule), contiguous blocks of
    ceil(Q / G) queries per GPU (SURVEY.md section 8e).  Every context writes its block straight into the shared host
    result arrays, so the output is in input order and byte-identical to the single-GPU output.  This is the in-process
    analogue of upstream's `mp.Pool(num_thread)` (run_apples.py:101-102); under torchrun the same split runs with one
    process per GPU and a final NCCL gather (apples_b200.parallel)."""

    def __init__(self, tree, reference=None, name_to_node_map=None, devices=(0,), matrix_tags=None):
        from concurrent.futures import ThreadPoolExecutor
        self.devices = [int(d) for d in devices]
        if not self.devices:
            raise ValueError('MultiGpuPlacer needs at least one device')
        self.pool = ThreadPoolExecutor(max_workers=len(self.devices))
        # contexts are built in parallel: each uploads its own replica of the reference
        self.placers = list(self.pool.map(
            lambda d: GpuPlacer(tree, reference, name_to_node_map, device=d, matrix_tags=matrix_tags), self.devices))
        p0 = self.placers[0]
        self.name_to_node, self.L, self.kind, self.ref_names = p0.name_to_node, p0.L, p0.kind, p0.ref_names
        self.matrix_tags = p0.matrix_tags
        self.params_from_options = p0.params_from_options

    def close(self):
        for p in self.placers:
            p.close()
        self.pool.shutdown(wait=True)

    def self_nodes(self, names):
        return self.placers[0].self_nodes(names)

    def _outputs(self, nq):
        return self.placers[0]._outputs(nq)

    def set_matrix_tags(self, tags):
        for p in self.placers:
            p.set_matrix_tags(tags)
        self.matrix_tags = self.placers[0].matrix_tags

    def _sharded(self, method, mat, self_node, params, keep):
        from .parallel import shard_bounds
        nq = int(mat.shape[0])
        out = self.placers[0]._outputs(nq)
        alt = self.placers[0]._alt_outputs(nq, check_keep(keep)) if keep > 1 else None
        bounds = shard_bounds(nq, len(self.placers))

        def run(i):
            b, e = bounds[i]
            if e > b:
                part = getattr(self.placers[i], method)(mat[b:e], None if self_node is None else self_node[b:e], params,
                                                        out=tuple(o[b:e] for o in out), keep=keep,
                                                        alt=None if alt is None else tuple(a[b:e] for a in alt))
                assert (part if alt is None else part[0])[0].ctypes.data == out[0][b:e].ctypes.data
        list(self.pool.map(run, range(len(self.placers))))
        return out if alt is None else (out, alt)

    def place_bytes(self, mat, self_node, params, keep=1):
        if not (mat.dtype == np.uint8 and mat.ndim == 2 and mat.strides[1] == 1):
            mat = np.ascontiguousarray(mat, dtype=np.uint8)
        return self._sharded('place_bytes', mat, self_node, params, keep)

    def place_rows(self, rows, self_node, params, keep=1):
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        return self._sharded('place_rows', rows, self_node, params, keep)

    def timings(self, reset=False):
        """Stage timers of the contexts: times are the maximum over the GPUs (they run side by side), counters the sum."""
        ts = [p.timings(reset) for p in self.placers]
        return {k: (max if k.endswith('_ms') or k.startswith('max_') or k.endswith('_mhz') else sum)(t[k] for t in ts)
                for k in ts[0]}


def visible_devices(first=0, count=0):
    """Device ordinals for `--device first --gpus count` (count 0 = every visible device from `first` on)."""
    n = _lib.device_count()
    if n <= 0:
        raise RuntimeError('no CUDA device is visible; apples_b200 has no CPU fallback')
    if count <= 0:
        count = n - first
    if first < 0 or count <= 0 or first + count > n:
        raise ValueError('--device %d --gpus %d does not fit the %d visible CUDA device(s)' % (first, count, n))
    return list(range(first, first + count))


def _distributed_world():
    """(rank, world) when torch.distributed has been initialised (torchrun: one process per GPU), else (0, 1)."""
    if 'torch' not in sys.modules:
        return 0, 1
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def place_arrays(reference, options, name_to_node_map, queries, tree=None, placer=None, device=0, devices=None, keep=1):
    """The device part of place_batch: returns (names, in_backbone, (edge, error, distal, pendant, status)) for ALL
    queries in input order, and the ranked records as a fourth item when keep > 1 (GpuPlacer.place_packed).  Inside an initialised torch.distributed job every rank places its contiguous block of
    ceil(Q / world) queries on its own GPU and the blocks are exchanged with one all-gather of 32-byte records
    (apples_b200.parallel); otherwise the queries are sharded over `devices` inside this process."""
    keep = check_keep(keep)
    names = [q[0] for q in queries]
    rank, world = _distributed_world()
    lo, hi = 0, len(queries)
    if world > 1:
        from .parallel import shard_bounds
        lo, hi = shard_bounds(len(queries), world)[rank]
    own = placer is None
    if placer is None:
        if tree is None:
            raise ValueError('place_batch needs the BackboneTree (tree=) or a GpuPlacer (placer=)')
        devs = [int(d) for d in devices] if devices else [int(device)]
        devs = devs[:max(1, min(len(devs), hi - lo))]
        if len(devs) > 1:
            placer = MultiGpuPlacer(tree, reference, name_to_node_map, devices=devs)
        else:
            placer = GpuPlacer(tree, reference, name_to_node_map, device=devs[0])
    try:
        t_before = placer.timings()
        in_backbone = [n in placer.name_to_node for n in names]
        # upstream decides per query (`if obs_dist` in runquery, PoolQueryWorker.py:40); one batch is one mode here
        matrix = bool(queries[0][2])
        for q in queries:
            if bool(q[2]) != matrix:
                raise ValueError('place_batch: query %s mixes distance-matrix and alignment input in one batch' % q[0])
        mine = queries[lo:hi]
        self_node = placer.self_nodes(names[lo:hi])
        if matrix:
            params = placer.params_from_options(options)
            # distance-matrix mode: every row is a {tag: float} dict in header order
            tags = list(queries[0][2].keys())
            seen = set(tags)
            for q in queries[1:]:
                for t in q[2].keys():
                    if t not in seen:
                        seen.add(t)
                        tags.append(t)
            if placer.matrix_tags != tags:
                placer.set_matrix_tags(tags)
            rows = np.full((len(mine), len(tags)), -1.0, dtype=np.float64)
            col = {t: j for j, t in enumerate(tags)}
            for i, q in enumerate(mine):
                if len(q[2]) == len(tags) and list(q[2]) == tags:  # same header order (run_apples.py:43-54)
                    rows[i] = np.fromiter(q[2].values(), dtype=np.float64, count=len(tags))
                else:
                    for t, v in q[2].items():
                        rows[i, col[t]] = v
            res = placer.place_rows(rows, self_node, params, keep=keep) if mine else _empty_outputs(placer, keep)
        else:
            params = placer.params_from_options(options, reference)
            mat = _fasta.as_byte_matrix([q[1] for q in mine], placer.L)
            res = placer.place_bytes(mat, self_node, params, keep=keep) if mine else _empty_outputs(placer, keep)
        log_stage_times(placer, len(mine), t_before)
        if world > 1:
            from .parallel import gather_placements
            res = gather_placements(res, len(queries)) if keep == 1 else gather_placements(res[0], len(queries), alt=res[1])
        return (names, in_backbone, res) if keep == 1 else (names, in_backbone) + tuple(res)
    finally:
        if own:
            placer.close()


def log_stage_times(placer, n_queries, before=None):
    """The reference logs two lines per query (PoolQueryWorker.py:134-139: time of the distance stage, time of the dynamic
    programming).  A batch has no per-query times; the same two lines are logged once per batch from the device stage
    timers (distances = packing + count kernels + selection, dynamic programming = placement kernels)."""
    import logging
    import time
    t = placer.timings()
    if before:   # a caller-owned placer accumulates over its calls: this call's share
        t = {k: t[k] - before.get(k, 0.0) for k in t}
    logging.info('[%s] Distances are computed for %d queries in %.3f seconds.\n'
                 '[%s] Dynamic programming is completed for %d queries in %.3f seconds.'
                 % (time.strftime('%H:%M:%S'), n_queries, 1e-3 * (t['transpose_ms'] + t['rep_distance_ms'] + t['selection_ms']),
                    time.strftime('%H:%M:%S'), n_queries, 1e-3 * t['placement_ms']))


def log_messages(names, in_backbone, out, exclude_intplace=False):
    """The warnings / stderr lines PoolQueryWorker.runquery emits (PoolQueryWorker.py:63-70, 97-98, 121-130), from the
    result arrays: only the special records are visited.  Raises on degenerate systems like results_to_jplace."""
    st_arr = np.asarray(out[4])
    bad = np.flatnonzero(st_arr & _lib.FLAG_DEGENERATE)
    if bad.size:
        raise ZeroDivisionError('float division by zero: the least-squares system of query %s is singular on at least '
                                'one edge (the reference raises in util.solve2_2 as well)' % names[int(bad[0])])
    code = st_arr & _lib.STATUS_CODE_MASK
    inb = np.asarray(in_backbone, dtype=bool)
    for i in np.flatnonzero(inb | (code == _lib.TOO_FEW_DISTANCES) | (code == _lib.PLACED_MISPLACEMENT_FLAG)).tolist():
        name = names[i]
        if inb[i]:
            logging.warning('The query named %s exists in the backbone. Changing its name to %s-query.' % (name, name))
            name = name + '-query'
        if code[i] == _lib.TOO_FEW_DISTANCES:
            sys.stderr.write('Taxon {} cannot be placed. At least three non-infinity distances '
                             'should be observed to place a taxon. '
                             'Consequently, this taxon is ignored (no output).\n'.format(name))
        elif code[i] == _lib.PLACED_MISPLACEMENT_FLAG:
            ignored = ' Consequently, this sequence is ignored (no output).' if exclude_intplace else ''
            logging.warning('Best placement for query sequence %s has zero pendant edge length and placed at '
                            'an internal node with a non-zero least squares error. This is a potential '
                            'misplacement.%s' % (name, ignored))


def place_alignment(reference, options, name_to_node_map, names, mat, tree=None, placer=None, device=0, devices=None,
                    keep=1):
    """Array-level twin of place_batch for alignment input: `names` (list of str) and `mat` (uint8 [n, L] alignment bytes
    as fasta2dic / the native reader leave them, e.g. FastaMatrix.matrix).  Returns (in_backbone, (edge, error, distal,
    pendant, status)) for all queries in input order -- no per-query Python objects, so a million queries cost
    milliseconds of host time -- and the ranked records as a third item when keep > 1 (GpuPlacer.place_packed).
    Sharding over `devices` / torch.distributed ranks as in place_arrays."""
    keep = check_keep(keep)
    rank, world = _distributed_world()
    n = len(names)
    lo, hi = 0, n
    if world > 1:
        from .parallel import shard_bounds
        lo, hi = shard_bounds(n, world)[rank]
    own = placer is None
    if placer is None:
        if tree is None:
            raise ValueError('place_alignment needs the BackboneTree (tree=) or a GpuPlacer (placer=)')
        devs = [int(d) for d in devices] if devices else [int(device)]
        devs = devs[:max(1, min(len(devs), hi - lo))]
        if len(devs) > 1:
            placer = MultiGpuPlacer(tree, reference, name_to_node_map, devices=devs)
        else:
            placer = GpuPlacer(tree, reference, name_to_node_map, device=devs[0])
    try:
        t_before = placer.timings()
        n2n = placer.name_to_node
        in_backbone = np.fromiter((nm in n2n for nm in names), dtype=bool, count=n)
        self_node = np.full(hi - lo, -1, np.int32)
        for i in np.flatnonzero(in_backbone[lo:hi]).tolist():
            self_node[i] = n2n[names[lo + i]]
        params = placer.params_from_options(options, reference)
        if mat.shape[1] != placer.L:
            raise ValueError('query alignment has %d columns, reference has %d' % (mat.shape[1], placer.L))
        res = placer.place_bytes(mat[lo:hi], self_node, params, keep=keep) if hi > lo else _empty_outputs(placer, keep)
        log_stage_times(placer, hi - lo, t_before)
        if world > 1:
            from .parallel import gather_placements
            res = gather_placements(res, n) if keep == 1 else gather_placements(res[0], n, alt=res[1])
        return (in_backbone, res) if keep == 1 else (in_backbone,) + tuple(res)
    finally:
        if own:
            placer.close()


def _empty_outputs(placer, keep):
    out = placer._outputs(0)
    return out if keep == 1 else (out, GpuPlacer._alt_outputs(0, keep))


def place_batch(reference, options, name_to_node_map, queries, tree=None, placer=None, device=0, devices=None, keep=1):
    """Drop-in for `pool.starmap(queryworker.runquery, queries)` (run_apples.py:94-102).

    queries yields (query_name, query_seq 'S1' row or None, obs_dist dict or None) exactly as run_apples.py builds
    them (:43-54 distance matrix, :85-89 alignment).  Returns the list of jplace dicts in input order.
    `tree` is the BackboneTree the name_to_node_map belongs to (or pass an existing GpuPlacer / MultiGpuPlacer).
    `devices` = list of CUDA ordinals to shard the queries over (default: the single `device`); the result does not
    depend on it.  Under torchrun (torch.distributed initialised) every rank returns the full list.
    keep > 1 (--keep-at-most): the 'p' list of a query placed by least squares holds its best `keep` placements in
    criterion order (results_to_jplace).
    """
    queries = list(queries)
    if not queries:
        return []
    keep = check_keep(keep)
    names, in_backbone, out, *alt = place_arrays(reference, options, name_to_node_map, queries, tree=tree, placer=placer,
                                                 device=device, devices=devices, keep=keep)
    log = _distributed_world()[0] == 0   # messages once per job
    return results_to_jplace(names, in_backbone, out, getattr(options, 'exclude_intplace', False), log=log,
                             alt=alt[0] if alt else None)
