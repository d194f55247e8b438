"""GPU (-m gpu): the line minima of the count stage and the selection that reads only the key lines they call for.

A line is the 32 keys [32 l, 32 l + 32) of a query's key row; its minimum is the key of smallest ratio mismatch / valid
among the keys the selection can use (valid >= max(vmin, 1), 4 mismatch < 3 valid), the smallest column on equal ratios,
or 0x00000001 when none qualifies.  The minima are a pure function of the keys, so they are checked bit for bit against
numpy on the keys the same call returns, in both dense modes, on tile edges, ragged sub-batches, overlap gates, all-gap
lines and ratio ties.

The selection that the minima drive is checked against an independent one: the same data in a byte-mode context, whose
selection (select_kernel<SEL_NUCW>) scans every key of the row.  Exotic bytes sit only in columns where every query has a
gap, so both contexts count the same pairs; observed sets, counts and placements must agree bit for bit.
"""
import numpy as np
import pytest

from tests.test_gpu_count_kernels import GAP, _nuc_rows, _placer, _set_singletons

pytestmark = pytest.mark.gpu

LINE_NONE = 1


def _vmin(L, overlap):
    """smallest valid count v with not (v / L < overlap) (api.cu overlap_vmin)"""
    for v in range(L + 1):
        if not (v / L < overlap):
            return v
    return L + 1


def _minima_np(keys, vmin):
    """line minima of a [nq, n] uint32 key matrix"""
    nq, n = keys.shape
    nl = (n + 31) // 32
    k = np.zeros((nq, nl * 32), np.uint32)
    k[:, :n] = keys
    m, v = (k & 0xffff).astype(np.int64), (k >> 16).astype(np.int64)
    usable = (v >= max(vmin, 1)) & (4 * m < 3 * v)
    # m / v with m, v <= 65535: distinct ratios give distinct doubles and equal ratios the identical one
    ratio = np.where(usable, m / np.maximum(v, 1), np.inf).reshape(nq, nl, 32)
    j = np.argmin(ratio, axis=2)                  # first occurrence: the smallest column on ties
    pick = np.take_along_axis(k.reshape(nq, nl, 32), j[..., None], axis=2)[..., 0]
    return np.where(np.isfinite(ratio.min(axis=2)), pick, np.uint32(LINE_NONE)).astype(np.uint32)


def _check_minima(L, r, qs, overlap=0.001, max_subbatch=0, tag=''):
    from apples_b200 import _lib, fasta
    params = _lib.make_params(overlap_frac=overlap)
    vmin = _vmin(L, overlap)
    got = {}
    for mode in (1, 0):
        pl = _placer(mode)
        try:
            _set_singletons(pl, fasta.NUC, L, fasta.pack_nucleotide(r))
            if max_subbatch:
                pl.set_limits(max_subbatch=max_subbatch)
            got[mode] = []
            for q in qs:
                keys, kind, mins = pl.count_keys(fasta.pack_nucleotide(q), params, line_minima=True)
                assert kind == 0 and mins.shape == (len(q), (len(r) + 31) // 32), (tag, kind, mins.shape)
                exp = _minima_np(keys, vmin)
                bad = np.argwhere(mins != exp)
                assert not bad.size, '%s mode %d: %d of %d minima wrong, first (query, line) %s: got %#x expected %#x' % (
                    tag, mode, len(bad), exp.size, tuple(bad[0]), mins[tuple(bad[0])], exp[tuple(bad[0])])
                got[mode].append(mins)
        finally:
            pl.close()
    for a, b in zip(got[1], got[0]):
        assert a.tobytes() == b.tobytes(), tag
    return got


@pytest.mark.parametrize('nq,n_rep', [(256, 256), (17 * 256, 13 * 256), (300, 1000), (257, 33)],
                         ids=['one_tile', '17x13_tiles', 'ragged', 'one_line_and_a_key'])
def test_line_minima_against_numpy(nq, n_rep):
    L = 300
    rng = np.random.default_rng(nq + n_rep)
    r = _nuc_rows(n_rep, L, rng, 'r')
    r[32:64] = GAP                                        # an all-gap line: the sentinel
    _check_minima(L, r, [_nuc_rows(nq, L, rng, 'q')], tag='%d x %d' % (nq, n_rep))


def test_line_minima_ragged_sub_batches():
    L = 200
    rng = np.random.default_rng(7)
    r = _nuc_rows(700, L, rng, 'r')
    _check_minima(L, r, [_nuc_rows(300, L, rng, 'q'), _nuc_rows(129, L, rng, 'q')], max_subbatch=128, tag='sub-batches')


def test_line_minima_overlap_gate_and_ties():
    """queries whose overlap with every representative is vmin - 1 / vmin / vmin + 1, and lines where keys tie on the
    ratio with different (mismatch, valid): 3 / 60 against 4 / 80 in either column order"""
    L, overlap = 160, 0.5
    vmin = _vmin(L, overlap)
    rng = np.random.default_rng(11)
    base = np.frombuffer(b'ACGT', np.uint8)[rng.integers(0, 4, L)]
    comp = np.frombuffer(b'ACGT', np.uint8)[(np.searchsorted(np.frombuffer(b'ACGT', np.uint8), base) + 1) % 4]
    r = np.tile(base, (96, 1))
    r[:, :60] = comp[:60]                                 # ratio 60 / 160 everywhere else
    for c, (valid, mism) in {1: (60, 3), 5: (80, 4), 33: (80, 4), 40: (60, 3), 70: (80, 4), 71: (60, 3)}.items():
        r[c] = base
        r[c, valid:] = GAP
        r[c, :mism] = comp[:mism]
    r[64:69, :] = GAP                                     # all-gap columns inside a line
    q = np.tile(base, (8, 1))
    for i, v in enumerate([vmin - 1, vmin, vmin + 1]):
        q[i, v:] = GAP
    q[3:, :] = _nuc_rows(5, L, rng, 'q')
    gate = _check_minima(L, r, [q], overlap=overlap, tag='overlap gate')[1][0]
    assert (gate[0] == LINE_NONE).all() and (gate[1] != LINE_NONE).all()
    # equal ratios: the smaller column wins whichever (mismatch, valid) it has
    ties = _check_minima(L, r, [base[None]], tag='ties')[1][0][0]
    assert ties.tolist() == [3 | 60 << 16, 4 | 80 << 16, 4 | 80 << 16]


# ---------------------------------------------------------------------------------------- selection against a full scan
def _case(seed, n_leaves=1500, L=400, n_queries=600, dup=150, n_exotic_cols=24):
    """a backbone with duplicated sequences (so that representatives tie on the ratio and the index decides), queries
    with zero-distance copies of references, and a byte-mode twin of the reference: exotic bytes only in the last
    columns, where every query has a gap"""
    from apples_b200 import synth
    from apples_b200.reference import ReducedReference
    from apples_b200.tree import BackboneTree
    tree = BackboneTree.from_newick(synth.random_tree(n_leaves, seed=seed))
    refs, states = synth.evolve_alignment(tree, L, seed=seed + 1)
    names = list(refs)
    rng = np.random.default_rng(seed)
    for a, b in rng.choice(len(names), (dup, 2), replace=False).tolist():   # copies far apart in the index order
        refs[names[b]] = refs[names[a]].copy()
    queries, _ = synth.make_queries(tree, states, n_queries, seed=seed + 2)
    qmat = np.stack([np.frombuffer(bytes(np.asarray(s).tobytes()), np.uint8)[:L] for s in queries.values()]).copy()
    qmat[:40] = np.stack([np.frombuffer(np.asarray(refs[names[i]]).tobytes(), np.uint8)[:L] for i in range(40)])
    qmat[:, L - n_exotic_cols:] = GAP
    exotic = {k: v.copy() for k, v in refs.items()}
    for i in rng.choice(len(names), 30, replace=False).tolist():
        exotic[names[i]][L - 1 - (i % n_exotic_cols)] = b'?'
    mk = lambda rf: ReducedReference(None, False, None, 0.02, 1, tree=tree, refs=rf)
    return tree, mk(refs), mk(exotic), qmat


@pytest.fixture(scope='module')
def selection_case():
    return _case(900)


def _results(tree, ref, qmat, params, mode, slot_cap):
    from apples_b200.placer import GpuPlacer
    pl = GpuPlacer(tree, None, tree.name_to_node, device=0)
    try:
        if mode is not None:
            pl.set_dense_mode(mode)
        pl.set_reference(ref, on_device=True)
        if slot_cap:
            pl.set_limits(slot_cap=slot_cap)
        packed = pl.pack_queries(qmat)
        nq = packed.shape[0]
        self_node = np.full(nq, -1, np.int32)
        pl.timings(reset=True)
        count, node, dist = pl.observed_sets(params, packed=packed, cap=4096)
        t = pl.timings()
        placed = pl.place_packed(packed, self_node, params)
        K, V, _ = pl.last_counts(nq)
        return dict(count=count, node=node, dist=dist, placed=placed, K=K, V=V, t=t)
    finally:
        pl.close()


@pytest.mark.parametrize('b,thr', [(25, 0.2), (200, 0.2), (1000, 0.2), (25, 0.6), (25, -1.0), (200, -1.0)],
                         ids=['b25', 'b200', 'b1000', 'many_near', 'nothing_near', 'nothing_near_b200'])
@pytest.mark.parametrize('mode', [1, 0], ids=['tensor', 'intpipe'])
def test_observed_sets_match_full_scan(selection_case, b, thr, mode):
    from apples_b200 import _lib
    tree, ref, exotic_ref, qmat = selection_case
    params = _lib.make_params('FM', 'MLSE', base_observation_threshold=b, filt_threshold=thr)
    slot_cap = 32 if b == 200 else 0                       # overflow: stash reruns and second-level reruns
    got = _results(tree, ref, qmat, params, mode, slot_cap)
    exp = _results(tree, exotic_ref, qmat, params, None, slot_cap)
    assert got['t']['tensor_core_launches'] == (got['t']['rep_distance_launches'] if mode == 1 else 0)
    assert exp['t']['fallback_queries'] > 0 and exp['t']['key_lines_read'] == 0
    assert got['t']['key_lines_read'] > 0
    for k in ('count', 'node', 'K', 'V'):
        assert np.array_equal(got[k], exp[k]), k
    placed = got['V'] > 0       # distances are final only for the queries that go on to placement
    assert np.array_equal(got['dist'][placed].view(np.uint64), exp['dist'][placed].view(np.uint64))
    for x, y in zip(got['placed'], exp['placed']):
        assert np.array_equal(np.asarray(x).view(np.uint8), np.asarray(y).view(np.uint8))
    assert (got['count'] > 0).any()
