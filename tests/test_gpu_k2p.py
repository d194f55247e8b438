"""GPU (-m gpu): placement under the Kimura two-parameter model (--model K2P, apples_ctx_set_model).

The K2P instantiation of the fp4 count kernel sends the y slice of every site into a third fp32 accumulator; the keys
(ts | tv << 16 | valid << 32) are checked bit for bit against numpy, first on one-tile launches whose pairs sit at the
extremes of the three accumulators up to FP4_MAX_L, then on the kernel's edges: 128-query and 160-representative tiles,
64-site stages, the length limit and ragged sub-batches.  Then the missing-distance gate, the placements against the
oracle's K2P run (tests/k2p_oracle.py) and the composition with the other features; last the errors.
"""
import json
import os
import types

import numpy as np
import pytest

from tests import util
from tests import k2p_oracle as ko
from tests.test_gpu_count_fp4 import FP4_MAX_L
from tests.test_gpu_count_kernels import GAP, _anchor, _nuc_rows
from tests.test_gpu_parity import _check_p

pytestmark = pytest.mark.gpu

A, C, G, T = (ord(x) for x in 'ACGT')
TRANSITION = np.zeros(256, np.uint8)
TRANSVERSION = np.zeros(256, np.uint8)
TRANSVERSION2 = np.zeros(256, np.uint8)
for _x, _ts, _tv, _tv2 in ((A, G, C, T), (G, A, T, C), (C, T, A, G), (T, C, G, A)):
    TRANSITION[_x], TRANSVERSION[_x], TRANSVERSION2[_x] = _ts, _tv, _tv2


def _small_tree_placer(model='K2P'):
    from apples_b200.placer import GpuPlacer
    from apples_b200.tree import BackboneTree
    tree = BackboneTree.from_newick('((A:0.1,B:0.2):0.05,C:0.3,D:0.4);')
    return GpuPlacer(tree, None, tree.name_to_node, device=0, model=model)


def _set_singletons(pl, L, rows):
    from apples_b200 import fasta
    p = fasta.pack_nucleotide(rows)
    n = p.shape[0]
    pl.set_reference_arrays(fasta.NUC, L, ['r%d' % i for i in range(n)], p, np.full(n, -1, np.int32), p,
                            np.arange(n + 1, dtype=np.int32), np.arange(n, dtype=np.int32))


def _expected(q, r):
    """exact (ts, tv, valid) of every pair as K2P keys, from one-hot float32 products (integers below 2^24: exact)"""
    def hot(x, b):
        return (x == b).astype(np.float32)
    valid = (q != GAP).astype(np.float32) @ (r != GAP).astype(np.float32).T
    match = sum(hot(q, b) @ hot(r, b).T for b in (A, C, G, T))
    ts = sum(hot(q, b) @ hot(r, TRANSITION[b]).T for b in (A, C, G, T))
    valid, match, ts = (x.astype(np.int64) for x in (valid, match, ts))
    tv = valid - match - ts
    return ts.astype(np.uint64) | (tv.astype(np.uint64) << np.uint64(16)) | (valid.astype(np.uint64) << np.uint64(32))


def _check_keys(L, r, qs, max_subbatch=0, tag=''):
    from apples_b200 import _lib, fasta
    params = _lib.make_params()
    pl = _small_tree_placer()
    out = []
    try:
        _set_singletons(pl, L, r)
        if max_subbatch:
            pl.set_limits(max_subbatch=max_subbatch)
        for q in qs:
            pl.timings(reset=True)
            keys, kind = pl.count_keys(fasta.pack_nucleotide(q), params)
            t = pl.timings()
            assert kind == 3, tag
            exp = _expected(q, r)
            bad = np.argwhere(keys != exp)
            if bad.size:
                i, j = bad[0]
                fields = lambda k: (int(k) & 0xffff, (int(k) >> 16) & 0xffff, int(k) >> 32)
                raise AssertionError('%s nq=%d: %d of %d keys wrong; first (query %d, representative %d): got (ts, tv, valid) '
                                     '%s, expected %s' % (tag, len(q), len(bad), exp.size, i, j, fields(keys[i, j]),
                                                          fields(exp[i, j])))
            assert t['k2p_launches'] == t['rep_distance_launches'] == t['fp4_launches'] == t['tensor_core_launches'] > 0, t
            out.append((keys, t))
    finally:
        pl.close()
    return out


# ------------------------------------------------------------------------------------- exact fp32 accumulation (one tile)
def _extreme_rows(L, side):
    a = _anchor(L)
    s = np.arange(L)
    ts, tv, tv2 = TRANSITION[a], TRANSVERSION[a], TRANSVERSION2[a]
    rows = [a, ts, tv, np.full(L, GAP, np.uint8)]
    if side == 'q':
        gaps = a.copy()
        gaps[s % 3 == 0] = GAP
        tail = ts.copy()
        tail[L // 2:] = GAP
        rows += [np.where(s % 2 == 0, a, ts), np.where(s % 2 == 0, a, tv), np.where(s % 2 == 0, ts, tv),
                 np.where((s // 4096) % 2 == 0, tv, ts), gaps, tail]
    else:
        late = a.copy()
        late[: L - L // 4] = tv[: L - L // 4]
        rows += [tv2, late]
    return np.stack(rows)


@pytest.mark.parametrize('L', [5000, 21846, 33816])
def test_k2p_accumulation_is_exact(L):
    """all-match (D1' = 2 L, D3 = L), all-transition (D1' = -2 L), all-transversion (D3 = -L) pairs, alternating and
    long-run mixtures and gaps in one 128 x 160 tile, against exact counts"""
    if L > FP4_MAX_L:
        pytest.skip('beyond the fp4 kernel (FP4_MAX_L = %d)' % FP4_MAX_L)
    rng = np.random.default_rng(L)
    q = np.concatenate([_extreme_rows(L, 'q'), _nuc_rows(8, L, rng, 'q')])
    r = np.concatenate([_extreme_rows(L, 'r'), _nuc_rows(8, L, rng, 'r')])
    keys = _check_keys(L, r, [q], tag='L=%d' % L)[0][0]
    assert (keys & 0xffff).max() == L and ((keys >> 16) & 0xffff).max() == L and (keys >> 32).max() == L


# ------------------------------------------------------------------------------------------------ tile and stage edges
@pytest.mark.parametrize('n_rep', [159, 160, 161, 319, 320, 321])
def test_k2p_keys_across_tile_shapes(n_rep):
    """127 / 128 / 129 queries x one to three 160-row representative tiles"""
    L = 97
    rng = np.random.default_rng(n_rep)
    r = _nuc_rows(n_rep, L, rng, 'r')
    _check_keys(L, r, [_nuc_rows(nq, L, rng, 'q') for nq in (127, 128, 129)], tag='n_rep=%d' % n_rep)


@pytest.mark.parametrize('L', [1, 32, 33, 63, 64, 65, 129, 4999, 5000, 33816])
def test_k2p_keys_across_lengths(L):
    """one word, whole and partial 64-site stages, odd and even word counts, the length limit"""
    rng = np.random.default_rng(3000 + L)
    _check_keys(L, _nuc_rows(161, L, rng, 'r'), [_nuc_rows(129, L, rng, 'q')], tag='L=%d' % L)


def test_k2p_ragged_sub_batches():
    """1000 queries as 384-query sub-batches and a ragged last one, against 3 x 160 - 1 representatives"""
    L = 300
    rng = np.random.default_rng(1001)
    res = _check_keys(L, _nuc_rows(479, L, rng, 'r'), [_nuc_rows(1000, L, rng, 'q')], max_subbatch=384)
    assert res[0][1]['rep_distance_launches'] == 3


# ------------------------------------------------------------------------------------------------ missing-distance gate
def _caterpillar(n, workdir, tag):
    s = 'L0:0.01'
    for i in range(1, n):
        s = '(%s,L%d:0.01):0.01' % (s, i)
    tfp = os.path.join(workdir, '%s.nwk' % tag)
    open(tfp, 'w').write(s.rsplit(':', 1)[0] + ';')
    return tfp


def _gate_rows(v):
    """rows of v sites whose (ts, tv) against the anchor sit on w1 = 1 - 2P - Q = 0 or w2 = 1 - 2Q = 0 and one count
    either side"""
    trip = set()
    for ts in sorted(set(np.linspace(0, v // 2, 12).astype(int).tolist())):
        for d in (-1, 0, 1):
            trip.add((ts, v - 2 * ts + d))
    for tv in (v // 2, (v + 1) // 2):
        for ts in (0, 1, 2, v - 2 * tv + 1):
            for d in (-1, 0, 1):
                trip.add((ts, tv + d))
    trip = sorted((ts, tv) for ts, tv in trip if ts >= 0 and tv >= 0 and ts + tv <= v)
    a = _anchor(v)
    rows = []
    for ts, tv in trip:
        r = a.copy()
        r[:ts] = TRANSITION[a[:ts]]
        r[ts:ts + tv] = TRANSVERSION[a[ts:ts + tv]]
        rows.append(r)
    return a, np.stack(rows), trip


@pytest.mark.parametrize('v', [9, 10, 1000, 1001, 33816])
def test_k2p_missing_distance_gate(v, workdir):
    """every leaf is its own representative and the threshold takes them all: a leaf is observed exactly when the
    oracle's K2P distance is not missing, with the oracle's distance"""
    from apples_b200 import _lib, fasta
    from apples_b200.placer import GpuPlacer
    from apples_b200.tree import BackboneTree
    a, rows, trip = _gate_rows(v)
    n = len(rows)
    tree = BackboneTree.from_newick(_caterpillar(n, workdir, 'gate%d' % v))
    names = ['L%d' % i for i in range(n)]
    pl = GpuPlacer(tree, None, tree.name_to_node, device=0, model='K2P')
    p = fasta.pack_nucleotide(rows)
    pl.set_reference_arrays(fasta.NUC, v, names, p, np.array([tree.name_to_node[x] for x in names], np.int32), p,
                            np.arange(n + 1, dtype=np.int32), np.arange(n, dtype=np.int32))
    pl.set_limits(slot_cap=16)    # the larger sets go through the overflow reruns
    params = _lib.make_params('FM', 'MLSE', False, 5, 1e9)
    count, node, dist = pl.observed_sets(params, packed=fasta.pack_nucleotide(a[None, :]), cap=n)
    pl.close()
    got = dict(zip(node[0, :count[0]].tolist(), dist[0, :count[0]].tolist()))
    qa = a.view('S1')
    for i, (ts, tv) in enumerate(trip):
        d = ko.k2p(qa, rows[i].view('S1'), 0.001)
        assert d == ko.k2p_from_counts(ts, tv, v, v, 0.001)
        u = tree.name_to_node[names[i]]
        assert (u in got) == (d >= 0), (v, ts, tv, d)
        if d >= 0:
            assert util.close(got[u], d, 1e-9, 0.0), (v, ts, tv, got[u], d)


# ------------------------------------------------------------------------------------------------ placements vs oracle
def _k2p_opts(options):
    o = types.SimpleNamespace(**vars(options))
    o.model = 'K2P'
    return o


@pytest.mark.parametrize('case', [c for c in util.golden_names('c1_align_*')])
def test_golden_fixtures_under_k2p(case, workdir):
    from apples_b200.placer import place_batch
    ci = util.CaseInputs(case, workdir)
    tree, ref = ci.product_state()
    res = place_batch(ref, _k2p_opts(ci.options), tree.name_to_node, ci.queries, tree=tree, device=0)
    octx = ko.oracle_context(ci)
    for q, r in zip(ci.queries, res):
        exp, _ = octx.runquery(q[0], q[1], None)
        assert r['placements'][0]['n'] == exp['placements'][0]['n']
        _check_p(case, q[0], r['placements'][0]['p'][0], exp['placements'][0]['p'][0], False, octx, (q[0], q[1], None))


def test_randomized_alignment_cases(workdir):
    """120 seeded random nucleotide cases (random gaps, clusterings incl. singletons, -V / -b / -f / -n, every method
    and criterion, copies of references and own-name queries, small slots for overflow reruns) against the oracle's
    K2P run: observed sets identical, distances within 1e-9, edges identical (score ties excepted)"""
    from oracle import apples_oracle as orc
    from apples_b200 import synth
    from apples_b200.placer import GpuPlacer, results_to_jplace
    from apples_b200.reference import ReducedReference
    from apples_b200.tree import BackboneTree
    rng = np.random.default_rng(2718281)
    checked = ties = zeros = overflows = 0
    for case in range(120):
        n = int(rng.integers(5, 70))
        L = int(rng.integers(40, 700))
        nwk = synth.random_tree(n, seed=int(rng.integers(1, 1 << 30)), mean_edge=float(rng.choice([0.01, 0.03, 0.08])),
                                polytomy_frac=float(rng.choice([0.0, 0.3])))
        tfp = os.path.join(workdir, 'k2pa_%d.nwk' % case)
        open(tfp, 'w').write(nwk)
        tree = BackboneTree.from_newick(tfp)
        refs, states = synth.evolve_alignment(tree, L, seed=int(rng.integers(1, 1 << 30)),
                                              gap_frac=float(rng.choice([0.0, 0.05, 0.4])), edge_frac=float(rng.choice([0.0, 0.3])))
        qd, _ = synth.make_queries(tree, states, int(rng.integers(1, 7)), seed=int(rng.integers(1, 1 << 30)),
                                   mean_extra=float(rng.choice([0.0, 0.03, 0.2])), gap_frac=float(rng.choice([0.0, 0.1, 0.6])))
        queries = [(k, v, None) for k, v in qd.items()]
        names = list(refs.keys())
        queries.append(('copy', refs[names[int(rng.integers(0, n))]], None))
        own = names[int(rng.integers(0, n))]
        queries.append((own, refs[own], None))
        tsv = os.path.join(workdir, 'k2pa_%d.tsv' % case)
        with open(tsv, 'w') as f:
            f.write('SequenceName\tClusterNumber\n')
            for nm in names:
                f.write('%s\t%d\n' % (nm, -1 if rng.random() < 0.35 else int(rng.integers(1, max(2, n // 3)))))
        thr = float(rng.choice([0.05, 0.2, 0.6]))
        ref = ReducedReference(None, False, tfp, thr, 1, cluster_tsv=tsv, tree=tree, refs=refs)
        opt = types.SimpleNamespace(method_name=str(rng.choice(['FM', 'OLS', 'BME', 'BE'])),
                                    criterion_name=str(rng.choice(['MLSE', 'ME', 'HYBRID'])),
                                    negative_branch=bool(rng.random() < 0.2), base_observation_threshold=int(rng.choice([2, 5, 25])),
                                    filt_threshold=thr, minimum_alignment_overlap=float(rng.choice([0.001, 0.2, 0.5])),
                                    exclude_intplace=False)
        pl = GpuPlacer(tree, ref, tree.name_to_node, device=0, model='K2P')
        if rng.random() < 0.3:
            pl.set_limits(slot_cap=4)
        params = pl.params_from_options(opt)
        qn = [q[0] for q in queries]
        sn = pl.self_nodes(qn)
        packed = pl.pack_queries([q[1] for q in queries])
        out = pl.place_packed(packed, sn, params)
        overflows += pl.timings()['overflow_queries'] > 0
        count, node, dist = pl.observed_sets(params, packed=packed, self_node=sn, cap=256)
        res = results_to_jplace(qn, [x in tree.name_to_node for x in qn], out, log=False, degenerate='keep')
        pl.close()
        otree, onames = orc.load_tree(tfp)
        octx = orc.OracleContext(otree, onames, refs=refs, representatives=orc.representatives_from_tsv(tsv, refs, False),
                                 method=opt.method_name, criterion=opt.criterion_name, negative_branch=opt.negative_branch,
                                 filt_threshold=thr, baseobs=opt.base_observation_threshold,
                                 overlap=opt.minimum_alignment_overlap)
        octx.dist_fn = ko.k2p
        for qi, (q, r) in enumerate(zip(queries, res)):
            det = {}
            ctx = (case, q[0], vars(opt))
            try:
                exp, st = octx.runquery(q[0], q[1], None, detail=det)
            except (ZeroDivisionError, AssertionError):
                assert int(out[4][qi]) & 0x200, ('the reference raises on a singular system, no APPLES_FLAG_DEGENERATE', ctx)
                continue
            except (FloatingPointError, OverflowError):
                continue
            assert not (int(out[4][qi]) & 0x200), ctx
            eobs = {tree.name_to_node[k]: v for k, v in det['observed']}
            assert int(count[qi]) == len(eobs), ctx
            zeros += st == 1
            if st in (0, 3):
                k = int(count[qi])
                assert node[qi, :k].tolist() == sorted(eobs), ctx
                for u, d in zip(node[qi, :k].tolist(), dist[qi, :k].tolist()):
                    assert util.close(d, eobs[u], 1e-9, 0.0), ctx
            g, e = r['placements'][0]['p'][0], exp['placements'][0]['p'][0]
            assert r['placements'][0]['n'] == exp['placements'][0]['n'], ctx
            if any(isinstance(x, float) and (x != x or abs(x) == float('inf')) for x in e[1:]):
                continue
            if _check_p('k2pa', q[0], g, e, False, octx, q) == 'tie':
                ties += 1
            checked += 1
    assert checked > 500 and ties <= 5 and zeros > 0 and overflows > 0, (checked, ties, zeros, overflows)


# ------------------------------------------------------------------------------------------------ composition
def _c1(workdir):
    ci = util.CaseInputs('c1_align_FM_MLSE', workdir)
    tree, ref = ci.product_state()
    return ci, tree, ref


def test_keep_at_most_under_k2p(workdir):
    """--keep-at-most 4: record 0 and the five arrays are bit-identical to the single-record call"""
    from apples_b200.placer import GpuPlacer
    ci, tree, ref = _c1(workdir)
    pl = GpuPlacer(tree, ref, tree.name_to_node, device=0, model='K2P')
    params = pl.params_from_options(ci.options, ref)
    sn = pl.self_nodes([q[0] for q in ci.queries])
    packed = pl.pack_queries([q[1] for q in ci.queries])
    base = pl.place_packed(packed, sn, params)
    out, (cnt, edge, err, distal, pend, int0) = pl.place_packed(packed, sn, params, keep=4)
    pl.close()
    for x, y in zip(base, out):
        assert x.tobytes() == y.tobytes()
    assert (edge[:, 0] == out[0]).all() and err[:, 0].tobytes() == out[1].tobytes()
    assert distal[:, 0].tobytes() == out[2].tobytes() and pend[:, 0].tobytes() == out[3].tobytes()
    assert (cnt > 1).any()


def test_packed_and_byte_input_agree(workdir):
    """the device packer and ragged sub-batches give the packed input's results"""
    from apples_b200 import fasta
    from apples_b200.placer import GpuPlacer
    ci, tree, ref = _c1(workdir)
    seqs = [q[1] for q in ci.queries] * 37
    pl = GpuPlacer(tree, ref, tree.name_to_node, device=0, model='K2P')
    params = pl.params_from_options(ci.options, ref)
    a = pl.place_packed(pl.pack_queries(seqs), None, params)
    b = pl.place_bytes(fasta.as_byte_matrix(seqs, pl.L), None, params)
    pl.set_limits(max_subbatch=128)
    c = pl.place_bytes(fasta.as_byte_matrix(seqs, pl.L), None, params)
    assert pl.timings()['k2p_launches'] > 0
    pl.close()
    for x, y, z in zip(a, b, c):
        assert x.tobytes() == y.tobytes() == z.tobytes()


def test_two_gpus_equal_one(workdir):
    from apples_b200 import _lib, fasta
    from apples_b200.placer import GpuPlacer, MultiGpuPlacer
    if _lib.device_count() < 2:
        pytest.skip('needs two GPUs')
    ci, tree, ref = _c1(workdir)
    seqs = [q[1] for q in ci.queries] * 41
    params = GpuPlacer.params_from_options(ci.options, ref)
    one = GpuPlacer(tree, ref, tree.name_to_node, device=0, model='K2P')
    two = MultiGpuPlacer(tree, ref, tree.name_to_node, devices=(0, 1), model='K2P')
    mat = fasta.as_byte_matrix(seqs, one.L)
    a, b = one.place_bytes(mat, None, params), two.place_bytes(mat, None, params)
    one.close()
    two.close()
    for x, y in zip(a, b):
        assert x.tobytes() == y.tobytes()


def test_cli(workdir):
    """--model JC69 writes the bytes of a run without the flag; --model K2P writes the oracle's K2P placements, alone and
    with --keep-at-most 3"""
    import run_apples
    ref, qry, tree = (util.gunzip_to(n, workdir) for n in ('ref.fa', 'query.fa', 'backbone.nwk'))
    tsv = os.path.join(util.GOLD, 'c1_clusters.tsv')
    argv = ['-s', ref, '-q', qry, '-t', tree, '-D', '--clusters', tsv]
    base, jc, k2p, k2p3 = (os.path.join(workdir, 'k2pcli_%s.jplace' % t) for t in ('base', 'jc69', 'k2p', 'k2p3'))
    run_apples.main(argv + ['-o', base])
    run_apples.main(argv + ['-o', jc, '--model', 'JC69'])
    run_apples.main(argv + ['-o', k2p, '--model', 'K2P'])
    run_apples.main(argv + ['-o', k2p3, '--model', 'K2P', '--keep-at-most', '3'])
    assert open(base).read() == open(jc).read().replace(' --model JC69', '')
    ci = util.CaseInputs('c1_align_FM_MLSE', workdir)
    octx = ko.oracle_context(ci)
    by_name = {q[0]: q for q in ci.queries}
    j, j3 = json.load(open(k2p)), json.load(open(k2p3))
    assert len(j['placements']) == len(ci.queries)
    for p, p3 in zip(j['placements'], j3['placements']):
        q = by_name[p['n'][0].replace('-query', '')]
        exp, _ = octx.runquery(q[0], q[1], None)
        _check_p('cli', q[0], p['p'][0], exp['placements'][0]['p'][0], False, octx, q)
        assert p3['p'][0] == p['p'][0]


# ------------------------------------------------------------------------------------------------ errors
def test_errors(workdir):
    """each case the K2P model does not cover fails with its message; the context stays usable"""
    from apples_b200 import fasta
    from apples_b200.placer import GpuPlacer
    pl = _small_tree_placer()
    rng = np.random.default_rng(5)
    with pytest.raises(RuntimeError, match='model must be'):
        pl._check(pl.lib.apples_ctx_set_model(pl.h, 7))
    with pytest.raises(ValueError, match='--model'):
        GpuPlacer(pl.tree, None, pl.tree.name_to_node, device=0, model='F81')
    aa = fasta.pack(np.frombuffer(b'ARND' * 10, np.uint8).reshape(4, 10), fasta.AA)
    with pytest.raises(RuntimeError, match='nucleotide'):
        pl.set_reference_arrays(fasta.AA, 10, ['a', 'b', 'c', 'd'], aa, np.full(4, -1, np.int32), aa,
                                np.arange(5, dtype=np.int32), np.arange(4, dtype=np.int32))
    with pytest.raises(RuntimeError, match='at most %d columns' % FP4_MAX_L):
        _set_singletons(pl, FP4_MAX_L + 1, _nuc_rows(3, FP4_MAX_L + 1, rng, 'r'))
    pl.set_dense_mode(0)
    with pytest.raises(RuntimeError, match='dense mode 1'):
        _set_singletons(pl, 50, _nuc_rows(3, 50, rng, 'r'))
    pl.set_dense_mode(1)
    bad = np.frombuffer(b'ACGTN' * 10, np.uint8).reshape(1, 50).repeat(3, 0)
    with pytest.raises(RuntimeError, match='A,C,G,T,-'):
        pl.set_reference_bytes(fasta.NUC, 50, ['r0', 'r1', 'r2'], bad, np.full(3, -1, np.int32), np.arange(4, dtype=np.int32),
                               np.arange(3, dtype=np.int32))
    pl.close()
    # a query row with other bytes: the place call names the first one; the next call on the context works
    ci, tree, ref = _c1(workdir)
    pl = GpuPlacer(tree, ref, tree.name_to_node, device=0, model='K2P')
    params = pl.params_from_options(ci.options, ref)
    mat = fasta.as_byte_matrix([q[1] for q in ci.queries] * 3, pl.L)
    good = pl.place_bytes(mat, None, params)
    mat2 = mat.copy()
    mat2[17, 5] = ord('N')
    mat2[23, 9] = ord('?')
    with pytest.raises(RuntimeError, match='query row 17 '):
        pl.place_bytes(mat2, None, params)
    again = pl.place_bytes(mat, None, params)
    pl.close()
    for x, y in zip(good, again):
        assert x.tobytes() == y.tobytes()


def test_matrix_mode_ignores_the_model(workdir):
    from apples_b200.placer import GpuPlacer
    ci = util.CaseInputs('c2_matrix_FM_MLSE', workdir)
    tree, _ = ci.product_state()
    tags = list(ci.queries[0][2].keys())
    rows = np.array([[q[2][t] for t in tags] for q in ci.queries], dtype=np.float64)
    out = {}
    for model in ('JC69', 'K2P'):
        pl = GpuPlacer(tree, None, tree.name_to_node, device=0, matrix_tags=tags, model=model)
        out[model] = pl.place_rows(rows, None, pl.params_from_options(ci.options))
        pl.close()
    for x, y in zip(out['JC69'], out['K2P']):
        assert x.tobytes() == y.tobytes()
