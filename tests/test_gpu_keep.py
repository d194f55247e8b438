"""GPU (-m gpu): --keep-at-most K, the ranked records of apples_set_alternatives, against the K-record oracle
(tests/keep_oracle.py) and against the single-record path.

Record 0 must be bit-identical to the single-record call.  The edge order follows the oracle's; as for the single
placement (DESIGN.md section 5, deviation 3), a different edge at a position is accepted only when the oracle scores the
two edges' keys within the tolerance.  In matrix mode x_1 / x_2 are bit-exact, so the ME order must be identical there.
"""
import json
import math
import os
import types

import numpy as np
import pytest

from tests import util
from tests import keep_oracle as ko

pytestmark = pytest.mark.gpu

REL, FLOOR = 1e-9, 1e-12
KEEPS = (2, 5, 16)


def _key(det, criterion, edge):
    x1, _, err = det['edges'][edge]
    return x1 if criterion in ('ME', 'HYBRID') else err


def _check_records(ctx, got, exp, det, criterion, matrix):
    """got / exp: the 'p' lists of one query (device, oracle).  det: the oracle's per-edge detail."""
    assert len(got) == len(exp), ctx
    if len(exp) == 1 or det is None:
        return
    for j, (g, e) in enumerate(zip(got, exp)):
        assert g[2] == (1 if j == 0 else 0), ctx
        if g[0] != e[0]:
            assert not (matrix and criterion == 'ME'), ('ME order differs in matrix mode', j, ctx, got, exp)
            assert g[0] in det['edges'], ctx
            assert util.close(_key(det, criterion, g[0]), _key(det, criterion, e[0]), REL, FLOOR), ('not a tie', j, ctx)
            continue
        assert [isinstance(x, int) for x in g] == [isinstance(x, int) for x in e], (j, ctx, g, e)
        assert util.close(g[1], e[1], REL, FLOOR), (j, ctx, g, e)
        if matrix:
            assert g[3] == e[3] and g[4] == e[4], (j, ctx, g, e)
        else:
            assert util.close(g[3], e[3], REL, 1e-15) and util.close(g[4], e[4], REL, 1e-15), (j, ctx, g, e)


def _expected_count(det, criterion, keep):
    V = det['num_nodes']
    return min(keep, math.floor(math.log2(V))) if criterion == 'HYBRID' else min(keep, V)


def _oracle_k(octx, q, keep):
    det = {}
    exp, st = ko.runquery_k(octx, q[0], q[1], dict(q[2]) if q[2] else None, keep)
    if st in (0, 3):
        octx.runquery(q[0], q[1], dict(q[2]) if q[2] else None, detail=det)
    return exp, st, (det or None)


def _compare_batch(tag, octx, queries, res1, resk, keep, criterion, matrix, exclude=False):
    """resk (keep records) against res1 (single record: record 0 bit-identical) and the oracle"""
    n = 0
    for q, r1, rk in zip(queries, res1, resk):
        p1, pk = r1['placements'][0]['p'], rk['placements'][0]['p']
        assert rk['placements'][0]['n'] == r1['placements'][0]['n']
        assert json.dumps(pk[0]) == json.dumps(p1[0]), (tag, q[0], pk[0], p1[0])
        try:
            exp, st, det = _oracle_k(octx, q, keep)
        except (ZeroDivisionError, AssertionError, FloatingPointError, OverflowError):
            continue
        pe = exp['placements'][0]['p']
        if any(isinstance(x, float) and (x != x or abs(x) == float('inf')) for rec in pe for x in rec[1:]):
            continue
        ctx = (tag, q[0], keep, criterion)
        if det is not None and not (st == 3 and exclude):
            assert len(pk) == _expected_count(det, criterion, keep), (ctx, len(pk))
        if pk[0][0] != pe[0][0]:
            continue   # a tie of the first placement: test_gpu_parity accepts it, the rankings then start apart
        _check_records(ctx, pk, pe, det, criterion, matrix)
        n += 1
    return n


@pytest.mark.parametrize('case', util.golden_names())
def test_golden_cases(case, workdir):
    from apples_b200.placer import place_batch
    ci = util.CaseInputs(case, workdir)
    tree, ref = ci.product_state()
    octx = ci.oracle_context()
    res1 = place_batch(ref, ci.options, tree.name_to_node, ci.queries, tree=tree, device=0)
    n = 0
    for keep in KEEPS:
        resk = place_batch(ref, ci.options, tree.name_to_node, ci.queries, tree=tree, device=0, keep=keep)
        n += _compare_batch(case, octx, ci.queries, res1, resk, keep, ci.options.criterion_name, ci.refs is None,
                            ci.options.exclude_intplace)
    assert n > 0


def test_keep_one_and_record_zero_are_the_single_record_call(workdir):
    """keep 1 through the new path, and the five arrays of a keep > 1 call, are bit-identical to a plain call; the
    count and the unused slots follow the header"""
    from apples_b200.placer import GpuPlacer
    for case in ('c1_align_FM_MLSE', 'c2_matrix_OLS_HYBRID_f100', 'syn300_BME_ME_pos', 'c3_prot_FM_MLSE'):
        ci = util.CaseInputs(case, workdir)
        tree, ref = ci.product_state()
        pl = GpuPlacer(tree, ref, tree.name_to_node, device=0)
        params = pl.params_from_options(ci.options, ref)
        sn = pl.self_nodes([q[0] for q in ci.queries])
        if ci.refs is None:
            tags = list(ci.queries[0][2].keys())
            pl.set_matrix_tags(tags)
            src = np.array([[q[2][t] for t in tags] for q in ci.queries], dtype=np.float64)
            place = pl.place_rows
        else:
            src = pl.pack_queries([q[1] for q in ci.queries])
            place = pl.place_packed
        base = place(src, sn, params)
        one = place(src, sn, params, keep=1)
        for x, y in zip(base, one):
            assert x.tobytes() == y.tobytes()
        for keep in KEEPS:
            out, (cnt, edge, err, distal, pend, int0) = place(src, sn, params, keep=keep)
            for x, y in zip(base, out):
                assert x.tobytes() == y.tobytes(), (case, keep)
            code = out[4] & 0xff
            assert (edge[:, 0] == out[0]).all() and (err[:, 0].tobytes() == out[1].tobytes())
            assert distal[:, 0].tobytes() == out[2].tobytes() and pend[:, 0].tobytes() == out[3].tobytes()
            assert (int0[:, 0] == ((out[4] >> 8) & 1)).all()
            assert ((cnt == 1) | (code == 0) | (code == 3)).all() and (cnt >= 1).all() and (cnt <= keep).all()
            for i in range(len(cnt)):
                assert (edge[i, cnt[i]:] == -1).all() and not err[i, cnt[i]:].any()
        # a place call takes the registration: the next call without keep has no ranked records
        assert isinstance(place(src, sn, params)[0], np.ndarray)
        pl.close()


def test_randomized_matrix_cases(workdir):
    """300 seeded random distance-matrix cases (the generator of test_gpu_parity): every method x criterion x -n, random
    -b / -f / --exclude, keep 2 / 5 / 16"""
    from oracle import apples_oracle as orc
    from apples_b200.placer import place_batch
    from tests.test_gpu_parity import _random_matrix_case
    rng = np.random.default_rng(8675309)
    n = 0
    for case in range(300):
        tfp, tree, queries = _random_matrix_case(rng, workdir, 'k%d' % case)
        method = str(rng.choice(['FM', 'OLS', 'BME', 'BE']))
        criterion = str(rng.choice(['MLSE', 'ME', 'HYBRID']))
        neg = bool(rng.random() < 0.25)
        b = int(rng.choice([1, 3, 5, 25, 1000]))
        f = float(rng.choice([0.0, 0.05, 0.2, 100.0]))
        keep = int(rng.choice(KEEPS))
        opt = types.SimpleNamespace(method_name=method, criterion_name=criterion, negative_branch=neg,
                                    base_observation_threshold=b, filt_threshold=f, minimum_alignment_overlap=0.001,
                                    exclude_intplace=bool(rng.random() < 0.3))
        otree, onames = orc.load_tree(tfp)
        octx = orc.OracleContext(otree, onames, method=method, criterion=criterion, negative_branch=neg,
                                 filt_threshold=f, baseobs=b, exclude_intplace=opt.exclude_intplace)
        try:
            res1 = place_batch(None, opt, tree.name_to_node, queries, tree=tree, device=0)
        except ZeroDivisionError:
            continue   # singular systems: the reference raises (test_gpu_parity)
        resk = place_batch(None, opt, tree.name_to_node, queries, tree=tree, device=0, keep=keep)
        n += _compare_batch('rndm%d' % case, octx, queries, res1, resk, keep, criterion, True, opt.exclude_intplace)
    assert n > 800


def test_randomized_alignment_cases(workdir):
    """120 seeded random alignment cases (nucleotide and protein, random gaps, clusterings, -V / -b / -f)"""
    from oracle import apples_oracle as orc
    from apples_b200 import synth
    from apples_b200.placer import place_batch
    from apples_b200.reference import ReducedReference
    from apples_b200.tree import BackboneTree
    rng = np.random.default_rng(5551212)
    n = 0
    for case in range(120):
        protein = bool(rng.random() < 0.3)
        nl = int(rng.integers(5, 70))
        L = int(rng.integers(40, 700))
        nwk = synth.random_tree(nl, seed=int(rng.integers(1, 1 << 30)), mean_edge=float(rng.choice([0.01, 0.03, 0.08])),
                                polytomy_frac=float(rng.choice([0.0, 0.3])))
        tfp = os.path.join(workdir, 'rndka_%d.nwk' % case)
        open(tfp, 'w').write(nwk)
        tree = BackboneTree.from_newick(tfp)
        refs, states = synth.evolve_alignment(tree, L, seed=int(rng.integers(1, 1 << 30)), protein=protein,
                                              gap_frac=float(rng.choice([0.0, 0.05, 0.4])))
        qd, _ = synth.make_queries(tree, states, int(rng.integers(1, 7)), seed=int(rng.integers(1, 1 << 30)), protein=protein,
                                   mean_extra=float(rng.choice([0.0, 0.03, 0.2])), gap_frac=float(rng.choice([0.0, 0.1, 0.6])))
        queries = [(k, v, None) for k, v in qd.items()]
        names = list(refs.keys())
        queries.append(('copy', refs[names[int(rng.integers(0, nl))]], None))
        tsv = os.path.join(workdir, 'rndka_%d.tsv' % case)
        with open(tsv, 'w') as fh:
            fh.write('SequenceName\tClusterNumber\n')
            for nm in names:
                fh.write('%s\t%d\n' % (nm, -1 if rng.random() < 0.35 else int(rng.integers(1, max(2, nl // 3)))))
        thr = float(rng.choice([0.05, 0.2, 0.6]))
        ref = ReducedReference(None, protein, tfp, thr, 1, cluster_tsv=tsv, tree=tree, refs=refs)
        opt = types.SimpleNamespace(method_name=str(rng.choice(['FM', 'OLS', 'BME', 'BE'])),
                                    criterion_name=str(rng.choice(['MLSE', 'ME', 'HYBRID'])),
                                    negative_branch=bool(rng.random() < 0.2), base_observation_threshold=int(rng.choice([2, 5, 25])),
                                    filt_threshold=thr, minimum_alignment_overlap=float(rng.choice([0.001, 0.2, 0.5])),
                                    exclude_intplace=False)
        keep = int(rng.choice(KEEPS))
        octx = orc.OracleContext(*orc.load_tree(tfp), refs=refs, representatives=orc.representatives_from_tsv(tsv, refs, protein),
                                 protein=protein, method=opt.method_name, criterion=opt.criterion_name,
                                 negative_branch=opt.negative_branch, filt_threshold=thr, baseobs=opt.base_observation_threshold,
                                 overlap=opt.minimum_alignment_overlap)
        try:
            res1 = place_batch(ref, opt, tree.name_to_node, queries, tree=tree, device=0)
        except ZeroDivisionError:
            continue
        resk = place_batch(ref, opt, tree.name_to_node, queries, tree=tree, device=0, keep=keep)
        n += _compare_batch('rndka%d' % case, octx, queries, res1, resk, keep, opt.criterion_name, False)
    assert n > 300


def _same_alt(a, b):
    for x, y in zip(a[0] + a[1], b[0] + b[1]):
        assert x.tobytes() == y.tobytes()


def test_pipeline_paths(workdir):
    """The ranked records through every placement launch: the block class (V + 1 > 512) with the default scratch limit
    and with one query per chunk, overflow reruns with a small slot capacity, byte-compare fallback queries and a
    ragged last sub-batch -- identical to the default limits and to the oracle."""
    from oracle import apples_oracle as orc
    from apples_b200 import _lib, fasta
    from apples_b200.placer import GpuPlacer, results_to_jplace
    from apples_b200.reference import ReducedReference
    from apples_b200.tree import BackboneTree
    keep = 5
    # ---- block class: a 700-leaf caterpillar from a distance matrix with the filter off (V = 2 * 700 - 2)
    rng = np.random.default_rng(31)
    nl = 700
    s = 'L0:%.5f' % rng.uniform(0.001, 0.02)
    for i in range(1, nl):
        s = '(%s,L%d:%.5f):%.5f' % (s, i, rng.uniform(0.001, 0.02), rng.uniform(0.0005, 0.01))
    tfp = os.path.join(workdir, 'kcat.nwk')
    open(tfp, 'w').write(s.rsplit(':', 1)[0] + ';')
    tree = BackboneTree.from_newick(tfp)
    depth = np.zeros(tree.num_nodes)
    for u in range(tree.num_nodes - 2, -1, -1):
        depth[u] = depth[tree.parent[u]] + tree.edge_length[u]
    names = ['L%d' % i for i in range(nl)]
    leaf = np.array([tree.name_to_node[x] for x in names])

    def pathdist(a, b):
        x, y = a, b
        while x != y:
            if x < y:
                x = tree.parent[x]
            else:
                y = tree.parent[y]
        return depth[a] + depth[b] - 2 * depth[x]
    rows = []
    for anchor in (50, 300, 650):
        d = np.array([pathdist(leaf[anchor], leaf[j]) for j in range(nl)]) + 0.013
        rows.append(np.maximum(np.round(d * (1 + 0.02 * rng.standard_normal(nl)), 6), 0.001))
    rows = np.array(rows)
    queries = [('q%d' % i, None, dict(zip(names, r.tolist()))) for i, r in enumerate(rows)]
    for crit in ('MLSE', 'HYBRID', 'ME'):
        params = _lib.make_params('FM', crit, False, 25, 100.0)
        pl = GpuPlacer(tree, None, tree.name_to_node, device=0, matrix_tags=names)
        a = pl.place_rows(rows, None, params, keep=keep)
        assert pl.timings()['placed_block'] == 3
        pl.set_limits(scratch_bytes=1, slot_cap=8)   # one query per chunk, overflow reruns through the block class
        b = pl.place_rows(rows, None, params, keep=keep)
        _same_alt(a, b)
        pl.close()
        octx = orc.OracleContext(*orc.load_tree(tfp), method='FM', criterion=crit, filt_threshold=100.0)
        res1 = results_to_jplace([q[0] for q in queries], [False] * 3, a[0], log=False)
        resk = results_to_jplace([q[0] for q in queries], [False] * 3, a[0], log=False, alt=a[1])
        assert _compare_batch('kcat', octx, queries, res1, resk, keep, crit, True) == 3
    # ---- overflow reruns, exotic bytes, ragged sub-batches: config 1 queries with symbols outside A,C,G,T,-
    ci = util.CaseInputs('c1_align_FM_MLSE', workdir)
    tree, _ = ci.product_state()
    rng = np.random.default_rng(99)
    queries = []
    for i, (qn, qs, _) in enumerate(ci.queries * 30):
        s = qs.copy()
        if i % 7 == 0:
            for pos in rng.integers(0, len(s), 3):
                s[pos] = rng.choice([b'.', b'*', b'?'])
        queries.append(('%s_%d' % (qn, i), s, None))
    ref = ReducedReference(None, False, ci.tree_fp, 0.2, 1, cluster_tsv=ci.tsv, tree=tree, refs=ci.refs)
    ref.set_baseobs(25)
    mat = fasta.as_byte_matrix([q[1] for q in queries], len(queries[0][1]))
    for crit in ('MLSE', 'ME', 'HYBRID'):
        opt = types.SimpleNamespace(method_name='FM', criterion_name=crit, negative_branch=False, base_observation_threshold=25,
                                    filt_threshold=0.2, minimum_alignment_overlap=0.001, exclude_intplace=False)
        pl = GpuPlacer(tree, ref, tree.name_to_node, device=0)
        params = pl.params_from_options(opt, ref)
        a = pl.place_bytes(mat, None, params, keep=keep)
        assert pl.timings()['fallback_queries'] > 0
        pl.set_limits(max_subbatch=128, slot_cap=8, scratch_bytes=1)   # ragged sub-batches, overflow reruns
        b = pl.place_bytes(mat, None, params, keep=keep)
        assert pl.timings()['overflow_queries'] > 0
        _same_alt(a, b)
        pl.close()
        octx = orc.OracleContext(*orc.load_tree(ci.tree_fp), refs=ci.refs,
                                 representatives=orc.representatives_from_tsv(ci.tsv, ci.refs, False), method='FM', criterion=crit)
        qn = [q[0] for q in queries]
        res1 = results_to_jplace(qn, [False] * len(qn), a[0], log=False)
        resk = results_to_jplace(qn, [False] * len(qn), a[0], log=False, alt=a[1])
        pick = list(range(0, len(queries), 7))[:12] + [1, 2, 3]
        assert _compare_batch('kpaths', octx, [queries[i] for i in pick], [res1[i] for i in pick], [resk[i] for i in pick],
                              keep, crit, False) >= 10


def test_two_gpus_equal_one(workdir):
    from apples_b200 import _lib, fasta
    from apples_b200.placer import GpuPlacer, MultiGpuPlacer
    if _lib.device_count() < 2:
        pytest.skip('needs two GPUs')
    ci = util.CaseInputs('c1_align_FM_MLSE', workdir)
    tree, ref = ci.product_state()
    seqs = [q[1] for q in ci.queries] * 41
    params = GpuPlacer.params_from_options(ci.options, ref)
    one = GpuPlacer(tree, ref, tree.name_to_node, device=0)
    two = MultiGpuPlacer(tree, ref, tree.name_to_node, devices=(0, 1))
    mat = fasta.as_byte_matrix(seqs, one.L)
    _same_alt(one.place_bytes(mat, None, params, keep=5), two.place_bytes(mat, None, params, keep=5))
    one.close()
    two.close()


def test_cli(workdir):
    """--keep-at-most 1 writes the file of a run without the flag; --keep-at-most 4 lists the oracle's records, in
    alignment and distance-matrix mode, with and without --exclude"""
    import run_apples
    ref, qry, tree, mat = (util.gunzip_to(n, workdir) for n in ('ref.fa', 'query.fa', 'backbone.nwk', 'dist.mat'))
    tsv = os.path.join(util.GOLD, 'c1_clusters.tsv')
    runs = [('c1_align_FM_MLSE', ['-s', ref, '-q', qry, '-t', tree, '-D', '--clusters', tsv]),
            ('c1_align_BME_HYBRID', ['-s', ref, '-q', qry, '-t', tree, '-D', '--clusters', tsv, '-m', 'BME', '-c', 'HYBRID']),
            ('c2_matrix_FM_MLSE', ['-d', mat, '-t', tree]),
            ('c2_matrix_BME_ME_b5', ['-d', mat, '-t', tree, '-m', 'BME', '-c', 'ME', '-b', '5', '-f', '0.05', '--exclude'])]
    for case, argv in runs:
        base, k1, k4 = (os.path.join(workdir, '%s_%s.jplace' % (case, t)) for t in ('base', 'k1', 'k4'))
        run_apples.main(argv + ['-o', base])
        run_apples.main(argv + ['-o', k1, '--keep-at-most', '1'])
        run_apples.main(argv + ['-o', k4, '--keep-at-most', '4'])
        assert open(base).read() == open(k1).read().replace(' --keep-at-most 1', '')
        j = json.load(open(k4))
        txt = open(k4).read()
        assert txt == json.dumps(j, sort_keys=True, indent=4) + '\n'
        ci = util.CaseInputs(case, workdir)
        octx = ci.oracle_context()
        octx.exclude_intplace = '--exclude' in argv
        jb = json.load(open(base))
        assert [p['n'] for p in j['placements']] == [p['n'] for p in jb['placements']]
        by_name = {q[0]: q for q in ci.queries}
        for pl, pb in zip(j['placements'], jb['placements']):
            assert pl['p'][0] == pb['p'][0]
            q = by_name[pl['n'][0].replace('-query', '')]
            exp, st, det = _oracle_k(octx, q, 4)
            pe = exp['placements'][0]['p']
            if pe[0][0] != pl['p'][0][0]:
                continue
            if st == 3 and octx.exclude_intplace or det is None:
                assert len(pl['p']) == 1
                continue
            _check_records((case, q[0]), pl['p'], pe, det, octx.criterion, ci.refs is None)
