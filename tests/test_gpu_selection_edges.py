"""GPU (-m gpu): the observed sets of the selection kernels against exact expectations, on the long key rows and at the
decision edges where the selection can go wrong.

The selection decides which leaves a query observes (Reference.py:117-157 for alignments, PoolQueryWorker.py:44-59 for
distance-matrix rows); V, the restricted subtree and the placement follow from that set.  Each case here builds its
expectation on the host from inputs the test knows exactly, with `expected_observed` (the reference's two-phase rule on
exact decisions), and compares it with GpuPlacer.observed_sets: the count, the node list, the distances and the status.

A. Distance-matrix rows of 5 000 and 4 113 columns (select_kernel<SEL_MATRIX>): values on a 1/64 grid, a lane class of
   equal smallest values (the far-phase refill with ties), +-0.0, +inf, negatives, columns not in the tree, the query's
   own column; the reference is orc.observed_matrix itself.
B. Protein at config-3 shape (select_kernel<SEL_AA>) with first- and second-level overflow reruns, a ragged last
   sub-batch, and packed / byte / resident input; K2P (select_kernel<SEL_K2P>) through the same harness.  Sampled
   queries against the oracle's fp64 distances, member distances also against exact pair counts.
C. The JC69 guard band: keys designed onto the edges of the 16.16 fixed-point gate and inside the band, in dense modes
   1 and 0, through the stash rerun and in byte mode; near decided in 50-digit decimal arithmetic.
D. Rows of 1 250 key lines (40 000 singleton representatives) in select_nuc_kernel, against the keys of count_keys and
   against the byte-mode twin.
"""
import decimal
import math
import os
from fractions import Fraction

import numpy as np
import pytest


pytestmark = pytest.mark.gpu

GAP = ord('-')
BASES = np.frombuffer(b'ACGT', np.uint8)
PLACED, ZERO_DIST_LEAF, TOO_FEW_DISTANCES = 0, 1, 2
TIE_REL = 1e-12


# ------------------------------------------------------------------------------------------------------- references
def overlap_vmin(L, overlap):
    """api.cu overlap_vmin: the smallest valid count v >= 1 with not (v / L < overlap)"""
    for v in range(1, L + 1):
        if not (v / L < overlap):
            return v
    return L + 1


def make_gate(thr):
    """api.cu make_gate restated: (P_lo, P_hi) of the 16.16 guard band; (m << 16) <= P_lo v is near, >= P_hi v far"""
    if not (thr >= 0.0):
        return 0, 0
    pstar = 0.75 * (1.0 - math.exp(-4.0 * thr / 3.0))
    lo = math.floor(pstar * (1.0 - 1e-9) * 65536.0) - 1.0
    hi = math.ceil(pstar * (1.0 + 1e-9) * 65536.0) + 1.0
    p_lo = int(max(0.0, min(lo, 49152.0)))
    p_hi = int(max(1.0, min(hi, 49153.0)))
    return (49152 if p_lo >= 49151 else p_lo), p_hi


def pstar_exact(thr):
    """p* = 0.75 (1 - exp(-4 thr / 3)) in 50-digit decimal: jc69(m, v) <= thr  <=>  m / v <= p*"""
    with decimal.localcontext() as c:
        c.prec = 50
        t = decimal.Decimal(thr)
        return decimal.Decimal('0.75') * (1 - (-4 * t / 3).exp())


def jc69(m, v, vmin=1):
    """the oracle's fp64 jc69_from_counts (distance.py:735-745) without the length argument"""
    if v == 0 or v < vmin:
        return -1.0
    p = np.float64(m * 1.0 / v)
    if p - np.finfo(float).eps < 0:
        return 0.0
    loc = 1 - (4 * p / 3)
    if 0 >= loc:
        return -1.0
    return float(-0.75 * np.log(loc))


def expected_observed(order, near, members_of, baseobs, self_node=-1):
    """Reference.py:141-157 / PoolQueryWorker.py:44-59 and :63-79 on decisions made exactly by the caller.

    order: the valid units in ascending (distance, index) order; near[i]: the verdict on order[i]; members_of(u): the
    (node, distance) pairs of the members of unit u whose distance is not missing, in group order.  Units are taken in
    order while `near or n_obs < baseobs`.  Returns (observed {node: distance} without the own entry, status, the far
    units taken, the number of units taken)."""
    obs, far, n_obs, k = {}, [], 0, 0
    for i, u in enumerate(order):
        if not (near[i] or n_obs < baseobs):
            break
        if not near[i]:
            far.append(int(u))
        for node, d in members_of(int(u)):
            obs[node] = d
            n_obs += 1
        k = i + 1
    if self_node >= 0:
        obs.pop(self_node, None)
    if any(d == 0 for d in obs.values()):
        status = ZERO_DIST_LEAF
    elif len(obs) <= 2:
        status = TOO_FEW_DISTANCES
    else:
        status = PLACED
    return obs, status, far, k


def refill_classes(far):
    """largest number of far units taken from one lane class (units u = lane mod 32) of select_kernel"""
    return int(np.bincount(np.asarray(far, np.int64) % 32, minlength=32).max()) if len(far) else 0


def check_observed(tag, exp, got, dist_ok):
    """exp: per query (observed {node: d}, status); got: observed_sets + status codes + V.  The node list and distances
    are final for the queries that reach placement; the others must hold the same set."""
    count, node, dist, status, V = got
    for qi, (obs, st) in enumerate(exp):
        if obs is None:
            continue
        ctx = (tag, qi)
        k = int(count[qi])
        assert k == len(obs), ctx + (k, len(obs))
        code = int(status[qi]) & 0xff
        if st == PLACED:
            assert code in (0, 3) and V[qi] > 0, ctx + (code, int(V[qi]))
            nodes = node[qi, :k].tolist()
            assert nodes == sorted(obs), ctx
            dist_ok(ctx, dist[qi, :k], np.array([obs[u] for u in nodes]))
        else:
            assert code == st and V[qi] == 0, ctx + (code, st)
            assert sorted(node[qi, :k].tolist()) == sorted(obs), ctx


def bit_identical(ctx, got, exp):
    assert got.view(np.uint64).tolist() == exp.view(np.uint64).tolist(), ctx


def within_ulps(ctx, got, exp, n=2):
    """device log and numpy log are each within 1 ulp: the same counts give distances at most 2 ulp apart, different
    counts of a different ratio are ~1e-5 apart"""
    assert (np.abs(got - exp) <= n * np.spacing(np.abs(exp))).all(), ctx + (got[:4], exp[:4])


def within_rel(rel):
    def check(ctx, got, exp):
        bad = np.abs(got - exp) > rel * np.abs(exp)
        assert not bad.any(), ctx + (got[bad][:4], exp[bad][:4])
    return check


def _placer(tree, mode=None, model='JC69'):
    from apples_b200.placer import GpuPlacer
    pl = GpuPlacer(tree, None, tree.name_to_node, device=0, model=model)
    if mode is not None:
        pl.set_dense_mode(mode)
    return pl


def _write_tree(workdir, name, nwk):
    tfp = os.path.join(workdir, name)
    with open(tfp, 'w') as f:
        f.write(nwk)
    return tfp


# ---------------------------------------------------------------------------------------- A. distance-matrix rows
def _path_lengths(parent, el, a):
    """path length from leaf a to every node (ids are post-order ranks: a parent has a larger id than its children)"""
    M = len(parent)
    d = [-1.0] * M
    x, acc = a, 0.0
    d[a] = 0.0
    while x != M - 1:
        acc += el[x]
        x = parent[x]
        d[x] = acc
    for u in range(M - 2, -1, -1):
        if d[u] < 0:
            d[u] = d[parent[u]] + el[u]
    return np.array(d)


@pytest.fixture(scope='module')
def matrix_case(workdir):
    """a 5 000-leaf backbone and two batches of 48 rows (5 000 and 4 096 + 17 columns).  Values are path lengths with
    noise on a 1/64 grid (ties everywhere).  Row roles by i % 8: 1, 5, 7: the columns = 7 mod 32 hold one equal smallest
    value (one lane class of ties); 2: one 0.0; 3: one -0.0; 4, 5: named like a backbone leaf whose column is present;
    6: a coarser 1/8 grid.  In every row ~1 % +inf and ~3 % negative values.  NaN is left out: the oracle's sort of a
    row is undefined on NaN."""
    from apples_b200 import synth
    from apples_b200.tree import BackboneTree
    nwk = synth.random_tree(5000, seed=5150)
    tfp = _write_tree(workdir, 'sel_matrix.nwk', nwk)
    tree = BackboneTree.from_newick(tfp)
    rng = np.random.default_rng(5151)
    leaves = [tree.label[u] for u in tree.leaf_ids.tolist()]
    parent, el = tree.parent.tolist(), np.abs(tree.edge_length).tolist()
    batches = []
    for width, n_ghost in ((5000, 100), (4096 + 17, 63)):
        tags = [leaves[i] for i in rng.permutation(len(leaves))[:width - n_ghost]] + ['ghost%d' % i for i in range(n_ghost)]
        rng.shuffle(tags)
        col_node = np.array([tree.name_to_node.get(t, -1) for t in tags])
        in_tree = np.flatnonzero(col_node >= 0)
        rows, names = np.empty((48, width)), []
        for i in range(48):
            anchor = tree.name_to_node[leaves[int(rng.integers(0, len(leaves)))]]
            pl = _path_lengths(parent, el, anchor)
            d = np.where(col_node >= 0, pl[np.maximum(col_node, 0)], rng.uniform(0, 0.5, width)) + 0.01
            d *= 1 + 0.05 * rng.standard_normal(width)
            grid = 8 if i % 8 == 6 else 64
            d = np.maximum(np.round(d * grid) / grid, 2 / 64)
            if i % 8 in (1, 5, 7):
                d[7::32] = 1 / 64
            u = rng.random(width)
            d[u < 0.01] = np.inf
            d[(u >= 0.01) & (u < 0.025)] = -1.0
            d[(u >= 0.025) & (u < 0.04)] = -1 / 64
            name = 'rq%d' % i
            if i % 8 == 2:
                d[int(rng.choice(in_tree))] = 0.0
            if i % 8 == 3:
                d[int(rng.choice(in_tree))] = -0.0
            if i % 8 in (4, 5):
                c = int(rng.choice(in_tree))
                name = tags[c]
                d[c] = 3 / 64
            rows[i] = d
            names.append(name)
        batches.append((tags, rows, names))
    return tfp, tree, batches


def _matrix_expected(tree, tags, rows, names, thr, b):
    """orc.observed_matrix on every row, then the own-entry removal and the status of PoolQueryWorker.py:63-79"""
    from oracle import apples_oracle as orc
    col = {t: j for j, t in enumerate(tags)}
    exp, refill = [], 0
    for row, name in zip(rows, names):
        obs = orc.observed_matrix(dict(zip(tags, row.tolist())), tree.name_to_node, thr, b)
        refill += refill_classes([col[t] for t, v in obs.items() if v > thr]) >= 3
        obs.pop(name, None)
        o = {tree.name_to_node[t]: v for t, v in obs.items()}
        st = ZERO_DIST_LEAF if any(v == 0 for v in o.values()) else (TOO_FEW_DISTANCES if len(o) <= 2 else PLACED)
        exp.append((o, st))
    return exp, refill


def _matrix_run(tree, tags, rows, names, params, slot_cap):
    pl = _placer(tree)
    try:
        pl.set_matrix_tags(tags)
        if slot_cap:
            pl.set_limits(slot_cap=slot_cap)
        sn = pl.self_nodes(names)
        pl.timings(reset=True)
        count, node, dist = pl.observed_sets(params, rows=rows, self_node=sn, cap=8192)
        out = pl.place_rows(rows, sn, params)
        _, V, _ = pl.last_counts(len(rows))
        return (count, node, dist, out[4], V), out, pl.timings()
    finally:
        pl.close()


def test_matrix_rows_against_observed_matrix(matrix_case):
    """every -b / -f / slot setting: observed sets, distances (bit for bit), status; with slot_cap 32 the queries
    overflow and their rows are gathered from the host for the reruns"""
    from apples_b200 import _lib
    _, tree, batches = matrix_case
    refill = overflow = 0
    for b in (1, 25, 300, 3000):
        for thr in (-1.0, 0.0, 0.05, np.inf):
            params = _lib.make_params('FM', 'MLSE', base_observation_threshold=b, filt_threshold=thr)
            for tags, rows, names in batches:
                exp, r = _matrix_expected(tree, tags, rows, names, thr, b)
                refill += r
                for slot_cap in (0, 32):
                    got, _, t = _matrix_run(tree, tags, rows, names, params, slot_cap)
                    overflow += t['overflow_queries']
                    check_observed(('matrix', len(tags), b, thr, slot_cap), exp, got, bit_identical)
    print('matrix: %d (query, setting) pairs take >= 3 far units of one lane class; %d overflow queries'
          % (refill, overflow))
    assert refill >= 20 and overflow > 0


def test_matrix_placements_against_the_oracle(matrix_case):
    """32 rows of the 5 000-column batch at -b 300 -f 0.05 with reruns: placements against the oracle"""
    from oracle import apples_oracle as orc
    from apples_b200 import _lib
    from tests.test_gpu_parity import _check_p
    tfp, tree, batches = matrix_case
    tags, rows, names = batches[0]
    rows, names = rows[:32], names[:32]
    b, thr = 300, 0.05
    params = _lib.make_params('FM', 'MLSE', base_observation_threshold=b, filt_threshold=thr)
    _, (edge, error, distal, pendant, status), _ = _matrix_run(tree, tags, rows, names, params, 32)
    otree, onames = orc.load_tree(tfp)
    octx = orc.OracleContext(otree, onames, method='FM', criterion='MLSE', filt_threshold=thr, baseobs=b)
    placed = 0
    for i, name in enumerate(names):
        q = (name, None, dict(zip(tags, rows[i].tolist())))
        res, st = octx.runquery(*q)
        p = res['placements'][0]['p'][0]
        assert int(status[i]) & 0xff == st, (i, status[i], st)
        if st in (0, 3):
            got = [int(edge[i]), float(error[i]), 1, float(distal[i]), 0 if status[i] & 0x100 else float(pendant[i])]
            assert _check_p('sel_matrix', name, got, p, True, octx, q) == 'ok'
            placed += 1
        elif st == ZERO_DIST_LEAF:
            assert int(edge[i]) == p[0]
    assert placed >= 16


# ------------------------------------------------------------------------------------- B. protein and K2P alignments
_POOL = {}   # what the fork-pool workers read


def _alignment_expect(qi):
    """expected observed set of query qi from the oracle's fp64 distances (_POOL['dist_fn']), with the oracle's
    placement of that set; 'tie' when two units on either side of the -b cut, or a unit and the threshold, are within
    1e-12 relative (either outcome is then accepted)"""
    from oracle import apples_oracle as orc
    c = _POOL
    q = c['qmat'][qi].view('S1')
    reps, refs, thr = c['reps'], c['refs'], c['thr']
    d = np.array([c['dist_fn'](q, cons, 0.001) for cons, _ in reps])
    valid = np.flatnonzero(d >= 0)
    order = valid[np.lexsort((valid, d[valid]))]
    near = d[order] <= thr

    def members_of(u):
        out = []
        for name in reps[u][1]:
            dm = c['dist_fn'](q, refs[name], 0.001)
            if not dm < 0:
                out.append((c['node_of'][name], dm))
        return out
    obs, st, far, k = expected_observed(order, near, members_of, c['b'])
    ds = d[order]
    tie = bool((np.abs(ds - thr) <= TIE_REL * np.maximum(np.abs(ds), abs(thr))).any()) if np.isfinite(thr) else False
    if 0 < k < len(order) and not near[k] and ds[k] - ds[k - 1] <= TIE_REL * ds[k]:
        tie = True
    name_of = c['name_of']
    det = {}
    res, ost = orc.place_from_observed('Q%d' % qi, {name_of[u]: v for u, v in obs.items()}, c['onames'], detail=det)
    exact = None
    if c['exact'] is not None and obs:
        exact = c['exact'](c['qmat'][qi], [name_of[u] for u in sorted(obs)])
    return dict(obs=obs, st=st, far=far, tie=tie, p=res['placements'][0]['p'][0], ost=ost, V=det.get('num_nodes'),
                exact=exact)


def _aa_exact(qrow, names):
    """member distances from exact pair counts (math.fsum of counts x BLOSUM45) and 1 - tot / v of each"""
    from tests.test_gpu_count_kernels import _scoredist_expected
    L = len(qrow)
    rows = np.stack([_POOL['refs'][n].view(np.uint8) for n in names])
    d, _ = _scoredist_expected(qrow[None], rows, L, 0.001)
    return d[0]


def _alignment_case(workdir, tag, n_leaves, L, protein, seed):
    from apples_b200 import synth
    from apples_b200.reference import ReducedReference
    from apples_b200.tree import BackboneTree
    nwk = synth.random_tree(n_leaves, seed=seed, mean_edge=0.02)
    tfp = _write_tree(workdir, tag + '.nwk', nwk)
    tree = BackboneTree.from_newick(tfp)
    refs, states = synth.evolve_alignment(tree, L, seed=seed + 1, protein=protein)
    qd, _ = synth.make_queries(tree, states, 2000, seed=seed + 2, protein=protein)
    qmat = np.stack([np.asarray(s).view(np.uint8) for s in qd.values()]).copy()
    ref = ReducedReference(None, protein, None, 0.2, 1, tree=tree, refs=refs)
    return tfp, tree, refs, ref, qmat


def _run_alignment_settings(tag, case, settings, dist_fn, model='JC69', exact=None, max_subbatch=512):
    """for each (-f, -b): one context with slot_cap 32 and ragged sub-batches gives observed sets and placements from
    packed, byte and resident input, which must equal a default context's; a seeded sample of up to 16 overflowed and
    ordinary queries (64 in all) is compared with the oracle.  Returns (refill queries, overflow queries, ties)."""
    import multiprocessing as mp
    from oracle import apples_oracle as orc
    from apples_b200 import _lib
    from tests.test_gpu_parity import _check_p
    tfp, tree, refs, ref, qmat = case
    nq = len(qmat)
    x, y = _placer(tree, model=model), _placer(tree, model=model)
    try:
        x.set_reference(ref, on_device=True)
        y.set_reference(ref, on_device=True)
        x.set_limits(max_subbatch=max_subbatch, slot_cap=32)
        packed = x.pack_queries(qmat)
        otree, onames = orc.load_tree(tfp)
        node_of = {n: tree.name_to_node[n] for n in refs}
        refill = overflow = ties = 0
        for thr, b in settings:
            params = _lib.make_params('FM', 'MLSE', base_observation_threshold=b, filt_threshold=thr)
            x.timings(reset=True)
            count, node, dist = x.observed_sets(params, packed=packed, cap=4096)
            t = x.timings()
            out = x.place_packed(packed, None, params)
            K, V, over = x.last_counts(nq)
            outs = [x.place_bytes(qmat, None, params), y.place_packed(packed, None, params)]
            x.upload_queries(packed)
            x.place_resident(params)
            outs.append(x.download_results())
            for o in outs:
                for a, c in zip(out, o):
                    assert a.tobytes() == c.tobytes(), (tag, thr, b)
            assert (count == K).all(), (tag, thr, b)
            assert t['overflow_queries'] > 0 and t['rep_distance_launches'] >= 4, (tag, thr, b, t)
            overflow += int(t['overflow_queries'])
            rng = np.random.default_rng(int(thr * 1000) + b)
            o1, o0 = np.flatnonzero(over == 1), np.flatnonzero(over == 0)
            s1 = rng.choice(o1, min(16, len(o1)), replace=False)
            rest = np.setdiff1d(np.arange(nq), s1)
            pool0 = o0 if len(o0) >= 64 - len(s1) else rest
            sample = np.concatenate([s1, rng.choice(pool0, 64 - len(s1), replace=False)]).tolist()
            _POOL.clear()
            _POOL.update(qmat=qmat, reps=ref.representatives, refs=refs, thr=thr, b=b, dist_fn=dist_fn,
                         node_of=node_of, name_of={v: k for k, v in node_of.items()}, onames=onames, exact=exact)
            with mp.get_context('fork').Pool(min(len(sample), os.cpu_count() or 1)) as pool:
                exp = pool.map(_alignment_expect, sample, chunksize=1)
            octx = orc.OracleContext(otree, onames, refs=refs, representatives=ref.representatives, filt_threshold=thr,
                                     baseobs=b)
            octx.dist_fn = dist_fn
            for qi, e in zip(sample, exp):
                ctx = (tag, thr, b, qi)
                if e['tie']:
                    ties += 1
                    continue
                refill += refill_classes(e['far']) >= 3
                st = e['st']
                assert st == (PLACED if e['ost'] in (0, 3) else e['ost']), ctx + (st, e['ost'])
                got = (count[qi:qi + 1], node[qi:qi + 1], dist[qi:qi + 1], out[4][qi:qi + 1], V[qi:qi + 1])
                check_observed(ctx, [(e['obs'], st)], got, within_rel(1e-9))
                if st != PLACED:
                    continue
                assert int(V[qi]) == e['V'], ctx + (int(V[qi]), e['V'])
                if e['exact'] is not None:
                    k = int(count[qi])
                    ex = e['exact']
                    x1 = np.exp(-ex / 1.3)                     # 1 - tot / v
                    rel = 8 * qmat.shape[1] * np.finfo(float).eps / x1
                    assert (np.abs(dist[qi, :k] - ex) <= rel * np.abs(ex) + 1e-300).all(), ctx
                q = ('Q%d' % qi, qmat[qi].view('S1'), None)
                g = [int(out[0][qi]), float(out[1][qi]), 1, float(out[2][qi]),
                     0 if out[4][qi] & 0x100 else float(out[3][qi])]
                if _check_p(tag, q[0], g, e['p'], False, octx, q) == 'tie':
                    ties += 1
        return refill, overflow, ties
    finally:
        x.close()
        y.close()


def test_protein_selection_and_reruns_against_the_oracle(workdir):
    """4 000 leaves, 1 638 sites, ~440 representatives at 0.2, 2 000 queries; -f 0.05 / 0.6 x -b 25 / 300"""
    from oracle import apples_oracle as orc
    case = _alignment_case(workdir, 'sel_prot', 4000, 1638, True, 3030)
    assert 350 <= len(case[3].groups) <= 500
    refill, overflow, ties = _run_alignment_settings('prot', case, [(0.05, 25), (0.05, 300), (0.6, 25), (0.6, 300)],
                                                     orc.scoredist, exact=_aa_exact)
    print('protein: %d refill queries, %d overflow queries, %d ties' % (refill, overflow, ties))
    assert refill >= 20 and ties <= 2


def test_k2p_selection_and_reruns_against_the_oracle(workdir):
    """5 000 leaves, 1 500 sites, -b 300, slot_cap 32: select_kernel<SEL_K2P> with refills and reruns"""
    from tests.k2p_oracle import k2p
    case = _alignment_case(workdir, 'sel_k2p', 5000, 1500, False, 4040)
    refill, overflow, ties = _run_alignment_settings('k2p', case, [(0.2, 300)], k2p, model='K2P')
    print('k2p: %d refill queries, %d overflow queries, %d ties' % (refill, overflow, ties))
    assert refill >= 1 and ties <= 2


# ------------------------------------------------------------------------------------------- C. the JC69 guard band
BAND_THRESHOLDS = (0.0, 1e-6, 0.02, 0.2, 10.0, np.inf, -1.0)


def _near_table(thr, vs):
    """{v: largest m with m / v <= p*} in exact arithmetic (-1: none)"""
    if not (thr >= 0.0):
        return {v: -1 for v in vs}
    ps = pstar_exact(thr)
    with decimal.localcontext() as c:
        c.prec = 50
        return {v: int((ps * v).to_integral_value(rounding=decimal.ROUND_FLOOR)) for v in vs}


def _designed_pairs(L, n_rep, seed):
    """(m, v) pairs with 1 <= m, 4 m < 3 v, v <= L - 1: on the two edges of classify() (m << 16 = P_lo v where v allows
    it, else the largest m below; m << 16 = P_hi v, else the smallest m above), adjacent pairs (m, v), (m + 1, v)
    around p* for v near the length limit, and the ratios closest to p* (1 +- 1e-8) over all v; then random pairs up
    to n_rep"""
    vmax = L - 1
    top = list(range(vmax - 11, vmax + 1))
    pairs = set()
    for thr in BAND_THRESHOLDS:
        p_lo, p_hi = make_gate(thr)
        if p_hi == 0:
            continue
        for P in (p_lo, p_hi):
            step = 65536 // math.gcd(P, 65536) if P else 65536
            pairs.update(((P * v) >> 16, v) for v in range(step, vmax + 1, step)[-3:])
        for v in top:
            pairs.add(((p_lo * v) >> 16, v))
            pairs.add((-((-p_hi * v) >> 16), v))
        if np.isfinite(thr):
            nt = _near_table(thr, top)
            for v in top:
                pairs.update(((nt[v], v), (nt[v] + 1, v)))
            ps = Fraction(pstar_exact(thr))
            for s in (1 - Fraction(1, 10 ** 8), 1 + Fraction(1, 10 ** 8)):
                target = ps * s
                vs = np.arange(vmax // 2, vmax + 1)
                m = np.floor(float(target) * vs + 0.5).astype(np.int64)
                err = np.abs(m / vs - float(target))
                for i in np.argsort(err)[:6].tolist():
                    pairs.add((int(m[i]), int(vs[i])))
    pairs = sorted((m, v) for m, v in pairs if 1 <= m and 4 * m < 3 * v and v <= vmax)
    rng = np.random.default_rng(seed)
    while len(pairs) < n_rep:
        v = int(rng.integers(vmax // 2, vmax + 1))
        m = int(rng.integers(1, (3 * v - 1) // 4 + 1))
        if (m, v) not in pairs:
            pairs.append((m, v))
    pairs = [pairs[i] for i in rng.permutation(len(pairs))]    # band keys spread over lines and lanes
    return pairs


def _band_rows(L, pairs, seed):
    """the query: random bases with a gap in column 0; representative i: the query with m mismatches in columns
    1..m, gaps from column v + 1 on (valid = v), any base in column 0"""
    rng = np.random.default_rng(seed)
    q = BASES[rng.integers(0, 4, L)]
    q[0] = GAP
    comp = BASES[(np.searchsorted(BASES, q) + 1) % 4]
    reps = np.tile(q, (len(pairs), 1))
    reps[:, 0] = ord('A')
    for i, (m, v) in enumerate(pairs):
        reps[i, 1:1 + m] = comp[1:1 + m]
        reps[i, 1 + v:] = GAP
    return q, reps


def _band_expected(pairs, nodes, thr, vmin, edge=None):
    """-b 1: the near set plus the smallest far unit, ordered by the exact ratio m / v then index.  edge = (m0, v0):
    the threshold is the distance of that key bit for bit, so near is m / v <= m0 / v0 (jc69 grows with the ratio, and
    equal ratios give the identical double)"""
    nt = _near_table(thr, sorted({v for _, v in pairs}))
    valid = [u for u, (m, v) in enumerate(pairs) if v >= vmin and 4 * m < 3 * v]
    order = sorted(valid, key=lambda u: (Fraction(*pairs[u]), u))
    if edge is None:
        near = [pairs[u][0] <= nt[pairs[u][1]] for u in order]
    else:
        near = [Fraction(*pairs[u]) <= Fraction(*edge) for u in order]
    return expected_observed(order, near, lambda u: [(nodes[u], jc69(*pairs[u]))], 1)


def test_jc69_guard_band():
    """Designed keys on the edges of the fixed-point gate and inside its band, at -b 1, for seven thresholds; then one
    more threshold equal to the device's distance of a designed band key, so that the fp64 comparison in the band
    decides on equality (`dist <= threshold`: the key is near)."""
    from apples_b200 import _lib, fasta, synth
    from apples_b200.tree import BackboneTree
    n_rep = 320
    tree = BackboneTree.from_newick(synth.random_tree(n_rep, seed=606))
    nodes = tree.leaf_ids.tolist()
    names = [tree.label[u] for u in nodes]
    node_arr = np.array(nodes, np.int32)
    csr = np.arange(n_rep + 1, dtype=np.int32)
    runs = [('fp4', 33816, 1, 0), ('intpipe', 33816, 0, 0), ('intpipe', 65535, 0, 0), ('stash', 33816, 1, 4),
            ('bytes', 33816, None, 0)]
    band = {}
    for tag, L, mode, slot_cap in runs:
        pairs = _designed_pairs(L, n_rep, L)
        assert len(pairs) == n_rep, len(pairs)
        q, reps = _band_rows(L, pairs, L)
        vmin = overlap_vmin(L, 0.001)
        # fp64 and exact verdicts agree because no designed distance lies within 4 ulp of a threshold
        for thr in BAND_THRESHOLDS:
            nt = _near_table(thr, sorted({v for _, v in pairs}))
            for m, v in pairs:
                d = jc69(m, v)
                if np.isfinite(thr) and thr >= 0:
                    assert abs(d - thr) >= 4 * np.spacing(thr), (m, v, thr)
                assert (d <= thr) == (m <= nt[v]), (m, v, thr)
        if tag in ('fp4', 'intpipe'):
            for thr in BAND_THRESHOLDS:
                p_lo, p_hi = make_gate(thr)
                nt = _near_table(thr, sorted({v for _, v in pairs}))
                inb = [(m, v) for m, v in pairs if v >= vmin and p_lo * v < (m << 16) < p_hi * v]
                band.setdefault(thr, [0, 0, 0])
                band[thr][0] += len(inb)
                band[thr][1] += sum(m <= nt[v] for m, v in inb)
                band[thr][2] += sum(m > nt[v] for m, v in inb)
        qmat = np.tile(q, (3, 1))
        pl = _placer(tree, mode)
        try:
            if tag == 'bytes':
                # an exotic byte where the query has a gap: byte mode, select_kernel<SEL_NUCW>, the same counts
                exotic = reps.copy()
                exotic[::3, 0] = ord('?')
                pl.set_reference_bytes(fasta.NUC, L, names, exotic, node_arr, csr, csr[:-1])
            else:
                packed = fasta.pack_nucleotide(reps)
                pl.set_reference_arrays(fasta.NUC, L, names, packed, node_arr, packed, csr, csr[:-1])
            if slot_cap:
                pl.set_limits(slot_cap=slot_cap)
            pq = pl.pack_queries(qmat)
            keys, kind = pl.count_keys(pq, _lib.make_params())
            sh = 32 if kind == 1 else 16
            k64 = keys.astype(np.uint64)
            want = np.array([m | (v << sh) for m, v in pairs], np.uint64)
            assert (k64 == want[None, :]).all(), tag
            assert kind == (1 if tag == 'bytes' else 0)
            overflow = 0
            for thr in BAND_THRESHOLDS:
                params = _lib.make_params('FM', 'MLSE', base_observation_threshold=1, filt_threshold=thr)
                pl.timings(reset=True)
                count, node, dist = pl.observed_sets(params, packed=pq, cap=512)
                t = pl.timings()
                overflow += t['overflow_queries']
                out = pl.place_packed(pq, None, params)
                _, V, _ = pl.last_counts(len(qmat))
                obs, st, _, _ = _band_expected(pairs, nodes, thr, vmin)
                check_observed((tag, L, thr), [(obs, st)] * len(qmat), (count, node, dist, out[4], V), within_ulps)
                if thr == 0.2:
                    d_dev = dict(zip(node[0, :int(count[0])].tolist(), dist[0, :int(count[0])].tolist()))
            # the largest near band key at 0.2; its distance as the device computes it becomes the threshold
            p_lo, p_hi = make_gate(0.2)
            nt = _near_table(0.2, sorted({v for _, v in pairs}))
            u0 = max((u for u, (m, v) in enumerate(pairs) if p_lo * v < (m << 16) < p_hi * v and m <= nt[v]),
                     key=lambda u: Fraction(*pairs[u]))
            thr = d_dev[nodes[u0]]
            p_lo, p_hi = make_gate(thr)
            m0, v0 = pairs[u0]
            assert p_lo * v0 < (m0 << 16) < p_hi * v0
            params = _lib.make_params('FM', 'MLSE', base_observation_threshold=1, filt_threshold=thr)
            count, node, dist = pl.observed_sets(params, packed=pq, cap=512)
            out = pl.place_packed(pq, None, params)
            _, V, _ = pl.last_counts(len(qmat))
            obs, st, _, _ = _band_expected(pairs, nodes, thr, vmin, edge=(m0, v0))
            assert nodes[u0] in obs
            check_observed((tag, L, 'equal', thr), [(obs, st)] * len(qmat), (count, node, dist, out[4], V), within_ulps)
            if tag == 'stash':
                assert overflow > 0
        finally:
            pl.close()
    print('guard band keys per threshold (in band, near, far):', band)
    for thr in (1e-6, 0.02, 0.2, 10.0):
        assert band[thr][0] > 0, thr
    for thr in (0.0, -1.0):
        assert band[thr][0] == 0, thr                 # P_hi = 1 or P_hi = 0: the band holds no count key
    assert band[0.02][1] > 0 and band[0.02][2] > 0 and band[0.2][1] > 0 and band[0.2][2] > 0


# ------------------------------------------------------------------------------------- D. more than 1024 key lines
@pytest.fixture(scope='module')
def singleton_case():
    """40 000 leaves, each its own representative (1 250 key lines), 300 columns, 600 queries; the byte-mode twin holds
    '?' in the last 8 columns, where every query has a gap"""
    from apples_b200 import synth
    from apples_b200.tree import BackboneTree
    tree = BackboneTree.from_newick(synth.random_tree(40000, seed=7070))
    refs, states = synth.evolve_alignment(tree, 300, seed=7071)
    qd, _ = synth.make_queries(tree, states, 600, seed=7072)
    names = list(refs)
    rmat = np.stack([refs[n].view(np.uint8) for n in names]).copy()
    qmat = np.stack([np.asarray(s).view(np.uint8) for s in qd.values()]).copy()
    qmat[:, -8:] = GAP
    qmat[:30] = rmat[np.arange(30) * 1000]            # zero-distance queries
    qmat[:30, -8:] = GAP
    exotic = rmat.copy()
    hit = np.arange(0, len(names), 97)
    exotic[hit, -1 - hit % 8] = ord('?')
    return tree, names, rmat, exotic, qmat


def _singleton_placer(tree, names, rows, byte_mode, slot_cap):
    from apples_b200 import fasta
    pl = _placer(tree)
    n = len(names)
    nodes = np.array([tree.name_to_node[x] for x in names], np.int32)
    csr = np.arange(n + 1, dtype=np.int32)
    if byte_mode:
        pl.set_reference_bytes(fasta.NUC, rows.shape[1], names, rows, nodes, csr, csr[:-1])
    else:
        packed = fasta.pack_nucleotide(rows)
        pl.set_reference_arrays(fasta.NUC, rows.shape[1], names, packed, nodes, packed, csr, csr[:-1])
    if slot_cap:
        pl.set_limits(slot_cap=slot_cap)
    return pl


def test_rows_of_more_than_1024_key_lines(singleton_case):
    from apples_b200 import _lib
    tree, names, rmat, exotic, qmat = singleton_case
    n_rep, L = len(names), rmat.shape[1]
    n_kl = (n_rep + 31) // 32
    assert n_kl > 1024, n_kl
    nodes = np.array([tree.name_to_node[x] for x in names])
    vmin = overlap_vmin(L, 0.001)
    pl = _singleton_placer(tree, names, rmat, False, 0)
    try:
        pq = pl.pack_queries(qmat)
        keys, kind = pl.count_keys(pq, _lib.make_params())
    finally:
        pl.close()
    assert kind == 0
    m_all, v_all = (keys & 0xffff).astype(np.int64), (keys >> 16).astype(np.int64)
    for thr in (0.2, -1.0):
        nt = _near_table(thr, range(L + 1))
        mmax = np.array([nt[v] for v in range(L + 1)])
        for b in (25, 1000):
            exp = []
            for qi in range(len(qmat)):
                m, v = m_all[qi], v_all[qi]
                valid = np.flatnonzero((v >= vmin) & (4 * m < 3 * v))
                # m / v as doubles orders exactly: distinct ratios of counts <= 65 535 differ by more than 2e-10
                order = valid[np.lexsort((valid, m[valid] / v[valid]))]
                near = m[order] <= mmax[v[order]]
                obs, st, _, _ = expected_observed(order, near, lambda u: [(int(nodes[u]), jc69(int(m[u]), int(v[u])))], b)
                exp.append((obs, st))
            got = {}
            for slot_cap in (0, 32):
                for byte_mode in (False, True):
                    pl = _singleton_placer(tree, names, exotic if byte_mode else rmat, byte_mode, slot_cap)
                    try:
                        params = _lib.make_params('FM', 'MLSE', base_observation_threshold=b, filt_threshold=thr)
                        pl.timings(reset=True)
                        count, node, dist = pl.observed_sets(params, packed=pq, cap=4096)
                        t = pl.timings()
                        out = pl.place_packed(pq, None, params)
                        _, V, _ = pl.last_counts(len(qmat))
                    finally:
                        pl.close()
                    tag = ('lines', thr, b, slot_cap, byte_mode)
                    assert (t['key_lines_read'] > 0) != byte_mode, (tag, t)
                    big = max(len(o) for o, _ in exp) > (slot_cap or 256)
                    assert (t['overflow_queries'] > 0) == big, (tag, t)
                    check_observed(tag, exp, (count, node, dist, out[4], V), within_ulps)
                    got[byte_mode] = (count, node, dist, out)
                # the twin: the same sets, distances and placements bit for bit
                (c1, n1, d1, o1), (c0, n0, d0, o0) = got[False], got[True]
                assert np.array_equal(c1, c0) and np.array_equal(n1, n0)
                for a, c in zip(o1, o0):
                    assert a.tobytes() == c.tobytes()
