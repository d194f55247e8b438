"""GPU (-m gpu): the keys of the count stage, read straight out of the hot path (apples_count_keys), against exact counts
computed from the alignment BYTES -- not from the bit-planes, so the reference does not share the packer with the device.

The three count kernels are each checked where they go wrong: the tensor-core kernel (dense_tc_kernel, the default), the
integer-pipe kernel (dense_nuc_kernel<false>, dense mode 0 and every alignment beyond 33 816 columns), the byte-compare
fallback (beyond 65 535 columns, exotic reference bytes) and the protein kernel (dense_aa_kernel).  Shapes sit on the
edges of the tiles (256 x 256 tensor-core tiles, 128 x 64 integer-pipe tiles, 8 x 256 protein tiles), of the K pipeline
(3 stages of one 32-site word, 32-word image chunks, 64-site protein stages, the limb fold every 1024 sites) and of the
length limits (33 816 / 33 817 / 65 535 columns); rows at the first and last row of a tile are the extreme ones: all
match, all mismatch, all gap, gaps only in the last partial word, every (query, reference) base pair.

Contexts hold singleton clusters, so the representatives are exactly the given rows, and a 4-leaf tree; nothing is
placed.  Nucleotide keys must be bit-identical in both dense modes, and the kernel that ran is asserted from the
launch counters.  Protein keys are within 1e-9 relative of scoredist evaluated from exact pair counts with math.fsum.
"""
import math
import os
import types

import numpy as np
import pytest

from tests import util

pytestmark = pytest.mark.gpu

TC_MAX_L = 33816                 # longest alignment of the tensor-core kernel (dense_tc.cu TC_MAX_L)
GAP = ord('-')
BASES = np.frombuffer(b'ACGT', np.uint8)
AA_LETTERS = np.frombuffer(b'ARNDCQEGHILKMFPSTWYV', np.uint8)   # a2i order (distance.py:418-678)


def _placer(mode=None):
    from apples_b200.placer import GpuPlacer
    from apples_b200.tree import BackboneTree
    tree = BackboneTree.from_newick('((A:0.1,B:0.2):0.05,C:0.3,D:0.4);')
    pl = GpuPlacer(tree, None, tree.name_to_node, device=0)
    if mode is not None:
        pl.set_dense_mode(mode)
    return pl


def _set_singletons(pl, kind, L, packed_reps):
    n = packed_reps.shape[0]
    pl.set_reference_arrays(kind, L, ['r%d' % i for i in range(n)], packed_reps, np.full(n, -1, np.int32), packed_reps,
                            np.arange(n + 1, dtype=np.int32), np.arange(n, dtype=np.int32))


def _edge_rows(n, tiles):
    """row indices on tile edges, most important first: first and last row, then the rows either side of each tile
    boundary, then the second and second-to-last row"""
    pos = [0, n - 1]
    for t in tiles:
        pos += [t - 1, t]
    pos += [1, n - 2]
    out = []
    for p in pos:
        if 0 <= p < n and p not in out:
            out.append(p)
    return out


# --------------------------------------------------------------------------------------------------------- nucleotides
def _anchor(L):
    """a gap-free row shared by the query and the representative side"""
    return BASES[np.random.default_rng(L).integers(0, 4, L)]


def _nuc_special(name, L, side):
    a = _anchor(L)
    s = np.arange(L)
    if name == 'same':
        return a
    if name == 'comp':                         # A->C->G->T->A: every site mismatches
        return BASES[(np.searchsorted(BASES, a) + 1) % 4]
    if name == 'allgap':
        return np.full(L, GAP, np.uint8)
    if name == 'tailgap':                      # gaps only in the last (partial) 32-site word
        r = a.copy()
        r[(L - 1) // 32 * 32 if L % 32 else max(0, L - 5):] = GAP
        return r
    if name == 'pairs':                        # query s % 4 against reference s // 4 % 4: all 16 base pairs
        return BASES[s % 4] if side == 'q' else BASES[(s // 4) % 4]
    raise KeyError(name)


def _nuc_rows(n, L, rng, side):
    """n rows of L alignment bytes: random rows with 0 / 5 / 40 % gaps; the rows on tile edges are the special rows"""
    rows = BASES[rng.integers(0, 4, (n, L))]
    gap = rng.random((n, L)) < np.array([0.0, 0.05, 0.4])[np.arange(n) % 3][:, None]
    rows[gap] = GAP
    specials = (['same', 'allgap', 'tailgap', 'pairs', 'same', 'comp'] if side == 'q' else
                ['same', 'comp', 'allgap', 'tailgap', 'pairs', 'same'])
    for i, p in enumerate(_edge_rows(n, (64, 128, 256))):
        rows[p] = _nuc_special(specials[i % len(specials)], L, side)
    return rows


def _nuc_expected(q, r):
    """exact (mismatch, valid) of every pair, from the bytes (distance.py:733-737): one-hot products in float32, exact
    because every partial sum is an integer below 2^24"""
    qv, rv = (q != GAP).astype(np.float32), (r != GAP).astype(np.float32)
    valid = qv @ rv.T
    match = np.zeros_like(valid)
    for b in np.union1d(np.unique(q), np.unique(r)).tolist():
        if b != GAP:
            match += (q == b).astype(np.float32) @ (r == b).astype(np.float32).T
    valid, match = valid.astype(np.int64), match.astype(np.int64)
    return valid - match, valid


def _expected_keys(q, r, shift):
    mism, valid = _nuc_expected(q, r)
    assert valid.max() < (1 << shift)
    return mism.astype(np.uint64) | (valid.astype(np.uint64) << np.uint64(shift))


def _assert_keys(keys, exp, shift, tag):
    got = keys.astype(np.uint64)
    assert got.shape == exp.shape, (tag, got.shape, exp.shape)
    bad = np.argwhere(got != exp)
    if bad.size:
        i, j = bad[0]
        mask, sh = np.uint64((1 << shift) - 1), np.uint64(shift)
        raise AssertionError('%s: %d of %d keys wrong; first (query %d, representative %d): got mismatch %d valid %d, '
                             'expected %d %d' % (tag, len(bad), exp.size, i, j, int(got[i, j] & mask), int(got[i, j] >> sh),
                                                 int(exp[i, j] & mask), int(exp[i, j] >> sh)))


def _run_nuc(L, r, qs, max_subbatch=0, tag=''):
    """keys of each query block of qs against the representatives r, in dense mode 1 and 0; asserts the kernel that ran
    and returns {mode: [keys]}"""
    from apples_b200 import fasta, _lib
    params = _lib.make_params()
    out = {}
    for mode in (1, 0):
        pl = _placer(mode)
        try:
            _set_singletons(pl, fasta.NUC, L, fasta.pack_nucleotide(r))
            if max_subbatch:
                pl.set_limits(max_subbatch=max_subbatch)
            out[mode] = []
            for q in qs:
                pl.timings(reset=True)
                keys, kind = pl.count_keys(fasta.pack_nucleotide(q), params)
                t = pl.timings()
                assert kind == 0, (tag, kind)
                assert t['rep_distance_launches'] >= 1, (tag, t)
                tc = mode == 1 and L <= TC_MAX_L
                assert t['tensor_core_launches'] == (t['rep_distance_launches'] if tc else 0), (tag, mode, L, t)
                out[mode].append((keys.copy(), t))
        finally:
            pl.close()
    for q, (k1, _), (k0, _) in zip(qs, out[1], out[0]):
        exp = _expected_keys(q, r, 16)
        _assert_keys(k1, exp, 16, '%s nq=%d mode 1' % (tag, len(q)))
        _assert_keys(k0, exp, 16, '%s nq=%d mode 0' % (tag, len(q)))
        assert k1.tobytes() == k0.tobytes()
    return out


@pytest.mark.parametrize('L', [1, 31, 32, 33, 96, 97, 128, 129, 1024, 1025, 1056, 1057])
def test_nucleotide_keys_across_lengths(L):
    """n_w = 1..4 words against the 3 tensor-core stages, plane rows rounded to 4 words, the 32-word chunk of
    tc_image_kernel and the 32-word stage of the integer-pipe kernel (DT_WC), at 257 x 257 (partial tiles of both)."""
    rng = np.random.default_rng(1000 + L)
    _run_nuc(L, _nuc_rows(257, L, rng, 'r'), [_nuc_rows(257, L, rng, 'q')], tag='L=%d' % L)


@pytest.mark.parametrize('L', [TC_MAX_L, TC_MAX_L + 1, 65535])
def test_nucleotide_keys_at_the_length_limits(L):
    """33 816 columns: the longest the tensor-core decode takes (all-match pairs reach S = 63503 * 33 816); 33 817: the
    context must switch to the integer-pipe kernel; 65 535: the last length of 16-bit counts, where D and E1 of the
    integer-pipe accumulator (mismatch + one-sided sites, one-sided sites) reach 65 535 (all-gap against gap-free rows)."""
    rng = np.random.default_rng(L)
    q, r = _nuc_rows(257, L, rng, 'q'), _nuc_rows(257, L, rng, 'r')
    out = _run_nuc(L, r, [q], tag='L=%d' % L)
    keys = out[1][0][0]
    mism, valid = keys & 0xffff, keys >> 16
    assert valid.max() == L and mism.max() == L      # the all-match and all-mismatch pairs are there


@pytest.mark.parametrize('n_rep', [1, 255, 256, 257])
def test_nucleotide_keys_across_tile_shapes(n_rep):
    """{1, 255, 256, 257} queries x representatives: partial 256 x 256 tensor-core tiles, partial 128 x 64 integer-pipe
    tiles."""
    L = 97
    rng = np.random.default_rng(n_rep)
    r = _nuc_rows(n_rep, L, rng, 'r')
    _run_nuc(L, r, [_nuc_rows(nq, L, rng, 'q') for nq in (1, 255, 256, 257)], tag='n_rep=%d' % n_rep)


@pytest.mark.parametrize('max_subbatch', [0, 1000])
def test_nucleotide_keys_many_tiles_and_sub_batches(max_subbatch):
    """4097 queries x 3073 representatives at 100 columns: 17 x 13 tensor-core tiles, more than there are SMs, so the
    persistent CTAs loop over tiles with stage and accumulator parity carried across them, and the last band and column
    of 12 x 12 super-tiles are thin.  With max_subbatch = 1000 the batch runs as 896-query sub-batches and a ragged last
    one of 513, reusing the query images and the key matrix."""
    L = 100
    rng = np.random.default_rng(4097)
    q, r = _nuc_rows(4097, L, rng, 'q'), _nuc_rows(3073, L, rng, 'r')
    out = _run_nuc(L, r, [q], max_subbatch=max_subbatch, tag='max_subbatch=%d' % max_subbatch)
    for mode in (0, 1):
        assert out[mode][0][1]['rep_distance_launches'] == (5 if max_subbatch else 1)


@pytest.mark.parametrize('L', [65536, 70001])
def test_byte_mode_keys_beyond_16_bit_counts(L):
    """Beyond 65 535 columns the context runs the byte-compare fallback with 64-bit keys mismatch | valid << 32."""
    from apples_b200 import fasta, _lib
    rng = np.random.default_rng(L)
    q, r = _nuc_rows(65, L, rng, 'q'), _nuc_rows(70, L, rng, 'r')
    pl = _placer()
    try:
        _set_singletons(pl, fasta.NUC, L, fasta.pack_nucleotide(r))
        keys, kind = pl.count_keys(fasta.pack_nucleotide(q), _lib.make_params())
        t = pl.timings()
    finally:
        pl.close()
    assert kind == 1
    assert t['tensor_core_launches'] == 0 and t['fallback_queries'] == len(q)
    _assert_keys(keys, _expected_keys(q, r, 32), 32, 'L=%d' % L)
    assert (keys >> np.uint64(32)).max() == L


def _consensus(rows, groups):
    """PoolRepresentativeWorker.py:30-85: column-wise majority over [A, C, G, T, -], first maximum; bytes outside the
    alphabet count for nothing, so a column of them alone becomes 'A'"""
    alpha = np.frombuffer(b'ACGT-', np.uint8)
    out = np.empty((len(groups), rows.shape[1]), np.uint8)
    for g, members in enumerate(groups):
        cnt = (rows[members][:, :, None] == alpha).sum(axis=0)     # [L, 5]
        out[g] = alpha[np.argmax(cnt, axis=1)]
    return out


def test_byte_mode_keys_of_an_exotic_reference():
    """References holding '?', '.', '*' put the context in byte mode (apples_set_reference_bytes); its representatives
    are the device's consensus rows, checked against a numpy consensus through the keys."""
    from apples_b200 import fasta, _lib
    L, n_ref = 300, 90
    rng = np.random.default_rng(300)
    refs = _nuc_rows(n_ref, L, rng, 'r')
    exotic = np.frombuffer(b'?.*', np.uint8)
    hit = rng.random(refs.shape) < 0.05
    refs[hit] = exotic[rng.integers(0, 3, int(hit.sum()))]
    refs[:3, :40] = exotic[rng.integers(0, 3, (3, 40))]     # whole columns of exotic bytes in the first cluster
    rest = (3 + rng.permutation(n_ref - 3)).tolist()
    groups, i = [[0, 1, 2]], 0
    while i < len(rest):                                      # clusters of 1, 3, 5, 2, 4, 1, ... members
        s = [1, 3, 5, 2, 4][len(groups) % 5]
        groups.append(rest[i:i + s])
        i += s
    offs = np.cumsum([0] + [len(g) for g in groups]).astype(np.int32)
    members = np.concatenate([np.array(g, np.int32) for g in groups])
    reps = _consensus(refs, groups)
    assert (reps[0, :40] == ord('A')).all()
    q = _nuc_rows(37, L, rng, 'q')
    pl = _placer()
    try:
        pl.set_reference_bytes(fasta.NUC, L, ['r%d' % i for i in range(n_ref)], refs, np.full(n_ref, -1, np.int32),
                               offs, members)
        keys, kind = pl.count_keys(fasta.pack_nucleotide(q), _lib.make_params())
    finally:
        pl.close()
    assert kind == 1 and keys.shape == (37, len(groups))
    _assert_keys(keys, _expected_keys(q, reps, 32), 32, 'exotic reference')


# ------------------------------------------------------------------------------------------------------------- protein
def _blosum21():
    from oracle import apples_oracle as orc
    b = np.zeros((21, 21))
    b[:20, :20] = orc.BLOSUM45.reshape(20, 20)
    return b


def _aa_rows(n, L, rng, side, base):
    """n protein rows: mutants of `base` at 10 / 30 / 60 % of the sites with 0 / 5 / 40 % gaps (so that scoredist is
    mostly defined); the rows on tile edges are the special rows: identical to base, all gap, and half of the sites on
    the pair with the table's largest entry (tot / valid ~ 0.92: large limb sums, scoredist still defined)"""
    codes = np.tile(base, (n, 1))
    i = np.arange(n)
    mut = rng.random((n, L)) < np.array([0.1, 0.3, 0.6])[i % 3][:, None]
    codes[mut] = rng.integers(0, 20, int(mut.sum()))
    codes[rng.random((n, L)) < np.array([0.0, 0.05, 0.4])[(i // 3) % 3][:, None]] = 20
    b = _blosum21()
    a_max, b_max = np.unravel_index(np.argmax(b), b.shape)
    half = base.copy()
    half[::2] = a_max if side == 'q' else b_max
    specials = [base, np.full(L, 20), half] if side == 'q' else [base, half, np.full(L, 20)]
    for k, p in enumerate(_edge_rows(n, (8, 16, 128, 256) if side == 'q' else (128, 256))):
        codes[p] = specials[k % len(specials)]
    return np.where(codes == 20, GAP, AA_LETTERS[np.minimum(codes, 19)]).astype(np.uint8)


def _aa_codes(rows):
    lut = np.full(256, 20, np.int64)
    lut[AA_LETTERS] = np.arange(20)
    return lut[rows]


def _scoredist_expected(q, r, L, overlap):
    """distance.py:681-715 from exact per-pair counts: the 21 x 21 matrix of (query, reference) symbol pairs, its dot
    product with BLOSUM45 by math.fsum, the overlap gate and the correction in fp64"""
    b = _blosum21().ravel()
    qc, rc = _aa_codes(q), _aa_codes(r)
    nq, nr = len(qc), len(rc)
    idx = (np.arange(nq * nr, dtype=np.int64).reshape(nq, nr, 1) * 441 + qc[:, None, :] * 21 + rc[None, :, :]).ravel()
    counts = np.bincount(idx, minlength=nq * nr * 441).reshape(nq, nr, 21, 21)
    valid = counts[:, :, :20, :20].sum(axis=(2, 3))
    flat = counts.reshape(nq, nr, 441)
    d = np.empty((nq, nr))
    for i in range(nq):
        for j in range(nr):
            v = int(valid[i, j])
            if v == 0 or v / L < overlap:
                d[i, j] = -1.0
                continue
            nz = np.flatnonzero(flat[i, j])
            tot = math.fsum((flat[i, j, nz] * b[nz]).tolist())
            x = 1.0 - tot / v
            d[i, j] = -1.0 if 0.0 >= x else -math.log(x) * 1.3
    return d, valid


def _assert_scoredist(got, q, r, L, overlap, tag):
    exp, valid = _scoredist_expected(q, r, L, overlap)
    assert got.shape == exp.shape
    gate = exp == -1.0
    assert ((got == -1.0) == gate).all(), (tag, np.argwhere((got == -1.0) != gate)[:5].tolist())
    rel = np.abs(got - exp) / np.maximum(np.abs(exp), 1e-300)
    worst = np.unravel_index(np.argmax(np.where(gate, 0.0, rel)), rel.shape)
    assert rel[worst] <= 1e-9 or gate[worst], (tag, worst, got[worst], exp[worst])
    return exp, valid


def _run_aa(L, r, qs, overlap=0.001):
    from apples_b200 import fasta, _lib
    params = _lib.make_params(overlap_frac=overlap)
    pl = _placer()
    try:
        _set_singletons(pl, fasta.AA, L, fasta.pack_protein(r))
        res = []
        for q in qs:
            keys, kind = pl.count_keys(fasta.pack_protein(q), params)
            assert kind == 2
            res.append(keys.copy())
    finally:
        pl.close()
    return res


@pytest.mark.parametrize('L', [1, 15, 16, 17, 63, 64, 65, 1023, 1024, 1025, 1088, 2049, 4097])
def test_protein_keys_across_lengths(L):
    """Partial and whole 64-site stages; the limb sums are folded into 64-bit totals every 16 stages (1024 sites), so
    1088, 2049 and 4097 sites run several fold groups with a partial last one.  17 queries x 257 representatives."""
    rng = np.random.default_rng(2000 + L)
    base = rng.integers(0, 20, L)
    q, r = _aa_rows(17, L, rng, 'q', base), _aa_rows(257, L, rng, 'r', base)
    (keys,) = _run_aa(L, r, [q])
    exp, _ = _assert_scoredist(keys, q, r, L, 0.001, 'L=%d' % L)
    # mostly defined distances, not the -1 gate; with a single site a pair of different residues is defined only when its
    # table entry is below 1
    assert (exp > 0).sum() > (exp.size // 4 if L > 1 else 0)
    if L >= 64:
        # the pairs of `half` rows: tot / valid = max(BLOSUM45) * ceil(L / 2) / L ~ 0.92
        x = 1.0 - _blosum21().max() * ((L + 1) // 2) / L
        assert np.isclose(keys, -math.log(x) * 1.3, rtol=1e-9, atol=0.0).sum() >= 4


@pytest.mark.parametrize('n_rep', [1, 255, 256, 257])
def test_protein_keys_across_tile_shapes(n_rep):
    """{1, 7, 8, 9, 17} queries x {1, 255, 256, 257} representatives: partial 8 x 256 tiles, at 1025 sites."""
    L = 1025
    rng = np.random.default_rng(n_rep)
    base = rng.integers(0, 20, L)
    r = _aa_rows(n_rep, L, rng, 'r', base)
    qs = [_aa_rows(nq, L, rng, 'q', base) for nq in (1, 7, 8, 9, 17)]
    for q, keys in zip(qs, _run_aa(L, r, qs)):
        _assert_scoredist(keys, q, r, L, 0.001, 'nq=%d n_rep=%d' % (len(q), n_rep))


def test_protein_overlap_gate():
    """distance.py:698-699: a pair counts only if valid / L >= overlap_frac; queries with exactly vmin - 1, vmin and
    vmin + 1 non-gap sites against gap-free representatives."""
    L, overlap = 1025, 0.5
    vmin = next(v for v in range(1, L + 1) if not v / L < overlap)
    rng = np.random.default_rng(7)
    base = rng.integers(0, 20, L)
    codes = np.tile(base, (40, 1))                 # gap-free mutants of base at 20 % of the sites: defined distances
    mut = rng.random(codes.shape) < 0.2
    codes[mut] = rng.integers(0, 20, int(mut.sum()))
    r = AA_LETTERS[codes]
    q = []
    for v in (vmin - 1, vmin, vmin + 1):
        row = AA_LETTERS[base].copy()
        row[rng.permutation(L)[v:]] = GAP
        q.append(row)
    q = np.array(q)
    (keys,) = _run_aa(L, r, [q], overlap)
    exp, valid = _assert_scoredist(keys, q, r, L, overlap, 'overlap gate')
    assert (valid == np.array([vmin - 1, vmin, vmin + 1])[:, None]).all()
    assert (keys[0] == -1.0).all() and (keys[1:] >= 0.0).all()


# -------------------------------------------------------------------------------------------------------- end to end
@pytest.mark.parametrize('L', [TC_MAX_L, TC_MAX_L + 1, 65535])
def test_placements_at_the_length_limits(L, workdir):
    """A 40-leaf backbone and 5 queries through place_batch on either side of the tensor-core limit and at the last
    length of 16-bit counts, against the oracle."""
    from apples_b200 import synth
    from apples_b200.placer import GpuPlacer, place_batch
    from apples_b200.reference import ReducedReference
    from apples_b200.tree import BackboneTree
    from tests.test_gpu_parity import _oracle_check
    nwk = synth.random_tree(40, seed=L, mean_edge=0.03)
    tfp = os.path.join(workdir, 'limit_%d.nwk' % L)
    with open(tfp, 'w') as f:
        f.write(nwk)
    tree = BackboneTree.from_newick(tfp)
    refs, states = synth.evolve_alignment(tree, L, seed=L + 1, edge_frac=0.0)
    qd, _ = synth.make_queries(tree, states, 5, seed=L + 2, edge_frac=0.0)
    queries = [(k, v, None) for k, v in qd.items()]
    ref = ReducedReference(None, False, None, 0.2, 1, tree=tree, refs=refs)
    ref.set_baseobs(25)
    opt = types.SimpleNamespace(method_name='OLS', criterion_name='MLSE', negative_branch=False, base_observation_threshold=25,
                                filt_threshold=0.2, minimum_alignment_overlap=0.001, exclude_intplace=False)
    pl = GpuPlacer(tree, ref, tree.name_to_node, device=0)
    try:
        res = place_batch(ref, opt, tree.name_to_node, queries, placer=pl)
        t = pl.timings()
    finally:
        pl.close()
    assert (t['tensor_core_launches'] > 0) == (L <= TC_MAX_L), t
    assert _oracle_check('limit%d' % L, tree, tfp, refs, ref.representatives, queries, res, opt) <= 1
