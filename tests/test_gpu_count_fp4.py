"""GPU (-m gpu): the block-scaled fp4 count kernel (dense_fp4_kernel, tcgen05.mma kind::mxf4 with all scale factors 1.0).

The kernel is only correct if the fp32 accumulators of the fp4 tensor-core path sum small integers EXACTLY:
D1 = 3 match - mismatch reaches 3 L and -L, D2 = valid reaches L.  Fewer accumulator bits than fp32's 24 would show
first on one-tile launches whose rows sit at those extremes (all match, all mismatch), alternate between them, or mix
them with gaps, so those are checked up to the kernel's length limit FP4_MAX_L.  Then keys and line minima are checked
bit for bit against numpy on the kernel's own edges: 128-query and 224-representative tiles, 64-site stages (an odd
word count pads the last stage with gap sites), the length limit on either side and ragged sub-batches.
"""
import os
import re

import numpy as np
import pytest

from tests.test_gpu_count_kernels import BASES, GAP, TC_MAX_L, _anchor, _assert_keys, _expected_keys, _nuc_rows, _placer, \
    _set_singletons
from tests.test_gpu_line_minima import _minima_np, _vmin

pytestmark = pytest.mark.gpu

_SRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'apples_b200', 'csrc', 'dense_tc.cu')
FP4_MAX_L = min(int(re.search(r'#define FP4_MAX_L_V (\d+)', open(_SRC).read()).group(1)), TC_MAX_L)


def _count(L, r, qs, overlap=0.001, max_subbatch=0):
    """keys, line minima and timings of each query block of qs against the representatives r (dense mode 1)"""
    from apples_b200 import _lib, fasta
    params = _lib.make_params(overlap_frac=overlap)
    pl = _placer(1)
    out = []
    try:
        _set_singletons(pl, fasta.NUC, L, fasta.pack_nucleotide(r))
        if max_subbatch:
            pl.set_limits(max_subbatch=max_subbatch)
        for q in qs:
            pl.timings(reset=True)
            keys, kind, mins = pl.count_keys(fasta.pack_nucleotide(q), params, line_minima=True)
            assert kind == 0
            out.append((keys.copy(), mins.copy(), pl.timings()))
    finally:
        pl.close()
    return out


def _check(L, r, qs, overlap=0.001, max_subbatch=0, tag=''):
    vmin = _vmin(L, overlap)
    res = _count(L, r, qs, overlap, max_subbatch)
    for q, (keys, mins, t) in zip(qs, res):
        _assert_keys(keys, _expected_keys(q, r, 16), 16, '%s nq=%d' % (tag, len(q)))
        exp = _minima_np(keys, vmin)
        bad = np.argwhere(mins != exp)
        assert not bad.size, '%s nq=%d: %d line minima wrong, first %s' % (tag, len(q), len(bad), bad[0])
        fp4 = L <= FP4_MAX_L
        assert t['fp4_launches'] == (t['rep_distance_launches'] if fp4 else 0), (tag, L, t)
        assert t['tensor_core_launches'] == (t['rep_distance_launches'] if L <= TC_MAX_L else 0), (tag, L, t)
    return res


# ------------------------------------------------------------------------------------- exact fp32 accumulation (one tile)
def _extreme_rows(L, side):
    """rows whose pair counts sit at the ends of the accumulator ranges, and mixtures of them"""
    a = _anchor(L)
    comp = BASES[(np.searchsorted(BASES, a) + 1) % 4]        # mismatches the anchor at every site
    s = np.arange(L)
    rows = [a, comp, np.full(L, GAP, np.uint8)]
    if side == 'q':
        alt = np.where(s % 2 == 0, a, comp)                    # match, mismatch, match, ...
        blocks = np.where((s // 4096) % 2 == 0, a, comp)       # long runs: D1 climbs, then falls
        gaps = a.copy()
        gaps[s % 3 == 0] = GAP
        tail = a.copy()
        tail[L // 2:] = GAP                                    # half the row is gap
        head = comp.copy()
        head[:L // 3] = GAP
        rows += [alt, blocks, gaps, tail, head]
    else:
        late = a.copy()
        late[: L - L // 4] = comp[: L - L // 4]                 # mismatches first, the matches at the end
        rows += [late]
    return np.stack(rows)


@pytest.mark.parametrize('L', [5000, 5462, 21846, 33816])
def test_fp4_accumulation_is_exact(L):
    """All-match pairs (D1 = 3 L), all-mismatch pairs (D1 = -L), alternating and long-run mixtures and gaps, in one
    128 x 224 tile, against exact counts.  An accumulator that kept fewer bits than fp32 would lose units once D1
    passes 2^14 (L = 5000 stays below, 5462 is above) or 2^16 (L = 21 846), and the test names the first pair whose
    counts differ."""
    if L > FP4_MAX_L:
        pytest.skip('beyond the fp4 kernel (FP4_MAX_L = %d)' % FP4_MAX_L)
    rng = np.random.default_rng(L)
    q = np.concatenate([_extreme_rows(L, 'q'), _nuc_rows(8, L, rng, 'q')])
    r = np.concatenate([_extreme_rows(L, 'r'), _nuc_rows(8, L, rng, 'r')])
    keys = _check(L, r, [q], tag='L=%d' % L)[0][0]
    assert (keys >> 16).max() == L and (keys & 0xffff).max() == L


# ------------------------------------------------------------------------------------------------ tile and stage edges
@pytest.mark.parametrize('n_rep', [223, 224, 225, 447, 448, 449])
def test_fp4_keys_across_tile_shapes(n_rep):
    """127 / 128 / 129 queries (one and two 128-row tiles) x 223 .. 449 representatives (one to three 224-row tiles)."""
    L = 97
    rng = np.random.default_rng(n_rep)
    r = _nuc_rows(n_rep, L, rng, 'r')
    _check(L, r, [_nuc_rows(nq, L, rng, 'q') for nq in (127, 128, 129)], tag='n_rep=%d' % n_rep)


@pytest.mark.parametrize('L', [1, 32, 33, 63, 64, 65, 129, 4999, 5000])
def test_fp4_keys_across_lengths(L):
    """one word, a whole and a partial 64-site stage, odd and even word counts, the lengths around the benchmark's."""
    rng = np.random.default_rng(2000 + L)
    _check(L, _nuc_rows(225, L, rng, 'r'), [_nuc_rows(129, L, rng, 'q')], tag='L=%d' % L)


@pytest.mark.parametrize('dL', [0, 1])
def test_fp4_length_limit(dL):
    """FP4_MAX_L runs the fp4 kernel; one column more runs the next kernel (kind::i8, or the integer pipes beyond
    33 816 columns), with the same keys."""
    L = FP4_MAX_L + dL
    rng = np.random.default_rng(L)
    _check(L, _nuc_rows(225, L, rng, 'r'), [_nuc_rows(129, L, rng, 'q')], tag='L=%d' % L)


@pytest.mark.parametrize('overlap', [0.001, 0.5])
def test_fp4_ragged_sub_batches(overlap):
    """1000 queries as 384-query sub-batches and a ragged last one of 232, against 3 x 224 - 1 representatives, the
    query images and key matrix reused across them; with overlap 0.5 the line minima skip the keys under the overlap
    gate."""
    L = 300
    rng = np.random.default_rng(1000)
    q, r = _nuc_rows(1000, L, rng, 'q'), _nuc_rows(671, L, rng, 'r')
    res = _check(L, r, [q], overlap=overlap, max_subbatch=384, tag='overlap=%g' % overlap)
    assert res[0][2]['rep_distance_launches'] == 3
