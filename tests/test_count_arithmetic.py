"""CPU: the integer arithmetic the count kernels rely on, with the constants parsed from the CUDA sources, so that a
change of a constant that breaks an overflow bound fails here before any GPU run.

* dense_tc.cu decodes one s32 accumulator S = 63503 * match - mismatch per pair; the decode adds 63502 in int32, which
  bounds the alignment length the tensor-core kernel may take (TC_MAX_L).
* dense_aa_kernel sums 22-bit fixed-point limbs in uint32 registers and folds them into 64-bit totals every 16 stages;
  no limb sum may wrap in between.
"""
import os
import re

import numpy as np

from tests import util

CSRC = os.path.join(util.ROOT, 'apples_b200', 'csrc')
INT32_MAX = 2 ** 31 - 1


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _const(src, name):
    m = re.search(r'constexpr int %s = (\d+);' % name, src)
    assert m, name
    return int(m.group(1))


def _tc_constants():
    src = _src('dense_tc.cu')
    return _const(src, 'TC_W'), _const(src, 'TC_MAX_L')


def _decode(S, tc_w):
    """dense_tc_kernel's epilogue in int32 / uint32 arithmetic: (match, mismatch, valid)."""
    S = np.asarray(S, np.int64)
    t = S + (tc_w - 1)
    assert (t <= INT32_MAX).all() and (t >= -2 ** 31).all(), 'S + (TC_W - 1) leaves int32'
    match = (t & 0xffffffff) // tc_w                  # (uint32_t)(S + (TC_W - 1)) / (uint32_t)TC_W
    prod = ((tc_w - 1) * match) & 0xffffffff          # (int)((TC_W - 1) * match) - S, as uint32
    prod = np.where(prod > INT32_MAX, prod - 2 ** 32, prod)
    mism = (prod - S) & 0xffffffff
    return match, mism, match + mism


def test_tensor_core_embedding_contributions():
    """The simplex embedding of tc_image_kernel: a matching site adds TC_W - 1, a mismatching one -1, a gap 0."""
    tc_w, _ = _tc_constants()
    src = _src('dense_tc.cu')
    assert '0x82u : 0x7eu' in src                      # -126 / +126
    api = _src('api.cu')
    assert re.search(r'launch_tc_image\(\(const uint32_t\*\)d_q, nb, .*, 125, ', api)
    assert re.search(r'launch_tc_image\(\(const uint32_t\*\)ctx->reps_rm\.p, .*, 127, ', api)

    def vec(code, vw):
        lo, hi = code & 1, code >> 1
        x, y, z = (-126 if hi else 126), (-126 if lo else 126), (-126 if lo ^ hi else 126)
        return np.array([x, y, z, vw], np.int64)

    for a in range(4):
        for b in range(4):
            d = int(vec(a, 125) @ vec(b, 127))
            assert d == (tc_w - 1 if a == b else -1), (a, b, d)
    assert tc_w - 1 == 3 * 126 ** 2 + 125 * 127


def test_tensor_core_decode_limit():
    tc_w, tc_max_l = _tc_constants()
    assert tc_w - 1 == 63503
    assert (tc_w - 1) * tc_max_l + (tc_w - 2) <= INT32_MAX < (tc_w - 1) * (tc_max_l + 1) + (tc_w - 2)
    # api.cu sends longer alignments to the integer-pipe kernel
    assert re.search(r'ctx->L > dense_tc_max_sites\(\)', _src('api.cu'))


def test_tensor_core_decode_exact():
    """Every (match, mismatch) split at valid = 0, 1 and TC_MAX_L, and a random sample below TC_MAX_L, decodes back."""
    tc_w, tc_max_l = _tc_constants()
    rng = np.random.default_rng(3)
    for valid in (0, 1, tc_max_l):
        match = np.arange(valid + 1, dtype=np.int64)
        mism = valid - match
        m, x, v = _decode((tc_w - 1) * match - mism, tc_w)
        assert (m == match).all() and (x == mism).all() and (v == valid).all()
    valid = rng.integers(0, tc_max_l + 1, 200000)
    match = (rng.random(valid.size) * (valid + 1)).astype(np.int64)
    mism = valid - match
    m, x, v = _decode((tc_w - 1) * match - mism, tc_w)
    assert (m == match).all() and (x == mism).all() and (v == valid).all()
    # the 32-bit key mismatch | valid << 16 holds both counts
    assert tc_max_l < 2 ** 16


def _blosum_inc():
    src = _src('blosum45.inc')
    vals = [float(x) for x in re.findall(r'-?\d+\.\d*(?:e-?\d+)?', src.split('\n', 1)[1])]
    assert len(vals) == 441
    return np.array(vals).reshape(21, 21)


def _limb_tables():
    """aa_build_tables: v = (uint64)(x * 2^43 + 0.5), high = v >> 22, low = v & (2^22 - 1)."""
    common = _src('common.cuh')
    limb, frac = _const(common, 'AA_LIMB'), _const(common, 'AA_FRAC')
    assert frac == 43
    assert '8796093022208.0 + 0.5' in _src('distance.cu')            # 2^43
    b = _blosum_inc()
    v = [[int(x * 8796093022208.0 + 0.5) for x in row] for row in b.tolist()]
    hi = np.array([[x >> limb for x in row] for row in v], np.int64)
    lo = np.array([[x & ((1 << limb) - 1) for x in row] for row in v], np.int64)
    return b, hi, lo


def _flush_sites():
    """sites between two folds of the limb sums in dense_aa_kernel: (c & F) == F -> F + 1 stages of AA_CH sites."""
    m = re.search(r'if \(\(c & (\d+)\) == \1 \|\| c \+ 1 == a\.n_chunks\)', _src('distance.cu'))
    assert m, 'dense_aa_kernel flush condition not found'
    return (int(m.group(1)) + 1) * _const(_src('common.cuh'), 'AA_CH')


def test_protein_limb_sums_cannot_wrap():
    b, hi, lo = _limb_tables()
    from oracle import apples_oracle as orc
    # the table the kernel carries is the oracle's BLOSUM45 with a zero gap row and column
    assert (b[:20, :20] == orc.BLOSUM45.reshape(20, 20)).all() and (b[20] == 0).all() and (b[:, 20] == 0).all()
    sites = _flush_sites()
    assert sites == 1024
    assert hi.max() == 3844397 and lo.max() == 4158118
    assert hi.max() * sites < 2 ** 32 and lo.max() * sites < 2 ** 32
    # the margin: the high limb sum of all-maximal sites wraps only after 1117 sites
    assert (2 ** 32 - 1) // hi.max() == 1117
    # the limbs recombine to the fixed-point value, whose rounding is at most 2^-44 per site
    v = (hi << 22) + lo
    assert (np.abs(v / 2.0 ** 43 - b) <= 2.0 ** -44).all()
