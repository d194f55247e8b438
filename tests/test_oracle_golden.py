"""CPU: the oracle (oracle/apples_oracle.py) against the committed golden vectors, which were produced by the
unmodified reference (oracle/gen_golden.py), and against the reference's own known answers (SURVEY.md 8c)."""
import json

import numpy as np
import pytest

from tests import util
from oracle import apples_oracle as orc

CASES = util.golden_names()
# the full grid is large; keep the CPU suite to a few minutes
FAST = [c for c in CASES if c.startswith('small_')] + [
    'c2_matrix_FM_MLSE', 'c2_matrix_OLS_HYBRID_f100', 'c2_matrix_BME_ME_b5', 'c2_matrix_BE_MLSE_neg',
    'c1_align_FM_MLSE', 'c1_align_special', 'c1_align_special_exclude', 'c1_align_FM_MLSE_f045_b5',
    'syn300_FM_MLSE_pos', 'syn300_OLS_MLSE_neg', 'syn300_BME_HYBRID_pos', 'syn300_BE_ME_pos',
]


@pytest.mark.parametrize('case', FAST)
def test_oracle_reproduces_reference(case, workdir):
    ci = util.CaseInputs(case, workdir)
    ctx = ci.oracle_context()
    for (qname, qseq, row), rec in zip(ci.queries, ci.g['queries']):
        det = {}
        res, status = ctx.runquery(qname, qseq, dict(row) if row else None, detail=det)
        p = res['placements'][0]['p'][0]
        exp = [util.unhex(x) for x in rec['p']]
        assert p == exp, (case, qname)
        assert [isinstance(a, int) for a in p] == [isinstance(b, int) for b in exp]  # int 0 vs float 0.0
        assert status == rec['status']
        assert res['placements'][0]['n'] == [rec['out_name']]
        if 'edges' in rec:
            got = {str(k): [float(v[0]).hex() if not isinstance(v[0], int) else v[0],
                            float(v[1]).hex() if not isinstance(v[1], int) else v[1], float(v[2]).hex()]
                   for k, v in det['edges'].items()}
            exp_e = {k: [v[0], v[1], v[2]] for k, v in rec['edges'].items()}
            assert got == exp_e
            assert det['num_nodes'] == rec['num_nodes']


def test_protein_case(workdir):
    ci = util.CaseInputs('c3_prot_FM_MLSE', workdir)
    ctx = ci.oracle_context()
    for (qname, qseq, row), rec in list(zip(ci.queries, ci.g['queries']))[:3]:
        res, status = ctx.runquery(qname, qseq, None)
        assert res['placements'][0]['p'][0] == [util.unhex(x) for x in rec['p']]
    sd = ci.g['scoredist_q0']
    for n, d in zip(sd['refs'], sd['d']):
        assert orc.scoredist(ci.queries[0][1], ci.refs[n], 0.001) == util.unhex(d)


def test_dist_mat_known_answer(workdir):
    """data/dist.mat == jc69 of the example alignment to 8 decimals (SURVEY.md section 4 / 8c item 1)."""
    ci = util.CaseInputs('c1_align_FM_MLSE', workdir)
    rows = util.read_dismat(util.gunzip_to('dist.mat', workdir))
    worst = 0.0
    for (qname, qseq, _), (mname, _, row) in zip(ci.queries, rows):
        assert qname == mname
        for tag, v in row.items():
            if tag in ci.refs:
                worst = max(worst, abs(orc.jc69(qseq, ci.refs[tag], 0.001) - v))
    assert worst <= 5.1e-9


def test_counts_golden(workdir):
    """mismatch / valid counts of config 1 (distance.py:733-737) and jc69_from_counts == jc69."""
    ci = util.CaseInputs('c1_align_FM_MLSE', workdir)
    names = ci.g['ref_names']
    for qi, (qname, qseq, _) in enumerate(ci.queries[:3]):
        for ri in range(0, len(names), 7):
            m, v = orc.nuc_counts(qseq, ci.refs[names[ri]])
            assert [m, v] == ci.g['counts'][qi][ri]
            a = orc.jc69(qseq, ci.refs[names[ri]], 0.001)
            b = orc.jc69_from_counts(m, v, len(qseq), 0.001)
            assert a == b


def test_survey_known_answers(workdir):
    """SURVEY.md section 8(c) items 2 and 3."""
    g = util.load_golden('c2_matrix_FM_MLSE')
    first = g['queries'][0]
    assert first['name'] == 'L379065'
    p = [util.unhex(x) for x in first['p']]
    assert p == [334, 0.0413224794640108, 1, 0.09494873497159563, 0.10096288502840432]
    edges = [q['p'][0] for q in g['queries']]
    assert edges == [334, 634, 547, 73, 547, 406, 506, 604, 263, 619]
    s = util.load_golden('small_FM_MLSE_pos')['queries'][0]
    assert [util.unhex(x) for x in s['p']] == [3, 0.0, 1, 0.1, 0.10000000000000005]
    s = util.load_golden('small_FM_ME_pos')['queries'][0]
    assert [util.unhex(x) for x in s['p']] == [4, 3.2704081632653055, 1, 0.2, 0]
    s = util.load_golden('small_BE_HYBRID_pos')['queries'][0]
    assert [util.unhex(x) for x in s['p']] == [6, 0.29090909090909056, 1, 0.2, 0.045454545454545414]


def test_alignment_and_matrix_agree():
    """config 1 and config 2 choose identical edges (SURVEY.md section 4)."""
    a = util.load_golden('c1_align_FM_MLSE')
    b = util.load_golden('c2_matrix_FM_MLSE')
    # (scores differ slightly: the observed sets are cut at different ties, SURVEY.md section 7 "hard parts")
    assert [q['p'][0] for q in a['queries']] == [q['p'][0] for q in b['queries']]


def test_golden_recipe_reproduces_committed_vectors():
    """oracle/gen_golden.py --check: the committed recipe, fed with the committed input fixtures and run against the
    UNMODIFIED reference, regenerates every tests/golden/*.json byte for byte (and asserts oracle == reference bit for
    bit on the way).  Catches drift between recipe, fixtures and oracle; runs only where the environment variable
    APPLES_REFERENCE names a checkout of the original APPLES (its apples/ package and data/ directory)."""
    import os
    import subprocess
    import sys
    if not os.path.isdir(os.path.join(os.environ.get('APPLES_REFERENCE', ''), 'apples')):
        pytest.skip('needs the original APPLES sources: set APPLES_REFERENCE to a checkout of them')
    r = subprocess.run([sys.executable, os.path.join(util.ROOT, 'oracle', 'gen_golden.py'), '--check'],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:]
    assert 'check ok' in r.stdout
