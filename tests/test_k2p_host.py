"""CPU: the K2P definition (tests/k2p_oracle.py), the --model option, and the JC69 count kernel left as it was.

The JC69 instantiation of dense_fp4_kernel and the fp4 operand-image kernel must compile to the SASS they had before the
K2P instantiation was added; the digests below are those of the parent build (CUDA 12.9, sm_100a), with the kernel
names and instruction encodings left out.
"""
import hashlib
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from oracle import apples_oracle as orc
from tests import k2p_oracle as ko

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PURINE = {b'A', b'G'}


def _k2p_loop(a, b, overlap):
    """per-site classification of every pair"""
    valid = ts = tv = 0
    for x, y in zip(a.tolist(), b.tolist()):
        if x == b'-' or y == b'-':
            continue
        valid += 1
        if x != y:
            if (x in PURINE) == (y in PURINE):
                ts += 1
            else:
                tv += 1
    if not valid or valid / len(a) < overlap:
        return -1.0
    if ts + tv == 0:
        return 0.0
    P, Q = ts / valid, tv / valid
    w1, w2 = 1 - 2 * P - Q, 1 - 2 * Q
    if w1 <= 0 or w2 <= 0:
        return -1.0
    return -0.5 * np.log(w1) - 0.25 * np.log(w2)


def test_k2p_against_a_per_site_loop():
    rng = np.random.default_rng(7)
    sym = np.array([b'A', b'C', b'G', b'T', b'-'], dtype='S1')
    seen = set()
    for case in range(400):
        L = int(rng.integers(1, 300))
        gap = float(rng.choice([0.0, 0.1, 0.5, 0.95]))
        a = sym[rng.integers(0, 4, L)]
        a[rng.random(L) < gap] = b'-'
        b = a.copy()
        mut = rng.random(L) < float(rng.choice([0.0, 0.05, 0.3, 0.8]))
        b[mut] = sym[rng.integers(0, 4, int(mut.sum()))]
        b[rng.random(L) < gap] = b'-'
        if case % 5 == 0:      # overlap only at the ends
            a[L // 4: L - L // 4] = b'-'
        overlap = float(rng.choice([0.001, 0.2, 0.5]))
        d = ko.k2p(a, b, overlap)
        assert d == _k2p_loop(a, b, overlap), (case, L)
        ts, tv, v = ko.k2p_counts(a, b)
        assert d == ko.k2p_from_counts(ts, tv, v, L, overlap)
        seen.add('missing' if d < 0 else 'zero' if d == 0 else 'positive')
    assert seen == {'missing', 'zero', 'positive'}


def test_k2p_equals_jc69_when_tv_is_twice_ts():
    """1 - 2P - Q = 1 - 2Q = 1 - 4 ts / v = the JC69 loc when tv = 2 ts, so d = -0.75 ln(loc) in exact arithmetic"""
    n = 0
    for v in range(1, 2001):
        for ts in range(0, v // 3 + 1):
            k = ko.k2p_from_counts(ts, 2 * ts, v, v, 0.001)
            j = orc.jc69_from_counts(3 * ts, v, v, 0.001)
            assert (k < 0) == (j < 0), (ts, v, k, j)
            assert abs(k - j) <= 1e-12 * abs(j), (ts, v, k, j)
            n += 1
    assert n > 600000


def test_model_option():
    from apples_b200.options import options_config_run
    base = ['-t', 'backbone.nwk', '-s', 'ref.fa', '-q', 'query.fa', '-D']
    assert options_config_run(base)[0].model == 'JC69'
    assert options_config_run(base + ['--model', 'JC69'])[0].model == 'JC69'
    o = options_config_run(base + ['--model', 'K2P', '--keep-at-most', '4'])[0]
    assert (o.model, o.keep_at_most) == ('K2P', 4)
    with pytest.raises(ValueError, match='--model must be JC69 or K2P'):
        options_config_run(base + ['--model', 'k2p'])
    with pytest.raises(ValueError, match='-p'):
        options_config_run(base + ['-p', '--model', 'K2P'])
    with pytest.raises(ValueError, match='-d'):
        options_config_run(['-t', 'backbone.nwk', '-d', 'dist.mat', '--model', 'JC69'])
    assert options_config_run(['-t', 'backbone.nwk', '-d', 'dist.mat'])[0].model == 'JC69'


def test_placer_checks_the_model():
    from apples_b200 import placer
    assert placer.check_model('K2P') == 'K2P'
    with pytest.raises(ValueError, match='--model'):
        placer.check_model('TN93')


# the JC69 count kernel and the operand-image kernel as the parent commit compiled them
PARENT_SASS = {
    '_Z16dense_fp4_kernelILb0EEv6TcArgs': '866e83d8acba89b8c5e8c4da88f84bdac91a03bb58c89b501c7579e55bf11300',
    '_Z16fp4_image_kernelPKjiiiiP5uint4': '8b75fd295f10d8842235fde34c737ccbec4d8f49c5e908ef6cb4cacb4534cdcb',
}


def _sass_digests(path):
    """sha256 of each kernel's SASS: instructions with their offsets, encodings and the function header dropped"""
    tool = shutil.which('cuobjdump') or '/usr/local/cuda/bin/cuobjdump'
    out = subprocess.run([tool, '-sass', path], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r'\s*Function : (\S+)', line)
        if m:
            cur = funcs.setdefault(m.group(1), [])
            continue
        line = re.sub(r'/\* 0x[0-9a-f]+ \*/', '', line).strip()
        if cur is not None and line and not line.startswith('.'):
            cur.append(line)
    return {k: hashlib.sha256('\n'.join(v).encode()).hexdigest() for k, v in funcs.items()}


def test_jc69_count_kernels_compile_as_before():
    lib = os.path.join(ROOT, 'apples_b200', 'libapples_b200.so')
    if not os.path.isfile(lib):
        pytest.skip('the library is not built')
    if not (shutil.which('cuobjdump') or os.path.isfile('/usr/local/cuda/bin/cuobjdump')):
        pytest.skip('cuobjdump is not installed')
    try:
        version = subprocess.run([shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc', '--version'], capture_output=True,
                                 text=True).stdout
    except OSError:
        version = ''
    if 'release 12.9' not in version:
        pytest.skip('the digests are those of CUDA 12.9')
    got = _sass_digests(lib)
    for name, digest in PARENT_SASS.items():
        assert got.get(name) == digest, name
