"""CPU: --keep-at-most K without a device -- the K-record oracle against brute force and against choose_edge, the native
K-record jplace writer against json.dumps, the option's bounds, and the gloo gather of K-record blocks."""
import json
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests import util
from tests import keep_oracle as ko
from oracle import apples_oracle as orc
from apples_b200 import parallel

FIXTURES = [c for c in util.golden_names() if c.startswith(('small_', 'syn300_', 'c1_', 'c2_', 'c3_'))]


def _brute(post, criterion, V, keep):
    """the definition spelled out: explicit (key, edge_index) sort keys instead of sort stability"""
    rows = [(orc.edge_error(e), e.x1, e.edge_index, e) for e in post]
    if criterion == 'HYBRID':
        cand = sorted(rows, key=lambda r: (r[0], r[2]))[:math.floor(math.log2(V))]
        ranked = [t[2][3] for t in sorted(((r[1], i, r) for i, r in enumerate(cand)), key=lambda t: (t[0], t[1]))]
    elif criterion == 'ME':
        ranked = [r[3] for r in sorted(rows, key=lambda r: (r[1], r[2]))]
    else:
        ranked = [r[3] for r in sorted(rows, key=lambda r: (r[0], r[2]))]
    return [e.edge_index for e in ranked[:keep]]


@pytest.mark.parametrize('case', FIXTURES)
def test_choose_edges_is_the_stable_sort(case, workdir):
    """choose_edges(keep=1)[0] is choose_edge's record; for every criterion x -n it is the stable sort by the key, on
    every query of the fixture."""
    ci = util.CaseInputs(case, workdir)
    octx = ci.oracle_context()
    n = 0
    for qname, qseq, row in ci.queries:
        if row:
            obs = orc.observed_matrix(dict(row), octx.name_to_node, octx.filt_threshold, octx.baseobs)
        else:
            obs = orc.observed_alignment(qseq, octx.representatives, octx.refs, octx.dist_fn, octx.filt_threshold,
                                         octx.baseobs, octx.overlap)
        obs.pop(qname, None)
        if len(obs) <= 2 or any(v == 0 for v in obs.values()):
            continue
        for criterion in ('MLSE', 'ME', 'HYBRID'):
            for neg in (False, True):
                def check(post, V):
                    one, _ = orc.choose_edge(post, criterion, V)
                    assert ko.choose_edges(post, criterion, V, 1)[0] == one, (case, qname, criterion, neg)
                    for keep in (2, 5, 16, len(post) + 3):
                        recs = ko.choose_edges(post, criterion, V, keep)
                        assert [r[0] for r in recs] == _brute(post, criterion, V, keep), (case, qname, criterion, neg, keep)
                        assert recs[0] == one and all(r[2] == 0 for r in recs[1:])
                    return None
                ko.solved_edges(obs, octx.name_to_node, octx.method, neg, check)
                n += 1
    assert n > 0


def test_place_from_observed_k_keeps_single_records(workdir):
    """zero-distance, too-few and --exclude queries keep their one record; record 0 of a placed query is the
    single-record result"""
    ci = util.CaseInputs('small_FM_MLSE_pos', workdir)
    octx = ci.oracle_context()
    q = ci.queries[0]
    row = dict(q[2])
    obs = orc.observed_matrix(row, octx.name_to_node, 0.2, 25)
    one, st = orc.place_from_observed(q[0], obs, octx.name_to_node)
    many, st2 = ko.place_from_observed_k(q[0], obs, octx.name_to_node, keep=4)
    assert st == st2 and many['placements'][0]['p'][0] == one['placements'][0]['p'][0]
    assert len(many['placements'][0]['p']) == 4
    k0 = next(iter(obs))
    zero = dict(obs)
    zero[k0] = 0.0
    assert len(ko.place_from_observed_k(q[0], zero, octx.name_to_node, keep=4)[0]['placements'][0]['p']) == 1
    few = dict(list(obs.items())[:2])
    assert ko.place_from_observed_k(q[0], few, octx.name_to_node, keep=4)[0]['placements'][0]['p'] == [[-1, 0, 1, 0, 0]]


def _random_records(n, keep, first_bad, seed):
    rng = np.random.default_rng(seed)
    vals = [0.0, -0.0, 1e-5, 1e-4, 1e16, 1.5e-7, float('nan'), float('inf'), -float('inf'), 5e-324, 0.1, 1 / 3, 2.0]
    names = ['q%d' % i for i in range(n)]
    if n > 3:
        names[1], names[2], names[3] = 'na\u00efve "q"\\t\u2603', '\U0001F600x', 'tab\there\x7f'

    def col(shape):
        a = rng.random(shape) * rng.choice([1e-18, 1e-9, 1e-3, 1.0, 1e6], shape)
        flat = a.reshape(-1)
        k = min(flat.size, len(vals))
        flat[:k] = vals[:k]
        rng.shuffle(flat)
        return a
    status = rng.choice([0, 0, 0, 0, 1, 2, 3, 0x100, 0x103], n).astype(np.int32)
    if first_bad:
        status[0] = 2
    edge = rng.integers(0, 1000, n).astype(np.int32)
    out = (edge, col(n), col(n), col(n), status)
    count = rng.integers(1, keep + 1, n).astype(np.int32)
    a_edge = rng.integers(0, 1000, (n, keep)).astype(np.int32)
    a_edge[:, 0] = edge
    alt = (count, a_edge, col((n, keep)), col((n, keep)), col((n, keep)), (rng.random((n, keep)) < 0.3).astype(np.uint8))
    return names, rng.random(n) < 0.1, out, alt


def test_native_k_writer_is_json_dumps(tmp_path):
    """apples_jplace_write_k == json.dumps(assemble(results_to_jplace(..., alt)), sort_keys=True, indent=4), byte for
    byte: int-0 pendants, unplaceable first records, --exclude, escaped names, NaN / infinity; with keep 1 it writes
    what apples_jplace_write writes."""
    from apples_b200 import jplace
    from apples_b200.placer import results_to_jplace
    fp = str(tmp_path / 'k.jplace')
    for n, keep, fb, ex, seed in [(1, 3, False, False, 1), (1, 3, True, False, 2), (2, 2, True, True, 3),
                                  (40, 5, False, False, 4), (40, 16, True, True, 5), (9000, 4, False, True, 6),
                                  (3, 2, True, False, 7)]:
        names, inb, out, alt = _random_records(n, keep, fb, seed)
        res = results_to_jplace(names, inb.tolist(), out, ex, log=False, degenerate='keep', alt=alt)
        doc = jplace.assemble(res, '((a,b),c);', argv=['run_apples.py', '-x'])
        ref = json.dumps(doc, sort_keys=True, indent=4) + '\n'
        assert jplace.dumps(doc) + '\n' == ref
        for th in (1, 3, 0):
            nw = jplace.write_arrays(fp, names, inb, out, '((a,b),c);', ex, argv=['run_apples.py', '-x'], threads=th, alt=alt)
            assert open(fp, encoding='utf-8').read() == ref, (n, keep, fb, ex, th)
            assert nw == len(doc['placements'])
        # keep 1: the single-record writer's file
        one = tuple(a[:, :1] if a.ndim == 2 else a for a in alt)
        jplace.write_arrays(fp, names, inb, out, '((a,b),c);', ex, argv=['run_apples.py', '-x'], alt=one)
        k1 = open(fp, encoding='utf-8').read()
        jplace.write_arrays(fp, names, inb, out, '((a,b),c);', ex, argv=['run_apples.py', '-x'])
        assert k1 == open(fp, encoding='utf-8').read()


@pytest.mark.parametrize('k', [0, 17, -1])
def test_keep_at_most_out_of_range_is_rejected(k, workdir):
    from apples_b200.options import options_config_run
    from apples_b200.placer import check_keep
    tfp = util.gunzip_to('small_backbone.nwk', workdir)
    with pytest.raises(ValueError, match='keep-at-most'):
        options_config_run(['-t', tfp, '-d', 'x.mat', '--keep-at-most', str(k)])
    with pytest.raises(ValueError, match='keep-at-most'):
        check_keep(k)
    assert options_config_run(['-t', tfp, '-d', 'x.mat'])[0].keep_at_most == 1
    assert options_config_run(['-t', tfp, '-d', 'x.mat', '--keep-at-most', '16'])[0].keep_at_most == 16


def _k_block(b, e, keep):
    """deterministic K-record shard of queries b..e (what a rank's placer would return)"""
    rng = np.random.default_rng(1000 + b)
    n = e - b
    out = (np.arange(b, e, dtype=np.int32), rng.random(n), rng.random(n), rng.random(n),
           rng.choice([0, 1, 2, 3, 0x100, 0x103], n).astype(np.int32))
    a_edge = rng.integers(0, 5000, (n, keep)).astype(np.int32)
    a_edge[:, 0] = out[0]
    a_edge[:, keep - 1] = -1
    err, dis, pen = rng.random((n, keep)), rng.random((n, keep)), rng.random((n, keep))
    err[:, 0], dis[:, 0], pen[:, 0] = out[1], out[2], out[3]
    int0 = (rng.random((n, keep)) < 0.5).astype(np.uint8)
    int0[:, 0] = (out[4] >> 8) & 1
    return out, (rng.integers(1, keep + 1, n).astype(np.int32), a_edge, err, dis, pen, int0)


def _worker(rank, world, port, n, keep, q):
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        b, e = parallel.shard_bounds(n, world)[rank]
        out, alt = _k_block(b, e, keep)
        main, alt_all = parallel.gather_placements(out, n, alt=alt)
        q.put((rank, [a.tolist() for a in main], [a.tolist() for a in alt_all]))
    finally:
        dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.parametrize('world,n,keep', [(2, 11, 5), (3, 10, 2)])
def test_gloo_gather_of_k_records(world, n, keep):
    """K records per query in the one all-gather, ragged last rank: every rank gets all records in input order"""
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n, keep, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = [q.get(timeout=180) for _ in range(world)]
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    parts = [_k_block(b, e, keep) for b, e in parallel.shard_bounds(n, world)]
    main = [np.concatenate([p[0][i] for p in parts]).tolist() for i in range(5)]
    alt = [np.concatenate([p[1][i] for p in parts]).tolist() for i in range(6)]
    for rank, m, a in got:
        assert m == main, rank
        assert a == alt, rank
