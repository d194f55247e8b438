#!/usr/bin/env python3
"""Cost of --keep-at-most K on the bench workload (config 5: 200 000-leaf backbone, 5000 sites, 125 000 queries, FM + MLSE,
plus HYBRID and ME): placement-stage device time (apples_get_timings slot 4) and the time of one place_bytes call, for
K = 1, 4, 16 alternating in one process, with the card's name and power limit read in the same run.

    python tools/keep_probe.py [--reps 5] [--out DIR]      (writes DIR/keep_probe.json)
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--keeps', default='1,4,16')
    ap.add_argument('--criteria', default='MLSE,HYBRID,ME')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    import torch
    import bench
    from apples_b200 import _lib
    from apples_b200.placer import GpuPlacer
    args = bench.parse([])
    tree, arrays, _, q_bytes, info, _ = bench.build_workload(args, 'cuda:0', 0, False)
    q_host = q_bytes.cpu().numpy()
    pl = GpuPlacer(tree, None, tree.name_to_node, device=0)
    pl.set_reference_arrays(**arrays)
    card = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    keeps = [int(k) for k in a.keeps.split(',')]
    res = {'card': card, 'power_limit': power, 'queries': int(q_host.shape[0]), 'leaves': args.leaves, 'sites': args.sites,
           'reps': a.reps, 'setup': info, 'runs': {}}
    for crit in a.criteria.split(','):
        params = _lib.make_params('FM', crit)
        for k in keeps:                        # warm-up of every shape
            pl.place_bytes(q_host, None, params, keep=k)
        place_ms = {k: [] for k in keeps}
        step_ms = {k: [] for k in keeps}
        ref = None
        for _ in range(a.reps):
            for k in keeps:                    # alternating K inside every repetition
                pl.timings(reset=True)
                t0 = time.perf_counter()
                r = pl.place_bytes(q_host, None, params, keep=k)
                step_ms[k].append(1e3 * (time.perf_counter() - t0))
                place_ms[k].append(pl.timings()['placement_ms'])
                out = r if k == 1 else r[0]
                if ref is None:
                    ref = [x.copy() for x in out]
                assert all(x.tobytes() == y.tobytes() for x, y in zip(ref, out)), 'record 0 differs between K values'
        res['runs'][crit] = {str(k): {'placement_ms_median': float(np.median(place_ms[k])), 'placement_ms': place_ms[k],
                                      'step_ms_median': float(np.median(step_ms[k])), 'step_ms': step_ms[k]} for k in keeps}
    pl.close()
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'keep_probe.json'), 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
