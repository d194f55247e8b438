#!/usr/bin/env python3
"""Cost of --model K2P on the bench workload (config 5: 200 000-leaf backbone, 5000 sites, 125 000 queries, FM + MLSE):
a JC69 context and a K2P context in one process, place_bytes alternating between them for every repetition.  Reports the
step (wall time of one place_bytes call, which ends in a device synchronise) and the device stage timers (count =
rep_distance_ms, selection, placement) as medians and raw values, with the card's name and power limit read in the
same run.

    python tools/k2p_probe.py [--reps 5] [--out FILE]      (e.g. --out profiles/k2p_r05.json)
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

STAGES = ('rep_distance_ms', 'selection_ms', 'placement_ms', 'transpose_ms')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    import torch
    import bench
    from apples_b200 import _lib
    from apples_b200.placer import GpuPlacer
    args = bench.parse([])
    tree, arrays, _, q_bytes, info, _ = bench.build_workload(args, 'cuda:0', 0, False)
    q_host = q_bytes.cpu().numpy()
    card = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        power = 'unknown'
    models = ('JC69', 'K2P')
    placers = {}
    for m in models:
        placers[m] = GpuPlacer(tree, None, tree.name_to_node, device=0, model=m)
        placers[m].set_reference_arrays(**arrays)
    params = _lib.make_params('FM', 'MLSE')
    for m in models:                           # warm-up of both contexts
        placers[m].place_bytes(q_host, None, params)
    raw = {m: {k: [] for k in ('step_ms',) + STAGES + ('overflow_queries', 'k2p_launches')} for m in models}
    for _ in range(a.reps):
        for m in models:                       # alternating inside every repetition
            pl = placers[m]
            pl.timings(reset=True)
            t0 = time.perf_counter()
            pl.place_bytes(q_host, None, params)
            raw[m]['step_ms'].append(1e3 * (time.perf_counter() - t0))
            t = pl.timings()
            for k in STAGES + ('overflow_queries', 'k2p_launches'):
                raw[m][k].append(t[k])
    for pl in placers.values():
        pl.close()
    res = {'card': card, 'power_limit': power, 'queries': int(q_host.shape[0]), 'leaves': args.leaves,
           'sites': args.sites, 'reps': a.reps, 'setup': info,
           'runs': {m: {'median': {k: float(np.median(v)) for k, v in raw[m].items()}, 'raw': raw[m]} for m in models}}
    text = json.dumps(res, indent=1)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
