"""Shared-memory and tensor roofline of the block-scaled fp4 count kernel (dense_fp4_kernel) from a bench.py result line.

bench.py's `roofline.smem` models the kind::i8 tile (256 x 256, 32 sites per stage: 64 KB of fills + 96 KB of operand
reads).  The fp4 kernel's tile is 128 queries x 224 representatives with 64 sites per stage:
    fills  (TMA into shared memory)   (128 + 224) x 128 B                     = 44 KB per tile and stage
    reads  (tensor-core operands)     4 MMAs x (128 + 224) rows x 32 B (K=64)  = 44 KB per tile and stage
against 128 B per clock and SM of the shared-memory crossbar, i.e. 1.57 B per pair and 32-site word instead of 2.5.

    python bench.py --gpus 1 --no-cpu-baseline --no-cli > line.json && python tools/fp4_roofline.py line.json
"""
import json
import math
import sys

TM, TN, KS = 128, 224, 128     # tile rows (queries, representatives), K bytes per row and stage (64 sites)


def fp4_roofline(line, sites=5000):
    rl = line['roofline']
    launches = rl['launches']
    q = line['config']['queries_per_step'] / line['n_gpus'] * line['steps'] / launches   # queries per launch
    r = line['config']['n_representatives']
    ms = rl['avg_launch_ms']
    mhz = (line.get('clocks') or {}).get('sm_max_mhz') or 1965.0
    n_c = math.ceil(math.ceil(sites / 32) / 2)
    tiles = math.ceil(q / TM) * math.ceil(r / TN)
    fills = tiles * n_c * (TM + TN) * KS
    reads = tiles * n_c * 4 * (TM + TN) * 32
    peak = 148 * 128 * mhz * 1e6
    rate = (fills + reads) / (ms * 1e-3)
    ops = 2.0 * q * r * n_c * 256            # fp4 multiply-adds of the unpadded pairs (K = 4 x 64 per stage)
    return {'kernel': 'dense_fp4_kernel (tcgen05.mma kind::mxf4, 128 x 224 tile, 64 sites per stage)',
            'avg_launch_ms': ms, 'launches': launches, 'queries_per_launch': q, 'representatives': r, 'sites': sites,
            'fill_bytes_per_launch': fills, 'operand_read_bytes_per_launch': reads,
            'bytes_per_pair_and_word': (fills + reads) / (tiles * TM * TN * n_c * 2),
            'smem': {'achieved_GBps': rate / 1e9, 'peak_GBps': peak / 1e9, 'frac': rate / peak,
                     'peak_source': 'shared-memory crossbar 128 B/clk/SM x 148 SMs x %.0f MHz (max SM clock of the run)' % mhz},
            'tensor': {'achieved_TOPs': ops / (ms * 1e-3) / 1e12, 'nominal_TOPs': 9000.0,
                       'frac': ops / (ms * 1e-3) / 9e15, 'peak_source': 'nominal dense fp4 of one B200 (data sheet)'}}


def main(argv):
    sites = 5000
    if '--sites' in argv:
        i = argv.index('--sites')
        sites = int(argv[i + 1])
        argv = argv[:i] + argv[i + 2:]
    text = open(argv[0]).read() if argv else sys.stdin.read()
    line = [json.loads(s) for s in text.splitlines() if s.startswith('{')][-1]
    print(json.dumps(fp4_roofline(line, sites), indent=1))


if __name__ == '__main__':
    main(sys.argv[1:])
