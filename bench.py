#!/usr/bin/env python3
"""bench.py -- queries placed per second on the 200 000-leaf backbone (BASELINE.json metric, config 5).

    python bench.py --gpus N --steps K --warmup W                 (N > 1: launched under torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W  the CPU arm (rank 0 only)
    ... --dump-outputs DIR      also write the last timed step's placements (all ranks' queries) to DIR/*.npy

Workload (SURVEY.md section 8d, config 5): synthetic 200 000-leaf Yule backbone, 5000-site nucleotide alignment
evolved under JC69 with gaps, max-diameter clusters at 1.2 x 0.2, FM + MLSE, -f 0.2 -b 25 -V 0.001.  One "step" places
125 000 queries per GPU (1 M queries at 8 GPUs: weak scaling, queries shard with no data-path collective; the only
collective is the final NCCL all-gather of the placements, which is inside the timed region).

`value` is measured with the packed queries already resident in HBM (apples_place_resident); `e2e` goes through the
reference-facing C-ABI call apples_place_batch with pinned HOST buffers, host<->device copies inside the timed region.
The roofline object describes the dominant kernel (dense query x representative distance kernel); the CPU baseline is
the oracle port of the reference's Python path (kind "port": the reference itself is Python and cannot travel to the
GPU box) run through a fork pool on all host cores on a bounded sample of the same queries.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='config5', choices=['config5', 'protein'],
                    help="config5 = BASELINE.json's metric workload (default); protein = config 3 scaled up (4038-leaf "
                         "backbone, 1638 amino-acid sites, 100 000 queries, scoredist + BLOSUM45): a side measurement of the "
                         "amino-acid kernel, not the headline")
    ap.add_argument('--leaves', type=int, default=None)
    ap.add_argument('--sites', type=int, default=None)
    ap.add_argument('--queries-per-gpu', type=int, default=None)
    ap.add_argument('--method', default='FM')
    ap.add_argument('--criterion', default='MLSE')
    ap.add_argument('--cpu-sample', type=int, default=0, help='queries in the CPU-baseline sample (0 = auto)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--dense', default='tensor', choices=['tensor', 'intpipe'],
                    help='kernel of the representative counts: tcgen05 tensor-core kernel (default) or the integer-pipe '
                         'LOP3/POPC kernel (identical results)')
    ap.add_argument('--no-cli', action='store_true', help='skip the run_apples.py command-line measurement (cli_e2e)')
    ap.add_argument('--slot-cap', type=int, default=0, help='observed-list slots per query before a rerun (0 = library default)')
    ap.add_argument('--sub-batch', type=int, default=0, help='queries per dense/selection launch (0 = library default)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the placements of the last timed step as DIR/<name>.npy (float64), so that two builds can '
                         'be compared output for output on the same seeded inputs')
    a = ap.parse_args(argv)
    prot = a.workload == 'protein'
    a.leaves = a.leaves or (4038 if prot else 200000)
    a.sites = a.sites or (1638 if prot else 5000)
    a.queries_per_gpu = a.queries_per_gpu or (100000 if prot else 125000)
    a.filt = 0.6 if prot else 0.2     # -f of the reference's protein example (README) / default
    return a


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None
        self.t_begin = 0.0

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '200'], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(',')]))

    def mark_begin(self):
        self.t_begin = time.time()

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        t_end = time.time()
        inside = [r for t, r in self.rows if self.t_begin <= t <= t_end + 0.3]
        for r in (inside if inside else [r for _, r in self.rows[-3:]]):
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith('active'):
                        reasons.add(n)
            except Exception:
                pass
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


def build_workload(args, device, rank, want_host_refs):
    """Synthetic backbone + reference (identical on every rank) and this rank's queries.  Untimed setup."""
    import torch
    from apples_b200 import synth, synth_torch, treecluster, fasta
    from apples_b200.tree import BackboneTree
    t0 = time.time()
    prot = getattr(args, 'workload', 'config5') == 'protein'
    nwk = synth.random_tree(args.leaves, seed=2, mean_edge=0.06 if prot else 0.02)
    tree = BackboneTree.from_newick(nwk)
    ref_bytes, leaf_states = synth_torch.evolve_alignment(tree, args.sites, 5, device, protein=prot)
    q_bytes, src = synth_torch.make_queries(leaf_states, args.queries_per_gpu, 1000 + rank, device, protein=prot)
    del leaf_states
    ref_host = ref_bytes.cpu().numpy()
    if prot:
        packed_refs = fasta.pack_protein(ref_host)
        packed_q = torch.from_numpy(fasta.pack_protein(q_bytes.cpu().numpy()))
    else:
        packed_refs = synth_torch.pack_nucleotide(ref_bytes).cpu().numpy().view(np.uint32)
        packed_q = synth_torch.pack_nucleotide(q_bytes)
    del ref_bytes
    # clusters and consensus representatives (Reference.py:85-107 equivalent, build-time)
    clusters = treecluster.max_diameter_clusters(tree, getattr(args, 'filt', 0.2) * 1.2)
    leaf_row = {int(u): i for i, u in enumerate(tree.leaf_ids.tolist())}
    # the reference orders representatives by the cluster-id STRING with singletons ('-1') first (Reference.py:97)
    multi = [c for c in clusters if len(c) > 1]
    single = [c for c in clusters if len(c) == 1]
    keyed = sorted(((str(i + 1), c) for i, c in enumerate(multi)), key=lambda kc: kc[0])
    ordered = single + [c for _, c in keyed]
    from apples_b200.reference import consensus_rows
    reps = np.empty((len(ordered), args.sites), dtype=np.uint8)
    offs = np.zeros(len(ordered) + 1, dtype=np.int32)
    members = []
    for i, c in enumerate(ordered):
        rows = [leaf_row[u] for u in c]
        reps[i] = ref_host[rows[0]] if len(rows) == 1 else consensus_rows(ref_host[rows], prot)
        members.extend(rows)
        offs[i + 1] = len(members)
    packed_reps = fasta.pack(reps, fasta.AA if prot else fasta.NUC)
    arrays = dict(kind=fasta.AA if prot else fasta.NUC, L=args.sites, ref_names=[tree.label[u] for u in tree.leaf_ids.tolist()],
                  packed_refs=packed_refs, ref_node=tree.leaf_ids.astype(np.int32), packed_reps=packed_reps,
                  group_offsets=offs, group_members=np.asarray(members, dtype=np.int32))
    info = {'setup_s': round(time.time() - t0, 1), 'n_rep': len(ordered), 'max_level': int(tree.level.max())}
    host = None
    if want_host_refs:
        host = dict(nwk=nwk, ref_host=ref_host, reps=reps, ordered=ordered, clusters=clusters, leaf_row=leaf_row, q_bytes=q_bytes)
    return tree, arrays, packed_q, q_bytes, info, host


def cpu_context(args, tree, host):
    """Oracle-side state (the analogue of prepareTree + ReducedReference, built once, untimed like the reference's
    own setup: its timer brackets only the starmap call, run_apples.py:93-104)."""
    import tempfile
    from oracle import apples_oracle as orc
    tfp = os.path.join(tempfile.mkdtemp(prefix='apples_bench_'), 'backbone.nwk')
    with open(tfp, 'w') as f:
        f.write(host['nwk'])
    otree, onames = orc.load_tree(tfp)
    names = [tree.label[u] for u in tree.leaf_ids.tolist()]
    ref_host = host['ref_host']
    refs = {n: ref_host[i].view('S1') for i, n in enumerate(names)}
    reps = [(host['reps'][i].view('S1'), [names[host['leaf_row'][u]] for u in c]) for i, c in enumerate(host['ordered'])]
    return orc.OracleContext(otree, onames, refs=refs, representatives=reps, method=args.method, criterion=args.criterion,
                             protein=getattr(args, 'workload', 'config5') == 'protein', filt_threshold=getattr(args, 'filt', 0.2))


def cpu_baseline(ctx, q_host, threads):
    """The oracle port of the reference's Python path (PoolQueryWorker.runquery under a fork pool,
    run_apples.py:94-102) on the given queries.  Returns (queries/s, seconds, results)."""
    from oracle import apples_oracle as orc
    queries = [('Q%07d' % i, q_host[i].view('S1'), None) for i in range(len(q_host))]
    t0 = time.time()
    res = orc.run_pool(ctx, queries, threads)
    dt = time.time() - t0
    return len(queries) / dt, dt, res


def write_fasta(path, names, mat):
    """uint8 [n, L] rows + fixed-width names -> FASTA text, vectorised (setup, untimed)."""
    n, L = mat.shape
    w = max(len(x) for x in names)
    assert all(len(x) == w for x in names)
    out = np.empty((n, w + 2 + L + 1), dtype=np.uint8)
    out[:, 0] = ord('>')
    out[:, 1:1 + w] = np.frombuffer(''.join(names).encode(), dtype=np.uint8).reshape(n, w)
    out[:, 1 + w] = ord('\n')
    out[:, 2 + w:2 + w + L] = mat
    out[:, -1] = ord('\n')
    with open(path, 'wb') as f:
        f.write(out.tobytes())


DUMP_BYTES_MAX = 64 << 20
RESULT_NAMES = ('edge', 'error', 'distal', 'pendant', 'status')


def dump_outputs(path, arrays):
    """The five placement arrays of one step (edge, error, distal, pendant, status) -> <path>/<name>.npy in float64, which
    holds the int32 edge and status exactly.  Above DUMP_BYTES_MAX in all, the same seeded sample of queries is written
    every run, with the sampled query indices as query_index.npy."""
    os.makedirs(path, exist_ok=True)
    arrays = [np.asarray(a) for a in arrays]
    n = len(arrays[0])
    idx = None
    if 8 * n * len(arrays) > DUMP_BYTES_MAX:
        k = (DUMP_BYTES_MAX - (64 << 10)) // (8 * (len(arrays) + 1))   # 64 KB left for the .npy headers
        idx = np.sort(np.random.default_rng(0).choice(n, k, replace=False))
        np.save(os.path.join(path, 'query_index.npy'), idx.astype(np.float64))
    for name, a in zip(RESULT_NAMES, arrays):
        np.save(os.path.join(path, name + '.npy'), (a if idx is None else a[idx]).astype(np.float64))


def cli_e2e(args, tree, host, q_bytes, device):
    """run_apples.py as a user runs it: reference FASTA + tree + cluster TSV + query FASTA on disk in, jplace on disk out.
    The files are written first (untimed); everything run_apples.main does is timed, stage by stage (its own timers)."""
    import shutil
    import tempfile
    import run_apples
    from apples_b200 import treecluster
    wd = tempfile.mkdtemp(prefix='apples_cli_')
    try:
        names = [tree.label[u] for u in tree.leaf_ids.tolist()]
        write_fasta(os.path.join(wd, 'ref.fa'), names, host['ref_host'])
        q_host = q_bytes.cpu().numpy()
        write_fasta(os.path.join(wd, 'query.fa'), ['Q%07d' % i for i in range(q_host.shape[0])], q_host)
        with open(os.path.join(wd, 'backbone.nwk'), 'w') as f:
            f.write(host['nwk'])
        treecluster.write_cluster_tsv(tree, host['clusters'], os.path.join(wd, 'clusters.tsv'))
        out = os.path.join(wd, 'out.jplace')
        argv = ['-s', os.path.join(wd, 'ref.fa'), '-q', os.path.join(wd, 'query.fa'), '-t', os.path.join(wd, 'backbone.nwk'),
                '--clusters', os.path.join(wd, 'clusters.tsv'), '-D', '-m', args.method, '-c', args.criterion, '-o', out,
                '-f', str(args.filt), '--device', str(device), '--gpus', '1'] + (['-p'] if args.workload == 'protein' else [])
        import logging
        lvl = logging.getLogger().level
        logging.getLogger().setLevel(logging.ERROR)
        t0 = time.time()
        run_apples.main(argv)
        wall = time.time() - t0
        logging.getLogger().setLevel(lvl)
        t = dict(run_apples.LAST_TIMINGS)
        nq = int(t.get('queries', 0))
        qpath = t.get('read_queries_s', 0.0) + t.get('place_s', 0.0) + t.get('write_s', 0.0)
        return {'queries': nq, 'wall_s': wall, 'queries_per_s': nq / wall,
                'query_path_s': qpath, 'query_path_queries_per_s': nq / qpath if qpath else None,
                'stages_s': {k: round(v, 3) for k, v in t.items() if k.endswith('_s')},
                'jplace_bytes': os.path.getsize(out),
                'note': 'setup_s = tree parsing, reference FASTA, clustering file, options (once per run); query path = '
                        'native FASTA reader -> apples_place_batch_bytes (context creation + reference upload included) -> '
                        'native jplace writer'}
    finally:
        shutil.rmtree(wd, ignore_errors=True)


def main():
    # the contract is ONE JSON line on stdout: libraries (NCCL prints its version banner to stdout) are redirected to
    # stderr at the file-descriptor level and the JSON line is written to the saved descriptor at the end
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + '\n').encode())

    args = parse()
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    threads = os.cpu_count() or 1
    prot = args.workload == 'protein'
    workload = ('synthetic %d-leaf Yule backbone, %d-site %s alignment (%s + gaps), %d queries per GPU per '
                'step, APPLES-2 clusters at 1.2x%g, %s+%s, -f %g -b 25' % (args.leaves, args.sites,
                                                                          'amino-acid' if prot else 'nucleotide',
                                                                          '20-state symmetric model' if prot else 'JC69',
                                                                          args.queries_per_gpu, args.filt, args.method,
                                                                          args.criterion, args.filt))
    import torch

    if args.impl == 'reference':
        if rank != 0:
            return 0
        dev = 'cuda:0' if torch.cuda.is_available() else 'cpu'
        tree, arrays, packed_q, q_bytes, info, host = build_workload(args, dev, 0, True)
        n_sample = args.cpu_sample or max(threads * 4, 32)
        q_host = q_bytes[:n_sample * (args.steps + args.warmup)].cpu().numpy()
        rates = []
        octx = cpu_context(args, tree, host)
        for s in range(args.warmup + args.steps):
            qs = q_host[s * n_sample:(s + 1) * n_sample]
            r, dt, res = cpu_baseline(octx, qs, threads)
            if s >= args.warmup:
                rates.append((r, dt))
        if args.dump_outputs:
            p = [x[0]['placements'][0]['p'][0] for x in res]
            dump_outputs(args.dump_outputs, ([q[0] for q in p], [q[1] for q in p], [q[3] for q in p], [q[4] for q in p],
                                             [x[1] for x in res]))
        tot_t = sum(dt for _, dt in rates)
        val = n_sample * len(rates) / tot_t
        line = {'impl': 'reference', 'metric': 'queries placed/sec', 'value': val, 'unit': 'queries/s',
                'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * tot_t / len(rates),
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'u32 popcount + f64',
                'data': 'synthetic', 'config': {'workload': workload, 'sample_queries_per_step': n_sample},
                'cpu_baseline': {'value': val, 'unit': 'queries/s', 'cores': threads, 'kind': 'port',
                                 'sample': '%d queries per step through the oracle port of PoolQueryWorker.runquery, '
                                           'fork pool of %d processes' % (n_sample, threads)},
                'e2e': {'value': val, 'unit': 'queries/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
        emit(line)
        return 0

    # ------------------------------------------------------------------------------------------------ our arm
    import torch.distributed as dist
    from apples_b200 import _lib
    from apples_b200.placer import GpuPlacer
    if not torch.cuda.is_available():
        raise RuntimeError('bench.py needs a CUDA device; the hot path has no CPU fallback')
    torch.cuda.set_device(local_rank)
    device = 'cuda:%d' % local_rank
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device(device))
    want_host = rank == 0 and world == 1 and not (args.no_cpu_baseline and args.no_cli)
    tree, arrays, packed_q, q_bytes, info, host = build_workload(args, device, rank, want_host)
    nq = args.queries_per_gpu
    pl = GpuPlacer(tree, None, tree.name_to_node, device=local_rank)
    pl.set_dense_mode(0 if args.dense == 'intpipe' else 1)
    pl.set_reference_arrays(**arrays)
    if args.slot_cap or args.sub_batch:
        pl.set_limits(max_subbatch=args.sub_batch, slot_cap=args.slot_cap)
    params = _lib.make_params(args.method, args.criterion, filt_threshold=args.filt)
    packed_host = torch.empty(packed_q.shape, dtype=packed_q.dtype).pin_memory()
    packed_host.copy_(packed_q)
    del packed_q
    pl.upload_queries(packed_host)
    stream = torch.cuda.ExternalStream(pl.stream, device=device)
    # device buffers of the final gather of placements: the five result arrays are packed into 32-byte records and
    # exchanged with ONE all-gather (apples_b200.parallel, the same code the product path uses under torchrun)
    from apples_b200 import parallel
    send = (torch.empty(nq, dtype=torch.int32, device=device), torch.empty(nq, dtype=torch.float64, device=device),
            torch.empty(nq, dtype=torch.float64, device=device), torch.empty(nq, dtype=torch.float64, device=device),
            torch.empty(nq, dtype=torch.int32, device=device))
    recv = torch.empty((nq * world, 4), dtype=torch.int64, device=device) if world > 1 else None
    gathered = [None]

    def step_resident():
        pl.place_resident(params)
        if world > 1:
            pl.results_to_device(*send)
            gathered[0] = parallel.gather_records(parallel.pack_records(*send), nq * world, out=recv)
            # the gathered placements are this step's result: wait for them before the next step starts.  Left
            # asynchronous, the NCCL kernels of a rank that is ahead spin on its SMs while its next dense kernel (one
            # persistent CTA per SM, statically striped tiles) starts, and the CTAs that start late set the kernel time
            # (+12 % on every rank at 8 GPUs; handing tiles out dynamically instead costs 4.5 % at 1 GPU, DESIGN.md 8)
            torch.cuda.current_stream().synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the clock sampler (one nvidia-smi process per rank) is started BEFORE the warm-up: its NVML start-up attaches to
    # every GPU of the node and, started at the edge of the timed region by eight ranks at once, slowed the dense
    # kernel of all of them by ~10 % for the first second.  Only samples taken inside the timed region are kept.
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        step_resident()
    pl.timings(reset=True)
    barrier()
    sampler.mark_begin()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        step_resident()
    e1.record(stream)
    barrier()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    tm = pl.timings(reset=True)
    last_step = None
    if args.dump_outputs and rank == 0:
        # taken here: the end-to-end steps below place the same queries again through the same context
        last_step = ([t.cpu().numpy() for t in parallel.unpack_records(gathered[0])] if world > 1
                     else pl.download_results())
    per_rank = None
    if world > 1:
        # every rank's own step time, dense-kernel time and the SM clock measured inside the dense kernel (clock64 /
        # globaltimer), so that a slow rank or a clock nvidia-smi does not show is visible in the line
        mine = torch.tensor([ms / args.steps, tm['rep_distance_ms'] / args.steps, float(tm.get('rep_distance_sm_mhz') or 0.0),
                             1.0 if clocks.get('reasons') else 0.0], dtype=torch.float64, device=device)
        allr = torch.empty(world * 4, dtype=torch.float64, device=device)
        dist.all_gather_into_tensor(allr, mine)
        allr = allr.view(world, 4).cpu().tolist()
        per_rank = {'ms_per_step': [round(r[0], 2) for r in allr], 'rep_distance_ms': [round(r[1], 2) for r in allr],
                    'rep_distance_sm_mhz': [round(r[2], 1) for r in allr], 'throttled': [bool(r[3]) for r in allr]}
        t = torch.tensor([ms], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = nq * world * args.steps / (ms / 1e3)

    # ---- end to end through the C-ABI call with host buffers ----
    e2e = None
    if not args.no_e2e:
        # the reference-facing call: aligned query BYTES in (pinned) host memory, as fasta2dic leaves them; packing
        # happens on the device, host<->device copies are inside the timed region
        self_node = None
        bytes_host = torch.empty(q_bytes.shape, dtype=torch.uint8).pin_memory()
        bytes_host.copy_(q_bytes)
        bytes_np = bytes_host.numpy()
        for _ in range(min(args.warmup, 1)):
            out = pl.place_bytes(bytes_np, self_node, params)
            if world > 1:   # the gather's pinned buffer and first-use costs belong to the warm-up as well
                parallel.gather_placements(out, nq * world, device=device)
        pl.timings(reset=True)   # stage timers of the timed steps only
        barrier()
        e0.record(stream)
        t0 = time.time()
        t_place = t_gather = 0.0
        for _ in range(args.steps):
            ta = time.time()
            out = pl.place_bytes(bytes_np, self_node, params)
            tb = time.time()
            if world > 1:
                # the product's multi-process path ends here: every rank holds all placements (placer.place_arrays)
                out_all = parallel.gather_placements(out, nq * world, device=device)
            t_place += tb - ta
            t_gather += time.time() - tb
        e1.record(stream)
        barrier()
        ems = e0.elapsed_time(e1)
        place_ms_per_rank = None
        if world > 1:
            t = torch.tensor([ems], dtype=torch.float64, device=device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ems = float(t.item())
            # the gather is a synchronisation point: a rank whose host->device copies are slower (PCIe / NUMA position)
            # makes every other rank wait there
            tp = torch.tensor([1e3 * t_place / args.steps], dtype=torch.float64, device=device)
            tps = [torch.zeros_like(tp) for _ in range(world)]
            dist.all_gather(tps, tp)
            place_ms_per_rank = [round(float(x.item()), 2) for x in tps]
        e2e = {'value': nq * world * args.steps / (ems / 1e3), 'unit': 'queries/s',
               'h2d_bytes_per_step': (int(bytes_host.numel()) + (32 * nq if world > 1 else 0)) * world,
               'd2h_bytes_per_step': (32 * nq + (32 * nq * world if world > 1 else 0)) * world,
               'input': 'alignment bytes (uint8 per site) in pinned host memory, packed on the device',
               'wall_ms_per_step': 1e3 * (time.time() - t0) / args.steps,
               'rank0_place_call_ms_per_step': 1e3 * t_place / args.steps,
               'rank0_gather_ms_per_step': 1e3 * t_gather / args.steps, 'place_call_ms_per_rank': place_ms_per_rank}
        tme = pl.timings(reset=True)
        e2e['stage_ms_per_step'] = {k: tme[k] / args.steps for k in ('h2d_ms', 'transpose_ms', 'rep_distance_ms', 'selection_ms',
                                                                      'placement_ms', 'd2h_ms')}

    # sha1 of every rank's block of result records (block r = the queries generated from seed 1000 + r): block 0 of an
    # N-GPU run must carry the hash the 1-GPU run prints, block 1 the hash the 2-GPU run prints for it, and so on
    import hashlib
    if world > 1:
        rec_all = gathered[0]
    else:
        pl.results_to_device(*send)
        rec_all = parallel.pack_records(*send)
    rec_np = rec_all.cpu().numpy()
    block_hashes = [hashlib.sha1(rec_np[r * nq:(r + 1) * nq].tobytes()).hexdigest()[:16] for r in range(world)]
    if world > 1 and e2e is not None:
        # the end-to-end (host buffers + gather) result must be the same records
        e2e_rec = parallel.pack_records(*[torch.from_numpy(np.ascontiguousarray(a)) for a in out_all]).numpy()
        e2e['result_equals_resident_path'] = bool((e2e_rec == rec_np).all())

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel (dense representative distances), per launch ----
    peaks = {}
    pk = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(pk):
        peaks = json.load(open(pk))
    hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
    peak_src = 'measured (MEASURED_PEAKS.json)' if 'hbm_gbs' in peaks else 'fallback (B200_PROFILING.md)'
    n_dense = max(tm['rep_distance_launches'], 1.0)
    dense_ms = tm['rep_distance_ms'] / n_dense
    W = _lib.load().apples_words_per_row(args.sites)
    n_rep = info['n_rep']
    q_per_launch = nq * args.steps / n_dense
    alg_bytes = (q_per_launch + n_rep) * 3 * W * 4 + 4.0 * q_per_launch * n_rep
    ach = alg_bytes / (dense_ms * 1e-3) / 1e9
    cell_sites = q_per_launch * n_rep * args.sites
    cs_rate = cell_sites / (dense_ms * 1e-3)
    sm_max = clocks.get('sm_max_mhz') or float(peaks.get('sm_max_mhz', 1965.0))
    sm_cur = clocks.get('sm_mhz') or sm_max
    # integer-pipe ceilings per SM and clock (profiles/microbench_r01.txt: POPC 16 lanes/clk/SM on the XU pipe, LOP3 64
    # lanes/clk/SM on the ALU pipe).  Per 32-site word pair the counting needs 3 LOP3 + 2 POPC; every carry-save step
    # trades 1 POPC for 2 LOP3.  With k steps per word pair the pipes take (3 + 2k) / 64 and (2 - k) / 16 clk: the
    # pipe-balanced optimum is k = 5/6, 13.71 word pairs/clk/SM -- that is the roofline (`peak`).  The kernel runs
    # k = 0.5 + 0.5 * 13/16 (distance.cu: DT_MCSA = 13), i.e. 4.8125 LOP3 + 1.09375 POPC: its own binding pipe is the ALU.
    def ceiling(word_pairs_per_clk_sm, mhz):
        return 148 * word_pairs_per_clk_sm * 32 * mhz * 1e6
    k_opt = 5.0 / 6.0
    bal_peak = ceiling(64 / (3 + 2 * k_opt), sm_max)
    k_run = 0.5 + 0.5 * 13 / 16
    alu_peak = ceiling(64 / (3 + 2 * k_run), sm_max)
    xu_peak = ceiling(16 / (2 - k_run), sm_max)
    plain_peak = ceiling(16 / 2.0, sm_max)
    traffic = None
    tpath = os.path.join(ROOT, 'profiles', 'dense_traffic_r01.json')
    if os.path.isfile(tpath):
        tj = json.load(open(tpath))
        # dram bytes of one ncu --set full capture, scaled from the captured launch's pair count to this run's
        traffic = tj['dram_bytes'] * (q_per_launch * n_rep) / tj['pairs']
    # top level = the BINDING resource of the dominant kernel (integer pipes); its HBM figures are nested under `hbm`
    roofline = {'kernel': 'dense_nuc_kernel<false> (query x representative mismatch/valid counts)', 'bound': 'int_pipe',
                'achieved': cs_rate / 1e12, 'peak': bal_peak / 1e12, 'unit': 'Tcell-sites/s', 'frac': cs_rate / bal_peak,
                'traffic': traffic, 'avg_launch_ms': dense_ms, 'launches': n_dense,
                'peak_model': 'no integer-pipe peak exists in MEASURED_PEAKS.json: peak = ALU/XU pipe-balanced optimum of '
                              'the 3 LOP3 + 2 POPC per 32-site word pair counting with carry-save steps (1 POPC <-> 2 '
                              'LOP3), LOP3 64 and POPC 16 lanes/clk/SM as measured by tools/microbench.cu '
                              '(profiles/microbench_r02.txt): 148 SMs x 13.71 word pairs/clk x %.0f MHz (max clock; '
                              'observed %.0f MHz)' % (sm_max, sm_cur),
                'alu_peak_this_mix': alu_peak / 1e12, 'frac_of_alu_peak': cs_rate / alu_peak,
                'xu_peak_this_mix': xu_peak / 1e12, 'frac_of_xu_peak': cs_rate / xu_peak,
                'plain_popcount_peak': plain_peak / 1e12, 'frac_of_plain_popcount_peak': cs_rate / plain_peak,
                'hbm': {'achieved': ach, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach / hbm_peak,
                        'peak_source': peak_src, 'algorithmic_bytes_per_launch': alg_bytes}}
    used_tc = tm.get('tensor_core_launches', 0) > 0
    if used_tc and not prot:
        # tensor-core kernel: one int8 dot product of K = 4 components x 32-site words per (query, representative)
        n_w = (args.sites + 31) // 32
        ops = 2.0 * q_per_launch * n_rep * n_w * 128
        tops = ops / (dense_ms * 1e-3) / 1e12
        bf16_burst = float(peaks.get('bf16_tflops', 1590.0))
        bf16_sust = float(peaks.get('bf16_tflops_sustained', 1400.0))
        nominal = 4500.0
        img_bytes = (q_per_launch + n_rep) * n_w * 128.0 + 4.0 * q_per_launch * n_rep
        fill_bytes = -(-q_per_launch // 256) * -(-n_rep // 256) * n_w * 65536.0
        read_bytes = fill_bytes * 1.5
        tc_traffic = None
        tpath = os.path.join(ROOT, 'profiles', 'dense_tc_traffic_r02.json')
        if os.path.isfile(tpath):
            # dram bytes of one ncu --set full capture of this kernel, scaled from the captured launch's pair count to this
            # run's.  4.6x the algorithmic bytes: the operand images are re-read from DRAM when the 148 tiles in flight
            # drift apart in K (L2 hit rate 68 %); at 2.2 TB/s it is a third of the HBM peak and not what binds the kernel
            tj = json.load(open(tpath))
            tc_traffic = tj['dram_bytes'] * (q_per_launch * n_rep) / tj['pairs']
        roofline = {'kernel': 'dense_tc_kernel (tcgen05.mma kind::i8, query x representative mismatch/valid counts as one int8 dot '
                              'product per pair)', 'bound': 'tensor', 'achieved': tops, 'peak': nominal, 'unit': 'TOP/s (int8)',
                    'frac': tops / nominal, 'traffic': tc_traffic, 'avg_launch_ms': dense_ms, 'launches': n_dense,
                    'peak_source': 'nominal dense int8 (4.5 POP/s = 2 x nominal bf16): MEASURED_PEAKS.json holds no int8 figure; '
                                   'against 2 x the measured bf16 GEMM (%s) the fraction is %.2f burst (2 x %.0f) / %.2f '
                                   'sustained (2 x %.0f)' % (peak_src, tops / (2 * bf16_burst), bf16_burst,
                                                             tops / (2 * bf16_sust), bf16_sust),
                    'algorithmic_ops_per_launch': ops,
                    # the resource that actually runs out: shared-memory bandwidth.  Per 32-site word a 256 x 256 tile writes
                    # 64 KB of operand images into shared memory (TMA) and its 8 MMAs (M = 128, N = 256, K = 32 bytes) read
                    # 4 KB of A and 8 KB of B each = 96 KB; the crossbar moves 128 B per clock and SM
                    'smem': {'achieved': (fill_bytes + read_bytes) / (dense_ms * 1e-3) / 1e9, 'peak': 148 * 128 * sm_max * 1e6 / 1e9,
                             'unit': 'GB/s', 'frac': (fill_bytes + read_bytes) / (dense_ms * 1e-3) / (148 * 128 * sm_max * 1e6),
                             'fill_bytes_per_launch': fill_bytes, 'operand_read_bytes_per_launch': read_bytes,
                             'peak_source': 'shared-memory crossbar 128 B/clk/SM (B300_MICROARCH.md) x 148 SMs x max SM clock; '
                                            'fills checked against ncu l1tex__m_xbar2l1tex_read_bytes (84.06 GB per 24 320-query '
                                            'launch, profiles/dense_tc_traffic_r02.json); at the full tensor rate the kernel '
                                            'would need 159 B/clk/SM, so 0.80 of the tensor peak is this design point\'s ceiling '
                                            'if no operand byte is reused inside the tensor core'},
                    'cell_sites_per_s': cs_rate, 'vs_int_pipe_balanced_peak': cs_rate / bal_peak,
                    'hbm': {'achieved': img_bytes / (dense_ms * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                            'frac': img_bytes / (dense_ms * 1e-3) / 1e9 / hbm_peak, 'peak_source': peak_src,
                            'algorithmic_bytes_per_launch': img_bytes}}
    if prot:
        # amino-acid dense kernel: one BLOSUM45 lookup (two conflict-free 32-bit shared-memory loads) per (query,
        # representative, site).  Bound by the shared-memory pipe: 32 banks x 4 B per clock per SM = one 32-lane LDS.32
        # wavefront per clock, two per 32 lookups -> 16 lookups/clk/SM.
        lookups = q_per_launch * n_rep * args.sites
        lk_rate = lookups / (dense_ms * 1e-3)
        lk_peak = 148 * 16 * sm_max * 1e6
        aa_bytes = (q_per_launch + n_rep) * args.sites + 8.0 * q_per_launch * n_rep
        roofline = {'kernel': 'dense_aa_kernel (query x representative scoredist, BLOSUM45 in shared memory)', 'bound': 'smem_pipe',
                    'achieved': lk_rate / 1e12, 'peak': lk_peak / 1e12, 'unit': 'Tlookups/s', 'frac': lk_rate / lk_peak,
                    'traffic': None, 'avg_launch_ms': dense_ms, 'launches': n_dense,
                    'peak_model': 'two 32-lane LDS.32 wavefronts per 32 table lookups (44-bit fixed-point BLOSUM45 in two limb '
                                  'tables, conflict-free by layout): 148 SMs x 16 lookups/clk x %.0f MHz' % sm_max,
                    'hbm': {'achieved': aa_bytes / (dense_ms * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                            'frac': aa_bytes / (dense_ms * 1e-3) / 1e9 / hbm_peak, 'peak_source': peak_src,
                            'algorithmic_bytes_per_launch': aa_bytes}}
    # selection and placement kernels: per 125k-query step from the stage timers (CUDA events around their launches)
    n_steps = args.steps
    K_avg = tm['observed'] / (nq * n_steps)
    V_avg = tm['valid_nodes'] / (nq * n_steps)
    sel_ms = tm['selection_ms'] / n_steps
    pla_ms = tm['placement_ms'] / n_steps
    sel_bytes = nq * ((8.0 if prot else 4.0) * n_rep + K_avg * (args.sites if prot else 3 * W * 4) + 16.0 * K_avg)   # key row + member rows + observed list
    pla_bytes = nq * (12.0 * K_avg + 20.0 * V_avg + 36.0)
    pla_flops = nq * 110.0 * V_avg
    roofline_select = {'kernel': 'select_nuc_kernel (all launches of a step incl. overflow reruns)', 'bound': 'hbm',
                       'achieved': sel_bytes / (sel_ms * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                       'frac': sel_bytes / (sel_ms * 1e-3) / 1e9 / hbm_peak, 'traffic': None, 'ms_per_step': sel_ms,
                       'algorithmic_bytes_per_step': sel_bytes, 'peak_source': peak_src}
    roofline_place = {'kernel': 'place_kernel (all launches of a step incl. overflow reruns)', 'bound': 'hbm',
                      'achieved': pla_bytes / (pla_ms * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                      'frac': pla_bytes / (pla_ms * 1e-3) / 1e9 / hbm_peak, 'traffic': None, 'ms_per_step': pla_ms,
                      'algorithmic_bytes_per_step': pla_bytes, 'peak_source': peak_src,
                      'fp64_gflops': pla_flops / (pla_ms * 1e-3) / 1e9,
                      'note': 'bound in practice by the dependency chain over tree levels (DESIGN.md 3b), neither by '
                              'HBM nor by the fp64 pipe'}
    step_ms = ms / args.steps
    row_bytes = _lib.load().apples_aa_row_bytes(args.sites) if prot else 3 * W * 4
    stages = {k: tm[k] / args.steps for k in ('h2d_ms', 'transpose_ms', 'rep_distance_ms', 'selection_ms', 'placement_ms', 'd2h_ms')}
    line = {'metric': 'queries placed/sec', 'value': value, 'unit': 'queries/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': step_ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': ('u8 codes, 44-bit fixed-point table sums + f64' if prot else
                      ('int8 (s32 accumulate) + f64' if used_tc else 'u32 popcount + f64')), 'data': 'synthetic',
            'config': {'workload': workload, 'dense_kernel': 'tensor' if used_tc else ('lookup' if prot else 'intpipe'), 'n_representatives': n_rep, 'queries_per_step': nq * world,
                       'l2': 'inputs larger than L2 (packed queries %.0f MB + packed reference %.0f MB per GPU)'
                             % (nq * row_bytes / 1e6, (args.leaves + n_rep) * row_bytes / 1e6),
                       'parallelism': 'queries sharded over %d GPU(s), reference + tree replicated, final NCCL all-gather' % world},
            'distance_gcell_sites_per_s': (tm['pairs'] / args.steps) * args.sites / (step_ms * 1e-3) / 1e9 * world,
            'stage_ms_per_step': stages, 'rep_distance_sm_mhz': tm.get('rep_distance_sm_mhz'), 'per_rank': per_rank, 'pairs_per_query': tm['pairs'] / (nq * args.steps),
            'observed_per_query': tm['observed'] / (nq * args.steps), 'valid_nodes_per_query': tm['valid_nodes'] / (nq * args.steps),
            'overflow_queries_per_step': tm['overflow_queries'] / args.steps,
            'placement_classes_per_step': {k: tm[k] / args.steps for k in ('placed_smem64', 'placed_smem128', 'placed_smem256', 'placed_smem512', 'placed_block')}, 'max_observed': tm['max_observed'],
            'max_valid_nodes': tm['max_valid_nodes'], 'gpu_launches': int(tm['launches']), 'result_sha1_per_block': block_hashes, 'clocks': clocks, 'e2e': e2e, 'roofline': roofline, 'roofline_select': roofline_select,
            'roofline_place': roofline_place, 'setup': info}

    # ---- the command line end to end (rank 0, N = 1): FASTA text on disk -> run_apples.py -> jplace on disk ----
    if not args.no_cli and world == 1 and host is not None:
        line['cli_e2e'] = cli_e2e(args, tree, host, q_bytes, local_rank)

    # ---- CPU baseline (rank 0, N = 1 only): bounded sample of the same queries ----
    if not args.no_cpu_baseline and world == 1:
        n_sample = args.cpu_sample or max(threads * 8, 64)
        # the sample is drawn across the whole batch and always holds queries of the overflow set (observed set larger
        # than the slot: key-row stash, gather, rerun selection and placement)
        edge, error, distal, pendant, status = pl.download_results()
        Kq, Vq, over = pl.last_counts(nq)
        rng = np.random.default_rng(12345)
        ov_idx = np.flatnonzero(over == 1)
        n_ov = min(len(ov_idx), max(1, n_sample // 8))
        pick = np.concatenate([rng.choice(ov_idx, n_ov, replace=False) if n_ov else np.zeros(0, np.int64),
                               rng.choice(np.flatnonzero(over == 0), n_sample - n_ov, replace=False)]).astype(np.int64)
        q_host = q_bytes[torch.from_numpy(pick).to(q_bytes.device)].cpu().numpy()
        rate, dt, res = cpu_baseline(cpu_context(args, tree, host), q_host, threads)
        # parity of the timed GPU results on that sample: edge identical, error / distal / pendant within 1e-9
        def near(a, b, floor):
            return abs(a - b) <= 1e-9 * max(abs(a), abs(b)) + floor
        same = 0
        for i, r in zip(pick.tolist(), res):
            p = r[0]['placements'][0]['p'][0]
            pend = 0.0 if int(status[i]) & 0x100 else float(pendant[i])
            if (p[0] == int(edge[i]) and near(p[1], float(error[i]), 1e-12) and near(p[3], float(distal[i]), 1e-15)
                    and near(p[4], pend, 1e-15)):
                same += 1
        line['cpu_baseline'] = {'value': rate, 'unit': 'queries/s', 'cores': threads, 'kind': 'port',
                                'sample': '%d of this step\'s queries, drawn across the batch (%d of them from the '
                                          'overflow-rerun set), through the oracle port of PoolQueryWorker.runquery '
                                          'under a fork pool of %d processes (%.1f s)' % (n_sample, n_ov, threads, dt),
                                'parity_on_sample': '%d/%d identical edge; error, distal and pendant within 1e-9 '
                                                    '(%d overflow-rerun queries in the sample)' % (same, n_sample, n_ov)}
    if last_step is not None:
        dump_outputs(args.dump_outputs, last_step)
    emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    sys.exit(main())
