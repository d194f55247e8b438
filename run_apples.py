#!/usr/bin/env python3
"""run_apples.py with the per-query worker pool replaced by the B200 hot path.

Same options, inputs and jplace output as the reference's run_apples.py; the one changed call is
`pool.starmap(queryworker.runquery, queries)` (reference run_apples.py:94-102) -> apples_b200.placer.place_batch.
"""
import logging
import os

import numpy as np
import pickle
import re
import sys
import time

from apples_b200 import jplace
from apples_b200.fasta import read_alignment
from apples_b200.options import options_config_run
from apples_b200.placer import log_messages, place_alignment, place_batch, visible_devices
from apples_b200.reference import ReducedReference
from apples_b200.tree import prepare_tree


def read_dismat(f):
    """run_apples.py:43-54"""
    tags = list(re.split(r"\s+", f.readline().rstrip()))[1:]
    for line in f.readlines():
        dists = list(re.split(r"\s+", line.strip()))
        yield (dists[0], None, dict(zip(tags, map(float, dists[1:]))))


LAST_TIMINGS = {}   # wall-clock seconds of the stages of the last main() call (bench.py reports them as cli_e2e)


def main(argv=None):
    startb = time.time()
    LAST_TIMINGS.clear()
    options, args = options_config_run(argv)
    logging.info('[%s] Options are parsed.' % time.strftime('%H:%M:%S'))
    tree = name_to_node_map = extended_newick_string = None
    up = fdtb = None
    # One process per GPU under torchrun (WORLD_SIZE > 1): every rank places its block of queries on its own GPU, the
    # blocks are exchanged with one NCCL all-gather and rank 0 writes the output.  Otherwise the queries are sharded
    # over --gpus devices inside this process (0 = all visible: the analogue of upstream's -T 0 = all cores).
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = 0
    if world > 1:
        import torch
        import torch.distributed as dist
        local = int(os.environ.get('LOCAL_RANK', '0'))
        if torch.cuda.is_available():
            torch.cuda.set_device(local)
            dist.init_process_group('nccl', device_id=torch.device('cuda:%d' % local))
        else:
            dist.init_process_group('gloo')
        rank = dist.get_rank()
        devices = [local]
    else:
        devices = visible_devices(options.device, options.num_gpus)
    if options.database_fp:
        start = time.time()
        fdtb = open(options.database_fp, 'rb')
        up = pickle.Unpickler(fdtb)
        try:
            tree = up.load()
            name_to_node_map = up.load()
            extended_newick_string = up.load()
        except (ModuleNotFoundError, AttributeError, EOFError, pickle.UnpicklingError) as e:
            # upstream databases pickle treeswift.Tree / apples.Reference objects, which this build does not contain
            raise SystemExit('%s is not a database written by this build\'s build_applesdtb.py (%s); databases pickled '
                             'by upstream APPLES hold treeswift / apples.* objects and cannot be loaded here: rebuild it '
                             'with build_applesdtb.py' % (options.database_fp, e))
        if not hasattr(tree, 'parent') or not hasattr(tree, 'first'):
            raise SystemExit('%s does not hold a tree written by this build\'s build_applesdtb.py' % options.database_fp)
        logging.info('[%s] Tree is loaded from APPLES database in %.3f seconds.' % (time.strftime('%H:%M:%S'),
                                                                                   time.time() - start))
    if options.tree_fp:
        tree, name_to_node_map, extended_newick_string = prepare_tree(options.tree_fp)

    if options.dist_fp:
        reference = None
        start = time.time()
        with open(options.dist_fp) as f:
            queries = list(read_dismat(f))
    else:
        start = time.time()
        if options.ref_fp:
            reference = ReducedReference(options.ref_fp, options.protein_seqs, options.tree_fp, options.filt_threshold,
                                         options.num_thread, cluster_tsv=options.cluster_fp, tree=tree)
            logging.info('[%s] Reduced reference is computed in %.3f seconds.' % (time.strftime('%H:%M:%S'),
                                                                                  time.time() - start))
        else:
            try:
                reference = up.load()
            except (ModuleNotFoundError, AttributeError, EOFError, pickle.UnpicklingError) as e:
                raise SystemExit('%s: the reduced reference was not pickled by this build (%s); rebuild the database with '
                                 'build_applesdtb.py' % (options.database_fp, e))
            fdtb.close()
            logging.info('[%s] Reduced reference is loaded from APPLES database in %.3f seconds.'
                         % (time.strftime('%H:%M:%S'), time.time() - start))
        reference.set_baseobs(options.base_observation_threshold)
        LAST_TIMINGS['setup_s'] = time.time() - startb
        start = time.time()
        # native reader (hostio.cpp): the whole query file becomes one (pinned) byte matrix, no per-query objects
        # (pageable memory: pinning 5 GB for a single pass costs more than the staged copy it would save)
        fm = read_alignment(options.query_fp or options.extended_ref_fp, options.protein_seqs, options.mask_lowconfidence,
                            pinned=False)
        if not fm.uniform:
            raise ValueError('the sequences of %s do not all have the same length' % (options.query_fp or options.extended_ref_fp))
        q_names, q_mat = fm.names, fm.matrix
        if len(set(q_names)) != len(q_names):
            # duplicate names: a dict keeps the first position and the last sequence (fasta2dic.py:71)
            d = fm.as_dict(copy=False)
            q_names = list(d.keys())
            q_mat = np.vstack([d[k].view(np.uint8) for k in q_names]) if q_names else q_mat[:0]
        if not options.query_fp:
            keep = [i for i, k in enumerate(q_names) if k not in reference.refs]   # run_apples.py:82-83
            q_names = [q_names[i] for i in keep]
            q_mat = q_mat[np.asarray(keep, dtype=np.int64)] if keep else q_mat[:0]
        queries = None
    logging.info('[%s] Query sequences are prepared in %.3f seconds.' % (time.strftime('%H:%M:%S'), time.time() - start))
    LAST_TIMINGS['read_queries_s'] = time.time() - start

    startq = time.time()
    if queries is not None:
        # distance-matrix input: the per-query dict interface of the reference (pool.starmap(runquery) drop-in)
        results = place_batch(reference, options, name_to_node_map, queries, tree=tree, devices=devices,
                              keep=options.keep_at_most)
        n_q = len(queries)
    else:
        # alignment input: byte matrix -> result arrays -> jplace text, all native
        in_backbone, out, *alt = place_alignment(reference, options, name_to_node_map, q_names, q_mat, tree=tree,
                                                 devices=devices, keep=options.keep_at_most) \
            if len(q_names) else (np.zeros(0, bool), None)
        alt = alt[0] if alt else None   # ranked records (--keep-at-most > 1)
        n_q = len(q_names)
    logging.info('[%s] Processed all queries in %.3f seconds on %d GPU(s).' % (time.strftime('%H:%M:%S'),
                                                                               time.time() - startq, max(world, len(devices))))
    LAST_TIMINGS['place_s'] = time.time() - startq
    LAST_TIMINGS['queries'] = n_q
    startw = time.time()
    if rank == 0:
        if queries is not None or n_q == 0:
            if n_q == 0:
                raise IndexError('list index out of range')   # join_jplace(results)[0] of an empty list, as upstream
            jplace.write(jplace.assemble(results, extended_newick_string), options.output_fp)
        else:
            log_messages(q_names, in_backbone, out, options.exclude_intplace)
            if options.output_fp:
                jplace.write_arrays(options.output_fp, q_names, in_backbone, out, extended_newick_string, options.exclude_intplace,
                                    alt=alt)
            else:
                from apples_b200.placer import results_to_jplace
                res = results_to_jplace(q_names, in_backbone.tolist(), out, options.exclude_intplace, log=False, alt=alt)
                jplace.write(jplace.assemble(res, extended_newick_string), None)
        LAST_TIMINGS['write_s'] = time.time() - startw
        LAST_TIMINGS['total_s'] = time.time() - startb
        logging.warning('[%s] APPLES finished in %.3f seconds.' % (time.strftime('%H:%M:%S'), time.time() - startb))
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
