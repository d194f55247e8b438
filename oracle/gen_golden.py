"""Generates tests/golden/*.json by running the UNMODIFIED reference (a checkout of the original APPLES, named by the
environment variable APPLES_REFERENCE) and asserts that oracle/apples_oracle.py reproduces it bit for bit.  TEST
INFRASTRUCTURE.

Run:  APPLES_REFERENCE=<checkout of APPLES> python oracle/gen_golden.py

What is the reference here and what is substituted:
  * everything under $APPLES_REFERENCE/apples is imported unmodified;
  * `treeswift` (absent dependency) is oracle/treeswift_shim;
  * `TreeCluster.py` (absent dependency) cannot run, so the cluster TSV is produced by apples_b200.treecluster and
    fed to the reference's own parsing + PoolRepresentativeWorker code (Reference.py:94-107), i.e. a
    ReducedReference instance is assembled without calling its __init__ (which would shell out).
Floats are stored as float.hex() strings so the vectors are exact.

The INPUTS of every case are the committed fixtures under tests/golden/data/ (and tests/golden/c1_clusters*.tsv): the
script reads them, it does not regenerate them, so the vectors stay pinned whatever apples_b200.synth or
apples_b200.treecluster become.  `--regen-inputs` rebuilds the synthetic inputs (syn300*, prot_*) and the cluster TSVs
from their seeds first (only when a fixture is to be replaced on purpose).  `--check` writes nothing: it regenerates
every vector into a scratch directory and fails if any committed tests/golden/*.json would change
(tests/test_oracle_golden.py::test_golden_recipe_reproduces_committed_vectors runs it where APPLES_REFERENCE is set).
"""
import gzip
import itertools
import json
import os
import shutil
import sys
import types
import warnings

import numpy as np

warnings.filterwarnings('ignore')
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, '..'))
REFERENCE = os.environ.get('APPLES_REFERENCE', '')
sys.path.insert(0, os.path.join(HERE, 'treeswift_shim'))
sys.path.insert(0, REFERENCE)
sys.path.insert(0, ROOT)

from apples.PoolQueryWorker import PoolQueryWorker  # noqa: E402
from apples.PoolRepresentativeWorker import PoolRepresentativeWorker  # noqa: E402
from apples.Reference import ReducedReference  # noqa: E402
from apples.Subtree import Subtree  # noqa: E402
from apples import distance as ref_distance  # noqa: E402
from apples.fasta2dic import fasta2dic as ref_fasta2dic  # noqa: E402
from apples.prepareTree import prepareTree  # noqa: E402
from apples.jutil import join_jplace  # noqa: E402
from apples.FM import FM  # noqa: E402
from apples.OLS import OLS  # noqa: E402
from apples.BME import BME  # noqa: E402
from apples.BE import BE  # noqa: E402

from oracle import apples_oracle as orc  # noqa: E402
from apples_b200 import synth, treecluster  # noqa: E402
from apples_b200.tree import BackboneTree  # noqa: E402

GOLD = os.path.join(ROOT, 'tests', 'golden')
DATA = os.path.join(GOLD, 'data')
OUT = GOLD   # --check redirects the vectors to a scratch directory
REF_DATA = os.path.join(REFERENCE, 'data')
ALGS = {'FM': FM, 'OLS': OLS, 'BME': BME, 'BE': BE}


def hx(v):
    """exact encoding: ints stay ints, floats become hex strings"""
    if isinstance(v, (int, np.integer)) and not isinstance(v, bool):
        return int(v)
    return float(v).hex()


def make_options(tree_fp, method='FM', criterion='MLSE', negative=False, baseobs=25, filt=0.2, overlap=0.001,
                 exclude=False):
    o = types.SimpleNamespace()
    o.tree_fp = tree_fp
    o.reestimate_backbone = False
    o.method_name = method
    o.criterion_name = criterion
    o.negative_branch = negative
    o.base_observation_threshold = baseobs
    o.filt_threshold = filt
    o.minimum_alignment_overlap = overlap
    o.exclude_intplace = exclude
    return o


def reference_reduced(refs, prot, tsv, threshold, baseobs):
    """A reference ReducedReference built by the reference's own code from an explicit TreeCluster TSV."""
    r = ReducedReference.__new__(ReducedReference)
    r.refs = refs
    r.prot_flag = prot
    r.dist_function = ref_distance.scoredist if prot else ref_distance.jc69
    r.threshold = threshold
    with open(tsv) as tc_output:  # Reference.py:94-107
        tc_output.readline()
        lines = map(lambda x: x.strip().split('\t'), tc_output.readlines())
        lines_sorted = sorted(lines, key=lambda x: x[1])
        clusters = [(key, [i[0] for i in list(group)]) for key, group in itertools.groupby(lines_sorted, lambda x: x[1])]
    w = PoolRepresentativeWorker()
    w.set_class_attributes(refs, prot)
    results = [w.worker(c) for c in clusters]
    r.representatives = [item for sub in results for item in sub]
    r.set_baseobs(baseobs)
    return r


def run_case(name, tree_fp, options, queries, reference=None, prot=False, detail_n=3, extra=None):
    """queries: list of (name, seq or None, row-dict or None).  Runs the reference and the oracle."""
    first_tree, name_to_node, ext_newick = prepareTree(options)
    worker = PoolQueryWorker()
    worker.set_class_attributes(reference, options, name_to_node)
    # oracle side
    otree, onames = orc.load_tree(tree_fp)
    octx = orc.OracleContext(otree, onames, refs=None if reference is None else reference.refs,
                             representatives=None if reference is None else reference.representatives,
                             protein=prot, method=options.method_name, criterion=options.criterion_name,
                             negative_branch=options.negative_branch, filt_threshold=options.filt_threshold,
                             baseobs=options.base_observation_threshold, overlap=options.minimum_alignment_overlap,
                             exclude_intplace=options.exclude_intplace)
    out = {'case': name, 'options': vars(options).copy(), 'queries': []}
    out['options']['tree_fp'] = os.path.basename(tree_fp)
    if extra:
        out.update(extra)
    results = []
    stderr_keep = sys.stderr
    for qi, (qname, qseq, row) in enumerate(queries):
        # observed set exactly as runquery computes it (PoolQueryWorker.py:40-59)
        if row:
            obs_ref = orc_observed_matrix_via_reference(row, name_to_node, options)
        else:
            obs_ref = reference.get_obs_dist(qseq, qname, options.minimum_alignment_overlap)
        sys.stderr = open(os.devnull, 'w')
        try:
            res = worker.runquery(qname, qseq, dict(row) if row else None)
        finally:
            sys.stderr.close()
            sys.stderr = stderr_keep
        results.append(res)
        det = {}
        ores, ostatus = octx.runquery(qname, qseq, dict(row) if row else None, detail=det)
        assert json.dumps(ores, sort_keys=True) == json.dumps(res, sort_keys=True), (name, qname, ores, res)
        # observed order (before self removal) must match too
        if row:
            oobs = orc.observed_matrix(row, onames, options.filt_threshold, options.base_observation_threshold)
        else:
            oobs = orc.observed_alignment(qseq, reference.representatives, reference.refs, octx.dist_fn,
                                          options.filt_threshold, options.base_observation_threshold,
                                          options.minimum_alignment_overlap)
        assert list(oobs.items()) == list(obs_ref.items()), (name, qname)
        p = res['placements'][0]['p'][0]
        rec = {'name': qname, 'out_name': res['placements'][0]['n'][0], 'p': [hx(x) for x in p], 'status': ostatus,
               'observed': [[k, hx(v)] for k, v in obs_ref.items()]}
        if qi < detail_n and ostatus in (orc.PLACED, orc.PLACED_MISPLACEMENT_FLAG):
            # per-edge values from the reference's own classes (PoolQueryWorker.py:101-119)
            obs2 = dict(obs_ref)
            if qname in name_to_node:
                obs2.pop(qname, None)
            st = Subtree(obs2, name_to_node)
            alg = ALGS.get(options.method_name, OLS)(st)
            alg.dp_frag()
            alg.placement_per_edge(options.negative_branch)
            edges = {}
            for n in filter(lambda x: x.valid, st.traverse_postorder()):
                edges[n.edge_index] = [hx(n.x_1), hx(n.x_2), hx(alg.error_per_edge(n))]
            rec['num_nodes'] = st.num_nodes
            st.unroll_changes()
            oedges = {k: [hx(v[0]), hx(v[1]), hx(v[2])] for k, v in det['edges'].items()}
            assert oedges == edges, (name, qname)
            assert det['num_nodes'] == rec['num_nodes']
            rec['edges'] = {str(k): v for k, v in edges.items()}
        out['queries'].append(rec)
    joined = join_jplace([json.loads(json.dumps(r)) for r in results])
    out['joined_names'] = [pl['n'][0] for pl in joined['placements']]
    out['extended_newick_sha'] = __import__('hashlib').sha256(ext_newick.encode()).hexdigest()
    # product tree layout agrees with the reference's numbering / newick
    bt = BackboneTree.from_newick(tree_fp)
    assert bt.extended_newick() == ext_newick, name
    for lbl, node in name_to_node.items():
        assert bt.name_to_node[lbl] == node.edge_index and bt.level[node.edge_index] == node.level
    with open(os.path.join(OUT, name + '.json'), 'w') as f:
        json.dump(out, f, indent=0, sort_keys=True)
    print('wrote', name, len(out['queries']), 'queries')
    return out


def orc_observed_matrix_via_reference(row, name_to_node, options):
    """The reference's valid_dists is a closure inside runquery (PoolQueryWorker.py:44-59); re-evaluated here through
    the same statements to record the observed set it produces."""
    tx = 0
    out = {}
    for k, v in sorted(row.items(), key=lambda kv: kv[1]):
        if v < 0 or k not in name_to_node:
            continue
        tx += 1
        if tx > options.base_observation_threshold and v > options.filt_threshold:
            break
        out[k] = v
    return out


def read_dismat(path):
    import re
    with open(path) as f:
        tags = list(re.split(r"\s+", f.readline().rstrip()))[1:]
        rows = []
        for line in f.readlines():
            d = list(re.split(r"\s+", line.strip()))
            rows.append((d[0], None, dict(zip(tags, map(float, d[1:])))))
    return rows


def copy_data():
    os.makedirs(DATA, exist_ok=True)
    for rel in ['ref.fa', 'query.fa', 'backbone.nwk', 'dist.mat', 'small_backbone.nwk', 'small_dist.mat',
                'prot/backbone.nwk']:
        dst = os.path.join(DATA, rel.replace('/', '_') + '.gz')
        with open(os.path.join(REF_DATA, rel), 'rb') as fi, gzip.GzipFile(dst, 'wb', mtime=0) as fo:
            shutil.copyfileobj(fi, fo)


def save_gz(src_path, name):
    with open(src_path, 'rb') as fi, gzip.GzipFile(os.path.join(DATA, name + '.gz'), 'wb', mtime=0) as fo:
        shutil.copyfileobj(fi, fo)


def cluster_tsv_for(tree_fp, threshold, out_path):
    bt = BackboneTree.from_newick(tree_fp)
    cl = treecluster.max_diameter_clusters(bt, threshold * 1.2)
    treecluster.write_cluster_tsv(bt, cl, out_path)
    return bt


def gunzip_to(name, workdir):
    dst = os.path.join(workdir, name)
    with gzip.open(os.path.join(DATA, name + '.gz'), 'rb') as fi, open(dst, 'wb') as fo:
        fo.write(fi.read())
    return dst


def regen_inputs(tmp):
    """Rebuilds the synthetic inputs and cluster TSVs from their seeds (replaces committed fixtures: on purpose only)."""
    copy_data()
    tree_fp = os.path.join(REF_DATA, 'backbone.nwk')
    cluster_tsv_for(tree_fp, 0.2, os.path.join(GOLD, 'c1_clusters.tsv'))
    cluster_tsv_for(tree_fp, 0.45, os.path.join(GOLD, 'c1_clusters_f045.tsv'))
    nwk = synth.random_tree(300, seed=11, polytomy_frac=0.15, zero_frac=0.05, neg_frac=0.03)
    tfp = os.path.join(tmp, 'syn300.nwk')
    open(tfp, 'w').write(nwk + '\n')
    bt = BackboneTree.from_newick(tfp)
    srefs, leaf_states = synth.evolve_alignment(bt, 600, seed=12)
    sq, _ = synth.make_queries(bt, leaf_states, 40, seed=13)
    cluster_tsv_for(tfp, 0.2, os.path.join(tmp, 'syn300.tsv'))
    synth.write_fasta(srefs, os.path.join(tmp, 'syn300_ref.fa'))
    synth.write_fasta(sq, os.path.join(tmp, 'syn300_query.fa'))
    ptree = os.path.join(REF_DATA, 'prot', 'backbone.nwk')
    pbt = BackboneTree.from_newick(ptree)
    prefs, pstates = synth.evolve_alignment(pbt, 400, seed=21, protein=True)
    pq, _ = synth.make_queries(pbt, pstates, 12, seed=22, protein=True)
    cluster_tsv_for(ptree, 0.6, os.path.join(tmp, 'prot.tsv'))
    synth.write_fasta(prefs, os.path.join(tmp, 'prot_ref.fa'))
    synth.write_fasta(pq, os.path.join(tmp, 'prot_query.fa'))
    for fn in ['syn300.nwk', 'syn300.tsv', 'syn300_ref.fa', 'syn300_query.fa', 'prot.tsv', 'prot_ref.fa', 'prot_query.fa']:
        save_gz(os.path.join(tmp, fn), fn)


def main(argv=None):
    global OUT
    argv = sys.argv[1:] if argv is None else argv
    check = '--check' in argv
    tmp = '/tmp/apples_golden'
    os.makedirs(tmp, exist_ok=True)
    if '--regen-inputs' in argv:
        if check:
            raise SystemExit('--check and --regen-inputs exclude each other')
        regen_inputs(tmp)
    if check:
        OUT = os.path.join(tmp, 'check')
        shutil.rmtree(OUT, ignore_errors=True)
        os.makedirs(OUT)
    # the reference's own example files must still be what the fixtures hold
    for rel in ['ref.fa', 'query.fa', 'backbone.nwk', 'dist.mat', 'small_backbone.nwk', 'small_dist.mat', 'prot/backbone.nwk']:
        with open(os.path.join(REF_DATA, rel), 'rb') as fi, gzip.open(os.path.join(DATA, rel.replace('/', '_') + '.gz'), 'rb') as fg:
            assert fi.read() == fg.read(), 'fixture %s differs from the reference file' % rel

    # ---------------- small 5-leaf case: every method x criterion x negative (SURVEY 8c item 3)
    small_tree = os.path.join(REF_DATA, 'small_backbone.nwk')
    small_rows = read_dismat(os.path.join(REF_DATA, 'small_dist.mat'))
    for m in ['FM', 'OLS', 'BME', 'BE']:
        for c in ['MLSE', 'ME', 'HYBRID']:
            for neg in [False, True]:
                run_case('small_%s_%s_%s' % (m, c, 'neg' if neg else 'pos'), small_tree,
                         make_options(small_tree, m, c, neg), small_rows, detail_n=1)

    # ---------------- config 2: data/dist.mat
    tree_fp = os.path.join(REF_DATA, 'backbone.nwk')
    rows = read_dismat(os.path.join(REF_DATA, 'dist.mat'))
    run_case('c2_matrix_FM_MLSE', tree_fp, make_options(tree_fp), rows)
    run_case('c2_matrix_OLS_HYBRID_f100', tree_fp, make_options(tree_fp, 'OLS', 'HYBRID', filt=100.0), rows, detail_n=1)
    run_case('c2_matrix_BME_ME_b5', tree_fp, make_options(tree_fp, 'BME', 'ME', baseobs=5, filt=0.05), rows, detail_n=1)
    run_case('c2_matrix_BE_MLSE_neg', tree_fp, make_options(tree_fp, 'BE', 'MLSE', negative=True), rows, detail_n=1)

    # ---------------- config 1: data/ref.fa + query.fa, clusters from the committed TSV (TreeCluster.py is absent)
    refs = ref_fasta2dic(os.path.join(REF_DATA, 'ref.fa'), False, False)
    queries = ref_fasta2dic(os.path.join(REF_DATA, 'query.fa'), False, False)
    tsv = os.path.join(GOLD, 'c1_clusters.tsv')
    rr = reference_reduced(refs, False, tsv, 0.2, 25)
    qlist = [(k, v, None) for k, v in queries.items()]
    # raw counts for every query x reference pair (distance.py:733-737) -- pins kernel (a) bit-exactly
    names = list(refs.keys())
    counts = []
    for k, v in queries.items():
        row = []
        for n in names:
            b = refs[n]
            nd = np.logical_and(v != b'-', b != b'-')
            row.append([int(np.count_nonzero(np.logical_and(v != b, nd))), int(np.count_nonzero(nd))])
        counts.append(row)
    run_case('c1_align_FM_MLSE', tree_fp, make_options(tree_fp), qlist, rr, extra={'counts': counts, 'ref_names': names})
    rr = reference_reduced(refs, False, tsv, 0.2, 25)
    run_case('c1_align_OLS_MLSE', tree_fp, make_options(tree_fp, 'OLS'), qlist, rr, detail_n=1)
    run_case('c1_align_BME_HYBRID', tree_fp, make_options(tree_fp, 'BME', 'HYBRID'), qlist, rr, detail_n=1)
    run_case('c1_align_BE_ME', tree_fp, make_options(tree_fp, 'BE', 'ME'), qlist, rr, detail_n=1)
    tsv45 = os.path.join(GOLD, 'c1_clusters_f045.tsv')
    rr45 = reference_reduced(refs, False, tsv45, 0.45, 5)
    run_case('c1_align_FM_MLSE_f045_b5', tree_fp, make_options(tree_fp, baseobs=5, filt=0.45), qlist, rr45, detail_n=1)
    # a reference sequence used as a query under its own name (PoolQueryWorker.py:63-70) and a copy under a new name
    # (zero-distance shortcut, PoolQueryWorker.py:72-75), an all-gap query and a nearly-all-gap query
    some = names[17]
    gap = np.frombuffer(b'-' * len(refs[some]), dtype='S1')
    thin = gap.copy()
    thin[100:103] = refs[names[3]][100:103]
    special = [(some, refs[some], None), ('copy_of_' + names[40], refs[names[40]], None), ('allgap', gap, None),
               ('thin', thin, None)]
    rr = reference_reduced(refs, False, tsv, 0.2, 25)
    run_case('c1_align_special', tree_fp, make_options(tree_fp), special, rr, detail_n=4)
    run_case('c1_align_special_exclude', tree_fp, make_options(tree_fp, exclude=True), special + qlist[:3], rr, detail_n=0)

    # ---------------- synthetic nucleotide with polytomies, zero and negative edges (committed fixture inputs)
    tfp = gunzip_to('syn300.nwk', tmp)
    srefs = ref_fasta2dic(gunzip_to('syn300_ref.fa', tmp), False, False)
    sq = ref_fasta2dic(gunzip_to('syn300_query.fa', tmp), False, False)
    stsv = gunzip_to('syn300.tsv', tmp)
    sql = [(k, v, None) for k, v in sq.items()]
    gen = {'generator': {'tree': dict(n_leaves=300, seed=11, polytomy_frac=0.15, zero_frac=0.05, neg_frac=0.03),
                         'L': 600, 'aln_seed': 12, 'n_queries': 40, 'q_seed': 13, 'cluster_threshold': 0.2}}
    for m in ['FM', 'OLS', 'BME', 'BE']:
        for c in ['MLSE', 'ME', 'HYBRID']:
            for neg in ([False, True] if c == 'MLSE' else [False]):
                rr = reference_reduced(srefs, False, stsv, 0.2, 25)
                run_case('syn300_%s_%s_%s' % (m, c, 'neg' if neg else 'pos'), tfp,
                         make_options(tfp, m, c, neg), sql, rr, detail_n=2, extra=gen)

    # ---------------- protein: the reference's real 4038-leaf tree (polytomies, negative edges), synthetic alignment
    ptree = os.path.join(REF_DATA, 'prot', 'backbone.nwk')
    prefs = ref_fasta2dic(gunzip_to('prot_ref.fa', tmp), True, False)
    pq = ref_fasta2dic(gunzip_to('prot_query.fa', tmp), True, False)
    ptsv = gunzip_to('prot.tsv', tmp)
    pgen = {'generator': {'L': 400, 'aln_seed': 21, 'n_queries': 12, 'q_seed': 22, 'cluster_threshold': 0.6}}
    prr = reference_reduced(prefs, True, ptsv, 0.6, 25)
    pql = [(k, v, None) for k, v in pq.items()]
    # scoredist values for query 0 against the first 64 references (1e-9 parity target, BLAS summation order)
    pn = list(prefs.keys())[:64]
    sd = [hx(ref_distance.scoredist(pql[0][1], prefs[n], 0.001)) for n in pn]
    pgen['scoredist_q0'] = {'refs': pn, 'd': sd}
    run_case('c3_prot_FM_MLSE', ptree, make_options(ptree, filt=0.6), pql, prr, prot=True, detail_n=1, extra=pgen)
    run_case('c3_prot_OLS_MLSE', ptree, make_options(ptree, 'OLS', filt=0.6), pql, prr, prot=True, detail_n=1, extra=pgen)

    if check:
        committed = sorted(f for f in os.listdir(GOLD) if f.endswith('.json'))
        made = sorted(os.listdir(OUT))
        bad = [f for f in committed if f not in made]
        bad += [f for f in made if f not in committed]
        for f in made:
            if f in committed and open(os.path.join(OUT, f), 'rb').read() != open(os.path.join(GOLD, f), 'rb').read():
                bad.append(f)
        if bad:
            print('golden vectors that would change:', ' '.join(sorted(set(bad))))
            raise SystemExit(1)
        print('check ok: %d committed golden vectors are reproduced byte for byte by the unmodified reference' % len(made))


if __name__ == '__main__':
    main()
