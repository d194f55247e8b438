"""Command-line options: the same flags, defaults and validation as apples/OptionsBasic.py:7-92,
apples/OptionsRun.py:5-112 and apples/OptionsBuild.py:4-10, plus two additions that do not exist upstream:
  --clusters FILE   TreeCluster-format TSV to use instead of running a clustering (TreeCluster.py is an external
                    dependency of the reference, Reference.py:87-88)
  --device N        first CUDA device ordinal (default 0); -T/--threads is accepted and ignored (no CPU workers);
  --gpus N          GPUs to shard the queries over (0 = all visible: the analogue of upstream's -T 0 = all cores);
  --keep-at-most K  report the best K placements of each query (pplacer's name; default 1), ranked by the criterion;
  --model M         nucleotide distance of alignment input: JC69 (upstream's, default) or K2P (Kimura two-parameter).
Backbone re-estimation with FastTree (reestimateBackbone.py) is outside the hot path: it is never run here, as with
the reference's -D flag; without -D a warning says that results can differ from upstream's default.
"""
import logging
from optparse import OptionParser

__version__ = '2.0.11+b200'


def _basic(output_filetype):
    p = OptionParser()
    p.add_option('-t', '--tree', dest='tree_fp', help='path to the reference tree', metavar='FILE')
    p.add_option('-o', '--output', dest='output_fp', help='path for the output %s file' % output_filetype, metavar='FILE')
    p.add_option('-s', '--ref', dest='ref_fp', metavar='FILE',
                 help='path to the reference alignment file (FASTA), containing reference sequences')
    p.add_option('-p', '--protein', dest='protein_seqs', action='store_true', default=False,
                 help='input sequences are protein sequences')
    p.add_option('-T', '--threads', dest='num_thread', type=int, default=0, metavar='NUMBER',
                 help='accepted for compatibility; placement runs on the GPU')
    p.add_option('-f', '--filter', dest='filt_threshold', type=float, default=0.2, metavar='NUMBER',
                 help='ignores distances higher than the given threshold.')
    p.add_option('-D', '--disable-reestimation', dest='disable_reestimation', action='store_true', default=False,
                 help='accepted for compatibility; backbone re-estimation is never run by this build')
    p.add_option('--debug', dest='debug_mode', action='store_true', default=False, help='Enables debug mode.')
    p.add_option('-v', '--version', dest='print_version', action='store_true', default=False,
                 help='print APPLES version number. ')
    p.add_option('--clusters', dest='cluster_fp', metavar='FILE', help='TreeCluster-format cluster TSV')
    p.add_option('--device', dest='device', type=int, default=0, metavar='NUMBER', help='first CUDA device ordinal')
    p.add_option('--gpus', dest='num_gpus', type=int, default=0, metavar='NUMBER',
                 help='number of GPUs to shard the queries over (0 = all visible, like -T 0 = all cores upstream)')
    return p


def _parse(p, argv=None):
    options, args = p.parse_args(argv)
    if options.print_version:
        print('APPLES version ' + __version__, flush=True)
        raise SystemExit(0)
    # Upstream re-estimates the backbone branch lengths with FastTree unless -D is given (OptionsBasic.py:
    # reestimate_backbone = not disable_reestimation; reestimateBackbone.py).  That step is outside this build: the tree
    # is always used as given, i.e. -D semantics.  Say so instead of silently differing from upstream's default.
    options.reestimate_backbone = False
    if getattr(options, 'ref_fp', None) and getattr(options, 'tree_fp', None) and not options.disable_reestimation:
        logging.warning('Backbone branch-length re-estimation (FastTree, upstream default without -D) is not part of this '
                        'build: the tree is used as given, as with -D. Placements can differ from an upstream run made '
                        'without -D; pass -D to silence this warning.')
    if options.debug_mode:
        logging.getLogger().setLevel(logging.DEBUG)
    return options, args


def options_config_run(argv=None):
    """OptionsRun.options_config"""
    p = _basic('jplace')
    p.add_option('-a', '--database', dest='database_fp', metavar='FILE', help='path to the APPLES database')
    p.add_option('-d', '--distances', dest='dist_fp', metavar='FILE', help='path to the table of observed distances')
    p.add_option('-x', '--extendedref', dest='extended_ref_fp', metavar='FILE',
                 help='path to the extened reference alignment file (FASTA), containing reference and query sequences')
    p.add_option('-q', '--query', dest='query_fp', metavar='FILE',
                 help='path to the query alignment file (FASTA), containing query sequences')
    p.add_option('-m', '--method', dest='method_name', default='FM', metavar='METHOD',
                 help='name of the weighted least squares method (OLS, FM, BME, or BE)')
    p.add_option('-c', '--criterion', dest='criterion_name', default='MLSE', metavar='CRITERIA',
                 help='name of the placement selection criterion (MLSE, ME, or HYBRID')
    p.add_option('-n', '--negative', dest='negative_branch', action='store_true',
                 help='relaxes positivity constraint on new branch lengths, i.e. allows negative branch lengths')
    p.add_option('-b', '--base', dest='base_observation_threshold', type=int, default=25, metavar='NUMBER',
                 help='minimum number of observations kept for each query ignoring the filter threshold.')
    p.add_option('-V', '--overlap', dest='minimum_alignment_overlap', type=float, default=0.001, metavar='NUMBER',
                 help='minimum fraction of nongap sites needed for a valid pairwise distance.')
    p.add_option('-X', '--mask', dest='mask_lowconfidence', action='store_true', default=False,
                 help='masks low confidence characters in the alignments indicated by lowercase characters')
    p.add_option('--exclude', dest='exclude_intplace', action='store_true', default=False,
                 help='exclude queries placed on the internal nodes in jplace file.')
    p.add_option('--keep-at-most', dest='keep_at_most', type=int, default=1, metavar='NUMBER',
                 help='report the best NUMBER (1 to 16) placements of each query in criterion order; the extra ones have '
                      'like_weight_ratio 0')
    p.add_option('--model', dest='model', default=None, metavar='MODEL',
                 help='nucleotide distance model of alignment input: JC69 (default) or K2P (Kimura two-parameter)')
    options, args = _parse(p, argv)
    if not 1 <= options.keep_at_most <= 16:
        raise ValueError('--keep-at-most must be from 1 to 16, got %d' % options.keep_at_most)
    if options.model is not None:
        if options.model not in ('JC69', 'K2P'):
            raise ValueError('--model must be JC69 or K2P, got %r' % options.model)
        if options.protein_seqs:
            raise ValueError('--model chooses a nucleotide distance; it cannot be combined with -p')
        if options.dist_fp:
            raise ValueError('--model applies to alignment input; it cannot be combined with -d')
    else:
        options.model = 'JC69'
    # OptionsRun.py:88-110
    if options.dist_fp:
        if options.ref_fp:
            raise ValueError('Input should be either an alignment or a distance matrix, but not both!')
        if options.database_fp:
            logging.warning('Input contains both an APPLES database and a distance matrix. Database sequences '
                            'will be ignored. Database phylogeny will be used if user did not provide a phylogeny '
                            '(using -t option). ')
    if options.database_fp:
        if options.ref_fp:
            raise ValueError('Input should be either an alignment or a APPLES database file, but not both!')
        if options.tree_fp:
            logging.warning('Input contains both an APPLES database and a tree file. User provided tree has '
                            'higher priority and therefore will be used.')
    if not options.tree_fp and not options.database_fp:
        raise ValueError('No input backbone tree provided by user.')
    if options.query_fp and options.extended_ref_fp:
        raise ValueError('Input should be either an extended alignment or a query alignment, but not both!')
    return options, args


def options_config_build(argv=None):
    """OptionsBuild.options_config"""
    return _parse(_basic('APPLES database'), argv)
