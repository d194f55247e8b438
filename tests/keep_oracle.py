"""The ranked records of --keep-at-most K on the CPU: the definition the device's records are checked against.

An extension of the oracle (oracle/apples_oracle.py), which stays as it is: upstream's choice of ONE edge is a "first
minimum" (Algorithm.py:74-91, choose_edge), and Python's min and heapq.nsmallest keep the first of equal elements.  K
records extend that to a stable sort by the criterion's key in post-order (= edge_index) order, truncated to K:
  MLSE    sorted(valid_edges, key=error)[:K]
  ME      sorted(valid_edges, key=x_1)[:K]
  HYBRID  sorted(heapq.nsmallest(floor(log2 V), valid_edges, key=error), key=x_1)[:K]   (at most floor(log2 V) records)
Record 0 is choose_edge's record; every record is [edge_num, error, like_weight_ratio, distal, pendant] with
like_weight_ratio 1 for record 0 and 0 for the others.
"""
import heapq
import math

from oracle import apples_oracle as orc


def choose_edges(valids, criterion, num_nodes, keep):
    """The first `keep` records of the valid edges `valids` (post-order, solved) in criterion order."""
    if criterion == 'HYBRID':
        ranked = sorted(heapq.nsmallest(math.floor(math.log2(num_nodes)), valids, key=orc.edge_error), key=lambda e: e.x1)
    elif criterion == 'ME':
        ranked = sorted(valids, key=lambda e: e.x1)
    else:
        ranked = sorted(valids, key=orc.edge_error)
    return [[e.edge_index, orc.edge_error(e), 1 if j == 0 else 0, e.edge_length - e.x2, e.x1]
            for j, e in enumerate(ranked[:keep])]


def solved_edges(obs, name_to_node, method, negative_branch, fn):
    """fn(post-order valid nodes with x_1 / x_2 solved, V) on the restricted subtree of `obs` (place_from_observed's
    steps, PoolQueryWorker.py:101-120); the tree's valid flags are reset afterwards."""
    root, marked = orc.mark_subtree(obs, name_to_node)
    try:
        post = orc.postorder_valid(root)
        orc.compute_moments(method, root, obs, post, orc.preorder_valid(root))
        for n in post:
            orc.solve_edge(n, negative_branch)
        return fn(post, len(marked))
    finally:
        for n in marked:
            n.valid = False


def place_from_observed_k(query_name, obs, name_to_node, method='FM', criterion='MLSE', negative_branch=False,
                          exclude_intplace=False, keep=1):
    """orc.place_from_observed with K records: a query placed by least squares (PLACED, or PLACED_MISPLACEMENT_FLAG
    without exclude_intplace) carries choose_edges' records; every other query keeps its single record."""
    jp, status = orc.place_from_observed(query_name, obs, name_to_node, method, criterion, negative_branch,
                                         exclude_intplace)
    if status == orc.PLACED or (status == orc.PLACED_MISPLACEMENT_FLAG and not exclude_intplace):
        obs = dict(obs)
        if query_name in name_to_node:
            obs.pop(query_name, None)
        jp['placements'][0]['p'] = solved_edges(obs, name_to_node, method, negative_branch,
                                                lambda post, V: choose_edges(post, criterion, V, keep))
    return jp, status


def runquery_k(octx, query_name, query_seq, row, keep):
    """OracleContext.runquery with K records."""
    if row:
        obs = orc.observed_matrix(row, octx.name_to_node, octx.filt_threshold, octx.baseobs)
    else:
        obs = orc.observed_alignment(query_seq, octx.representatives, octx.refs, octx.dist_fn, octx.filt_threshold,
                                     octx.baseobs, octx.overlap)
    return place_from_observed_k(query_name, obs, octx.name_to_node, octx.method, octx.criterion, octx.negative_branch,
                                 octx.exclude_intplace, keep)
