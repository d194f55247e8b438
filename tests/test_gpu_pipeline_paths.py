"""GPU (-m gpu): the two placement paths that share their block-class code (the main pass and the overflow reruns), and a
context that installs one reference after another.  Results are compared bit for bit, so these tests guard the host
orchestration in api.cu: chunking, argument set-up and derived-state resets must not change what is computed."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

DEFAULT_SCRATCH = 6 << 30


def _backbone(n_leaves, L, n_queries, seed, protein=False):
    from apples_b200 import synth
    from apples_b200.reference import ReducedReference
    from apples_b200.tree import BackboneTree
    tree = BackboneTree.from_newick(synth.random_tree(n_leaves, seed=seed))
    refs, states = synth.evolve_alignment(tree, L, seed=seed + 1, protein=protein)
    queries, _ = synth.make_queries(tree, states, n_queries, seed=seed + 2, protein=protein)
    return tree, refs, states, ReducedReference(None, protein, None, 0.2, 1, tree=tree, refs=refs), queries


def _identical(a, b):
    return all(np.array_equal(x.view(np.uint8), y.view(np.uint8)) for x, y in zip(a, b))


@pytest.fixture(scope='module')
def block_case():
    from apples_b200.placer import GpuPlacer
    tree, _, _, ref, queries = _backbone(5000, 1500, 2000, 300)
    pl = GpuPlacer(tree, ref, tree.name_to_node, device=0)
    packed = pl.pack_queries(list(queries.values()))
    yield pl, packed, np.full(packed.shape[0], -1, np.int32)
    pl.close()


@pytest.mark.parametrize('slot_cap,overflowed', [(4096, 0), (32, 1)], ids=['main_pass', 'reruns'])
def test_block_class_chunking(block_case, slot_cap, overflowed):
    """Queries with V + 1 > 512 are placed one block per query, in chunks under the scratch limit.  With scratch_bytes=1
    every such query is a chunk of its own; the results must not change.  slot_cap 4096: they reach the main pass's block
    class without overflowing; slot_cap 32: they overflow and reach the reruns' block class."""
    from apples_b200 import _lib
    pl, packed, self_node = block_case
    nq = packed.shape[0]
    pl.set_limits(scratch_bytes=DEFAULT_SCRATCH, slot_cap=slot_cap)
    for thr in (0.2, 0.4, 0.8, 1.6):   # wider observed sets until enough queries land in the block class
        params = _lib.make_params('FM', 'MLSE', filt_threshold=thr)
        pl.timings(reset=True)
        whole = pl.place_packed(packed, self_node, params)
        _, V, ov = pl.last_counts(nq)
        hits = int(((V + 1 > 512) & (ov == overflowed)).sum())
        if hits >= 2:
            break
    assert hits >= 2, 'only %d block-class queries with overflowed=%d' % (hits, overflowed)
    assert pl.timings()['placed_block'] > 0
    try:
        pl.set_limits(scratch_bytes=1)
        pl.timings(reset=True)
        chunked = pl.place_packed(packed, self_node, params)
        assert pl.timings()['placed_block'] > 0
    finally:
        pl.set_limits(scratch_bytes=DEFAULT_SCRATCH)
    _, V2, ov2 = pl.last_counts(nq)
    assert (V2 == V).all() and (ov2 == ov).all()
    assert _identical(whole, chunked)


def test_reference_reinstall():
    """One context installs a tensor-core nucleotide reference, a byte-mode one (a byte outside ACGT-), a protein one
    and the first again from packed arrays.  Each placement equals that of a fresh context with only that reference."""
    from apples_b200 import _lib
    from apples_b200.placer import GpuPlacer
    from apples_b200.reference import ReducedReference
    tree, refs, states, nuc_ref, nuc_q = _backbone(600, 700, 300, 400)
    exotic = {k: v.copy() for k, v in refs.items()}
    first = next(iter(exotic))
    exotic[first][5] = b'N'
    exotic_ref = ReducedReference(None, False, None, 0.2, 1, tree=tree, refs=exotic)
    _, _, _, prot_ref, prot_q = _backbone(600, 300, 300, 400, protein=True)
    # (reference, install from bytes on the device, queries, tensor-core kernel expected)
    installs = [(nuc_ref, True, nuc_q, True), (exotic_ref, True, nuc_q, False), (prot_ref, True, prot_q, False),
                (nuc_ref, False, nuc_q, True)]
    params = _lib.make_params('FM', 'MLSE')
    pl = GpuPlacer(tree, None, tree.name_to_node, device=0)
    try:
        for ref, on_device, queries, tc in installs:
            pl.set_reference(ref, on_device=on_device)
            packed = pl.pack_queries(list(queries.values()))
            self_node = np.full(packed.shape[0], -1, np.int32)
            pl.timings(reset=True)
            got = pl.place_packed(packed, self_node, params)
            assert (pl.timings()['tensor_core_launches'] > 0) == tc
            fresh = GpuPlacer(tree, None, tree.name_to_node, device=0)
            try:
                fresh.set_reference(ref, on_device=on_device)
                exp = fresh.place_packed(packed, self_node, params)
            finally:
                fresh.close()
            assert _identical(got, exp)
    finally:
        pl.close()
