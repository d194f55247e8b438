"""Multi-GPU data parallelism over queries (SURVEY.md section 8e).

The reference's only parallelism is `mp.Pool.starmap` over queries with fork-inherited read-only state
(run_apples.py:20,94-102).  Here: one process per GPU, queries split into contiguous blocks of ceil(Q / G), the packed
reference + tree replicated on every GPU, no data-path collective; the single collective is the final all-gather of
the placements (ONE collective of 32-byte records: edge i32, status i32, error f64, distal f64, pendant f64; k of them per
query with --keep-at-most k), after which every rank
holds the results of all queries in input order -- so the N-GPU output is byte-identical to the 1-GPU output.

torch.distributed is plumbing here: `nccl` on GPUs (NVLink / NVSwitch), `gloo` in the CPU tests.
"""
import numpy as np


def shard_bounds(n_items, world):
    """Contiguous blocks of ceil(n / world): [(begin, end)] per rank (trailing ranks may be empty)."""
    per = -(-int(n_items) // int(world)) if n_items else 0
    return [(min(r * per, n_items), min((r + 1) * per, n_items)) for r in range(world)]


RECORD_BYTES = 32  # one placement: edge i32 | status i32 | error f64 | distal f64 | pendant f64


def pack_records(edge, error, distal, pendant, status):
    """Five result arrays (torch tensors on one device) -> one int64 [n, 4] tensor of 32-byte records, so that the final
    gather is ONE collective.  Word 0 = edge (low 32 bits) | status (high 32 bits), words 1-3 = the doubles' bit patterns."""
    import torch
    n = edge.shape[0]
    rec = torch.empty((n, 4), dtype=torch.int64, device=edge.device)
    rec[:, 0] = (edge.to(torch.int64) & 0xffffffff) | (status.to(torch.int64) << 32)
    rec[:, 1] = error.view(torch.int64)
    rec[:, 2] = distal.view(torch.int64)
    rec[:, 3] = pendant.view(torch.int64)
    return rec


def pack_alt_records(count, edge, error, distal, pendant, int0):
    """Ranked records [n, k] (GpuPlacer._alt_outputs, torch tensors on one device) -> int64 [n, 4 (k - 1)]: records
    1 .. k - 1 as 32-byte records, word 0 = edge (low 32 bits) | (pendant_int0 | count << 8) (high 32 bits).  Record 0
    is the placement pack_records carries."""
    import torch
    n, k = edge.shape
    rec = torch.empty((n, k - 1, 4), dtype=torch.int64, device=edge.device)
    hi = int0[:, 1:].to(torch.int64) | (count.to(torch.int64)[:, None] << 8)
    rec[:, :, 0] = (edge[:, 1:].to(torch.int64) & 0xffffffff) | (hi << 32)
    rec[:, :, 1] = error[:, 1:].contiguous().view(torch.int64)
    rec[:, :, 2] = distal[:, 1:].contiguous().view(torch.int64)
    rec[:, :, 3] = pendant[:, 1:].contiguous().view(torch.int64)
    return rec.reshape(n, 4 * (k - 1))


def unpack_alt_records(rec, main):
    """int64 [n, 4 (k - 1)] of pack_alt_records + the unpacked placements `main` -> (count i32 [n], edge i32, error f64,
    distal f64, pendant f64, pendant_int0 u8 [n, k]) tensors (same device)."""
    import torch
    edge0, error0, distal0, pendant0, status = main
    n = rec.shape[0]
    r = rec.reshape(n, -1, 4)
    w0 = r[:, :, 0]
    hi = w0 >> 32
    col = lambda x: x[:, None]   # noqa: E731
    f64 = lambda j: r[:, :, j].contiguous().view(torch.float64)   # noqa: E731
    return ((hi[:, 0] >> 8).to(torch.int32),
            torch.cat([col(edge0), (w0 << 32 >> 32).to(torch.int32)], 1),
            torch.cat([col(error0), f64(1)], 1), torch.cat([col(distal0), f64(2)], 1), torch.cat([col(pendant0), f64(3)], 1),
            torch.cat([col((status.to(torch.int64) >> 8) & 1), hi & 0xff], 1).to(torch.uint8))


def unpack_records(rec):
    """int64 [n, 4] records -> (edge i32, error f64, distal f64, pendant f64, status i32) tensors (same device)."""
    import torch
    w0 = rec[:, 0]
    edge = (w0 << 32 >> 32).to(torch.int32)   # arithmetic shift: sign-extends the low half (edge may be -1)
    status = (w0 >> 32).to(torch.int32)
    return (edge, rec[:, 1].contiguous().view(torch.float64), rec[:, 2].contiguous().view(torch.float64),
            rec[:, 3].contiguous().view(torch.float64), status)


def gather_records(rec, n_total=None, out=None):
    """All-gather of the ranks' record blocks (each rank holds the block of ceil(n_total / world) queries that
    shard_bounds gives it, the last ones possibly shorter).  Returns the records of all queries in input order on every
    rank.  `out` may be a preallocated [per * world, width] tensor (bench.py reuses it every step)."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return rec
    world = dist.get_world_size()
    if n_total is None:
        n_total = rec.shape[0] * world
    per = -(-int(n_total) // world)
    if rec.shape[0] < per:
        rec = torch.cat([rec, torch.zeros((per - rec.shape[0], rec.shape[1]), dtype=rec.dtype, device=rec.device)])
    full = out if out is not None else torch.empty((per * world, rec.shape[1]), dtype=rec.dtype, device=rec.device)
    dist.all_gather_into_tensor(full, rec.contiguous())
    return full[:n_total]


_GATHER_BUFFERS = {}   # device -> (capacity in records, device SoA buffer, pinned host twin); grown, never one per batch size


def _soa_views(buf, n):
    """The five result arrays as views of one byte buffer laid out [edge i32 n | status i32 n | error | distal | pendant f64 n]."""
    import torch
    e = buf[0:4 * n].view(torch.int32)
    s = buf[4 * n:8 * n].view(torch.int32)
    f = buf[8 * n:32 * n].view(torch.float64)
    return e, f[0:n], f[n:2 * n], f[2 * n:3 * n], s


def gather_placements(local, n_total, device=None, alt=None):
    """local: tuple (edge i32, error f64, distal f64, pendant f64, status i32) of this rank's shard as numpy arrays or
    torch tensors.  Returns the same tuple for all `n_total` queries in input order, as numpy arrays, after ONE
    all-gather of 32-byte records.  alt: the shard's ranked records (GpuPlacer._alt_outputs); they travel in the same
    all-gather, and the call returns (placements, ranked records of all queries).  With NCCL the gathered records are split into the five arrays on the device and come
    back in ONE copy into a pinned host buffer that is reused from call to call: the returned arrays are views of it,
    valid until the next call with the same shape (copy them to keep them)."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        main = tuple(np.asarray(a.cpu() if hasattr(a, 'cpu') else a) for a in local)
        return main if alt is None else (main, tuple(np.asarray(a.cpu() if hasattr(a, 'cpu') else a) for a in alt))
    if device is None:
        device = 'cuda' if dist.get_backend() == 'nccl' else 'cpu'
    import os
    import time
    trace = torch.device(device).type == 'cuda' and os.environ.get('APPLES_B200_GATHER_TRACE')
    t0 = time.time()
    def up(arrays):
        return [(a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))).to(device, non_blocking=True)
                for a in arrays]
    rec = pack_records(*up(local))
    if alt is not None:
        rec = torch.cat([rec, pack_alt_records(*up(alt))], 1)
    if trace:
        torch.cuda.synchronize(device)
        t1 = time.time()
    full = gather_records(rec, n_total)
    if trace:
        torch.cuda.synchronize(device)
        t2 = time.time()
    parts = unpack_records(full)
    alt_all = None if alt is None else tuple(t.cpu().numpy() for t in unpack_alt_records(full[:, 4:], parts))
    if torch.device(device).type != 'cuda':
        main = tuple(t.numpy() for t in parts)
        return main if alt is None else (main, alt_all)
    key = str(device)
    if key not in _GATHER_BUFFERS or _GATHER_BUFFERS[key][0] < n_total:
        _GATHER_BUFFERS[key] = (int(n_total), torch.empty(32 * n_total, dtype=torch.uint8, device=device),
                                torch.empty(32 * n_total, dtype=torch.uint8).pin_memory())
    _, dbuf, hbuf = _GATHER_BUFFERS[key]
    dbuf, hbuf = dbuf[:32 * n_total], hbuf[:32 * n_total]
    for dst, src in zip(_soa_views(dbuf, n_total), parts):
        dst.copy_(src)
    hbuf.copy_(dbuf, non_blocking=True)
    torch.cuda.current_stream(device).synchronize()
    if trace:
        import sys
        sys.stderr.write('[apples_b200] gather rank %d: upload + pack %.2f ms, all-gather %.2f ms, split + download %.2f ms\n'
                         % (dist.get_rank(), 1e3 * (t1 - t0), 1e3 * (t2 - t1), 1e3 * (time.time() - t2)))
    main = tuple(v.numpy() for v in _soa_views(hbuf, n_total))
    return main if alt is None else (main, alt_all)


def place_sharded(place_fn, n_total):
    """Run `place_fn(begin, end) -> result tuple` on this rank's block and gather every rank's results."""
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        rank, world = dist.get_rank(), dist.get_world_size()
    else:
        rank, world = 0, 1
    b, e = shard_bounds(n_total, world)[rank]
    local = place_fn(b, e)
    return gather_placements(local, n_total)
