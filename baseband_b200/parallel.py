"""Multi-GPU reading: contiguous frame ranges per rank, optional all-gather.

Frames are independent, so a stream shards with no collective on the data
path (SURVEY.md section 8(e)): rank ``r`` of ``W`` decodes frames
``[r*N/W, (r+1)*N/W)`` on its own GPU, reading only its own byte range of the
file.  Only when the caller wants the whole decoded stream on every device is
a collective used: one NCCL all-gather of the decoded shards over NVLink
(``gather=True``).  Gathering *decoded* float32 moves 16x the packed bytes for
2-bit data; prefer leaving the shards where they are.

The packed-byte consumer shards the same way, and its collective is tiny:
`state_counts_sharded` counts whole integration bins per rank and sums the
int64 count tables with one all-reduce (a few KB), so every rank ends up with
the counts of the whole stream.

One process per GPU (``torchrun``); ``torch.distributed`` is plumbing only.
"""
import os

import torch

__all__ = ['shard_bounds', 'shard_samples', 'gather_block', 'read_sharded',
           'state_counts_sharded']


def shard_bounds(nitem, rank, world):
    """[start, stop) of ``nitem`` items for ``rank``: contiguous, covering,
    sizes differing by at most one."""
    if not 0 <= rank < world:
        raise ValueError('rank {} outside world of size {}'.format(rank,
                                                                   world))
    return rank * nitem // world, (rank + 1) * nitem // world


def shard_samples(fh, rank, world):
    """Sample range [start, stop) of stream reader ``fh`` owned by ``rank``:
    whole frames, except that the last rank takes the tail (e.g. GUPPI's
    final overlap)."""
    f0, f1 = shard_bounds(fh._nframe, rank, world)
    spf = fh.samples_per_frame
    start = f0 * spf
    stop = fh.shape[0] if rank == world - 1 else f1 * spf
    return start, stop


def _dist_env(rank, world):
    if rank is None or world is None:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist.get_rank(), dist.get_world_size()
        return (int(os.environ.get('RANK', 0)),
                int(os.environ.get('WORLD_SIZE', 1)))
    return rank, world


def gather_block(fh, world):
    """Samples per rank for a gathered read: equal blocks of whole frames
    (the last ranks' blocks may be short or empty), so that rank r's shard
    sits at row ``r * block`` of the gathered array and the all-gather can
    write every shard straight to its final place."""
    spf = fh.samples_per_frame
    # from the sample count, so that a tail beyond the last whole frame
    # (GUPPI's final overlap) is covered too
    return -(-fh.shape[0] // (world * spf)) * spf


def read_sharded(fh, rank=None, world=None, gather=False, group=None):
    """Decode this rank's contiguous share of ``fh``.

    Returns ``(data, (start, stop))``: the decoded samples of the shard (on
    the reader's device when it was opened with ``device=``) and the sample
    range they cover.

    With ``gather=True`` every rank instead receives the whole stream.  The
    stream is then cut into equal blocks of whole frames (`gather_block`);
    each rank decodes its block directly into its place in the full-length
    result and ONE in-place ``all_gather_into_tensor`` (NCCL over NVLink for
    CUDA tensors) fills in the others: no padding pass, no list of pieces, no
    concatenation -- the only traffic besides the decode itself is the
    collective's.
    """
    rank, world = _dist_env(rank, world)
    if not gather or world == 1:
        start, stop = shard_samples(fh, rank, world)
        fh.seek(start)
        data = fh.read(stop - start)
        return data, (start, stop)
    import torch.distributed as dist
    import numpy as np
    total = fh.shape[0]
    block = gather_block(fh, world)
    start, stop = min(total, rank * block), min(total, (rank + 1) * block)
    on_device = getattr(fh, '_device_output', False)
    backend = dist.get_backend(group)
    if not on_device and backend == 'nccl':
        raise TypeError('gather=True over NCCL needs a reader with device '
                        'output (open(..., device=...)): NCCL moves device '
                        'tensors only.')
    # the reader's result type: float16 / bfloat16 readers gather half the
    # bytes of float32 ones
    dec = fh._dec_dtype
    t_dtype = fh._result_dtype(dec)
    reduced = dec != torch.float32
    shape = (world * block,) + tuple(fh.sample_shape) + fh._pair_axis(dec)
    if on_device:
        whole = torch.empty(shape, dtype=t_dtype, device=fh.device)
    else:
        whole = torch.empty(shape, dtype=t_dtype)
    mine = whole[rank * block:(rank + 1) * block]
    if stop > start:
        fh.seek(start)
        fh.read(out=mine[:stop - start] if on_device or reduced
                else mine[:stop - start].numpy())
    # rows past the end of the stream (short last blocks) are never looked at
    if on_device or backend != 'gloo':
        dist.all_gather_into_tensor(whole, mine, group=group)
    else:
        # gloo has no all_gather_into_tensor on every build: views of the
        # result serve as the output list (still no extra copy of our own)
        dist.all_gather([whole[r * block:(r + 1) * block]
                         for r in range(world)], mine.clone(), group=group)
    whole = whole[:total]
    if not on_device and not reduced:
        whole = whole.numpy()
    return whole, (0, total)


def state_counts_sharded(fh, samples_per_bin, rank=None, world=None,
                         reduce=True, group=None):
    """`tasks.state_counts` of ONE stream over all ranks: the integration
    bins are dealt out in contiguous ranges (`shard_bounds`), every rank
    ingests and counts only its own frames, and -- with ``reduce`` -- one
    all-reduce of the int64 count table (zeros outside the rank's bins)
    leaves the counts of the whole stream on every rank.

    Returns ``(counts, (bin0, bin1))``: the table (numpy; all bins with
    ``reduce``, else this rank's bins only) and the range of bins this rank
    counted.  The stream must hold whole bins from the current sample
    pointer on (a last partial bin is left out)."""
    from . import tasks
    rank, world = _dist_env(rank, world)
    start = fh.tell()
    nbin = (fh.shape[0] - start) // samples_per_bin
    if nbin <= 0:
        raise ValueError('the stream does not hold one whole bin')
    b0, b1 = shard_bounds(nbin, rank, world)
    mine = None
    if b1 > b0:
        fh.seek(start + b0 * samples_per_bin)
        mine = tasks.state_counts(fh, samples_per_bin,
                                  count=(b1 - b0) * samples_per_bin,
                                  device_output=reduce and world > 1)
    if not reduce or world == 1:
        return mine, (b0, b1)
    import torch.distributed as dist
    backend = dist.get_backend(group)
    dev = fh.device if backend == 'nccl' else torch.device('cpu')
    # every rank needs the shape of a bin's table, also one without bins
    shape = [None]
    if mine is not None:
        shape[0] = tuple(mine.shape[1:])
    shapes = [None] * world
    dist.all_gather_object(shapes, shape[0], group=group)
    bin_shape = next(s for s in shapes if s is not None)
    whole = torch.zeros((nbin,) + tuple(bin_shape), dtype=torch.int64,
                        device=dev)
    if mine is not None:
        whole[b0:b1] = mine.to(dev)
    dist.all_reduce(whole, op=dist.ReduceOp.SUM, group=group)
    fh.seek(start + nbin * samples_per_bin)
    return whole.cpu().numpy(), (b0, b1)
