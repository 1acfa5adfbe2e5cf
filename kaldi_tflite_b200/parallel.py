"""
Multi-GPU plumbing: one process per GPU (torchrun), torch.distributed for rendezvous.

* wav -> x-vector: utterances are independent, so they are sharded across ranks with NO
  data-path collective (`shard_range`); an optional final gather of the 128-d x-vectors is
  offered for callers that want one tensor (`gather_rows`).
* PLDA all-vs-all: ENROLLED vectors (score columns) are sharded by rank, the transformed TEST
  vectors are exchanged once with an all-gather over NCCL/NVLink, and every rank writes its own
  (n_test x n_enroll/G) block; the 10 GB score matrix is never gathered (SURVEY.md 8e).
"""

import torch
import torch.distributed as dist

from . import _native
from . import _tensor as T


def world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_range(n_items, rank=None, world_size=None):
    """Contiguous, balanced [start, stop) of `n_items` units for this rank."""
    r, w = world()
    rank = r if rank is None else rank
    world_size = w if world_size is None else world_size
    base, rem = divmod(n_items, world_size)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def gather_rows(local, counts=None):
    """All-gather of row blocks that may differ in length; returns the concatenation on every rank."""
    rank, w = world()
    if w == 1:
        return local
    n = torch.tensor([local.shape[0]], device=local.device, dtype=torch.int64)
    sizes = [torch.zeros_like(n) for _ in range(w)]
    dist.all_gather(sizes, n)
    sizes = [int(s.item()) for s in sizes]
    m = max(sizes)
    pad = torch.zeros((m,) + tuple(local.shape[1:]), device=local.device, dtype=local.dtype)
    pad[:local.shape[0]] = local
    bufs = [torch.empty_like(pad) for _ in range(w)]
    dist.all_gather(bufs, pad)
    return torch.cat([b[:s] for b, s in zip(bufs, sizes)], dim=0)


def exchange_test_vectors(u_test_local, test_counts=None):
    """
    The one collective of the PLDA path (SURVEY.md 8e): all-gather of the transformed test vectors.
    Returns (u_all, offsets, works): `works[r].wait()` makes the current stream wait for rank r's block; `u_all` may be
    read for block r only after that.

    NCCL: ONE asynchronous all-gather (`all_gather_into_tensor` on blocks padded to the largest shard -- shards from
    `shard_range` differ by at most one row); 25.6 MB at 50 k x 128 is ~35 us of NVLink time, so a single collective
    beats per-rank broadcasts, whose launch latencies add up (measured at 8 ranks: 0.63 ms for eight broadcasts).  It
    runs on NCCL's own stream: the caller scores its LOCAL rows (and transforms its enrolled vectors) underneath it.
    Other backends (gloo in the CPU / single-GPU tests) use one asynchronous broadcast per source rank.
    """
    rank, w = world()
    if test_counts is None:
        n = torch.tensor([u_test_local.shape[0]], device=u_test_local.device, dtype=torch.int64)
        sizes = [torch.zeros_like(n) for _ in range(w)]
        dist.all_gather(sizes, n)
        test_counts = [int(t.item()) for t in sizes]
    offs = [0]
    for c in test_counts:
        offs.append(offs[-1] + int(c))
    dim = u_test_local.shape[1]
    if dist.get_backend() == "nccl":
        per = max(int(c) for c in test_counts)
        if all(int(c) == per for c in test_counts):
            u_all = torch.empty((w * per, dim), device=u_test_local.device, dtype=u_test_local.dtype)
            work = dist.all_gather_into_tensor(u_all, u_test_local.contiguous(), async_op=True)
            return u_all, offs, [_Gathered(work)] * w
        padded = torch.zeros((per, dim), device=u_test_local.device, dtype=u_test_local.dtype)
        padded[:u_test_local.shape[0]].copy_(u_test_local)
        gathered = torch.empty((w * per, dim), device=u_test_local.device, dtype=u_test_local.dtype)
        work = dist.all_gather_into_tensor(gathered, padded, async_op=True)
        u_all = torch.empty((offs[-1], dim), device=u_test_local.device, dtype=u_test_local.dtype)

        def compact():                        # ragged shards: drop the padding rows once the gather has landed
            for r in range(w):
                u_all[offs[r]:offs[r + 1]].copy_(gathered[r * per:r * per + int(test_counts[r])])
        return u_all, offs, [_Gathered(work, compact)] * w
    u_all = torch.empty((offs[-1], dim), device=u_test_local.device, dtype=u_test_local.dtype)
    u_all[offs[rank]:offs[rank + 1]].copy_(u_test_local)
    works = [dist.broadcast(u_all[offs[r]:offs[r + 1]], src=r, async_op=True) if offs[r + 1] > offs[r] else None
             for r in range(w)]
    return u_all, offs, works


class _Gathered:
    """Work handle of the single NCCL all-gather, shared by every rank's block: the first wait() makes the current stream
    wait for the collective (and runs the optional compaction of ragged shards), later ones are free."""

    def __init__(self, work, after=None):
        self.work, self.after, self.done = work, after, False

    def wait(self):
        if not self.done:
            self.work.wait()
            if self.after is not None:
                self.after()
            self.done = True
        return True


def plda_score_sharded(plda, x_test_local, x_enroll_local, test_counts=None, out=None):
    """
    Sharded PLDA trial scoring.  Each rank holds a slice of the test x-vectors and a slice of the enrolled
    x-vectors (raw, (n, dim) float32).  Returns this rank's block scores[all tests, local enrolled] -- test
    rows ordered by rank -- plus the gathered transformed test vectors.

    The exchange is an all-gather of the transformed test vectors (`exchange_test_vectors`, SURVEY.md 8e).  Over NCCL it
    is one asynchronous collective: while it is in flight this rank transforms its enrolled vectors and scores its OWN
    test rows, then the rows above and below them in two more score GEMMs.  On backends without a GPU all-gather the
    per-rank broadcasts are consumed block by block.  `test_counts` (rows per rank) saves the small size exchange when
    the caller already knows the partition (e.g. from `shard_range`); `out` is an optional preallocated
    (n_test, n_enroll_local) score block.
    """
    rank, w = world()
    u_test_local = plda.transformVector(x_test_local.contiguous())
    if w == 1:
        u_enroll_local = plda.transformVector(x_enroll_local.contiguous())
        return plda.logLikelihoodRatio(u_test_local, u_enroll_local, out=out), u_test_local
    u_all, offs, works = exchange_test_vectors(u_test_local, test_counts)
    u_enroll_local = plda.transformVector(x_enroll_local.contiguous())
    if out is None:
        # row pitch padded to 16 bytes: the score kernel's boxed (TMA) stores need an aligned pitch
        ne = u_enroll_local.shape[0]
        out = torch.empty((offs[-1], (ne + 7) // 8 * 8), device=u_test_local.device, dtype=u_test_local.dtype)[:, :ne]
    scores = out
    if all(isinstance(wk, _Gathered) for wk in works):
        lo, hi = offs[rank], offs[rank + 1]
        if hi > lo:                           # local rows: no need to wait for anybody
            plda.logLikelihoodRatio(u_test_local, u_enroll_local, out=scores[lo:hi])
        works[0].wait()
        if lo > 0:
            plda.logLikelihoodRatio(u_all[:lo], u_enroll_local, out=scores[:lo])
        if offs[-1] > hi:
            plda.logLikelihoodRatio(u_all[hi:], u_enroll_local, out=scores[hi:])
        return scores, u_all
    for r in range(w):
        if works[r] is None:
            continue
        works[r].wait()                       # the compute stream waits for block r only
        plda.logLikelihoodRatio(u_all[offs[r]:offs[r + 1]], u_enroll_local, out=scores[offs[r]:offs[r + 1]])
    return scores, u_all


def plda_best_matches_sharded(plda, x_test_local, x_enroll_local, k, test_counts=None):
    """
    Sharded k-best trial search: `PLDA.bestMatches` of ALL test vectors against ALL enrolled vectors, where each rank
    holds a slice of both (raw, (n, dim) float32).  The transformed test vectors are all-gathered
    (`exchange_test_vectors`), the enrolled ones stay where they are: every rank finds the k best of its own enrolled
    shard for every test row, with indexes offset to the global enrolled numbering (shards in rank order), the ranks
    exchange these (n_test, k) lists once, and `ktf_topk_merge` reduces them on every rank.  Returns (scores, indexes),
    (n_test, k) each, test rows ordered by rank -- equal to `bestMatches` on the whole set.
    """
    rank, w = world()
    u_test_local = plda.transformVector(x_test_local.contiguous())
    if w == 1:
        return plda.bestMatches(u_test_local, plda.transformVector(x_enroll_local.contiguous()), k=k)
    u_all, offs, works = exchange_test_vectors(u_test_local, test_counts)
    u_enroll_local = plda.transformVector(x_enroll_local.contiguous())
    n = torch.tensor([u_enroll_local.shape[0]], device=u_enroll_local.device, dtype=torch.int64)
    sizes = [torch.zeros_like(n) for _ in range(w)]
    dist.all_gather(sizes, n)
    e_off = sum(int(s.item()) for s in sizes[:rank])
    for wk in works:
        if wk is not None:
            wk.wait()
    scores, index = plda.bestMatches(u_all, u_enroll_local, k=k)
    index = torch.where(index >= 0, index + e_off, index)
    # one exchange: the score bits ride in the int64 tensor next to the indexes
    local = torch.cat([scores.view(torch.int32).to(torch.int64), index], dim=1)
    lists = [torch.empty_like(local) for _ in range(w)]
    dist.all_gather(lists, local)
    lists = torch.stack(lists)                                     # (w, n_test, 2k)
    s_in = lists[:, :, :k].to(torch.int32).view(torch.float32).contiguous()
    i_in = lists[:, :, k:].contiguous()
    n_test = u_all.shape[0]
    out_s = torch.empty((n_test, k), device=u_all.device, dtype=torch.float32)
    out_i = torch.empty((n_test, k), device=u_all.device, dtype=torch.int64)
    _native.check(_native.lib().ktf_topk_merge(T.ptr(s_in), T.ptr(i_in), w, n_test, k, k, T.ptr(out_s), T.ptr(out_i),
                                               T.stream_ptr()))
    return out_s, out_i


def stream_batches(fn, host_in, chunk, host_out=None, depth=3):
    """
    Runs `fn` (any layer / model call taking a CUDA tensor of utterances and returning a CUDA tensor with
    the same leading dimension) over a HOST batch in chunks of `chunk` utterances, with the host->device
    copy of chunk i+1 and the device->host copy of result i-1 overlapped with the compute of chunk i
    (two side streams; PCIe is full duplex).  Utterances are independent on this path, so the result equals
    the one-shot call.  `host_in` should be pinned for the copies to be asynchronous; `host_out`, if given,
    is a pinned tensor that receives the results, otherwise the device results are concatenated.

    The audio lands in a ring of `depth` device staging buffers that is allocated once per (chunk shape, dtype) and
    reused: a slot is refilled only after the compute stream has finished the chunk that used it (event wait on the
    copy stream -- the HOST never blocks).  Nothing on this path synchronises with the host any more, so without the
    ring the host would run ahead and ask the allocator for a fresh 80 MB block per chunk.
    """
    dev = T.device()
    cur = torch.cuda.current_stream(dev)
    s_in, s_out = _side_streams(dev)
    s_in.wait_stream(cur)
    s_out.wait_stream(cur)
    outs = []
    n = host_in.shape[0]
    ring = _staging_ring(dev, (min(chunk, max(n, 1)),) + tuple(host_in.shape[1:]), host_in.dtype, depth)
    freed = [None] * depth                       # event: the compute stream is done with slot k

    def fetch(idx):
        i = idx * chunk
        m = min(chunk, n - i)
        k = idx % depth
        if freed[k] is not None:
            s_in.wait_event(freed[k])
        with torch.cuda.stream(s_in):
            x = ring[k][:m]
            x.copy_(host_in[i:i + m], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(s_in)
        return x, ev, k

    n_chunks = (n + chunk - 1) // chunk
    nxt = fetch(0) if n > 0 else None
    for idx in range(n_chunks):
        x, ev, k = nxt
        nxt = fetch(idx + 1) if idx + 1 < n_chunks else None   # the next copy is in flight before this chunk computes
        cur.wait_event(ev)
        y = fn(x)
        freed[k] = torch.cuda.Event()
        freed[k].record(cur)
        i = idx * chunk
        if host_out is None:
            outs.append(y)
        else:
            s_out.wait_stream(cur)
            with torch.cuda.stream(s_out):
                host_out[i:i + y.shape[0]].copy_(y, non_blocking=True)
            y.record_stream(s_out)
    cur.wait_stream(s_out)
    s_in.wait_stream(cur)                        # the ring may be refilled by the next call only after this one's compute
    return host_out if host_out is not None else torch.cat(outs, dim=0)


_SIDE = {}
_RINGS = {}


def _side_streams(dev):
    key = (dev.type, dev.index)
    if key not in _SIDE:
        _SIDE[key] = (torch.cuda.Stream(dev), torch.cuda.Stream(dev))
    return _SIDE[key]


def _staging_ring(dev, shape, dtype, depth):
    key = (dev.type, dev.index, tuple(shape), dtype, depth)
    if key not in _RINGS:
        if len(_RINGS) >= 4:                      # a handful of shapes per process; drop the oldest
            _RINGS.pop(next(iter(_RINGS)))
        _RINGS[key] = [torch.empty(shape, device=dev, dtype=dtype) for _ in range(depth)]
    return _RINGS[key]
