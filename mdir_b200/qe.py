"""alpha query expansion and database-side augmentation on top of the fused scan + top-k.

NOT in the reference (SURVEY.md App. E; parity unpinned): these follow the published
definitions restated in oracle/oracle.py:alpha_qe / dba.  Builder-chosen defaults:
alpha = 3, n_qe = 10, k_dba = 10, negative similarities clamped to 0, self included in DBA."""
import torch

from . import _lib
from .search import Index, ShardedIndex, WIDE_Q


DBA_BLOCK = 4096      # rows augmented per search() call (four wide scan passes; ONE status read-back per call instead of one per pass)
# Queries per scan pass: 1,024 as one WIDE launch (8 blocks of 128 queries per 256-row database tile, the blocks of a
# tile adjacent in the persistent round-robin): the tile comes from HBM once and from L2 seven times, so the pass is
# bound by the tensor pipe / L2 -> shared-memory ingest instead of HBM (128 queries per pass: AI = 128 FLOP per database
# byte, under the ~214 FLOP/B ridge).  One 256-query tile (all of TMEM) was the earlier attempt and measured slower
# than 2 x 128: three 64 KB stages and no accumulator double-buffering -- tools/time_wide.py.
DBA_QUERIES_PER_PASS = WIDE_Q


def _accumulate(index, idx, scores, alpha):
    n_q, n_qe = idx.shape
    acc = torch.empty((n_q, index.D), dtype=torch.float32, device=index.device)
    with torch.cuda.device(index.device):
        _lib.check(_lib.lib().mdir_qe_accumulate(_lib.ptr(index.db32), index.n, index.idx_base, index.D, _lib.ptr(idx.contiguous()),
                                                 _lib.ptr(scores.contiguous()), n_q, n_qe, float(alpha), _lib.ptr(acc), _lib.stream()),
                   "mdir_qe_accumulate")
    return acc


def _add_l2n(a, b):
    out = torch.empty_like(a)
    with torch.cuda.device(a.device):
        _lib.check(_lib.lib().mdir_add_l2n(_lib.ptr(a), _lib.ptr(b), a.shape[0], a.shape[1], _lib.ptr(out), _lib.stream()), "mdir_add_l2n")
    return out


def expand_queries(index, q, alpha=3.0, n_qe=10):
    """q' = normalise(q + sum_{i<=n_qe} max(s_i,0)^alpha x_i).  index: Index or ShardedIndex
    (shards contribute the rows they own; one all-reduce of N_q x D fp32 combines them)."""
    local = index.local if isinstance(index, ShardedIndex) else index
    if local.db32 is None:
        raise _lib.MdirError("query expansion needs the fp32 master copy (keep_fp32=True)")
    from .search import _as_dev_f32
    q32 = _as_dev_f32(q, local.device)
    s, i = index.search(q32, n_qe, precision="fp32")
    acc = _accumulate(local, i, s, alpha)
    if isinstance(index, ShardedIndex) and index.world > 1:
        index.dist.all_reduce(acc, group=index.group)
    return _add_l2n(q32, acc)


def search_qe(index, q, k, alpha=3.0, n_qe=10, precision="fp32"):
    """alpha-QE search: two similarity + top-k passes."""
    return index.search(expand_queries(index, q, alpha, n_qe), k, precision=precision)


def dba(index, alpha=3.0, k_dba=10, rows=None):
    """Database-side augmentation of a single-GPU Index: every row replaced by the normalised
    alpha-weighted sum of its own top-k_dba neighbours (self included).  Returns a new Index.
    Every 1,024 rows are one wide pass over the database (see DBA_QUERIES_PER_PASS).
    rows: augment only the first `rows` rows (the others are copied unchanged) -- bounded benchmarks."""
    if index.db32 is None:
        raise _lib.MdirError("DBA needs the fp32 master copy (keep_fp32=True)")
    index._require_all_live("qe.dba()")
    n_aug = index.n if rows is None else min(int(rows), index.n)
    out = torch.empty_like(index.db32) if n_aug == index.n else index.db32.clone()
    for r0 in range(0, n_aug, DBA_BLOCK):
        r1 = min(r0 + DBA_BLOCK, n_aug)
        s, i = index.search(index.db32[r0:r1], k_dba, precision="fp32", block_q=DBA_QUERIES_PER_PASS)
        out[r0:r1] = _add_l2n(_accumulate(index, i, s, alpha), None)
    return Index(out, device=index.device, keep_fp32=True, idx_base=index.idx_base)


def dba_sharded(sharded, alpha=3.0, k_dba=10):
    """DBA for a row-sharded database (one process per GPU): the shards are all-gathered once
    (bf16 operand + fp32 master: 12 B per element per GPU -- 24.6 GB for 1M x 2048 of the 180 GB),
    then every rank augments ITS OWN rows against the full database; the result is a new
    ShardedIndex with the same row ownership.  Tensor-side work per rank = N/G x N x D, no further
    collective."""
    dist = sharded.dist
    local = sharded.local
    if local.db32 is None:
        raise _lib.MdirError("DBA needs the fp32 master copy (keep_fp32=True)")
    local._require_all_live("qe.dba_sharded()")
    world = sharded.world
    if world == 1:
        out = dba(local, alpha, k_dba)
        return ShardedIndex.from_local(out, sharded.group)
    dev = local.device
    sizes = torch.zeros((world,), dtype=torch.int64, device=dev)
    sizes[dist.get_rank(sharded.group)] = local.n
    dist.all_reduce(sizes, group=sharded.group)
    sizes = [int(x) for x in sizes.tolist()]
    n_max, n_tot = max(sizes), sum(sizes)
    pad = torch.zeros((n_max, local.D), dtype=torch.float32, device=dev)
    pad[:local.n] = local.db32
    gathered = torch.empty((world * n_max, local.D), dtype=torch.float32, device=dev)
    dist.all_gather_into_tensor(gathered, pad, group=sharded.group)
    full = torch.cat([gathered[r * n_max:r * n_max + sizes[r]] for r in range(world)]) if any(s != n_max for s in sizes) else gathered
    del pad
    full_index = Index(full, device=dev, keep_fp32=True, idx_base=0)
    out = torch.empty_like(local.db32)
    for r0 in range(0, local.n, DBA_BLOCK):
        r1 = min(r0 + DBA_BLOCK, local.n)
        s, i = full_index.search(local.db32[r0:r1], k_dba, precision="fp32", block_q=DBA_QUERIES_PER_PASS)
        out[r0:r1] = _add_l2n(_accumulate(full_index, i, s, alpha), None)
    new_local = Index(out, device=dev, keep_fp32=True, idx_base=local.idx_base)
    return ShardedIndex.from_local(new_local, sharded.group)
