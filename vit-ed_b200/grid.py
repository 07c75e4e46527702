"""All-pairs grid drivers: what replaces the pair loops of evaluation.py:101-131 (puzzle) and hisfrag.py:161-296
(Hisfrag20), plus the integer bookkeeping around them (pair enumeration, row sharding, consumer layouts).

Multi-GPU: the grid shards by rows with no data-path collective; every rank encodes all items itself and scores its
row block; ONE all-gather of the score blocks at the end replaces the shared-filesystem polling of
hisfrag.py:251-276 (SURVEY 8e).
"""
import math

import numpy as np
import torch

from . import _lib


# --------------------------------------------------------------------------------------------- pair enumeration
def ordered_pairs(n):
    """[(i, j) for i for j if i != j], i-major (data/datasets/pieces_dataset.py:27-32) as int32 [n(n-1), 2]."""
    i = np.repeat(np.arange(n, dtype=np.int32), n)
    j = np.tile(np.arange(n, dtype=np.int32), n)
    keep = i != j
    return np.stack([i[keep], j[keep]], axis=1)


def ordered_pair_index(i, j, n):
    """entry index of (i, j) in ordered_pairs(n): i*(n-1) + (j if j < i else j-1)."""
    return i * (n - 1) + (j if j < i else j - 1)


def upper_tri_pairs(n):
    """torch.combinations(arange(n), r=2, with_replacement=True) (hisfrag.py:166-167): rows (a, b), a <= b, a-major."""
    a, b = np.triu_indices(n)
    return np.stack([a.astype(np.int32), b.astype(np.int32)], axis=1)


# --------------------------------------------------------------------------------------------- row sharding
def indicates_row_ranges(indexes, num_replicas):
    """Row boundaries computed exactly like DistributedIndicatesSampler (data/samplers.py:108-137): split the sorted
    first-column ``indexes`` into ceil(P/world)-sized chunks and snap each boundary to a row. Returns ``sizes`` with
    len(chunks)+1 entries; rank r owns rows [sizes[r], sizes[r+1]). (When a row straddles two chunks the reference
    moves the boundary to ``row - 1``; kept as is.)"""
    indexes = np.asarray(indexes)
    n_per = math.ceil(len(indexes) / num_replicas)
    starts = list(range(0, len(indexes), n_per))
    sizes = [0]
    for c in range(1, len(starts)):
        first = int(indexes[starts[c]])
        prev_last = int(indexes[starts[c] - 1])
        sizes.append(first - 1 if first == prev_last else first)
    sizes.append(int(indexes[-1]) + 1)
    return sizes


def hisfrag_row_ranges(n, num_replicas):
    """``indicates_row_ranges(upper_tri_pairs(n)[:, 0], num_replicas)`` in O(num_replicas) Python integer operations,
    without the n(n+1)/2-entry pair list (200 M pairs, gigabytes of host arrays, at 20,000 fragments). Row a of the
    upper-triangular grid holds pair indices [off(a), off(a + 1)) with off(a) = a*n - a(a-1)/2; the row of a pair index
    is the inverse of that quadratic (math.isqrt, then a +-1 fix-up for the rounding of the root)."""
    n_pairs = n * (n + 1) // 2
    n_per = -(-n_pairs // num_replicas)

    def off(a):
        return a * n - a * (a - 1) // 2

    def row(k):
        b = 2 * n + 1
        a = (b - math.isqrt(b * b - 8 * k)) // 2
        while a > 0 and off(a) > k:
            a -= 1
        while off(a + 1) <= k:
            a += 1
        return a

    starts = range(0, n_pairs, n_per)      # the reference's chunk starts (ValueError for an empty grid, as there)
    sizes = [0]
    for c in range(1, len(starts)):
        first, prev_last = row(starts[c]), row(starts[c] - 1)
        sizes.append(first - 1 if first == prev_last else first)
    sizes.append(row(n_pairs - 1) + 1)
    return sizes


def hisfrag_row_range(n, world, rank):
    """Rows of the upper-triangular grid owned by ``rank`` (hisfrag.py:166-170)."""
    sizes = hisfrag_row_ranges(n, world)
    if rank + 1 >= len(sizes):
        return n, n  # fewer chunks than ranks: this rank has nothing (the reference would raise IndexError)
    return sizes[rank], sizes[rank + 1]


def equal_row_range(n_rows, world, rank):
    """Contiguous equal split (every puzzle row has N-1 pairs, SURVEY 8e)."""
    per = math.ceil(n_rows / world)
    lo = min(rank * per, n_rows)
    return lo, min(lo + per, n_rows)


def puzzle_unit_ranges(n_pieces, world, rank):
    """BASELINE configs[2] sharding (SURVEY 8e): the (puzzle, row) units of a batch of puzzles -- every unit is one grid
    row of N_p - 1 pairs -- are numbered puzzle-major and split into ``world`` contiguous equal shares. Returns rank's
    share as [(puzzle, row_lo, row_hi), ...] (at most one segment per puzzle, puzzle ascending)."""
    starts = np.concatenate([[0], np.cumsum(np.asarray(n_pieces, dtype=np.int64))])
    lo, hi = equal_row_range(int(starts[-1]), world, rank)
    out = []
    for p in range(len(n_pieces)):
        a, b = max(lo, int(starts[p])), min(hi, int(starts[p + 1]))
        if a < b:
            out.append((p, a - int(starts[p]), b - int(starts[p])))
    return out


# --------------------------------------------------------------------------------------------- collectives
def _all_gather_rows(block, ranges, n_rows):
    """all-gather variable-height row blocks -> [n_rows, ...] on every rank (pads to the tallest block)."""
    import torch.distributed as dist
    world = dist.get_world_size()
    tallest = max(hi - lo for lo, hi in ranges)
    padded = block.new_zeros((tallest,) + tuple(block.shape[1:]))
    padded[:block.shape[0]] = block
    bufs = [torch.empty_like(padded) for _ in range(world)]
    dist.all_gather(bufs, padded)
    out = block.new_zeros((n_rows,) + tuple(block.shape[1:]))
    for (lo, hi), buf in zip(ranges, bufs):
        out[lo:hi] = buf[:hi - lo]
    return out


def _dist_info():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


# --------------------------------------------------------------------------------------------- grid entries
@torch.no_grad()
def score_puzzle(model, images, gather=True):
    """images [N,3,S,S] (all pieces, same on every rank) -> logits [N, N, C] fp32, logits[i, j] = model pair (i, j);
    the diagonal is zero (the reference never scores i == j). Replaces evaluation.py:101-107."""
    rank, world = _dist_info()
    n = images.shape[0]
    ranges = [equal_row_range(n, world, r) for r in range(world)]
    lo, hi = ranges[rank]
    block = model.score_grid(images, _lib.GRID_ORDERED_OFFDIAG, lo, hi)
    if world == 1 or not gather:
        return block
    return _all_gather_rows(block, ranges, n)


@torch.no_grad()
def score_puzzles(model, puzzles, n_pieces=None, gather=True, blocks_out=None):
    """A batch of puzzles, each scored all-pairs, the (puzzle, row) units sharded over the ranks (``puzzle_unit_ranges``)
    with no data-path collective and ONE all-gather of the score blocks at the end. Replaces the per-puzzle loop of
    evaluation.py:82-114 for a whole evaluation set.

    puzzles[p]: CUDA tensor [N_p, 3, S, S] of puzzle p's pieces, or a zero-argument callable returning it (called only
    on the ranks that own rows of puzzle p; ``n_pieces`` must then list every N_p). Returns a list with one
    [N_p, N_p, C] fp32 logits tensor per puzzle (diagonals zero); with ``gather=False`` (or a single rank's share)
    entries of puzzles this rank owns no rows of are None and partially owned puzzles hold the owned rows only,
    as ``(row_lo, row_hi, block)``."""
    rank, world = _dist_info()
    if n_pieces is None:
        n_pieces = [int(p.shape[0]) for p in puzzles]
    mine = puzzle_unit_ranges(n_pieces, world, rank)
    n_classes = model.num_classes
    owned = {p: (puzzles[p]() if callable(puzzles[p]) else puzzles[p]) for p, _, _ in mine}
    dev = next(iter(owned.values())).device if owned else next(model.parameters()).device
    # this rank's blocks, back to back in one flat buffer (what the all-gather moves)
    sizes = [(hi - lo) * n_pieces[p] * n_classes for p, lo, hi in mine]
    flat_len = [sum((hi - lo) * n_pieces[p] * n_classes for p, lo, hi in puzzle_unit_ranges(n_pieces, world, r))
                for r in range(world)]
    longest = max(flat_len) if flat_len else 0
    flat = blocks_out if blocks_out is not None else torch.zeros(longest, dtype=torch.float32, device=dev)
    if flat.numel() < longest or flat.dtype != torch.float32 or flat.device != dev:
        raise _lib.VitedError(f'score_puzzles: blocks_out must be a fp32 buffer of at least {longest} elements on {dev}')
    off = 0
    for (p, lo, hi), size in zip(mine, sizes):
        images = owned[p]
        if images.shape[0] != n_pieces[p]:
            raise _lib.VitedError(f'score_puzzles: puzzle {p} has {images.shape[0]} pieces, n_pieces says {n_pieces[p]}')
        block = flat[off:off + size].view(hi - lo, n_pieces[p], n_classes)
        block.zero_()                      # the diagonal is never written
        model.score_grid(images, _lib.GRID_ORDERED_OFFDIAG, lo, hi, out=block)
        off += size
    if world == 1 or not gather:
        out, off = [None] * len(n_pieces), 0
        for (p, lo, hi), size in zip(mine, sizes):
            block = flat[off:off + size].view(hi - lo, n_pieces[p], n_classes)
            out[p] = block if (lo, hi) == (0, n_pieces[p]) else (lo, hi, block)
            off += size
        return out
    import torch.distributed as dist
    gathered = torch.empty(world * longest, dtype=torch.float32, device=dev)
    dist.all_gather_into_tensor(gathered, flat[:longest])     # NCCL: one ncclAllGather over NVLink
    gathered = gathered.view(world, longest)
    out = [torch.zeros((n, n, n_classes), dtype=torch.float32, device=dev) for n in n_pieces]
    for r in range(world):
        off = 0
        for p, lo, hi in puzzle_unit_ranges(n_pieces, world, r):
            size = (hi - lo) * n_pieces[p] * n_classes
            out[p][lo:hi] = gathered[r, off:off + size].view(hi - lo, n_pieces[p], n_classes)
            off += size
    return out


@torch.no_grad()
def score_fragments(model, images, gather=True, resume_path=None, block_rows=64, save_every=5, remove_cache_file=False,
                    xsrc_budget_mb=None):
    """images [N,3,S,S] fp32, or the uint8 crops [N,S,S,3] of ``pieces.fragments_to_u8_device`` (same scores, a
    quarter of the memory) -> symmetric similarity logits [N, N] fp32 (raw logits, no sigmoid: hisfrag.py:230-231,
    :281-292). Rows are sharded as DistributedIndicatesSampler does (hisfrag.py:170).

    ``xsrc_budget_mb`` (None: leave the engine's setting) bounds the decoder input states of the grid columns held at
    once (``OPT_XSRC_BUDGET_MB``, default 32,000 MB = 20,345 Hisfrag fragments); a larger grid is scored in column
    windows of that size.

    ``resume_path`` switches on the crash-resume of the reference's test loop (hisfrag.py:181-195, :243-246): the
    rank's rows are then walked in blocks of ``block_rows`` rows (the reference's x1 batches), after every
    ``save_every`` blocks (SAVE_TMP_FREQ, config.py:225) and after the last one the rows scored so far go to
    ``resume_path.format(rank=rank)`` together with an ``is_finished`` flag, and a later call with the same grid picks up
    behind the last saved block (``remove_cache_file=True`` discards the file first, as in the reference). A file
    written for another grid size or row range is an error, not silently reused."""
    rank, world = _dist_info()
    n = images.shape[0]
    if xsrc_budget_mb is not None:
        model.set_option(_lib.OPT_XSRC_BUDGET_MB, xsrc_budget_mb)
    if world == 1:
        ranges = [(0, n)]
    else:
        sizes = hisfrag_row_ranges(n, world)
        if any(a > b for a, b in zip(sizes, sizes[1:])):
            # for grids of a dozen items the reference sampler's row snapping (samplers.py:113-134) yields boundaries
            # that run backwards; every rank sees the same `sizes`, so all of them stop here, before any collective
            raise _lib.VitedError(f'score_fragments: the reference sampler cannot split {n} items over {world} ranks '
                                  f'(row boundaries {sizes})')
        ranges = [(sizes[r], sizes[r + 1]) if r + 1 < len(sizes) else (n, n) for r in range(world)]
    lo, hi = ranges[rank]
    if resume_path is None:
        block = model.score_grid(images, _lib.GRID_UPPER_TRI_DIAG, lo, hi)[..., 0]
    else:
        block = _score_fragment_rows_resumable(model, images, lo, hi, str(resume_path).format(rank=rank), block_rows,
                                               save_every, remove_cache_file)
    if world > 1 and gather:
        upper = _all_gather_rows(block, ranges, n)
    elif world > 1:
        return block
    else:
        upper = block
    return mirror_upper(upper)


def _score_fragment_rows_resumable(model, images, lo, hi, path, block_rows, save_every, remove_cache_file):
    """Rows [lo, hi) of the upper-triangular grid in saved blocks (see score_fragments)."""
    import os
    if block_rows < 1 or save_every < 1:
        raise _lib.VitedError(f'score_fragments: block_rows={block_rows} and save_every={save_every} must be positive')
    n = images.shape[0]
    block = images.new_zeros((hi - lo, n), dtype=torch.float32)
    done = lo
    if os.path.exists(path):
        if remove_cache_file:
            os.unlink(path)
        else:
            data = torch.load(path, map_location='cpu')
            if data.get('n') != n or tuple(data.get('rows', ())) != (lo, hi):
                raise _lib.VitedError(f'score_fragments: {path} holds rows {data.get("rows")} of a {data.get("n")}-item grid, '
                                      f'this call scores rows {(lo, hi)} of {n} items')
            done = int(data['done'])
            block[:done - lo] = data['upper'].to(block.device)
            if data['is_finished']:
                return block

    def save(until, finished):
        tmp = path + '.tmp'
        torch.save({'n': n, 'rows': (lo, hi), 'done': until, 'upper': block[:until - lo].cpu(), 'is_finished': finished}, tmp)
        os.replace(tmp, path)      # a crash during the write leaves the previous file intact

    starts = list(range(done, hi, block_rows))
    for k, a in enumerate(starts):
        b = min(a + block_rows, hi)
        block[a - lo:b - lo] = model.score_grid(images, _lib.GRID_UPPER_TRI_DIAG, a, b)[..., 0]
        last = k == len(starts) - 1
        if k % save_every == 0 or last:
            save(b, last)
    if not starts:
        save(hi, True)             # an empty row range (more ranks than chunks) still reports "finished"
    return block


# --------------------------------------------------------------------------------------------- pair lists
def extension_pairs(is_new):
    """The pairs of ``upper_tri_pairs(N)`` that touch a new item: every (a, b) with a <= b and ``is_new[a] or
    is_new[b]``, a-major with b ascending, as int32 [P, 2]. What a scored collection of the old items lacks once the new
    ones are inserted at their sorted positions: N_old * N_new + N_new (N_new + 1) / 2 pairs."""
    is_new = np.asarray(is_new, dtype=bool)
    n = len(is_new)
    new_idx = np.flatnonzero(is_new).astype(np.int32)
    rows = []
    for a in range(n):
        cols = np.arange(a, n, dtype=np.int32) if is_new[a] else new_idx[np.searchsorted(new_idx, a):]
        if len(cols):
            rows.append(np.stack([np.full(len(cols), a, dtype=np.int32), cols], axis=1))
    return np.concatenate(rows) if rows else np.zeros((0, 2), dtype=np.int32)


def pair_shares(ctx_items, world):
    """Sharding of a pair list over ``world`` ranks: the pairs stable-sorted by context item (so that a rank encodes
    only the context items of its share), then split into contiguous shares of equal pair count. Returns ``order``
    (sorted position -> input position, int64) and ``bounds`` (rank r takes sorted positions [bounds[r], bounds[r+1]))."""
    ctx_items = np.asarray(ctx_items)
    order = np.argsort(ctx_items, kind='stable').astype(np.int64)
    per = -(-len(ctx_items) // world)
    bounds = [min(r * per, len(ctx_items)) for r in range(world + 1)]
    return order, bounds


def unpermute_shares(gathered, order, bounds):
    """Inverse of ``pair_shares``: ``gathered`` [world, longest, ...] holds rank r's scores in its first
    bounds[r+1] - bounds[r] rows; returns them as [P, ...] in input order."""
    shares = [gathered[r, :bounds[r + 1] - bounds[r]] for r in range(len(bounds) - 1)]
    flat = torch.cat(shares) if shares else gathered.new_zeros((0,) + tuple(gathered.shape[2:]))
    out = torch.empty_like(flat)
    out[torch.as_tensor(order, device=flat.device)] = flat
    return out


@torch.no_grad()
def score_pairs(model, images, pairs, gather=True):
    """Logits of a pair list -> [P, num_classes] fp32 in the list's order (``model.score_pairs`` on every rank's share,
    see ``pair_shares``), then ONE all-gather of the padded shares. ``images`` (either form of ``score_grid``) are
    the whole collection on every rank; ``pairs`` a [P, 2] int32 / int64 tensor or array (any device). With several
    ranks and ``gather=False``, returns this rank's share as (input positions int64 [P_r], logits [P_r, C])."""
    rank, world = _dist_info()
    dev = images.device
    if world == 1:
        return model.score_pairs(images, torch.as_tensor(pairs).to(dev))
    pairs_np = (pairs.cpu().numpy() if isinstance(pairs, torch.Tensor) else np.asarray(pairs)).astype(np.int64)
    if pairs_np.ndim != 2 or pairs_np.shape[1] != 2:
        raise ValueError(f'pairs must be [P, 2], got {pairs_np.shape}')
    order, bounds = pair_shares(pairs_np[:, 0], world)
    lo, hi = bounds[rank], bounds[rank + 1]
    mine = model.score_pairs(images, torch.from_numpy(pairs_np[order[lo:hi]]).to(dev))
    if not gather:
        return torch.from_numpy(order[lo:hi]), mine
    import torch.distributed as dist
    longest = max(b - a for a, b in zip(bounds, bounds[1:]))
    padded = mine.new_zeros((longest, model.num_classes))
    padded[:hi - lo] = mine
    gathered = mine.new_empty((world * longest, model.num_classes))
    dist.all_gather_into_tensor(gathered, padded)
    return unpermute_shares(gathered.view(world, longest, model.num_classes), order, bounds)


@torch.no_grad()
def extend_fragments(model, images, old_sim, is_new, gather=True):
    """Similarity logits [N, N] fp32 of a fragment collection grown by new items, without re-scoring the old ones.
    ``images`` is the whole collection in its sorted order (fp32 or the uint8 crops, as ``score_fragments``);
    ``is_new[k]`` marks the new items; ``old_sim`` is the ``score_fragments`` matrix of the old items in their relative
    order. Old x old entries are copied from ``old_sim``; every other entry is scored through
    ``score_pairs(extension_pairs(is_new))`` and mirrored as ``mirror_upper`` does. With several ranks and
    ``gather=False``, returns this rank's share of the extension pairs as ``score_pairs`` does."""
    is_new = np.asarray(is_new, dtype=bool)
    n = images.shape[0]
    if is_new.shape != (n,):
        raise ValueError(f'is_new has shape {is_new.shape}, the collection {n} items')
    old = np.flatnonzero(~is_new)
    if tuple(old_sim.shape) != (len(old), len(old)):
        raise ValueError(f'old_sim is {tuple(old_sim.shape)}, the collection has {len(old)} old items')
    pairs = extension_pairs(is_new)
    scores = score_pairs(model, images, pairs, gather=gather)
    if isinstance(scores, tuple):
        return scores
    dev = images.device
    upper = torch.zeros((n, n), dtype=torch.float32, device=dev)
    p = torch.from_numpy(pairs).to(dev).long()
    upper[p[:, 0], p[:, 1]] = scores[:, 0]
    sim = mirror_upper(upper)
    o = torch.from_numpy(old).to(dev)
    sim[o[:, None], o[None, :]] = old_sim.to(device=dev, dtype=torch.float32)
    return sim


def mirror_upper(upper):
    """sim[a, b] = sim[b, a] = score(a, b) for a <= b (hisfrag.py:291-292)."""
    tri = torch.triu(upper)
    return tri + torch.triu(upper, diagonal=1).transpose(0, 1)


# --------------------------------------------------------------------------------------------- consumer layouts
def puzzle_distance(logits):
    """1 - sigmoid(logit) (evaluation.py:109-114), fp32 [N, N, 4] on the host as numpy."""
    return (1.0 - torch.sigmoid(logits)).cpu().numpy()


def make_distance_function(distance, side_enum):
    """The closure of evaluation.py:116-131 as an array lookup. ``distance[i, j]`` is indexed by origin_piece_id;
    bin 0: i.right-j.left, 1: i.bottom-j.top, 2: i.left-j.right, 3: i.top-j.bottom; x1000; inf otherwise."""
    def distance_function(piece_i, piece_i_side, piece_j, piece_j_side):
        pred = distance[piece_i.origin_piece_id][piece_j.origin_piece_id]
        if piece_j_side == side_enum.left:
            if piece_i_side == side_enum.right:
                return pred[0] * 1000.
        if piece_j_side == side_enum.right:
            if piece_i_side == side_enum.left:
                return pred[2] * 1000.
        if piece_j_side == side_enum.top:
            if piece_i_side == side_enum.bottom:
                return pred[1] * 1000.
        if piece_j_side == side_enum.bottom:
            if piece_i_side == side_enum.top:
                return pred[3] * 1000.
        return float('inf')
    return distance_function


def similarity_to_distance(sim):
    """fp16 similarity matrix then ``1 - sim`` (hisfrag.py:281-296) -> numpy fp16 [N, N]."""
    sim16 = sim.detach().to('cpu').type(torch.float16)
    return (1 - sim16).numpy()


def retrieval_metrics(similarity, labels):
    """(mAP, top-1, Pr@10, Pr@100) of ``wi19_evaluate.get_metrics(1 - fp16(similarity), labels)`` (hisfrag.py:283-309,
    misc/wi19_evaluate.py:12-56), evaluated on the device from the fp32 similarity matrix that ``score_fragments``
    returns (C-ABI ``vited_retrieval_rows``: ranks of the relevant items by counting, no sort, no N x N host copy).
    labels: integer writer ids (``utils.list_to_idx`` output). Ties in distance are ordered by ascending index."""
    import ctypes

    import numpy as np
    from . import _lib
    if not (isinstance(similarity, torch.Tensor) and similarity.is_cuda and similarity.dtype == torch.float32
            and similarity.dim() == 2 and similarity.shape[0] == similarity.shape[1]):
        raise _lib.VitedError('retrieval_metrics: similarity must be a square CUDA fp32 tensor (there is no CPU path)')
    n = similarity.shape[0]
    dev = similarity.device
    labels_np = np.asarray(labels)
    if labels_np.shape != (n,):
        raise _lib.VitedError(f'retrieval_metrics: {labels_np.shape} labels for {n} items')
    similarity = similarity.contiguous()
    with torch.cuda.device(dev):
        lab = torch.from_numpy(labels_np.astype(np.int32)).to(dev)
        n_rel = torch.empty(n, dtype=torch.int32, device=dev)
        ap_sum = torch.empty(n, dtype=torch.float64, device=dev)
        top1 = torch.empty(n, dtype=torch.int32, device=dev)
        h10 = torch.empty(n, dtype=torch.int32, device=dev)
        h100 = torch.empty(n, dtype=torch.int32, device=dev)
        p = lambda t: ctypes.c_void_p(t.data_ptr())
        _lib.check(_lib.lib.vited_retrieval_rows(p(similarity), p(lab), n, p(n_rel), p(ap_sum), p(top1), p(h10), p(h100),
                                                 ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)),
                   'vited_retrieval_rows')
        n_rel, ap_sum, top1, h10, h100 = [t.cpu().numpy() for t in (n_rel, ap_sum, top1, h10, h100)]
    keep = n_rel > 0
    m_ap = (ap_sum[keep] / n_rel[keep]).mean()
    with np.errstate(invalid='ignore', divide='ignore'):       # singleton queries: 0 / 0 = nan, as in the reference
        pr10 = (h10 / np.minimum(n_rel, 10)).sum() / n
        pr100 = (h100 / np.minimum(n_rel, 100)).sum() / n
    return float(m_ap), float(top1.sum() / n), float(pr10), float(pr100)
