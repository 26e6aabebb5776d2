"""Multi-GPU host logic: one process per GPU (torch.distributed), shard the work, exchange only tiny results.

The path shards naturally (SURVEY 8e): strings of a batch are independent, and the start positions of a buffer
search are independent attempts.  No text ever crosses GPUs.

  batches   contiguous string ranges balanced by bytes (shard_strings); results stay sharded; one all-reduce
            of the per-rank match counts (8 bytes per rank).
  buffer    contiguous byte slabs plus a read-only halo behind each slab (attempts started in the slab may run
            into it) and 3 bytes in front (character-boundary look-back); each rank finds the smallest winning
            start of its slab; one all-reduce(MIN) of that 8-byte key; the owner of the winner computes the span;
            one broadcast of 16 bytes.

  buffer, linear time (statemap_search)
            contiguous byte slabs plus 64 bytes of look-back, no halo; each rank computes the state map of its slab
            (the chunked state-map scan of the single-GPU path, every state that can arrive at the slab as a key); one
            all-gather of the maps; every rank combines them into the end of the match; a backward walk from that end
            finds the start, handed to the rank in front by a 32-byte broadcast whenever it reaches its window's front
            edge; the last broadcast carries the span.  No attempt is replayed, so no pattern makes it quadratic.

Everything here is host logic over callbacks (`scan` / `finish`, `window_map` / `combine` / `back`), so it runs
unchanged on CPU with the gloo backend (tests/test_dist_gloo.py and tests/test_statemap_windows.py plug Python models of
the kernels in) and on GPUs with NCCL (plugs the C ABI in).
"""
import numpy as np

NO_START = (1 << 64) - 1
STATEMAP_LOOKBACK = 64                 # bytes in front of a slab the slab map reads (SM_LOOKBACK of the kernels)
STATEMAP_MAP_WORDS = 98                # FX_STATEMAP_MAP_WORDS: status, key count, 32 keys, 32 end states, 32 last accepts
STATEMAP_WALK_NEW, STATEMAP_WALK_DONE = -1, -2


def shard_strings(offsets, world, rank):
    """contiguous range [first, last) of strings for `rank`, balanced by bytes (offsets: n+1 ascending int64)"""
    offsets = np.asarray(offsets)
    n = len(offsets) - 1
    total = int(offsets[-1] - offsets[0])
    cuts = [0]
    for r in range(1, world):
        target = offsets[0] + (total * r) // world
        cuts.append(int(np.searchsorted(offsets[:n], target, side="left")))
    cuts.append(n)
    for i in range(1, len(cuts)):
        cuts[i] = max(cuts[i], cuts[i - 1])
    return cuts[rank], cuts[rank + 1]


def slab_bounds(length, world, rank, align=16):
    """contiguous byte slab [lo, hi) of a buffer of `length` bytes for `rank` (cut at multiples of `align`)"""
    per = -(-length // world)
    per = -(-per // align) * align
    lo = min(length, rank * per)
    hi = min(length, (rank + 1) * per)
    return lo, hi


def window_for_slab(length, lo, hi, halo):
    """the bytes a rank must hold to scan the starts [lo, hi): 3 bytes of look-back, `halo` bytes of look-ahead"""
    w_lo = max(0, lo - 3)
    w_hi = min(length, hi + halo)
    return w_lo, w_hi


def window_for_statemap_slab(length, lo, hi):
    """the bytes a rank must hold for the linear-time form over [lo, hi): STATEMAP_LOOKBACK bytes of look-back, no halo"""
    return max(0, lo - STATEMAP_LOOKBACK), hi


def all_reduce_int(value, op, group=None, device=None):
    """all-reduce of one integer (uint64 keys are shifted into int64 order for MIN)"""
    import torch
    import torch.distributed as dist
    t = torch.tensor([value], dtype=torch.int64, device=device)
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=op, group=group)
    return int(t.item())


def count_matches(local_count, group=None, device=None):
    import torch.distributed as dist
    return all_reduce_int(int(local_count), dist.ReduceOp.SUM, group, device)


def gather_ints(values, group=None, device=None):
    """all-gather of a short vector of integers: returns a world x len(values) list (the one collective of a scan)"""
    import torch
    import torch.distributed as dist
    t = torch.tensor([list(values)], dtype=torch.int64, device=device)
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        out = torch.empty((dist.get_world_size(group), len(values)), dtype=torch.int64, device=device)
        dist.all_gather_into_tensor(out, t, group=group)
        return out.cpu().tolist()
    return t.cpu().tolist()


def _k64(key):
    """uint64 start keys in int64 order: keys are < 2**63 except NO_START, which becomes the largest int64"""
    return key if key != NO_START else (1 << 63) - 1


def buffer_search(scan, finish, length, rank, world, slab, window=None, group=None, device=None, scan_all=None,
                  widen=None, max_widenings=40, stats=None):
    """Leftmost-longest search of one pattern in one buffer that is split across ranks.

    scan(start_lo, start_hi) -> (key, undecided[, occurrences]): smallest winning start of this rank's slab as a
        1-based position in NUL||text||NUL of the whole text (NO_START if none), the number of attempts that ran off
        the window and -- for a pattern with a prefix literal -- how many occurrences of the literal the slab holds.
    scan_all(start_lo, start_hi) -> (key, undecided): the same over EVERY character boundary.  Given for a pattern
        with a prefix literal: Forgex takes its candidate starts from the literal's occurrences, and from every
        boundary when the literal occurs nowhere in the text (api_internal_m.F90:76-104) -- "nowhere" is a property
        of the whole text, so it is decided on the gathered counts.
    finish(key) -> (from, to) computed by the rank whose slab holds the winning start, or (-1, -1) if its window ends
        before the match does.
    widen() -> bool: COLLECTIVE; every rank grows its look-ahead halo with bytes read from its successors (P2P) and
        returns True if some window grew.  Called when an attempt ran off a window (undecided > 0) or the winner's
        window is too short; without it such a search reports the undecided count instead of resolving it.
    Collectives per search: one all-gather of 3 integers per scan round, one 16-byte all-reduce for the span.
    Returns (from, to, undecided_total); every rank gets the same answer.
    """
    import torch
    import torch.distributed as dist
    lo, hi = slab
    active = hi > lo or (rank == 0 and length == 0)
    multi = dist.is_initialized() and world > 1
    every, widenings, carried = False, 0, 0
    while True:
        if active:
            res = scan_all(lo, hi) if every else scan(lo, hi)
        else:
            res = (NO_START, 0, 0)
        mine = (_k64(res[0]), int(res[1]), int(res[2]) if len(res) > 2 else 0)
        table = gather_ints(mine, group, device)
        undecided_total = sum(r[1] for r in table) + carried
        if stats is not None:
            stats["scan_rounds"] = stats.get("scan_rounds", 0) + 1
        if undecided_total > 0 and widen is not None and widenings < max_widenings and widen():
            widenings += 1          # some attempt (or literal occurrence) ran off a window: look further ahead, scan again
            every, carried = False, 0
            continue
        if scan_all is not None and not every and sum(r[2] for r in table) == 0:
            # the literal occurs in no slab: every boundary is a candidate.  An occurrence that straddles an open
            # window end was counted as undecided, not as an occurrence: keep that count
            every, carried = True, undecided_total
            continue
        break
    best = min(r[0] for r in table)
    if stats is not None:
        stats["widenings"] = widenings
    span = torch.zeros(2, dtype=torch.int64, device=device)
    while True:
        span.zero_()
        if best != (1 << 63) - 1:
            pos = best - 2                       # text index of the winning start (-1: the leading NUL)
            if (lo <= pos < hi) or (pos < 0 and rank == 0):
                f, t = finish(best)
                span[0], span[1] = f, t
            if multi:
                dist.all_reduce(span, group=group)      # SUM: every other rank holds zeros
        f, t = (int(x) for x in span.cpu().tolist())
        if f == -1 and t == -1 and widen is not None and widenings < max_widenings and widen():
            widenings += 1                       # the winner's window ends before its match does
            continue
        break
    return f, t, undecided_total


def statemap_search(window_map, combine, back, length, rank, world, slab, group=None, device=None, stats=None):
    """Leftmost-longest search of one pattern in one buffer split across ranks, in time linear in the text.

    window_map(lo, hi) -> STATEMAP_MAP_WORDS integers: the slab map of this rank's slab [lo, hi) (fx_statemap_window_dev).
    combine(maps) -> (end, declined): the slab maps of all ranks chained in text order (fx_statemap_combine).
    back(walk) -> walk: the backward walk advanced over this rank's window (fx_statemap_back_dev); walk = [pos, best,
        reverse state, end], started as [0, 0, STATEMAP_WALK_NEW, end], over when walk[2] == STATEMAP_WALK_DONE, and
        then walk[:2] = (from, to).
    Collectives per search: one all-gather of STATEMAP_MAP_WORDS + 2 integers, then one 32-byte broadcast per rank the
    walk visits -- the first from the rank that holds byte end - 1 (the last rank when the trailing NUL was consumed),
    one more per slab boundary the match crosses (stats["hops"]); the last one carries the span.  Nothing when there is
    no match.  Returns (from, to, declined); every rank gets the same answer.  declined: more than 32 states can arrive
    at some slab on the true path, (from, to) = (0, 0) is then no answer: search with buffer_search instead.
    """
    import torch
    import torch.distributed as dist
    lo, hi = slab
    multi = dist.is_initialized() and world > 1
    table = gather_ints(list(window_map(lo, hi)) + [lo, hi], group, device)
    maps = [row[:STATEMAP_MAP_WORDS] for row in table]
    slabs = [(row[STATEMAP_MAP_WORDS], row[STATEMAP_MAP_WORDS + 1]) for row in table]
    end, declined = combine(maps)
    hops = 0
    if stats is not None:
        stats["hops"] = 0
    if declined:
        return 0, 0, True
    if end <= 0:
        return 0, 0, False

    def owner(b):
        return next(r for r, (a, z) in enumerate(slabs) if a <= b < z)

    walker = owner(end - 1) if end <= length else len(slabs) - 1
    walk = torch.tensor([0, 0, STATEMAP_WALK_NEW, end], dtype=torch.int64, device=device)
    while True:
        if rank == walker:
            walk.copy_(torch.tensor(back(walk.cpu().tolist()), dtype=torch.int64))
        if multi:
            dist.broadcast(walk, src=walker if group is None else dist.get_global_rank(group, walker), group=group)
        pos, best, state, _ = walk.cpu().tolist()
        if state == STATEMAP_WALK_DONE:
            break
        nxt = owner(pos - 1)
        if nxt == walker:
            raise RuntimeError("backward walk stopped at %d inside the window of rank %d: the window lacks its look-back"
                               % (pos, walker))
        walker = nxt
        hops += 1
    if stats is not None:
        stats["hops"] = hops
    return pos, best, False


class _GpuWindow:
    """a rank's piece of the text on its GPU: slab + 3 bytes of look-back + a look-ahead halo that can grow"""

    def __init__(self, d_window, origin, length, rank, world, slab, group):
        self.t, self.origin, self.length = d_window, origin, length
        self.rank, self.world, self.slab, self.group = rank, world, slab, group

    def end(self):
        return self.origin + self.t.numel()

    def widen(self):
        """double every rank's halo with bytes read from the ranks that own them (P2P send/recv over NVLink)"""
        import torch
        import torch.distributed as dist
        ends = gather_ints((self.slab[0], self.slab[1], self.end()), self.group, self.t.device)
        want = []
        for r, (s_lo, s_hi, w_hi) in enumerate(ends):
            halo = max(w_hi - s_hi, 64)
            want.append((w_hi, min(self.length, w_hi + halo)))       # rank r asks for text[w_hi : w_hi + halo)
        if all(b <= a for a, b in want):
            return False
        ops, recv = [], []
        for r, (a, b) in enumerate(want):
            for src, (s_lo, s_hi, _) in enumerate(ends):
                x, y = max(a, s_lo), min(b, s_hi)
                if y <= x or src == r:
                    continue
                if src == self.rank:
                    ops.append(dist.P2POp(dist.isend, self.t[x - self.origin:y - self.origin].contiguous(), r, group=self.group))
                if r == self.rank:
                    buf = torch.empty(y - x, dtype=torch.uint8, device=self.t.device)
                    recv.append((x, buf))
                    ops.append(dist.P2POp(dist.irecv, buf, src, group=self.group))
        if ops:
            for w in dist.batch_isend_irecv(ops):
                w.wait()
        if recv:
            recv.sort(key=lambda e: e[0])
            self.t = torch.cat([self.t] + [b for _, b in recv])
        return True


def gpu_buffer_search(pattern_obj, d_window, window_origin, length, rank, world, slab, group=None, stats=None):
    """buffer_search over the C ABI: d_window is this rank's CUDA tensor holding text[window_origin : ...]"""
    import torch
    dev = d_window.device
    win = _GpuWindow(d_window, window_origin, length, rank, world, slab, group)
    best = torch.empty(3, dtype=torch.int64, device=dev)
    init = torch.tensor([-1, 0, 0], dtype=torch.int64, device=dev)
    ft = torch.zeros(2, dtype=torch.int64, device=dev)
    prefixed = bool(pattern_obj.info()["prefix_scan"])

    def run(lo, hi, every_boundary):
        best.copy_(init)                       # key = all ones, no undecided attempts, no occurrences
        wlen = win.t.numel()
        call = pattern_obj.buffer_scan_all_dev if every_boundary else pattern_obj.buffer_scan_dev
        call(win.t, wlen, lo - win.origin, hi - win.origin, win.origin, win.origin == 0, win.end() == length, best)
        b = best.cpu().numpy().view(np.uint64)
        return int(b[0]), int(b[1]), int(b[2])

    def scan(lo, hi):
        return run(lo, hi, False)

    def scan_all(lo, hi):
        return run(lo, hi, True)[:2]

    def finish(key):
        k = torch.tensor([key], dtype=torch.int64, device=dev)
        pattern_obj.buffer_finish_dev(win.t, win.t.numel(), win.origin, win.end() == length, k, ft)
        r = ft.cpu().numpy()
        return int(r[0]), int(r[1])

    return buffer_search(scan, finish, length, rank, world, slab, None, group, dev, scan_all if prefixed else None,
                         widen=win.widen if world > 1 else None, stats=stats)


def gpu_buffer_search_linear(pattern_obj, d_window, window_origin, length, rank, world, slab, group=None, stats=None):
    """statemap_search over the C ABI: d_window is this rank's CUDA tensor holding text[window_for_statemap_slab(...)].

    Patterns the linear-time form does not serve (a prefix literal, a literal-only pattern, no span path, the NFA
    engine) and searches it declines are answered by gpu_buffer_search on the same window, whose look-ahead halo starts
    empty and grows on demand (what that scan does not serve either -- a sequential candidate list, an NFA-engine
    handle -- raises its ForgexError).  stats["route"] = "statemap" or "scan".  Returns (from, to)."""
    import torch
    from .api import ForgexError
    from . import _lib
    lo, hi = slab
    assert (window_origin, window_origin + d_window.numel()) == window_for_statemap_slab(length, lo, hi), \
        "the window must come from window_for_statemap_slab"
    stats = {} if stats is None else stats
    dev = d_window.device
    try:
        pattern_obj.statemap_combine(np.zeros((0, STATEMAP_MAP_WORDS), dtype=np.int64), length)     # (host-only)
        served = True
    except ForgexError as e:
        if e.status not in (_lib.FX_ERR_DFA_STATE_CAP, _lib.FX_ERR_PREFILTER_UNSUPPORTED):
            raise
        served = False                  # a property of the pattern: every rank takes the same route
    if served:
        wlen = d_window.numel()
        d_map = torch.empty(STATEMAP_MAP_WORDS, dtype=torch.int64, device=dev)
        work = torch.empty(pattern_obj.buffer_work_bytes(hi - lo), dtype=torch.uint8, device=dev)
        d_walk = torch.empty(4, dtype=torch.int64, device=dev)

        def window_map(a, b):
            pattern_obj.statemap_window_dev(d_window, wlen, a - window_origin, b - window_origin, window_origin, d_map, work)
            return d_map.cpu().tolist()

        def combine(maps):
            out = pattern_obj.statemap_combine(np.array(maps, dtype=np.int64), length)
            return int(out[0]), bool(out[1])

        def back(walk):
            d_walk.copy_(torch.tensor(walk, dtype=torch.int64))
            pattern_obj.statemap_back_dev(d_window, wlen, window_origin, length, d_walk)
            return d_walk.cpu().tolist()

        f, t, declined = statemap_search(window_map, combine, back, length, rank, world, slab, group, dev, stats)
        if not declined:
            stats["route"] = "statemap"
            return f, t
    stats["route"] = "scan"
    f, t, _ = gpu_buffer_search(pattern_obj, d_window, window_origin, length, rank, world, slab, group, stats)
    return f, t
