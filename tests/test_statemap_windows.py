"""CPU tests of the linear-time window form (fx_statemap_*; forgex_b200.dist.statemap_search): a text split into
slabs, a state map per slab, the maps combined on the host, a backward walk handed from slab to slab.

The kernels are replaced by Python models on the product's own tables: SlabStateMapScan (the slab map of
k_statemap_regions + k_statemap_compose<WINDOW>, same look-back rule) and back_walk (k_statemap_back).  The combine is
the product's own host function.  What is checked: the compose of the slab maps equals the whole-text scan, the span
equals SpanLinear and the oracle, and the host logic of statemap_search over gloo.
"""
import os
import random
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import forgex_b200 as fx
from forgex_b200 import _lib
from forgex_b200 import dist as fxd
from tests import oracle_lib as O
from tests.table_model import StateMapScan
from tests.test_host_tables import gen_pattern, gen_text
from tools import synth

WORDS = _lib.FX_STATEMAP_MAP_WORDS
UNKNOWN = _lib.FX_STATEMAP_UNKNOWN
NEW, DONE = _lib.FX_STATEMAP_WALK_NEW, _lib.FX_STATEMAP_WALK_DONE


class SlabStateMapScan(StateMapScan):
    """StateMapScan over one slab [lo, hi) of a text: region 0's keys are every reachable state walked over the
    `lookback` bytes in front of the slab (all of them when fewer exist; the start state when the slab begins the
    text), sub-chunk 0 takes its candidates from the bytes in front; the map is returned in FX_STATEMAP_MAP_WORDS form"""

    _off = 0                                   # where the slab begins in the bytes handed to the base class

    def bnd(self, text, k):
        return self._off + StateMapScan.bnd(self, text[self._off:], k)

    def slab_map(self, text, lo, hi):
        words = [0] * WORDS
        words[66:98] = [-1] * 32
        if hi <= lo:
            words[0] = 2
            return words
        w0 = max(0, lo - self.lookback)
        s = text[w0:hi]
        self._off = lo - w0
        try:
            spr = max(1, self.region // self.sub)
            chain, reg = None, 0
            while reg * spr * self.sub < len(s) - self._off:
                self._k0, self._k1 = reg * spr, (reg + 1) * spr
                r0, r1 = self.bnd(s, self._k0), min(len(s), self.bnd(s, self._k1))
                m = self.region_map(s, r0, r1)
                if chain is None:
                    if not m:                  # declined (more than 32 states arrive), or no state at all
                        words[0] = 1
                        return words
                    chain = dict(m)
                else:
                    for k, (c, last) in chain.items():
                        if c == 0 or c is None:
                            continue
                        if m is None or c not in m:
                            chain[k] = (None, None)          # unknown
                        else:
                            e, nl = m[c]
                            chain[k] = (e, nl if nl is not None else last)
                reg += 1
        finally:
            self._off = 0
        words[1] = len(chain)
        for i, (k, (e, last)) in enumerate(chain.items()):
            words[2 + i] = k
            words[34 + i] = e if e is not None else 0
            words[66 + i] = UNKNOWN if e is None else -1 if last is None else last + w0
        return words


def compose(sl, maps, n):
    """what fx_statemap_combine computes, in Python: (end, declined)"""
    s = int(sl.t["start"])
    last = 0 if sl.t["start_acc"] else -1
    for m in maps:
        if s == 0:
            break
        if m[0] == 2:
            continue
        if m[0] != 0:
            return -1, 1
        keys = list(m[2:2 + m[1]])
        if s not in keys or m[66 + keys.index(s)] == UNKNOWN:
            return -1, 1
        k = keys.index(s)
        s = m[34 + k]
        if m[66 + k] >= 0:
            last = m[66 + k]
    return sl.end_of_text(s, n, last), 0


class _Window:
    """text[w_lo:w_hi] indexed in text positions; reading outside it is an error"""

    def __init__(self, text, w_lo, w_hi):
        self.text, self.lo, self.hi = text, w_lo, w_hi

    def __getitem__(self, i):
        assert self.lo <= i < self.hi, "read of text byte %d outside the window [%d, %d)" % (i, self.lo, self.hi)
        return self.text[i]


def back_walk(sl, text, w_lo, w_hi, walk, n):
    """k_statemap_back: the backward walk advanced over text[w_lo:w_hi]"""
    pos, best, state, end = walk
    if state == DONE:
        return walk
    s = _Window(text, w_lo, w_hi)
    rd = sl.t["rdelta"]
    nul = sl.cls(0)
    if state == NEW:
        blank = n == 0 or (n == 1 and w_lo == 0 and w_hi >= 1 and s[0] == 0x20)
        if blank or end <= 0:
            return [0, 0, DONE, end]
        r, pos, best = int(sl.t["rstart"]), end, -2
        if end > n:
            r, pos = int(rd[r, nul]) & 0x7FFF, n
    else:
        r = state
    while r != 0 and pos > 0 and (w_lo == 0 or pos - 4 >= w_lo):
        c = s[pos - 1]
        q, cp = pos - 1, c
        if c >= 0x80:
            cp = 0xFFFF
            if (c & 0xC0) == 0x80 and pos >= 2:
                d1 = s[pos - 2]
                if (d1 & 0xE0) == 0xC0:
                    cp, q = ((d1 & 0x1F) << 6) | (c & 0x3F), pos - 2
                elif (d1 & 0xC0) == 0x80 and pos >= 3:
                    d2 = s[pos - 3]
                    if (d2 & 0xF0) == 0xE0:
                        cp, q = ((d2 & 0x0F) << 12) | ((d1 & 0x3F) << 6) | (c & 0x3F), pos - 3
                    elif (d2 & 0xC0) == 0x80 and pos >= 4:
                        d3 = s[pos - 4]
                        if (d3 & 0xF8) == 0xF0:
                            cp, q = ((d3 & 0x07) << 18) | ((d2 & 0x3F) << 12) | ((d1 & 0x3F) << 6) | (c & 0x3F), pos - 4
        w = int(rd[r, sl.cls(cp)])
        r = w & 0x7FFF
        if r == 0:
            break
        pos = q
        if w & 0x8000:
            best = pos
    if r != 0 and pos > 0:
        return [pos, best, r, end]             # at the window's front edge: the holder of byte pos - 1 goes on
    if r != 0 and pos == 0:
        w = int(rd[r, nul])
        if (w & 0x7FFF) != 0 and (w & 0x8000):
            best = -1
    f = 0 if best == -2 else 1 if best < 0 else best + 1
    return [f, min(end, n) if f > 0 else 0, DONE, end]


def walk_slabs(sl, text, slabs, end):
    """the backward hops of statemap_search, slab after slab in one process: ((from, to), hops)"""
    n = len(text)
    if end <= 0:
        return (0, 0), 0
    owner = lambda b: next(i for i, (a, z) in enumerate(slabs) if a <= b < z)     # noqa: E731
    w = owner(end - 1) if end <= n else len(slabs) - 1
    walk, hops = [0, 0, NEW, end], 0
    while True:
        walk = back_walk(sl, text, *fxd.window_for_statemap_slab(n, *slabs[w]), walk, n)
        if walk[2] == DONE:
            return (walk[0], walk[1]), hops
        nxt = owner(walk[0] - 1)
        assert nxt != w, "the walk must leave the window it stopped in"
        w, hops = nxt, hops + 1


def served(p):
    inf = p.info()
    return p.status == 0 and inf["statemap"] and not inf["literal_only"] and not inf["literal_prefix_len"] and not inf["nfa_engine"]


def cut_points(rng, text, k):
    """k - 1 cut points, sorted, duplicates allowed (empty slabs): random, inside UTF-8 sequences, between CR and LF"""
    n = len(text)
    special = [i for i in range(1, n) if (text[i] & 0xC0) == 0x80 or (text[i - 1] == 13 and text[i] == 10)]
    cuts = []
    for _ in range(k - 1):
        r = rng.random()
        cuts.append(rng.choice(special) if special and r < 0.4 else rng.randint(0, n))
    cuts.sort()
    b = [0] + cuts + [n]
    return [(b[i], b[i + 1]) for i in range(k)]


def check_split(p, sm, text, slabs, exp_span, counts):
    sl = sm.sl
    n = len(text)
    maps = [sm.slab_map(text, lo, hi) for lo, hi in slabs]
    end, declined = compose(sl, maps, n)
    out = p.statemap_combine(np.array(maps, dtype=np.int64), n)
    assert (int(out[0]), int(out[1])) == (end, declined), (p.pattern, slabs)
    if declined:
        counts["declined"] += 1
        return None
    st, last = sl.forward(text)
    assert end == sl.end_of_text(st, n, last), (p.pattern, text, slabs)
    whole = sm.last(text)
    assert whole is None or whole == end
    span, hops = walk_slabs(sl, text, slabs, end)
    assert span == sl.regex(text) == exp_span, (p.pattern, text, slabs, span, exp_span)
    counts["ok"] += 1
    counts["hops"] += hops
    return span


@pytest.mark.parametrize("seed", range(6))
def test_slab_maps_of_generated_patterns(seed):
    """fuzz patterns of test_host_tables over random cuts (align 1, slabs shorter than the look-back, empty slabs, cuts
    inside UTF-8 sequences and between CR and LF): compose of the slab maps == the whole-text scan, the product's combine
    == the Python compose, maps + combine + backward hops == SpanLinear == the oracle wherever the model does not
    decline"""
    rng = random.Random(7100 + seed)
    counts = {"ok": 0, "declined": 0, "hops": 0, "patterns": 0}
    for _ in range(25):
        pat = gen_pattern(rng).encode()
        p = fx.Pattern(pat, "regex")
        if not served(p):
            continue
        counts["patterns"] += 1
        sm = SlabStateMapScan(p, lookback=rng.choice([6, 64]))
        texts = [b"\n".join(gen_text(rng) for _ in range(rng.randint(1, 40))) for _ in range(4)] + [b"", b" ", b"a"]
        for text in texts:
            exp = O.regex(pat, text)
            assert exp[4] == 0
            for k in (1, 2, 3, 5, 8):
                check_split(p, sm, text, cut_points(rng, text, k), (exp[2], exp[3]), counts)
    assert counts["patterns"] >= 8 and counts["ok"] >= 200, counts


def test_slab_maps_of_fixed_patterns():
    """the patterns of the single-GPU state-map scan tests, including anchors, `(|^)a` at the leading NUL, `$` before
    CR LF, UTF-8 classes; cut everywhere a slab of 1..3 bytes can be"""
    pats = [synth.PATTERNS["c4"], b"[a-z]+r", rb"\s\S+$", b"[xy]+a[ab]y", rb"[^a]{2,3}$", rb"^\w", b"(a|b)*a(a|b){3}",
            "[ぁ-ん]+a".encode(), rb"\d+-\d+", b"[ab].*c", b".+", b"^$", b"(|^)a", b"[ab]$", b"$"]
    texts = [b"ab\r\nxa\r\n", "xあんa b\r\n12-34 あ".encode(), b"xxay yay\nz\xc3", b"abc", b" ", b"",
             b"ERROR x timeout=12\r\nINFO\n", b"\xe3\x81\x82\xe3\x81\x82a\xf0\x9f\x98\x80a"]
    counts = {"ok": 0, "declined": 0, "hops": 0}
    for pat in pats:
        p = fx.Pattern(pat, "regex")
        assert served(p), pat
        sm = SlabStateMapScan(p, lookback=6)
        for text in texts:
            exp = O.regex(pat, text)
            n = len(text)
            for a in range(n + 1):
                for b in range(a, min(n, a + 3) + 1):
                    check_split(p, sm, text, [(0, a), (a, b), (b, n)], (exp[2], exp[3]), counts)
    assert counts["ok"] > 1000 and counts["declined"] == 0, counts


def test_combine_rejects_what_it_does_not_serve():
    """the codes of the patterns the form does not serve, from the host-only combine"""
    empty = np.zeros((0, WORDS), dtype=np.int64)
    for pat, code in ((b"foo(bar|baz)", _lib.FX_ERR_PREFILTER_UNSUPPORTED), (b"ERROR", _lib.FX_ERR_PREFILTER_UNSUPPORTED),
                      (b"a.*b", _lib.FX_ERR_PREFILTER_UNSUPPORTED), (b".*a(a|b){500}c{20}", _lib.FX_ERR_DFA_STATE_CAP)):
        p = fx.Pattern(pat, "regex")
        with pytest.raises(fx.ForgexError) as e:
            p.statemap_combine(empty, 10)
        assert e.value.status == code, pat
    p = fx.Pattern(b"[ab].*c", "regex")
    assert p.statemap_combine(empty, 0).tolist() == [-1, 0]       # no slab, empty text: no match
    bad = np.zeros((1, WORDS), dtype=np.int64)
    bad[0, :2] = (0, 1)
    bad[0, 2] = int(p.span_tables()["start"])
    bad[0, 34] = 1 << 20                                          # an end state the automaton does not have
    with pytest.raises(fx.ForgexError):
        p.statemap_combine(bad, 10)


DECLINE_PATTERN = b"[ax](b{34})*c"
DECLINE_TEXT = b"xa" + b"b" * 600


def test_a_wide_slab_start_declines():
    """`[ax](b{34})*c` behind 64 bytes of `b`: an attempt in each of 34 phases can be alive, more than the 32 keys a slab
    map holds -- the slab declines, and the combine says so"""
    p = fx.Pattern(DECLINE_PATTERN, "regex")
    assert served(p)
    sm = SlabStateMapScan(p, lookback=64)
    assert sm.slab_map(DECLINE_TEXT, 300, 602)[0] == 1
    maps = [sm.slab_map(DECLINE_TEXT, 0, 300), sm.slab_map(DECLINE_TEXT, 300, 602)]
    assert p.statemap_combine(np.array(maps), len(DECLINE_TEXT)).tolist()[1] == 1


# ---- statemap_search over gloo, the kernels replaced by the models -----------------------------------
def free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def worker(rank, world, port, cfg, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        text, n = cfg["text"], len(cfg["text"])
        p = fx.Pattern(cfg["pattern"], "regex")
        sm = SlabStateMapScan(p, sub=cfg.get("sub", 8), region=cfg.get("region", 40), lookback=fxd.STATEMAP_LOOKBACK)
        lo, hi = fxd.slab_bounds(n, world, rank, align=cfg.get("align", 16))
        w_lo, w_hi = fxd.window_for_statemap_slab(n, lo, hi)
        held = text[:w_hi]                  # (the models only read text[w_lo:w_hi]: _Window checks the walk)

        def window_map(a, b):
            assert (a, b) == (lo, hi)
            return sm.slab_map(held, a, b)

        def combine(maps):
            out = p.statemap_combine(np.array(maps, dtype=np.int64), n)
            return int(out[0]), bool(out[1])

        def back(walk):
            return back_walk(sm.sl, held, w_lo, w_hi, walk, n)
        stats = {}
        r = fxd.statemap_search(window_map, combine, back, n, rank, world, (lo, hi), stats=stats)
        ret[rank] = r + (stats["hops"],)
    finally:
        dist.destroy_process_group()


def run(world, cfg):
    m = mp.Manager()
    ret = m.dict()
    mp.spawn(worker, args=(world, free_port(), cfg, ret), nprocs=world, join=True)
    return [ret[r] for r in range(world)]


def oracle_span(pat, text):
    return O.Compiled(pat, 0).regex_buffer(np.frombuffer(text, dtype=np.uint8))


@pytest.mark.parametrize("world,match_at", [(2, 0.1), (2, 0.9), (3, 0.1), (3, 0.9), (2, None), (3, None)])
def test_statemap_search_c4(world, match_at):
    text = bytes(synth.gen_c4(6000, match_at))
    pat = synth.PATTERNS["c4"]
    res = run(world, {"text": text, "pattern": pat, "align": 1, "sub": 64, "region": 640})
    exp = oracle_span(pat, text)
    assert (exp[0] > 0) == (match_at is not None)
    assert all(r[:3] == (exp[0], exp[1], False) for r in res), (res, exp)
    assert len(set(res)) == 1


def test_statemap_search_match_across_three_slabs():
    """the match spans all three slabs: the walk starts on rank 2 and is handed to rank 1, then to rank 0"""
    text = b"xy" + b"a" * 300 + b"c" + b"z" * 40
    res = run(3, {"text": text, "pattern": b"[ab].*c", "align": 1})
    exp = oracle_span(b"[ab].*c", text)
    assert exp == (3, 303)
    assert all(r == (3, 303, False, 2) for r in res), res


@pytest.mark.parametrize("pat,text", [(b"(|^)a", b"abc" * 40), (rb"^\w", b"hello world\n" * 20), (rb"(|^)a\w*", b"a" + b"b" * 100)])
def test_statemap_search_leading_nul(pat, text):
    """matches that begin at the leading NUL (from = 1) or behind it"""
    res = run(2, {"text": text, "pattern": pat, "align": 1})
    exp = oracle_span(pat, text)
    assert exp[0] > 0
    assert all(r[:3] == (exp[0], exp[1], False) for r in res), (res, exp)


def test_statemap_search_no_c():
    """`[ab].*c` over a text of `a` only: no match, no walk"""
    res = run(3, {"text": b"a" * 3000, "pattern": b"[ab].*c", "align": 1, "sub": 64, "region": 640})
    assert all(r == (0, 0, False, 0) for r in res), res


def test_statemap_search_declines():
    res = run(2, {"text": DECLINE_TEXT, "pattern": DECLINE_PATTERN, "align": 1})
    assert all(r == (0, 0, True, 0) for r in res), res
