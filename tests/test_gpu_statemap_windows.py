"""GPU tests of the linear-time window form (fx_statemap_window_dev / fx_statemap_combine / fx_statemap_back_dev and
forgex_b200.dist.gpu_buffer_search_linear) against the CPU oracle and the single-buffer state-map scan.

One device: the "ranks" are slabs processed one after another, each through its own window tensor (the slab and
64 bytes in front of it) -- the way a rank holds its piece of the text.
"""
import os
import random
import socket
import time

import numpy as np
import pytest
import torch

import forgex_b200 as fx
from forgex_b200 import _lib
from forgex_b200 import dist as fxd
from tests import oracle_lib as O
from tools import synth

pytestmark = pytest.mark.gpu

WORDS, NEW, DONE = _lib.FX_STATEMAP_MAP_WORDS, _lib.FX_STATEMAP_WALK_NEW, _lib.FX_STATEMAP_WALK_DONE


def split_search(p, d_text, n, slabs):
    """slab maps, the host combine, the backward hops: ((from, to), declined, hops)"""
    dev = d_text.device
    windows = [fxd.window_for_statemap_slab(n, lo, hi) for lo, hi in slabs]
    work = torch.empty(p.buffer_work_bytes(max(hi - lo for lo, hi in slabs)), dtype=torch.uint8, device=dev)
    maps = torch.empty((len(slabs), WORDS), dtype=torch.int64, device=dev)
    for i, ((lo, hi), (w_lo, w_hi)) in enumerate(zip(slabs, windows)):
        win = d_text[w_lo:w_hi]
        p.statemap_window_dev(win, w_hi - w_lo, lo - w_lo, hi - w_lo, w_lo, maps[i], work)
    end, declined = (int(x) for x in p.statemap_combine(maps.cpu().numpy(), n))
    if declined:
        return (0, 0), True, 0
    if end <= 0:
        return (0, 0), False, 0
    owner = lambda b: next(i for i, (a, z) in enumerate(slabs) if a <= b < z)     # noqa: E731
    w = owner(end - 1) if end <= n else len(slabs) - 1
    walk = torch.tensor([0, 0, NEW, end], dtype=torch.int64, device=dev)
    hops = 0
    while True:
        w_lo, w_hi = windows[w]
        p.statemap_back_dev(d_text[w_lo:w_hi], w_hi - w_lo, w_lo, n, walk)
        pos, best, state, _ = walk.cpu().tolist()
        if state == DONE:
            return (pos, best), False, hops
        nxt = owner(pos - 1)
        assert nxt != w
        w, hops = nxt, hops + 1


def random_slabs(rng, n, k):
    cuts = sorted(rng.randint(0, n) for _ in range(k - 1))
    b = [0] + cuts + [n]
    return [(b[i], b[i + 1]) for i in range(k)]


def parity_cases():
    """the patterns and texts of test_gpu_parity.test_statemap_scan_against_the_oracle (same seeds)"""
    from tests.test_host_tables import gen_pattern, gen_text
    rng = random.Random(4242)
    nrng = np.random.default_rng(8)
    pieces = [b"a", b"z", b" ", "あ".encode(), "ん".encode(), "α".encode(), "　".encode(), b"\x80", b"\xc3", b"\xe3\x81", b"\xf0\x9f\x98",
              b"\xff", b"\xc0\x80", b"\n", b"\r\n", b"_", b"7", b"ERROR", b"timeout=", b"x" * 40, b"foo", b"bar"]
    texts = []
    for size in (700, 5000, 40000, 300000):
        t = b""
        while len(t) < size:
            t += pieces[int(nrng.integers(0, len(pieces)))]
        texts.append(t)
    texts += [b"\n".join(gen_text(rng) for _ in range(400)), bytes(synth.gen_c4(200000, 0.7)), bytes(synth.gen_c4(70000, None)),
              b"x" * 1500 + b"ab" + b"y" * 900, b"", b" ", b"a", b"\xe3\x81\x82" * 700]
    pats = [synth.PATTERNS["c4"], synth.PATTERNS["c3"], b"[a-z]+r", rb"\s\S+$", b"[xy]+a[ab]y", rb"[^a]{2,3}$", rb"^\w", b"(a|b)*a(a|b){3}",
            "[ぁ-ん]+a".encode(), rb"\d+-\d+", b"[ab].*c", b".+", b"^$", b"(|^)a"]
    pats += [gen_pattern(rng).encode() for _ in range(60)]
    return pats, texts


def served(p):
    inf = p.info()
    return p.status == 0 and inf["statemap"] and not inf["literal_only"] and not inf["literal_prefix_len"] and not inf["nfa_engine"]


def test_slabs_against_the_oracle(monkeypatch):
    """maps + combine + backward hops over 1, 2, 3, 5 and 8 slabs with unaligned cuts == the oracle == fx_regex_buffer
    with the state-map scan forced"""
    pats, texts = parity_cases()
    rng = random.Random(17)
    monkeypatch.setenv("FX_STATEMAP", "2")
    used, splits, hops_seen = 0, 0, 0
    for pat in pats:
        p = fx.Pattern(pat, "regex")
        if not served(p):
            continue
        c = O.Compiled(pat, 0)
        for text in texts:
            if len(text) > 6000 and pat not in pats[:2]:
                continue                       # (the oracle is quadratic in the worst case, see the parity test)
            arr = np.frombuffer(text, dtype=np.uint8)
            exp = c.regex_buffer(np.ascontiguousarray(arr))
            assert p.regex_buffer(arr) == exp, (pat, len(text))
            d = torch.from_numpy(np.frombuffer(b"#" + text, dtype=np.uint8).copy()).cuda()[1:]     # odd address
            for k in (1, 2, 3, 5, 8):
                slabs = random_slabs(rng, len(text), k)
                got, declined, hops = split_search(p, d, len(text), slabs)
                assert not declined, (pat, len(text), slabs)
                assert got == exp, (pat, len(text), slabs, got, exp)
                splits += 1
                hops_seen += hops
        used += 1
    assert used >= 25 and splits >= 1000 and hops_seen >= 10, (used, splits, hops_seen)


def test_c4_one_gib_in_eight_slabs(monkeypatch):
    """about 1 GiB of the C4 log in 8 slabs: the span known by construction (the planted line) and the single-buffer
    state-map scan's span"""
    import bench
    n = 1 << 30
    w = bench.build_workload(torch, "c4", n, 0, 1)
    p, buf = w["pattern_obj"], w["buf"]
    got, declined, _ = split_search(p, buf, n, [fxd.slab_bounds(n, 8, r, align=1) for r in range(8)])
    assert not declined and got == tuple(w["expect_span"]), (got, w["expect_span"])
    monkeypatch.setenv("FX_STATEMAP", "2")
    ft = torch.zeros(2, dtype=torch.int64, device="cuda")
    work = torch.zeros(p.buffer_work_bytes(n), dtype=torch.uint8, device="cuda")
    p.regex_buffer_dev(buf, n, ft, work)
    assert tuple(ft.cpu().tolist()) == got
    uneven = [(0, 1000), (1000, 1 << 28), (1 << 28, (1 << 29) + 7), ((1 << 29) + 7, n - 3), (n - 3, n)]
    assert split_search(p, buf, n, uneven)[:2] == (got, False)


def test_long_attempts_are_linear_time_across_slabs():
    """`[ab].*c` over 256 MiB of `a` in 4 slabs: no match, in milliseconds (the window scan runs the reference's
    quadratic loop here).  A `c` at the last byte of 4 MiB: (1, 4 MiB), the walk handed over three times"""
    p = fx.Pattern(b"[ab].*c", "regex")
    n = 256 << 20
    buf = torch.full((n,), ord("a"), dtype=torch.uint8, device="cuda")
    slabs = [fxd.slab_bounds(n, 4, r) for r in range(4)]
    split_search(p, buf, n, slabs)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    got = split_search(p, buf, n, slabs)
    dt = time.perf_counter() - t0
    assert got == ((0, 0), False, 0)
    assert dt < 0.25, "%.3f s for 256 MiB" % dt
    m = 4 << 20
    buf[m - 1] = ord("c")
    assert split_search(p, buf[:m], m, [fxd.slab_bounds(m, 4, r) for r in range(4)]) == ((1, m), False, 3)


def test_gpu_buffer_search_linear_one_rank():
    """world = 1: the route and the answer of fx_regex_buffer, for served patterns, patterns the form does not serve
    (prefix literal, literal only) and one it declines (more than 32 states behind a region cut).  An NFA-engine
    handle has no window form at all: FX_ERR_DFA_STATE_CAP (as a sequential candidate list gets
    FX_ERR_PREFILTER_UNSUPPORTED from the window scan)"""
    pats, texts = parity_cases()
    wide = b"xa" + b"b" * 40000
    cases = [(pat, texts[k]) for pat in pats[:14] for k in (0, 4, 7, 10)]
    cases += [(b"foo(bar|baz)", b"xx foobar foobaz"), (b"ERROR", b"x ERROR y"), (b"a.*[bc]", b"aaab"),
              (b"[ax](b{34})*c", wide), (b"[ax](b{34})*c", wide + b"c")]
    routes = set()
    for pat, text in cases:
        p = fx.Pattern(pat, "regex")
        arr = np.frombuffer(text, dtype=np.uint8)
        exp = p.regex_buffer(arr)
        d = torch.from_numpy(arr.copy()).cuda()
        stats = {}
        got = fxd.gpu_buffer_search_linear(p, d, 0, len(text), 0, 1, (0, len(text)), stats=stats)
        assert got == exp, (pat, len(text), got, exp)
        want = "statemap" if served(p) and text[:len(wide)] != wide else "scan"
        assert stats["route"] == want, (pat, stats)
        routes.add(stats["route"])
        if len(text) < 1000:
            assert got == O.Compiled(pat, 0).regex_buffer(arr), pat
    assert routes == {"statemap", "scan"}
    p = fx.Pattern(b".*a(a|b){500}c{20}", "regex")
    assert p.status == 0 and p.info()["nfa_engine"] == 1
    d = torch.zeros(8, dtype=torch.uint8, device="cuda")
    with pytest.raises(fx.ForgexError) as e:
        fxd.gpu_buffer_search_linear(p, d, 0, 8, 0, 1, (0, 8))
    assert e.value.status == _lib.FX_ERR_DFA_STATE_CAP
    p = fx.Pattern(b"a.*b", "regex")
    assert p.info()["prefix_scan"] == 0
    with pytest.raises(fx.ForgexError) as e:
        fxd.gpu_buffer_search_linear(p, d, 0, 8, 0, 1, (0, 8))
    assert e.value.status == _lib.FX_ERR_PREFILTER_UNSUPPORTED


def _nccl_worker(rank, world, port, ret):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    try:
        text = bytes(synth.gen_c4(4 << 20, 0.7))
        n = len(text)
        lo, hi = fxd.slab_bounds(n, world, rank)
        w_lo, w_hi = fxd.window_for_statemap_slab(n, lo, hi)
        d = torch.from_numpy(np.frombuffer(text, dtype=np.uint8)[w_lo:w_hi].copy()).cuda()
        p = fx.Pattern(synth.PATTERNS["c4"], "regex")
        stats = {}
        ret[rank] = fxd.gpu_buffer_search_linear(p, d, w_lo, n, rank, world, (lo, hi), stats=stats) + (stats["route"],)
    finally:
        dist.destroy_process_group()


def test_nccl_two_ranks():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs for an NCCL world of 2 (%d visible)" % torch.cuda.device_count())
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ret = mp.Manager().dict()
    mp.spawn(_nccl_worker, args=(2, port, ret), nprocs=2, join=True)
    text = bytes(synth.gen_c4(4 << 20, 0.7))
    exp = O.Compiled(synth.PATTERNS["c4"], 0).regex_buffer(np.frombuffer(text, dtype=np.uint8))
    assert exp[0] > 0
    assert ret[0] == ret[1] == exp + ("statemap",)
