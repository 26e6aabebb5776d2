"""fx_regex_all_batch(_dev): every match of every string of a ragged batch, as CSR rows + flat spans, against the oracle's
loop (`oracle_all`: regex(), then regex() again on text(to+1:), each call framed afresh).

The rows are the counts of k_regex_count scanned in place (k_scan_i64_sums / _carry / _apply, a fixed grid of at most
1024 blocks of 1024 values each); the spans come from k_regex_count's WRITE form, which walks each string again and
writes its k-th match at rows[i] + k below `capacity`.  The tests cover both k_regex_count forms (the span path and,
with FX_SPAN_LINEAR=0, the emulation), capacities around the total, the scan's tile and grid edges, device views at
every alignment on a side stream, NFA-engine handles, and one batch past 2^32 bytes whose match count passes 2^31.
The GPU tests free their device memory; the big one skips, naming the size, when the shared device has too little free.
"""
import functools
import random

import numpy as np
import pytest

import forgex_b200 as fx
from forgex_b200 import _lib as L
from tests import oracle_lib as O
from tests.test_gpu_all_matches import device, to_device  # noqa: F401  (device: the fixture)
from tests.test_gpu_parity import oracle_all, pack
from tools import synth

GiB = 1 << 30
B31, B32 = 1 << 31, 1 << 32
SCAN_TILE, SCAN_MAX_BLOCKS = 1024, 1024
SENTINEL = -7
C4 = synth.PATTERNS["c4"]


def dev_call(torch, p, d_buf, d_off, n, total, capacity, slack=8):
    """the _dev form with sentinels behind rows, spans and the work area: (rows, spans, launches).  Nothing past
    n + 1 rows, `capacity` spans or fx_regex_all_batch_work_bytes(n) bytes of scratch may be written."""
    d_rows = torch.full((n + 1 + slack,), SENTINEL, dtype=torch.int64, device="cuda")
    d_from = torch.full((capacity + slack,), SENTINEL, dtype=torch.int64, device="cuda")
    d_to = torch.full((capacity + slack,), SENTINEL, dtype=torch.int64, device="cuda")
    wb = p.all_batch_work_bytes(n)
    work = torch.full((wb + 64,), 0x5A, dtype=torch.uint8, device="cuda")
    before = fx.launch_count()
    p.regex_all_batch_dev(d_buf, d_off, n, total, d_rows, d_from, d_to, capacity, work[:wb])
    launches = fx.launch_count() - before
    torch.cuda.current_stream().synchronize()
    rows, f, t = d_rows.tolist(), d_from.tolist(), d_to.tolist()
    assert rows[n + 1:] == [SENTINEL] * slack, (p.pattern, n, "rows written past n + 1")
    assert f[capacity:] == [SENTINEL] * slack and t[capacity:] == [SENTINEL] * slack, (p.pattern, capacity, "past capacity")
    assert bool((work[wb:] == 0x5A).all()), (p.pattern, n, "scratch written past fx_regex_all_batch_work_bytes")
    return rows[:n + 1], list(zip(f[:capacity], t[:capacity])), launches


def expected_rows(exp):
    return [0] + np.cumsum([len(e) for e in exp], dtype=np.int64).tolist()


# ---- parity: the corpus of test_all_matches_and_counts plus fuzz patterns, one ragged batch per pattern -------------
@functools.lru_cache(maxsize=1)
def parity_corpus():
    """test_gpu_parity.py::test_all_matches_and_counts's 15 fixed and 25 generated patterns (same seed) and texts -- its
    long texts for the fixed patterns only, as there -- plus 30 more generated patterns and, in every batch, 60 generated
    texts, empty and lone-blank strings, line ends and UTF-8: (pattern, strings, the oracle's spans per string)"""
    from tests.test_host_tables import gen_pattern, gen_text
    rng = random.Random(99)
    log = bytes(synth.gen_c4(60000, 0.3)) + synth.C4_MATCH_LINE + b"\n" + bytes(synth.gen_c4_block(30000, 5)) + synth.C4_MATCH_LINE
    texts = [b"foobar foobaz fooba foobarfoobaz", b"abc\nabc\r\nabc", b"aaa", b"", b" ", b"x y  z", log,
             "あいう えお かきく".encode() * 50, b"\n".join(gen_text(rng) for _ in range(300)), b"a" * 5000, b"ab" * 3000 + b"\n" + b"ba" * 200]
    fixed = [b"foo(bar|baz)", b"^abc", b"abc$", b"a", b"[a-z]+", rb"\s", C4, "[ぁ-ん]+".encode(), b"a{1,7}", b"(ab)+", b"^", b".",
             b"[ab]{2,3}", b"ERROR", rb"\w+\s"]
    pats = fixed + [gen_pattern(rng).encode() for _ in range(25)]
    frng = random.Random(4242)
    pats += [gen_pattern(frng).encode() for _ in range(30)]
    extra = [gen_text(frng) for _ in range(60)] + [b"", b" ", b"\n", b"\r\n", b"  ", "あ".encode(), "α ω".encode(), b""]
    cases = []
    for pat in pats:
        p = fx.Pattern(pat, "regex")
        if p.status != 0:
            continue
        assert p.info()["nfa_engine"] == 0, pat
        c = O.Compiled(pat, 0)
        strings = [t for t in texts if len(t) <= 20000 or pat in fixed] + extra
        random.Random(len(cases)).shuffle(strings)
        cases.append((pat, strings, [oracle_all(c, s) for s in strings]))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("linear", ["1", "0"], ids=["default", "FX_SPAN_LINEAR=0"])
def test_parity_with_the_oracle_loop(device, monkeypatch, linear):
    """string i's spans[rows[i]:rows[i + 1]] == oracle_all(string i) == fx_regex_buffer_all(string i), and diff(rows) ==
    fx_regex_count_batch, for the host form and the _dev form"""
    torch = device
    monkeypatch.setenv("FX_SPAN_LINEAR", linear)
    cases = parity_corpus()
    assert len(cases) >= 60, len(cases)
    seen = set()
    for pat, strings, exp in cases:
        p = fx.Pattern(pat, "regex")
        inf = p.info()
        seen.update(k for k, on in (("literal only", inf["literal_only"]), ("prefix literal", inf["literal_prefix_len"] > 0),
                                    ("span path", inf["statemap"]), ("anchor", b"^" in pat or b"$" in pat)) if on)
        buf, off = pack(strings)
        want_rows = expected_rows(exp)
        flat = [s for e in exp for s in e]
        rows, f, t = p.regex_all_batch(buf, off, capacity=len(flat) + 1)
        assert rows.tolist() == want_rows, (pat, rows.tolist()[-1], want_rows[-1])
        spans = list(zip(f.tolist(), t.tolist()))
        for i, e in enumerate(exp):
            assert spans[rows[i]:rows[i + 1]] == e, (pat, i, strings[i][:20], spans[rows[i]:rows[i + 1]][:4], e[:4])
        assert np.diff(rows).tolist() == p.regex_count_batch(buf, off).tolist(), pat
        if linear == "1":
            for s, e in zip(strings, exp):
                bf, bt, cnt = p.regex_buffer_all(np.frombuffer(s, dtype=np.uint8), capacity=len(e) + 1)
                assert (list(zip(bf.tolist(), bt.tolist())), cnt) == (e, len(e)), (pat, s[:20])
        d_rows, d_spans, _ = dev_call(torch, p, to_device(torch, bytes(buf)), torch.from_numpy(off).cuda(), len(strings),
                                      int(off[-1]), len(flat))
        assert (d_rows, d_spans) == (want_rows, flat), pat
    assert seen == {"literal only", "prefix literal", "span path", "anchor"}, seen


# ---- capacity --------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_capacities_around_the_total(device):
    """capacity 0, 1, total - 1, total, total + 1 (and total_bytes, always enough): rows complete, the spans' prefix
    right, nothing written at or past capacity; capacity 0 launches no span pass"""
    torch = device
    strings = [b"a b c", b"", b" ", b"xyz", b"abc abc\nab", "あ a".encode(), b"c" * 40 + b" a", b"b", b"ab ab ab"]
    buf, off = pack(strings)
    n, nbytes = len(strings), int(off[-1])
    d_buf, d_off = to_device(torch, bytes(buf)), torch.from_numpy(off).cuda()
    for pat in (b"[a-c]+", b"ab", b"a(b|c)", rb"^\w"):
        p = fx.Pattern(pat, "regex")
        c = O.Compiled(pat, 0)
        exp = [oracle_all(c, s) for s in strings]
        want_rows, flat = expected_rows(exp), [s for e in exp for s in e]
        total = len(flat)
        assert total >= 3, pat
        launches = {}
        for cap in (0, 1, total - 1, total, total + 1, nbytes):
            rows, f, t = p.regex_all_batch(buf, off, capacity=cap)
            assert rows.tolist() == want_rows and list(zip(f.tolist(), t.tolist())) == flat[:cap], (pat, cap)
            d_rows, d_spans, launches[cap] = dev_call(torch, p, d_buf, d_off, n, nbytes, cap)
            k = min(cap, total)
            assert d_rows == want_rows and d_spans[:k] == flat[:k], (pat, cap)
            assert d_spans[k:] == [(SENTINEL, SENTINEL)] * (cap - k), (pat, cap)
        assert launches[0] == launches[1] - 1 and len(set(launches.values()) - {launches[0]}) == 1, launches


# ---- the scan's edges --------------------------------------------------------------------------------------------------
def dense_batch(counts):
    """string i = `a ` repeated counts[i] times: `[a-c]+` matches every `a`, at (2j + 1, 2j + 1) of its string"""
    counts = np.asarray(counts, dtype=np.int64)
    off = np.zeros(len(counts) + 1, dtype=np.int64)
    np.cumsum(2 * counts, out=off[1:])
    buf = np.frombuffer(b"a " * int(counts.sum()), dtype=np.uint8)
    rows = np.zeros(len(counts) + 1, dtype=np.int64)
    np.cumsum(counts, out=rows[1:])
    spans_from = 2 * (np.arange(rows[-1], dtype=np.int64) - np.repeat(rows[:-1], counts)) + 1
    return buf, off, rows, spans_from


SCAN_SIZES = [0, 1, 2, 31, SCAN_TILE - 1, SCAN_TILE, SCAN_TILE + 1, 3 * SCAN_TILE + 5, SCAN_TILE * SCAN_MAX_BLOCKS - 1,
              SCAN_TILE * SCAN_MAX_BLOCKS, SCAN_TILE * SCAN_MAX_BLOCKS + 1, 2 * SCAN_TILE * SCAN_MAX_BLOCKS + 3,
              3 * SCAN_TILE * SCAN_MAX_BLOCKS + 777]


@pytest.mark.gpu
def test_scan_edges(device):
    """n = 0, 1 and both sides of a scan tile (1024 values) and of the grid (1024 blocks; past it each block scans
    several tiles): rows and every span by construction.  Then all counts zero, and one string holding every match
    (first, middle, last)."""
    torch = device
    p = fx.Pattern(b"[a-c]+", "regex")
    rng = np.random.default_rng(7)
    for n in SCAN_SIZES:
        buf, off, rows, spans_from = dense_batch(rng.integers(0, 4, size=n))
        d_buf, d_off = to_device(torch, bytes(buf)), torch.from_numpy(off).cuda()
        d_rows = torch.full((n + 1,), SENTINEL, dtype=torch.int64, device="cuda")
        d_from = torch.zeros(int(rows[-1]) + 1, dtype=torch.int64, device="cuda")
        d_to = torch.zeros(int(rows[-1]) + 1, dtype=torch.int64, device="cuda")
        work = torch.zeros(p.all_batch_work_bytes(n), dtype=torch.uint8, device="cuda")
        p.regex_all_batch_dev(d_buf, d_off, n, len(buf), d_rows, d_from, d_to, int(rows[-1]), work)
        assert np.array_equal(d_rows.cpu().numpy(), rows), n
        assert np.array_equal(d_from[:-1].cpu().numpy(), spans_from) and torch.equal(d_from, d_to), n
        if n <= SCAN_TILE + 1:
            got_rows, f, t = p.regex_all_batch(buf, off, capacity=int(rows[-1]))
            assert np.array_equal(got_rows, rows) and np.array_equal(f, spans_from) and np.array_equal(t, spans_from), n
    # all counts zero
    for n in (1, SCAN_TILE + 1, SCAN_TILE * SCAN_MAX_BLOCKS + 1):
        strings = [b"x" * (i % 3) for i in range(n)]
        buf, off = pack(strings)
        rows, spans, _ = dev_call(torch, p, to_device(torch, bytes(buf)), torch.from_numpy(off).cuda(), n, len(buf), 4)
        assert rows == [0] * (n + 1) and spans == [(SENTINEL, SENTINEL)] * 4, n
    # one string holds every match
    n, m = SCAN_TILE * SCAN_MAX_BLOCKS + 1, 100000
    for j in (0, n // 2, n - 1):
        counts = np.zeros(n, dtype=np.int64)
        counts[j] = m
        buf, off, rows, spans_from = dense_batch(counts)
        d_rows = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
        d_from = torch.zeros(m, dtype=torch.int64, device="cuda")
        d_to = torch.zeros(m, dtype=torch.int64, device="cuda")
        work = torch.zeros(p.all_batch_work_bytes(n), dtype=torch.uint8, device="cuda")
        p.regex_all_batch_dev(to_device(torch, bytes(buf)), torch.from_numpy(off).cuda(), n, len(buf), d_rows, d_from, d_to, m, work)
        assert np.array_equal(d_rows.cpu().numpy(), rows), j
        assert np.array_equal(d_from.cpu().numpy(), spans_from) and torch.equal(d_from, d_to), j


# ---- device views, a side stream, NFA-engine handles ------------------------------------------------------------------
@pytest.mark.gpu
def test_dev_form_on_unaligned_views_and_a_side_stream(device):
    """the _dev form over text views at byte offsets 1..15 into a tensor, on a non-default torch stream: the host
    form's answer"""
    torch = device
    far = b"x" * 70000
    strings = [b"a b c" + far + b"abc", b"", b" ", bytes(synth.gen_c4(50000, 0.8, crlf=True)) + synth.C4_MATCH_LINE,
               "あいう えお".encode() * 20 + b" 12 abc", b"foobar foobaz x foobar", b"abc\nabc\r\nabc", b"\n"]
    buf, off = pack(strings)
    side = torch.cuda.Stream()
    for pat in (b"[a-c]+", rb"\d+", C4, "[ぁ-ん]+".encode(), b"foo(bar|baz)", b"abc"):
        p = fx.Pattern(pat, "regex")
        rows, f, t = p.regex_all_batch(buf, off)
        want = (rows.tolist(), list(zip(f.tolist(), t.tolist())))
        assert want[0][-1] > 0, pat
        with torch.cuda.stream(side):
            d_off = torch.from_numpy(off).cuda()
            for shift in range(1, 16):
                got = dev_call(torch, p, to_device(torch, bytes(buf), shift), d_off, len(strings), int(off[-1]), want[0][-1])
                assert got[:2] == want, (pat, shift)
        side.synchronize()


@pytest.mark.gpu
def test_nfa_engine_handles_are_refused(device, monkeypatch):
    """the batch form needs the table engine: an NFA-engine handle gets FX_ERR_DFA_STATE_CAP from both forms (the pattern
    whose eager automaton passes the cap, and any pattern under FX_STATE_CAP=3)"""
    torch = device
    buf, off = pack([b"ab aab c", b"", b"x"])
    d, d_off = to_device(torch, bytes(buf)), torch.from_numpy(off).cuda()
    handles = [fx.Pattern(b".*a(a|b){500}c{20}", "regex")]
    monkeypatch.setenv("FX_STATE_CAP", "3")
    handles.append(fx.Pattern(b"[a-c]+", "regex"))
    monkeypatch.delenv("FX_STATE_CAP")
    z = torch.zeros(8, dtype=torch.int64, device="cuda")
    work = torch.zeros(fx.Pattern.all_batch_work_bytes(3), dtype=torch.uint8, device="cuda")
    for p in handles:
        assert p.status == 0 and p.info()["nfa_engine"] == 1, p.pattern
        for call in (lambda: p.regex_all_batch(buf, off, capacity=4),
                     lambda: p.regex_all_batch_dev(d, d_off, 3, len(buf), z, z[4:], z[6:], 2, work)):
            with pytest.raises(fx.ForgexError) as e:
                call()
            assert e.value.status == L.FX_ERR_DFA_STATE_CAP, p.pattern


# ---- past 2^32 bytes and 2^31 matches ----------------------------------------------------------------------------------
BIG_TAILS = [b"", b"", b"", b"a", b" ", b"x", "あ".encode()]


def big_block(nstrings=4099, seed=3):
    """a seeded block of strings `a ` * k + tail (k < 2200, tails that add no span or one more `a`): `[a-c]+` matches
    every `a`, so every span has from == to, odd, and a string's count is about half its bytes.  (buf, offsets, counts)"""
    rng = np.random.default_rng(seed)
    ks, tails = rng.integers(0, 2200, size=nstrings), rng.integers(0, len(BIG_TAILS), size=nstrings)
    buf, off = pack([b"a " * int(k) + BIG_TAILS[int(t)] for k, t in zip(ks, tails)])
    return buf, off, ks + (np.array(BIG_TAILS, dtype=object)[tails] == b"a")


def test_big_block_against_the_oracle():
    """(CPU) the block's counts by construction are the oracle's, and tiled past 2^32 + 2^28 bytes it passes 2^31 matches"""
    hb, ho, counts = big_block()
    c = O.Compiled(b"[a-c]+", 0)
    for i in range(0, len(counts), 97):
        s = bytes(hb[ho[i]:ho[i + 1]])
        assert oracle_all(c, s) == [(2 * j + 1, 2 * j + 1) for j in range(int(counts[i]))], i
    reps = -(-(B32 + (1 << 28)) // int(ho[-1]))
    assert reps * int(ho[-1]) > B32 + (1 << 28) and reps * int(counts.sum()) > B31 + (1 << 26)


@pytest.mark.gpu
def test_past_4_gib_and_2_pow_31_matches(device):
    """a batch of 2^32 + 2^28 bytes with more than 2^31 matches, so that rows and span indices need 64 bits: rows ==
    the inclusive cumsum of fx_regex_count_batch_dev; every span odd with from == to; the strings around match index
    2^31 and around byte 2^32 against the oracle"""
    torch = device
    hb, ho, block_counts = big_block()
    reps = -(-(B32 + (1 << 28)) // int(ho[-1]))
    lens = np.diff(ho)
    n, nbytes, matches = reps * len(lens), reps * int(ho[-1]), reps * int(block_counts.sum())
    need = nbytes + 16 * matches + 32 * n + GiB
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip("needs %.1f GiB of free device memory, %.1f GiB free" % (need / GiB, free / GiB))
    p = fx.Pattern(b"[a-c]+", "regex")
    buf = torch.from_numpy(hb).cuda().repeat(reps)
    off = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    torch.cumsum(torch.from_numpy(lens).cuda().repeat(reps), 0, out=off[1:])
    counts = torch.empty(n, dtype=torch.int64, device="cuda")
    p.regex_count_batch_dev(buf, off, n, nbytes, counts)
    total = int(counts.sum())
    assert total == matches, (total, matches)
    rows = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    d_from = torch.empty(total, dtype=torch.int64, device="cuda")
    d_to = torch.empty(total, dtype=torch.int64, device="cuda")
    work = torch.empty(p.all_batch_work_bytes(n), dtype=torch.uint8, device="cuda")
    p.regex_all_batch_dev(buf, off, n, nbytes, rows, d_from, d_to, total, work)
    torch.cuda.synchronize()
    assert int(rows[0]) == 0 and torch.equal(rows[1:], torch.cumsum(counts, 0)), "rows != cumsum(counts)"
    del counts
    step = 1 << 28
    for a in range(0, total, step):
        f, t = d_from[a:a + step], d_to[a:a + step]
        assert torch.equal(f, t) and bool((f % 2 == 1).all()), a
    rows_h, off_h = rows.cpu().numpy(), off.cpu().numpy()
    c = O.Compiled(b"[a-c]+", 0)
    at_match = int(np.searchsorted(rows_h, B31, side="right")) - 1
    at_byte = int(np.searchsorted(off_h, B32, side="right")) - 1
    assert rows_h[at_match] <= B31 < rows_h[at_match + 1] and off_h[at_byte] <= B32 < off_h[at_byte + 1]
    for i in sorted(set(range(at_match - 2, at_match + 3)) | set(range(at_byte - 2, at_byte + 3))):
        s = bytes(buf[off_h[i]:off_h[i + 1]].cpu().numpy())
        r0, r1 = int(rows_h[i]), int(rows_h[i + 1])
        got = list(zip(d_from[r0:r1].tolist(), d_to[r0:r1].tolist()))
        assert got == oracle_all(c, s), (i, r0, r1)
    del buf, off, rows, d_from, d_to, work
