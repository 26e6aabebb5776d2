"""The all-matches entry points -- fx_regex_buffer_all(_dev) and fx_regex_count_batch(_dev) -- against the oracle's loop.

fx_regex_buffer_all is a host-driven loop over two steps.  The local step (k_buffer_all_local, one thread) walks the
forward span automaton at most FX_ALL_REACH bytes (65536) from the start of the rest and takes up to 1024 matches per
launch.  When the automaton is still alive after that, the far step runs the whole long-buffer search (K4 / K5 / K4L /
sequential) on the rest and k_buffer_all_take records its match.  These tests put matches on every hand-off between the
two: just past the reach, across it, on the 1024-per-launch boundary, after a far match whose loop then ends in the
local step, under the work budget, and past bytes 2^31 and 2^32 of one buffer.  Each case asserts which route its
pattern takes.  A pattern with the local step (the state-map scan, no prefix literal, not a literal) has a linear-time
stand-in for every search, so no call on it may answer FX_ERR_WORK_BUDGET.

The GPU tests free their device memory; the one over 2^32 bytes skips, naming the size, when the shared device has too
little free.  The CPU test checks that the layout of that buffer is what the oracle's loop finds.
"""
import ctypes as C
import functools
import gc
import random

import numpy as np
import pytest

import forgex_b200 as fx
from forgex_b200 import _lib as L
from tests import oracle_lib as O
from tests.test_gpu_parity import oracle_all, pack
from tools import synth

GiB = 1 << 30
B31, B32 = 1 << 31, 1 << 32
REACH = 1 << 16                      # FX_ALL_REACH's default: bytes the local step walks before it hands off
PER_LAUNCH = 1024                    # matches the local step takes per launch
C4 = synth.PATTERNS["c4"]
LINE = synth.C4_MATCH_LINE
SENTINEL = -7


def routes_locally(p):
    """the loop looks for this pattern's next match with the local step first"""
    inf = p.info()
    return inf["statemap"] == 1 and inf["literal_prefix_len"] == 0 and inf["literal_only"] == 0


def local_pattern(pat):
    p = fx.Pattern(pat, "regex")
    assert p.status == 0 and routes_locally(p), pat
    return p


def all_spans(p, text, capacity=1 << 20):
    """the host form: (spans, count).  FX_ERR_WORK_BUDGET from a pattern with the local step fails the test."""
    try:
        f, t, cnt = p.regex_buffer_all(np.frombuffer(text, dtype=np.uint8), capacity=capacity)
    except fx.ForgexError as e:
        assert not (e.status == L.FX_ERR_WORK_BUDGET and routes_locally(p)), \
            "%r over %d bytes: work budget from a pattern with a linear-time stand-in" % (p.pattern, len(text))
        raise
    return list(zip(f.tolist(), t.tolist())), cnt


def all_dev(torch, p, d_buf, length, capacity, slack=8):
    """the _dev form through the C ABI, so that the count also comes back with an error status: (status, count, spans).
    d_from / d_to hold capacity + slack sentinels; nothing past capacity may be written."""
    d_from = torch.full((capacity + slack,), SENTINEL, dtype=torch.int64, device="cuda")
    d_to = torch.full((capacity + slack,), SENTINEL, dtype=torch.int64, device="cuda")
    work = torch.zeros(p.buffer_work_bytes(length), dtype=torch.uint8, device="cuda")
    cnt = C.c_int64(SENTINEL)
    stream = torch.cuda.current_stream()
    rc = L.lib().fx_regex_buffer_all_dev(p.h, d_buf.data_ptr(), length, d_from.data_ptr(), d_to.data_ptr(), capacity,
                                         C.byref(cnt), work.data_ptr(), stream.cuda_stream)
    stream.synchronize()
    f, t = d_from.cpu().tolist(), d_to.cpu().tolist()
    assert f[capacity:] == [SENTINEL] * slack and t[capacity:] == [SENTINEL] * slack, (p.pattern, capacity, "written past capacity")
    assert not (rc == L.FX_ERR_WORK_BUDGET and routes_locally(p)), (p.pattern, length, "work budget")
    return rc, cnt.value, list(zip(f[:capacity], t[:capacity]))


def to_device(torch, text, offset=0):
    """text on the device at `offset` bytes into a fresh tensor (a view, unaligned for offset % 16 != 0)"""
    d = torch.zeros(len(text) + offset + 16, dtype=torch.uint8, device="cuda")
    if text:
        d[offset:offset + len(text)] = torch.frombuffer(bytearray(text), dtype=torch.uint8).cuda()
    return d[offset:]


@pytest.fixture
def device():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    yield torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


# ---- (a) a far match, then a loop that ends in the local step ---------------------------------------------------
# (pattern, one match, filler of n bytes that holds no match and keeps the automaton alive, three near matches)
FAR_CASES = [
    (b"[a-c]+", b"abc", lambda n: b"x" * n, b" a bb c"),
    (rb"\d+", b"123", lambda n: b"x" * n, b" 1 22 3"),
    (C4, LINE, lambda n: b"x" * (n - 1) + b"\n", LINE + b"\n" + LINE + b"\nERROR y timeout=5"),
    ("[ぁ-ん]+".encode(), "あいう".encode(), lambda n: b"x" * n, " あ いい う".encode()),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(FAR_CASES)), ids=[c[0].decode() for c in FAR_CASES])
def test_far_match_then_a_loop_that_ends_locally(device, case):
    """A far step finds the match, the local step then ends the loop: on an empty or blank rest, on a short rest
    without a match, or after near matches.  The far step's from_to once shared a word with the loop's work-budget
    flag, so these loops answered FX_ERR_WORK_BUDGET instead of their matches."""
    pat, match, filler, near = FAR_CASES[case]
    p = local_pattern(pat)
    c = O.Compiled(pat, 0)
    sep = b"\n" if pat == C4 else b""         # (C4's `$`: the tail begins a line of its own)
    tails = [b"", b" ", b"\n", b"xyzxyz-_.!", b"x" * 70000, near, b"x" * 70000 + sep + match]
    for gap in (REACH - 1, REACH, REACH + 1, 200000):
        for tail in tails:
            text = filler(gap) + match + (sep + tail if tail else b"")
            exp = oracle_all(c, text)
            assert exp and exp[0][0] == gap + 1 - len(sep), (pat, gap, tail[:12], exp[:2])   # (C4's span holds the LF before it)
            got, cnt = all_spans(p, text)
            assert (got, cnt) == (exp, len(exp)), (pat, gap, tail[:12], cnt, got[:4], exp[:4])


# ---- (b) a match across the reach --------------------------------------------------------------------------------
@pytest.mark.gpu
def test_a_match_across_the_reach(device):
    """A match that begins before byte `reach` of the rest and whose longest end lies after it: the local step gives
    up, the far step must find the same leftmost-longest span.  Runs of `a`, C4's line with its CR LF split across the
    boundary, and `^` at restarts (every rest is framed behind a fresh leading NUL)."""
    p, c = local_pattern(b"[a-c]+"), O.Compiled(b"[a-c]+", 0)
    for lead in (b"", b"abc"):                # the rest begins at byte 0, or behind a local match
        for lo, hi in ((REACH - 1, REACH + 1), (REACH - 5, REACH + 300), (REACH - 2000, REACH), (REACH, REACH + 3), (REACH - 3, REACH)):
            text = lead + b"x" * lo + b"a" * (hi - lo) + b" bc x"
            exp = oracle_all(c, text)
            run = (len(lead) + lo + 1, len(lead) + hi)
            assert run in exp, (lead, lo, hi, exp)
            assert all_spans(p, text) == (exp, len(exp)), (lead, lo, hi)
    # C4's line: its end on both sides of the reach, LF or CR LF, followed by log lines and a second line
    p, c = local_pattern(C4), O.Compiled(C4, 0)
    log = bytes(synth.gen_c4_block(3000, 3))
    for end in (REACH - 2, REACH - 1, REACH, REACH + 1, REACH + 40):
        for term in (b"\n", b"\r\n"):
            start = end - len(LINE)
            text = b"x" * (start - 1) + b"\n" + LINE + term + log + b"\n" + LINE + term + b"INFO x"
            exp = oracle_all(c, text)
            assert len(exp) == 2 and exp[0][0] == start, (end, term, exp)
            assert all_spans(p, text) == (exp, 2), (end, term)
    # `^` at the restart: only the fresh leading NUL of each rest lets `b` and `c` match
    for pat in (b"^[a-c]", rb"^\d", b"[a-c]+$"):
        p, c = local_pattern(pat), O.Compiled(pat, 0)
        for gap in (REACH - 2, REACH - 1, REACH, REACH + 1):
            for body in (b"\nabc", b"\n123", b"\nab\r\nc", b"\nabc\n"):
                text = b"x" * gap + body + b" xa"
                exp = oracle_all(c, text)
                assert all_spans(p, text) == (exp, len(exp)), (pat, gap, body)
    assert oracle_all(O.Compiled(b"^[a-c]", 0), b"x" * REACH + b"\nabc x") == [(REACH + 1, REACH + 2), (REACH + 3, REACH + 3), (REACH + 4, REACH + 4)]


# ---- (c) every match a hand-off -------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=1)
def handoff_corpus():
    """the patterns of test_gpu_parity.py::test_all_matches_and_counts (its 15 fixed and 25 generated ones, the same
    seed) that have the local step, over its texts cut to 500 bytes (the full log for C4) -- with the oracle's answers"""
    from tests.test_host_tables import gen_pattern, gen_text
    rng = random.Random(99)
    log = bytes(synth.gen_c4(60000, 0.3)) + LINE + b"\n" + bytes(synth.gen_c4_block(30000, 5)) + LINE
    texts = [b"foobar foobaz fooba foobarfoobaz", b"abc\nabc\r\nabc", b"aaa", b"", b" ", b"x y  z", log,
             "あいう えお かきく".encode() * 50, b"\n".join(gen_text(rng) for _ in range(300)), b"a" * 5000, b"ab" * 3000 + b"\n" + b"ba" * 200]
    pats = [b"foo(bar|baz)", b"^abc", b"abc$", b"a", b"[a-z]+", rb"\s", C4, "[ぁ-ん]+".encode(), b"a{1,7}", b"(ab)+", b"^", b".",
            b"[ab]{2,3}", b"ERROR", rb"\w+\s"]
    pats += [gen_pattern(rng).encode() for _ in range(25)]
    short = [t[:500] for t in texts]
    cases = []
    for pat in pats:
        p = fx.Pattern(pat, "regex")
        if p.status != 0 or not routes_locally(p):
            continue
        c = O.Compiled(pat, 0)
        ts = short + ([log] if pat == C4 else [])
        cases.append((pat, [(t, oracle_all(c, t)) for t in ts]))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize("local,reach", [(1, r) for r in (0, 1, 2, 3, 7, 64, 4097)] + [(0, REACH)])
def test_every_match_position_is_a_handoff(device, monkeypatch, local, reach):
    """FX_ALL_REACH from 0 (every search is a far step) to 4097, and FX_ALL_LOCAL=0 (no local step; the reach is then
    not read): with a small reach every match position is a hand-off somewhere.  Same spans as the oracle's loop."""
    monkeypatch.setenv("FX_ALL_LOCAL", str(local))
    monkeypatch.setenv("FX_ALL_REACH", str(reach))
    cases = handoff_corpus()
    assert len(cases) >= 18, len(cases)
    for pat, texts in cases:
        p = fx.Pattern(pat, "regex")
        for text, exp in texts:
            got, cnt = all_spans(p, text, capacity=len(exp) + 3)
            assert (got, cnt) == (exp, len(exp)), (pat, text[:20], len(text), cnt, len(exp), got[:3], exp[:3])


# ---- (d) the 1024-per-launch boundary, then a far step --------------------------------------------------------------
@pytest.mark.gpu
def test_full_launches_before_a_far_step(device):
    """N near matches (N = 1023 ... 2049 around multiples of the 1024 a launch takes), a gap longer than the reach,
    one far match.  Capacities 0, 1, k - 1, k, k + 1 of the k matches: the first `capacity` spans are returned, the
    count is k, and the _dev form writes nothing past capacity."""
    torch = device
    p, c = local_pattern(b"[a-c]+"), O.Compiled(b"[a-c]+", 0)
    gap = REACH + 100
    for n in (PER_LAUNCH - 1, PER_LAUNCH, PER_LAUNCH + 1, 2 * PER_LAUNCH, 2 * PER_LAUNCH + 1):
        text = b"a " * n + b"x" * gap + b"bc"
        exp = [(2 * i + 1, 2 * i + 1) for i in range(n)] + [(2 * n + gap + 1, 2 * n + gap + 2)]
        assert oracle_all(c, text) == exp
        k = len(exp)
        d = to_device(torch, text)
        for cap in (0, 1, k - 1, k, k + 1):
            assert all_spans(p, text, capacity=cap) == (exp[:cap], k), (n, cap)
            rc, cnt, got = all_dev(torch, p, d, len(text), cap)
            assert (rc, cnt) == (0, k) and got[:min(cap, k)] == exp[:cap], (n, cap, rc, cnt)
            assert got[k:] == [(SENTINEL, SENTINEL)] * (cap - min(cap, k)), (n, cap)


# ---- (e) the work budget in the middle of the loop ----------------------------------------------------------------
@pytest.mark.gpu
def test_work_budget_in_the_middle_of_the_loop(device):
    """`aa.*[xy]` has a bordered prefix literal: no local step and no linear-time stand-in.  Two lines with one match
    each, then 1 MiB of `a`: the third search spends its work budget.  The _dev form answers FX_ERR_WORK_BUDGET with the
    count and the spans found before it; the host form raises."""
    torch = device
    pat = b"aa.*[xy]"
    p = fx.Pattern(pat, "regex")
    inf = p.info()
    assert inf["literal_prefix_len"] == 2 and inf["prefix_scan"] == 0 and not routes_locally(p)
    head = b"aax\naay\n"
    before = oracle_all(O.Compiled(pat, 0), head)
    assert before == [(1, 3), (5, 7)]
    text = head + b"a" * (1 << 20)
    with pytest.raises(fx.ForgexError) as e:
        p.regex_buffer_all(np.frombuffer(text, dtype=np.uint8), capacity=8)
    assert e.value.status == L.FX_ERR_WORK_BUDGET
    d = to_device(torch, text)
    for cap in (0, 1, 2, 8):
        rc, cnt, got = all_dev(torch, p, d, len(text), cap)
        assert (rc, cnt) == (L.FX_ERR_WORK_BUDGET, 2) and got[:2] == before[:cap], (cap, rc, cnt, got)
    # the same handle and work area right afterwards: a loop within the budget
    assert all_dev(torch, p, d, len(head), 4)[:2] == (0, 2)


# ---- (f) one buffer past 2^31 and 2^32 bytes --------------------------------------------------------------------------
BIG_PATTERN = b"[a-c]+"
BIG_FILL = ord("x")


def big_layout(scale=1.0):
    """the planted matches of a buffer of 2^32 + 2^28 bytes of `x` for `[a-c]+`, its gaps multiplied by `scale`:
    (length, [(offset, bytes)], expected spans).  A far match across byte 2^31; 3000 near matches `a ` across 2^32, so
    that the local step runs past 2^32 and ends a full launch there; a far match 1000 bytes before the end; a tail of
    997 bytes without a match, which ends the loop in the local step."""
    length = int((B32 + (1 << 28)) * scale)
    b31, b32 = int(B31 * scale), int(B32 * scale)
    plants, spans = [], []
    o = b31 - 50
    plants.append((o, b"a" * 100))
    spans.append((o + 1, o + 100))
    o = b32 - 3000
    plants.append((o, b"a " * 3000))
    spans += [(o + 2 * i + 1, o + 2 * i + 1) for i in range(3000)]
    o = length - 1000
    plants.append((o, b"cab"))
    spans.append((o + 1, o + 3))
    return length, plants, spans


def test_big_layout_against_the_oracle():
    """(CPU) the layout of the big buffer, gaps shrunk: the oracle's loop finds exactly the constructed spans; at full
    scale the first match straddles 2^31, the near matches straddle 2^32 and reach past it by more than a launch"""
    length, plants, spans = big_layout(2.0 ** -14)
    text = bytearray([BIG_FILL]) * length
    for o, b in plants:
        text[o:o + len(b)] = b
    assert oracle_all(O.Compiled(BIG_PATTERN, 0), bytes(text)) == spans
    length, plants, spans = big_layout()
    assert length == B32 + (1 << 28) and len(spans) == 3002
    assert spans[0][0] <= B31 < spans[0][1]
    near = [f for f, _ in spans[1:-1]]
    assert near[0] <= B32 < near[-1] and sum(f > B32 for f in near) > PER_LAUNCH
    assert spans[-1][1] < length and length - spans[-1][1] < REACH
    assert all(a[1] < b[0] for a, b in zip(spans, spans[1:]))


@pytest.mark.gpu
def test_all_matches_past_4_gib(device):
    """the _dev form over one device buffer of 2^32 + 2^28 bytes: every constructed span, in 64-bit positions"""
    torch = device
    length, plants, spans = big_layout()
    need = length + GiB
    free, _ = torch.cuda.mem_get_info()
    if free < need:
        pytest.skip("needs %.1f GiB of free device memory, %.1f GiB free" % (need / GiB, free / GiB))
    p = local_pattern(BIG_PATTERN)
    buf = torch.full((length,), BIG_FILL, dtype=torch.uint8, device="cuda")
    for o, b in plants:
        buf[o:o + len(b)] = torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda()
    rc, cnt, got = all_dev(torch, p, buf, length, len(spans) + 1)
    assert (rc, cnt) == (0, len(spans))
    assert got[:-1] == spans and got[-1] == (SENTINEL, SENTINEL)
    del buf


# ---- (g) counts ----------------------------------------------------------------------------------------------------
def count_strings():
    far = b"-" * (REACH + 5000)
    return [bytes(synth.gen_c4(70000, 0.5)) + b"\n" + (LINE + b"\n") * 150 + "あいう えお".encode() * 150 + b" 12 abc", b"", b" ",
            far + b"abc 123 foobar ERROR x timeout=7 " + "かき".encode(),
            far + b"\n" + LINE, b"abc\nabc\r\nabc", "あいう".encode(), b"\n", b"a" * 3000 + b" b" * 40]


COUNT_SPAN = [b"[a-c]+", rb"\d+", C4, "[ぁ-ん]+".encode(), b"[a-z]+", rb"\s+", rb"^\w"]
COUNT_PREFIXED = [b"foo(bar|baz)", rb"ERROR.*timeout=\d+", b"ab*c?", b"timeout"]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["span", "span, FX_SPAN_LINEAR=0", "prefix literal"])
def test_counts_against_the_oracle_loop(device, monkeypatch, kind):
    """fx_regex_count_batch and its _dev form on a ragged batch: counts == the oracle's loop per string ==
    fx_regex_buffer_all's count.  Span patterns run k_regex_count<true>, or <false> with FX_SPAN_LINEAR=0; patterns
    with a prefix literal (or literals) always run <false>."""
    torch = device
    strings = count_strings()
    buf, off = pack(strings)
    if kind == "span, FX_SPAN_LINEAR=0":
        monkeypatch.setenv("FX_SPAN_LINEAR", "0")
    for pat in (COUNT_PREFIXED if kind == "prefix literal" else COUNT_SPAN):
        p = fx.Pattern(pat, "regex")
        assert p.status == 0
        if kind == "prefix literal":
            assert p.info()["literal_prefix_len"] > 0 and not routes_locally(p), pat
        else:
            assert routes_locally(p), pat
        c = O.Compiled(pat, 0)
        exp = [len(oracle_all(c, s)) for s in strings]
        assert exp[0] > 100 or kind == "prefix literal", (pat, exp)      # many matches in one string past 64 KB
        assert p.regex_count_batch(buf, off).tolist() == exp, pat
        assert [all_spans(p, s, capacity=1)[1] for s in strings] == exp, pat
        d_off = torch.from_numpy(off).cuda()
        for shift in (0, 5):
            d_counts = torch.full((len(strings) + 1,), SENTINEL, dtype=torch.int64, device="cuda")
            p.regex_count_batch_dev(to_device(torch, bytes(buf), shift), d_off, len(strings), int(off[-1]), d_counts)
            assert d_counts.cpu().tolist() == exp + [SENTINEL], (pat, shift)


@pytest.mark.gpu
def test_nfa_engine_handles_are_refused(device, monkeypatch):
    """counting and the all-matches loop need the table engine: an NFA-engine handle gets FX_ERR_DFA_STATE_CAP from all
    four entry points (the pattern whose eager automaton passes the cap, and any pattern under FX_STATE_CAP=3)"""
    torch = device
    text = b"ab aab c"
    buf, off = pack([text, b"", b"x"])
    d, d_off = to_device(torch, bytes(buf)), torch.from_numpy(off).cuda()
    handles = [fx.Pattern(b".*a(a|b){500}c{20}", "regex")]
    monkeypatch.setenv("FX_STATE_CAP", "3")
    handles.append(fx.Pattern(b"[a-c]+", "regex"))
    monkeypatch.delenv("FX_STATE_CAP")
    for p in handles:
        assert p.status == 0 and p.info()["nfa_engine"] == 1, p.pattern
        calls = [lambda: p.regex_count_batch(buf, off),
                 lambda: p.regex_count_batch_dev(d, d_off, 3, len(buf), torch.zeros(3, dtype=torch.int64, device="cuda")),
                 lambda: p.regex_buffer_all(np.frombuffer(text, dtype=np.uint8), capacity=4)]
        for call in calls:
            with pytest.raises(fx.ForgexError) as e:
                call()
            assert e.value.status == L.FX_ERR_DFA_STATE_CAP, p.pattern
        assert all_dev(torch, p, d, len(text), 4)[0] == L.FX_ERR_DFA_STATE_CAP, p.pattern


# ---- (h) device-resident forms: unaligned views, another stream ------------------------------------------------------
@pytest.mark.gpu
def test_dev_forms_on_unaligned_views_and_a_side_stream(device):
    """the _dev forms over views at byte offsets 1..15 into a tensor, on a non-default torch stream: the same answers
    as the host forms"""
    torch = device
    far = b"x" * (REACH + 77)
    texts = [b"a b c" + far + b"abc" + b" ab" * 1500 + far + "あい".encode() + b"\n12",
             bytes(synth.gen_c4(90000, 0.8, crlf=True)) + LINE]
    strings = count_strings()
    buf, off = pack(strings)
    side = torch.cuda.Stream()
    for pat in (b"[a-c]+", rb"\d+", C4, "[ぁ-ん]+".encode(), b"foo(bar|baz)"):
        p = fx.Pattern(pat, "regex")
        want = [all_spans(p, t) for t in texts]
        want_counts = p.regex_count_batch(buf, off).tolist()
        with torch.cuda.stream(side):
            d_off = torch.from_numpy(off).cuda()
            for shift in range(1, 16):
                for t, (spans, cnt) in zip(texts, want):
                    d = to_device(torch, t, shift)
                    d_from = torch.full((cnt + 1,), SENTINEL, dtype=torch.int64, device="cuda")
                    d_to = torch.full((cnt + 1,), SENTINEL, dtype=torch.int64, device="cuda")
                    work = torch.zeros(p.buffer_work_bytes(len(t)), dtype=torch.uint8, device="cuda")
                    assert p.regex_buffer_all_dev(d, len(t), d_from, d_to, cnt, work) == cnt, (pat, shift)
                    assert list(zip(d_from.tolist(), d_to.tolist())) == spans + [(SENTINEL, SENTINEL)], (pat, shift)
                d_counts = torch.zeros(len(strings), dtype=torch.int64, device="cuda")
                p.regex_count_batch_dev(to_device(torch, bytes(buf), shift), d_off, len(strings), int(off[-1]), d_counts)
                assert d_counts.tolist() == want_counts, (pat, shift)
        side.synchronize()
