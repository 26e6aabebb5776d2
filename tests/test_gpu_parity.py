"""GPU parity tests: the CUDA path, called through the C ABI, against the CPU oracle (bit-exact).

Run on the B200 box with `pytest -m gpu`.  Inputs are seeded (tools/synth.py) at sizes the oracle
finishes in seconds; the reference's own vectors go through the one-pattern-one-text entry points.
"""
import json
import os

import numpy as np
import pytest

import forgex_b200 as fx
from forgex_b200 import _lib
from tests import oracle_lib as O
from tools import synth

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
EAGER_CAP_PATTERNS = {b".*a(a|b){500}c{20}", b"[ab]*a[ab]{20}"}


def oracle_bool(pattern, op, buf, offsets=None, n=None, stride=None):
    c = O.Compiled(pattern, 1 if op == "match" else 0)
    o = 1 if op == "match" else 0
    return c.bool_batch(o, buf, offsets) if offsets is not None else c.bool_fixed(o, buf, n, stride)


def pack(strings):
    offsets = np.zeros(len(strings) + 1, dtype=np.int64)
    np.cumsum([len(s) for s in strings], out=offsets[1:])
    return np.frombuffer(b"".join(strings), dtype=np.uint8).copy(), offsets


# ---- the reference's own vectors through fx_in / fx_match / fx_regex ---------------------------
def test_reference_vectors_on_gpu():
    """all 997 API vectors of the reference's own tests through fx_in / fx_match / fx_regex.  Every one gets an answer:
    the two patterns whose eager automaton passes the state cap (Forgex only ever builds the few states their texts
    visit) run on the NFA engine"""
    with open(os.path.join(GOLD, "reference_api.json")) as fh:
        vecs = json.load(fh)["vectors"]
    bad, capped = [], 0
    for v in vecs:
        pat, text = bytes.fromhex(v["pattern"]), bytes.fromhex(v["text"])
        if v["kind"] == "match":
            ok = fx.op_match(pat, text) == v["expect"]
        elif v["kind"] == "in":
            ok = fx.op_in(pat, text) == v["expect"]
        else:
            ok = fx.regex_f(pat, text) == bytes.fromhex(v["expect"])
        capped += pat in EAGER_CAP_PATTERNS
        if not ok:
            bad.append("%s %s %r on %r" % (v["src"], v["kind"], pat, text[:40]))
    assert not bad, "\n".join(bad[:40])
    assert capped == 4
    for pat in EAGER_CAP_PATTERNS:
        assert fx.Pattern(pat, "match").info()["nfa_engine"] == 1


def test_nfa_engine_against_the_oracle(monkeypatch):
    """the NFA engine forced on ordinary patterns (FX_STATE_CAP=3: nearly every eager automaton passes that cap):
    `.in.`, `.match.`, spans, batches and the buffer path must still give the oracle's answers"""
    import random
    from tests.test_host_tables import gen_pattern, gen_text
    monkeypatch.setenv("FX_STATE_CAP", "3")
    rng = random.Random(515)
    texts = [gen_text(rng) for _ in range(150)] + [b"", b" ", b"foobar", b"abc\nabc", b"\xe3\x81\x82a\xff", b"aaaa"]
    buf, off = pack(texts)
    used = 0
    for pat in [b"foo(bar|baz)", rb"\d{3}-\d{4}", synth.PATTERNS["c3"], synth.PATTERNS["c4"], b"(a|b)*a(a|b){3}", b"a*", b"^$", b"aa[bc]", b"ab+c"] + \
               [gen_pattern(rng).encode() for _ in range(40)]:
        for op in ("in", "match", "regex"):
            p = fx.Pattern(pat, op)
            if p.status != 0 or not p.info()["nfa_engine"]:
                continue
            c = O.Compiled(pat, 1 if op == "match" else 0)
            if op == "regex":
                f, t = p.regex_batch(buf, off)
                ef, et = c.regex_batch(buf, off)
                assert np.array_equal(f, ef) and np.array_equal(t, et), (pat, np.nonzero((f != ef) | (t != et))[0][:5])
                joined = np.frombuffer(b"\n".join(texts[:40]), dtype=np.uint8)
                assert p.regex_buffer(joined) == c.regex_buffer(joined), (pat, "buffer")
            else:
                o = 1 if op == "match" else 0
                got = p.in_batch(buf, off) if op == "in" else p.match_batch(buf, off)
                assert np.array_equal(got, c.bool_batch(o, buf, off)), (pat, op)
            used += 1
    assert used > 60, used


def test_regex_out_arguments_like_reference():
    r = fx.regex(b"[d-f]{3}", b"abcdefghi")            # README.md:204-220
    assert (r.res, r.length, r.from_, r.to, r.status) == (b"def", 3, 4, 6, 0)
    r = fx.regex(b"(a", b"x")                           # forgex.F90:266-274
    assert (r.res, r.length, r.from_, r.to, r.status) == (b"", 0, -9999, -9999, 2)
    assert r.err_msg == O.error_message(2)
    r = fx.regex(b"zzz", b"abc")
    assert (r.res, r.length, r.from_, r.to, r.status) == (b"", 0, 0, 0, 0)


@pytest.mark.unpinned
def test_source_derived_expectations_on_gpu():
    """SURVEY 8c table: read off the reference source, never executed there; oracle and GPU must agree"""
    LF = b"\n"
    cases = [
        ("in", b"^", b"abc", False), ("in", b"^", b"a" + LF + b"b", False),
        ("in", rb"\s", b" ", False), ("match", rb"\s", b" ", True),
        ("match", b"^abc$", b"abc" + LF, True), ("match", b"abc$", b"abc" + LF, False),
        ("match", b"a{0}", b"a", True), ("in", b"aa[bc]", b"aaab", False),
        ("in", b"/", b"\xc0\xaf", False), ("in", b"[/x]", b"\xc0\xaf", True),
        ("match", b".", b"\t", False), ("match", b".", b"\xc8", True),
    ]
    for op, pat, text, exp in cases:
        got = fx.op_in(pat, text) if op == "in" else fx.op_match(pat, text)
        ora = O.op_in(pat, text) if op == "in" else O.op_match(pat, text)
        assert got == exp == bool(ora), (op, pat, text, got, ora)
    r = fx.regex(b"^abc$", b"def" + LF + b"abc")
    assert (r.res, r.from_, r.to) == (LF + b"abc", 4, 7)
    assert fx.regex_f(b"a{1,7}", b"aaa") == b"a" and fx.regex_f(b"[ab]{1,7}", b"aaa") == b"aaa"


# ---- config-shaped batches -----------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 31, 4097, 200000])
def test_c1_match_fixed(n):
    buf, n, stride = synth.gen_c1(n)
    p = fx.Pattern(synth.PATTERNS["c1"], "match")
    got = p.match_fixed(buf, n, stride)
    exp = oracle_bool(synth.PATTERNS["c1"], "match", buf, n=n, stride=stride)
    assert np.array_equal(got, exp)
    assert 0 < got.mean() < 1 or n < 31


@pytest.mark.parametrize("residency", ["auto", "global"])
@pytest.mark.parametrize("n", [1, 257, 30000])
def test_c2_in_ragged(n, residency):
    buf, off = synth.gen_c2(n)
    p = fx.Pattern(synth.PATTERNS["c2"], "in", residency=residency)
    got = p.in_batch(buf, off)
    exp = oracle_bool(synth.PATTERNS["c2"], "in", buf, offsets=off)
    assert np.array_equal(got, exp)
    info = p.info()
    assert info["residency"] == (_lib.FX_TABLE_GLOBAL if residency == "global" else _lib.FX_TABLE_SMEM)


def test_c2_overlong_and_prefix_candidates():
    """texts with bytes >= 0x80 take the exact prefix-candidate replay (api_internal_m.F90:76-104)"""
    strings = [b"xx\xc1\xa6oobar yy", b"\xc1\xa6oobar fooba!", b"foobax \xc1\xa6oobaz", b"foobar\xff", b"\xe3\x81\x82foobaz",
               b"fooba", b"foofoobar", b"", b" ", b"foobafoobar", b"\x00foobar\x00"]
    buf, off = pack(strings)
    p = fx.Pattern(synth.PATTERNS["c2"], "in")
    assert p.info()["prefix_mode"] == 1
    got = p.in_batch(buf, off)
    exp = oracle_bool(synth.PATTERNS["c2"], "in", buf, offsets=off)
    assert np.array_equal(got, exp), (got, exp)


@pytest.mark.parametrize("n", [1, 300, 20000])
def test_c3_regex_spans(n):
    buf, off = synth.gen_c3(n)
    p = fx.Pattern(synth.PATTERNS["c3"], "regex")
    f, t = p.regex_batch(buf, off)
    ef, et = O.Compiled(synth.PATTERNS["c3"], 0).regex_batch(buf, off)
    assert np.array_equal(f, ef) and np.array_equal(t, et)
    if n >= 300:
        assert 0.2 < (f > 0).mean() < 1.0


@pytest.mark.parametrize("match_at,crlf", [(0.001, False), (0.5, True), (0.999, False), (None, False)])
@pytest.mark.parametrize("nbytes", [4099, 3_000_001])
def test_c4_regex_buffer(nbytes, match_at, crlf):
    if nbytes < 10000 and match_at is not None and match_at < 0.01:
        match_at = 0.2
    buf = synth.gen_c4(nbytes, match_at, crlf=crlf)
    p = fx.Pattern(synth.PATTERNS["c4"], "regex")
    got = p.regex_buffer(buf)
    exp = O.Compiled(synth.PATTERNS["c4"], 0).regex_buffer(buf)
    assert got == exp
    if match_at is not None:
        # the span includes the line terminators the anchors consumed (SURVEY Q1)
        s = bytes(buf[got[0] - 1:got[1]])
        assert s.startswith(b"\n") or got[0] == 1
        assert synth.C4_MATCH_LINE in s and s.endswith(b"\n")
    else:
        assert got == (0, 0)


def test_c4_unaligned_and_tiny_buffers():
    p = fx.Pattern(synth.PATTERNS["c4"], "regex")
    c = O.Compiled(synth.PATTERNS["c4"], 0)
    line = synth.C4_MATCH_LINE
    for text in [b"", b" ", line, line + b"\n", b"x\n" + line, b"x\r\n" + line + b"\r\nrest", b"INFO a\nINFO b\n",
                 b"\n" * 40 + line, b"ERROR timeout=1", b"ERROR timeout=", b"\xe3\x81" + line + b"\xe3"]:
        for shift in (0, 1, 7):
            arr = np.frombuffer(b"#" * shift + text, dtype=np.uint8)[shift:]
            assert p.regex_buffer(arr) == c.regex_buffer(np.ascontiguousarray(arr)), (text, shift)


def test_buffer_one_byte_texts():
    for pat in [b"[a-z]+", b"a", b"ab*", b".", b"^", b"x|y"]:
        p = fx.Pattern(pat, "regex")
        c = O.Compiled(pat, 0)
        for text in [b"a", b"x", b" ", b"\n", b"\xff", b"b"]:
            arr = np.frombuffer(text, dtype=np.uint8)
            assert p.regex_buffer(arr) == c.regex_buffer(arr), (pat, text)


def test_buffer_patterns_with_a_prefix_literal():
    """candidates = the occurrences of the extracted prefix (api_internal_m.F90:76-104); every boundary when the
    literal occurs nowhere; FX_ERR_PREFILTER_UNSUPPORTED for a bordered prefix or a suffix literal"""
    rng = np.random.default_rng(23)
    filler = bytes(rng.integers(0x20, 0x7F, size=200000, dtype=np.uint8)).replace(b"foo", b"f0o").replace(b"ERR", b"E_R")
    texts = [b"xx foobar foobaz", b"fooba foobar", b"foobar", b"\xc1\xa6oobar", b"x\xc1\xa6oobar foobaz", b"zzz", b"", b" ", b"f",
             b"fooba", b"foobafoobar", filler + b"foobaz" + filler, filler + b"\xc1\xa6oobar" + filler, filler,
             filler[:70001] + b"fooba" + filler[:33] + b"foobar", b"foobar" + filler,
             b"ERROR x timeout=12 ERROR timeout=5", filler + b"ERROR a timeout=777\n" + filler, b"ERROR timeout=", b"ERROR"]
    used = 0
    for pat in [b"foo(bar|baz)", rb"ERROR.*timeout=\d+", b"ab+", b"hello (world|there)", "\u3042\u3044+".encode(), b"key=[0-9]*"]:
        p = fx.Pattern(pat, "regex")
        assert p.info()["prefix_scan"] == 1, pat
        c = O.Compiled(pat, 0)
        for text in texts + [b"hello there hello world", b"xabbb ab", "\u3042\u3044\u3044 \u3042".encode(), b"fooobar", b"key", b"a key=12 key="]:
            for shift in (0, 3):
                arr = np.frombuffer(b"#" * shift + text, dtype=np.uint8)[shift:]
                assert p.regex_buffer(arr) == c.regex_buffer(np.ascontiguousarray(arr)), (pat, text[:60], len(text), shift)
        used += 1
    assert used == 6
    # suffix literal / bordered prefix: the candidate list is sequential (non-overlapping occurrences, cut short by the
    # last suffix occurrence) -- one thread replays the reference's rule; the window forms decline
    import torch
    for pat in [b"ab+c", b"aab*", b"abab+", b"fo+bar", b"aa[bc]"]:
        p = fx.Pattern(pat, "regex")
        assert p.info()["prefix_scan"] == 0
        c = O.Compiled(pat, 0)
        for text in [b"xx aabab abc", b"aaab", b"aaaab aab", b"ababab abab", b"fobar foobar", b"abbbc abc c", b"", b"c", filler[:3000] + b"aaab abbc foobar",
                     b"ab" * 500 + b"c", b"a" * 301 + b"b"]:
            arr = np.frombuffer(text, dtype=np.uint8)
            assert p.regex_buffer(arr) == c.regex_buffer(arr), (pat, text[:40])
        win = torch.zeros(64, dtype=torch.uint8, device="cuda")
        best = torch.tensor([-1, 0, 0], dtype=torch.int64, device="cuda")
        with pytest.raises(fx.ForgexError) as e:
            p.buffer_scan_dev(win, 64, 0, 64, 0, True, True, best)
        assert e.value.status == _lib.FX_ERR_PREFILTER_UNSUPPORTED


@pytest.mark.parametrize("residency", ["auto", "global"])
@pytest.mark.parametrize("compact", ["1", "0"])
def test_c5_in_fixed_big_table(residency, compact, monkeypatch):
    """10252 byte-states x 16 classes (328 KB) fit neither shared memory nor L1.  K1c walks the ASCII columns alone
    (82 KB: from shared memory, or from global memory when that path is forced as BASELINE config 5 states it); with
    FX_COMPACT=0 the full class-compressed table is read through L1/L2 (K1).  Strings with bytes >= 0x80 always take
    the full table."""
    monkeypatch.setenv("FX_COMPACT", compact)
    buf, n, stride = synth.gen_c5(3000)
    buf = buf.copy()
    buf[5 * 64 + 7] = 0xC3; buf[5 * 64 + 8] = 0xA9        # a multi-byte character, a stray continuation byte, an overlong `a`
    buf[9 * 64 + 60] = 0x80
    buf[11 * 64 + 3] = 0xC1; buf[11 * 64 + 4] = 0xA1
    p = fx.Pattern(synth.PATTERNS["c5"], "in", residency=residency)
    got = p.in_fixed(buf, n, stride)
    exp = oracle_bool(synth.PATTERNS["c5"], "in", buf, n=n, stride=stride)
    assert np.array_equal(got, exp)
    info = p.info()
    if compact == "1":
        assert info["compact_used"] == (2 if residency == "global" else 1)
        assert info["residency"] == (_lib.FX_TABLE_GLOBAL if residency == "global" else _lib.FX_TABLE_SMEM)
    else:
        assert info["compact_used"] == 0 and info["residency"] == _lib.FX_TABLE_GLOBAL


# ---- edge cases: empty / ragged / long / unaligned -------------------------------------------------
def test_ragged_edge_cases(monkeypatch):
    rng = np.random.default_rng(7)
    strings = [b"", b" ", b"a", b"", b"", b"foobar", b"x" * 5000 + b"foobaz", b"y" * 70000, b"foobar" * 3, b"",
               bytes(rng.integers(0, 256, size=300, dtype=np.uint8)), b"\x00", b"\xe3\x81", b"fooba", b""]
    strings += [bytes(rng.integers(0x20, 0x7F, size=int(k), dtype=np.uint8)) for k in rng.integers(0, 40, size=500)]
    strings += [b"7" * 20000 + b"abcr" + b"7" * 3000, b"7" * 9000 + "\u3042\u3044 ab".encode() + b"7" * 9000]   # longer than a warp's tile
    strings += [b"", b""]
    buf, off = pack(strings)
    for pat, op in [(b"foo(bar|baz)", "in"), (rb"\d{3}-\d{4}", "match"), (b"[a-z]+", "in"), (b"", "match"), (b"a*", "in"),
                    (b"x*y+", "match"), (b"foobar", "in"), (b"foobar", "match"), (b"fo+bar", "match"), (b"^$", "in")]:
        p = fx.Pattern(pat, op)
        got = p.in_batch(buf, off) if op == "in" else p.match_batch(buf, off)
        exp = oracle_bool(pat, op, buf, offsets=off)
        assert np.array_equal(got, exp), (pat, op, np.nonzero(got != exp)[0][:10])
    # empty strings and a lone blank at both ends, a 3006-byte string, an overlong `C1 A6` start of `foobar`, 3000
    # short random strings, and C2 data: through the default route (K2c for `foo(bar|baz)`) and through K2 alone
    more = [b"", b"", b" ", b"foobar", b"x" * 3000 + b"foobaz", b"", b"fooba", b"\xc1\xa6oobar fooba!"]
    rng = np.random.default_rng(3)
    more += [bytes(rng.integers(0x20, 0x7F, size=int(k), dtype=np.uint8)) for k in rng.integers(0, 300, size=3000)]
    more += [b"foobaz", b"", b""]
    sets = [pack(more), synth.gen_c2(40000)]
    for sparse in ("1", "0"):
        monkeypatch.setenv("FX_SPARSE", sparse)
        for pat, op in [(b"foo(bar|baz)", "in"), (rb"\d{3}-\d{4}", "match"), (b"[a-z]+", "in"), (b"a*", "in"), (b"x*y+", "match")]:
            p = fx.Pattern(pat, op)
            for b_, o_ in sets:
                got = p.in_batch(b_, o_) if op == "in" else p.match_batch(b_, o_)
                info = p.info()
                assert info["sparse_used"] == (info["sparse"] if sparse == "1" else 0)
                exp = oracle_bool(pat, op, b_, offsets=o_)
                assert np.array_equal(got, exp), (sparse, pat, op, np.nonzero(got != exp)[0][:10])
    monkeypatch.delenv("FX_SPARSE")
    for pat in [b"[a-z]+", b"o+b", b"foobar", b"(foo|y+)$", b"^", b"\\s\\S+", b"aa[bc]", synth.PATTERNS["c3"]]:
        p = fx.Pattern(pat, "regex")
        f, t = p.regex_batch(buf, off)
        ef, et = O.Compiled(pat, 0).regex_batch(buf, off)
        assert np.array_equal(f, ef) and np.array_equal(t, et), pat
    # a pattern whose attempts run long (quadratic for the reference's brute force, hence for the oracle): only on
    # strings where every failing start dies at once; they are longer than a warp's tile and take the linear path
    # from global memory
    long_strings = [b"7" * 20000 + b"abcr" + b"7" * 3000, b"abc", b"7" * 30000, b"", b"7" * 6000 + b"zr", b"r" * 9]
    buf, off = pack(long_strings)
    for pat in [b"[a-z]+r", b"[a-z]*r7", rb"\d{3}r"]:
        f, t = fx.Pattern(pat, "regex").regex_batch(buf, off)
        ef, et = O.Compiled(pat, 0).regex_batch(buf, off)
        assert np.array_equal(f, ef) and np.array_equal(t, et), pat


def test_fixed_strides_and_alignment():
    rng = np.random.default_rng(11)
    for stride in (0, 1, 3, 8, 16, 24, 64, 100):
        n = 1000
        raw = rng.integers(0x20, 0x7F, size=n * max(stride, 1) + 16, dtype=np.uint8)
        raw[rng.random(raw.size) < 0.3] = ord("a")
        for shift in (0, 5):
            buf = raw[shift:shift + n * stride]
            for pat, op in [(b"a+b?", "in"), (b"[a-m ]*", "match"), (b"(a|b)*a(a|b){3}", "in")]:
                p = fx.Pattern(pat, op)
                got = p.in_fixed(buf, n, stride) if op == "in" else p.match_fixed(buf, n, stride)
                exp = oracle_bool(pat, op, np.ascontiguousarray(buf), n=n, stride=stride)
                assert np.array_equal(got, exp), (stride, shift, pat)


def test_utf8_and_invalid_bytes_batch():
    rng = np.random.default_rng(5)
    pieces = [b"a", b"z", b" ", "あ".encode(), "ん".encode(), "α".encode(), "　".encode(), b"\x80", b"\xbf", b"\xc3", b"\xe3\x81",
              b"\xf0\x9f\x98", b"\xff", b"\xc0\x80", b"\xc1\xa1", b"\xe0\x81\xa1", b"\xef\xbf\xbf", b"\xf4\x90\x80\x81", b"\n", b"\r\n", b"_", b"7"]
    strings = [b"".join(pieces[i] for i in rng.integers(0, len(pieces), size=int(k))) for k in rng.integers(0, 24, size=4000)]
    buf, off = pack(strings)
    for pat in [synth.PATTERNS["c3"], b"[a-z]+", b".+", rb"\S+", "[ぁ-ん]+".encode(), b"a.", rb"[^a]{2,3}$", rb"^\w"]:
        p = fx.Pattern(pat, "regex")
        f, t = p.regex_batch(buf, off)
        ef, et = O.Compiled(pat, 0).regex_batch(buf, off)
        assert np.array_equal(f, ef) and np.array_equal(t, et), pat
        for op in ("in", "match"):
            q = fx.Pattern(pat, op)
            got = q.in_batch(buf, off) if op == "in" else q.match_batch(buf, off)
            assert np.array_equal(got, oracle_bool(pat, op, buf, offsets=off)), (pat, op)


def test_device_pointer_entry_points():
    import torch
    buf, off = synth.gen_c2(50000)
    d_buf = torch.from_numpy(buf).cuda()
    d_off = torch.from_numpy(off).cuda()
    d_out = torch.empty(len(off) - 1, dtype=torch.uint8, device="cuda")
    p = fx.Pattern(synth.PATTERNS["c2"], "in")
    before = fx.launch_count()
    p.in_batch_dev(d_buf, d_off, len(off) - 1, int(off[-1]), d_out)
    torch.cuda.synchronize()
    assert fx.launch_count() == before + 1
    assert np.array_equal(d_out.cpu().numpy(), oracle_bool(synth.PATTERNS["c2"], "in", buf, offsets=off))
    # size-independent property: a line is true iff it holds foobar or foobaz (ASCII data, SURVEY 8-P)
    truth = np.array([(b"foobar" in bytes(buf[off[i]:off[i + 1]])) or (b"foobaz" in bytes(buf[off[i]:off[i + 1]]))
                      for i in range(2000)], dtype=np.uint8)
    assert np.array_equal(d_out[:2000].cpu().numpy(), truth)


def test_invalid_pattern_and_wrong_op_errors():
    p = fx.Pattern(b"(a", "in")
    assert p.status == 2
    with pytest.raises(fx.ForgexError):
        p.in_batch(np.zeros(4, np.uint8), np.array([0, 4], np.int64))
    q = fx.Pattern(b"a", "in")
    with pytest.raises(fx.ForgexError):
        q.match_batch(np.zeros(4, np.uint8), np.array([0, 4], np.int64))
    assert fx.op_in(b"(a", b"a") is False and fx.op_match(b"a)", b"a") is False


def test_sparse_start_kernel(monkeypatch):
    """K2c (linear sweep + candidate starts) against the oracle, and against K2 with the sparse path switched off"""
    monkeypatch.setenv("FX_SPARSE_MAX_FIRST", "128")      # every eligible pattern, however dense its first-byte set
    rng = np.random.default_rng(17)
    pieces = [b"a", b"z", b" ", b"f", b"foo", b"bar", b"foobar", "あ".encode(), "α".encode(), b"\x80", b"\xbf", b"\xc3", b"\xe3\x81",
              b"\xff", b"\xc0\x80", b"\xc1\xa6", b"\xe0\x81\xa6", b"\xf0\x80\x81\xa6", b"\n", b"\r\n", b"\r", b"\x00", b"7", b"-",
              b"ERROR", b"timeout=", b"x", b"h\xc3\xa9llo"]
    s1 = [b"".join(pieces[i] for i in rng.integers(0, len(pieces), size=int(k))) for k in rng.integers(0, 30, size=6000)]
    s2 = [b"", b" ", b"a", b"", b"", b"foobar", b"x" * 5000 + b"foobaz", b"y" * 70000 + b"foobar", b"foobar" * 3, b"",
          bytes(rng.integers(0, 256, size=300, dtype=np.uint8)), b"\x00", b"\xe3\x81", b"fooba", b"", b"f", b"\nfoobar", b"foobar\n"]
    s2 += [bytes(rng.integers(0x20, 0x7F, size=int(k), dtype=np.uint8)) for k in rng.integers(0, 400, size=3000)]
    s2 += [b"f" * 3000, b"", b""]
    sets = [pack(s1), pack(s2), synth.gen_c2(30000)]
    used = 0
    for pat in [b"foo(bar|baz)", b"^foo", b"a*", rb"\d{3}-\d{4}", b"[a-z]+r", b"x$", rb"^ERROR.*timeout=\d+$", "héllo|x".encode(),
                "[ぁ-ん]+a".encode(), b"(|^)a", b"f.*r$", b"(foo|bar)+", rb"\s\S+", b"^", b"$", b"f{2,}", b"z?y", b"(a|b)*a(a|b){3}"]:
        monkeypatch.setenv("FX_SPARSE", "1")
        p = fx.Pattern(pat, "in")
        for buf, off in sets:
            got = p.in_batch(buf, off)
            info = p.info()
            assert info["sparse_used"] == info["sparse"]
            exp = oracle_bool(pat, "in", buf, offsets=off)
            assert np.array_equal(got, exp), (pat, np.nonzero(got != exp)[0][:10])
        used += info["sparse_used"]
        if info["sparse"]:
            monkeypatch.setenv("FX_SPARSE", "0")
            buf, off = sets[0]
            assert np.array_equal(p.in_batch(buf, off), oracle_bool(pat, "in", buf, offsets=off))
            assert p.info()["sparse_used"] == 0
    assert used >= 10
    monkeypatch.setenv("FX_SPARSE", "1")
    monkeypatch.delenv("FX_SPARSE_MAX_FIRST")
    assert fx.Pattern(b"foo(bar|baz)", "in").info()["sparse"] == 1     # the C2 pattern takes this path by default
    assert fx.Pattern(rb"\w+@\w+", "in").info()["sparse"] == 0


def test_buffer_windows_like_two_gpus():
    """the window entry points (fx_buffer_scan_dev / fx_buffer_finish_dev) driven the way forgex_b200.dist drives
    them on 2..4 GPUs, here one slab after the other on one device"""
    import torch
    from forgex_b200 import dist as fxd
    p = fx.Pattern(synth.PATTERNS["c4"], "regex")
    c = O.Compiled(synth.PATTERNS["c4"], 0)
    for nbytes, match_at, world in [(200_000, 0.7, 2), (200_000, 0.2, 4), (50_001, None, 3), (300_000, 0.5001, 2)]:
        text = synth.gen_c4(nbytes, match_at)
        exp = c.regex_buffer(text)
        d_text = torch.from_numpy(text).cuda()
        keys, und = [], 0
        for rank in range(world):
            lo, hi = fxd.slab_bounds(nbytes, world, rank)
            w_lo, w_hi = fxd.window_for_slab(nbytes, lo, hi, 1024)
            win = d_text[w_lo:w_hi].clone()
            best = torch.tensor([-1, 0, 0], dtype=torch.int64, device="cuda")
            p.buffer_scan_dev(win, w_hi - w_lo, lo - w_lo, hi - w_lo, w_lo, w_lo == 0, w_hi == nbytes, best)
            b = best.cpu().numpy().view(np.uint64)
            keys.append(int(b[0]))
            und += int(b[1])
        assert und == 0
        key = min(keys)
        if key == fxd.NO_START:
            assert exp == (0, 0)
            continue
        owner = keys.index(key)
        lo, hi = fxd.slab_bounds(nbytes, world, owner)
        w_lo, w_hi = fxd.window_for_slab(nbytes, lo, hi, 1024)
        win = d_text[w_lo:w_hi].clone()
        ft = torch.zeros(2, dtype=torch.int64, device="cuda")
        p.buffer_finish_dev(win, w_hi - w_lo, w_lo, w_hi == nbytes, torch.tensor([key], dtype=torch.int64, device="cuda"), ft)
        assert tuple(ft.cpu().tolist()) == exp, (nbytes, match_at, world)


def test_prefix_literal_windows_like_two_gpus():
    """a pattern with a prefix literal over slabs: occurrences are counted per slab (d_best[2]); only when NO slab holds
    one does the search fall back to every boundary (fx_buffer_scan_all_dev) -- forgex_b200.dist.buffer_search's protocol"""
    import torch
    from forgex_b200 import dist as fxd
    pat = b"foo(bar|baz)"
    p = fx.Pattern(pat, "regex")
    c = O.Compiled(pat, 0)
    rng = np.random.default_rng(29)
    filler = bytes(rng.integers(0x20, 0x7F, size=90000, dtype=np.uint8)).replace(b"foo", b"f0o")
    cases = [filler + b"foobaz" + filler, filler + filler[:5000] + b"fooba!" + filler + b"foobar",
             filler + b"\xc1\xa6oobar" + filler,                      # the literal occurs nowhere: overlong start wins by brute force
             filler + b"\xc1\xa6oobar" + filler + b"fooba",           # ... but here it does occur, so the overlong start is never tried
             filler + filler, b"foobar" + filler]
    for text in cases:
        text = np.frombuffer(text, dtype=np.uint8)
        nbytes = len(text)
        exp = c.regex_buffer(text)
        d_text = torch.from_numpy(text.copy()).cuda()
        for world in (2, 3):
            def scan_all_ranks(every):
                keys, und, occ = [], 0, 0
                for rank in range(world):
                    lo, hi = fxd.slab_bounds(nbytes, world, rank)
                    w_lo, w_hi = fxd.window_for_slab(nbytes, lo, hi, 1024)
                    win = d_text[w_lo:w_hi].clone()
                    best = torch.tensor([-1, 0, 0], dtype=torch.int64, device="cuda")
                    call = p.buffer_scan_all_dev if every else p.buffer_scan_dev
                    call(win, w_hi - w_lo, lo - w_lo, hi - w_lo, w_lo, w_lo == 0, w_hi == nbytes, best)
                    b = best.cpu().numpy().view(np.uint64)
                    keys.append(int(b[0])); und += int(b[1]); occ += int(b[2])
                return keys, und, occ
            keys, und, occ = scan_all_ranks(False)
            assert occ == (0 if bytes(text).find(b"fooba") < 0 else occ) and (occ > 0) == (bytes(text).find(b"fooba") >= 0)
            if occ == 0:
                keys, und, _ = scan_all_ranks(True)
            assert und == 0
            key = min(keys)
            if key == fxd.NO_START:
                assert exp == (0, 0), (len(text), world)
                continue
            owner = keys.index(key)
            lo, hi = fxd.slab_bounds(nbytes, world, owner)
            w_lo, w_hi = fxd.window_for_slab(nbytes, lo, hi, 1024)
            win = d_text[w_lo:w_hi].clone()
            ft = torch.zeros(2, dtype=torch.int64, device="cuda")
            p.buffer_finish_dev(win, w_hi - w_lo, w_lo, w_hi == nbytes, torch.tensor([key], dtype=torch.int64, device="cuda"), ft)
            assert tuple(ft.cpu().tolist()) == exp, (len(text), world)


def test_sparse_start_kernel_fixed_stride(monkeypatch):
    """fixed-stride `.in.` batches take the sparse-start kernel too (a Fortran character array is one)"""
    monkeypatch.setenv("FX_SPARSE_MAX_FIRST", "128")
    rng = np.random.default_rng(31)
    for stride in (1, 3, 8, 16, 24, 64, 100, 160, 4099):
        n = 3000 if stride < 1000 else 40
        raw = rng.integers(0x20, 0x7F, size=n * stride + 64, dtype=np.uint8)
        raw[rng.random(raw.size) < 0.05] = ord("f")
        for k in rng.integers(0, max(1, n * stride - 8), size=n // 3):
            raw[k:k + 6] = np.frombuffer(b"foobar" if k & 1 else b"fooba!", dtype=np.uint8)
        raw[rng.random(raw.size) < 0.002] = 0xC1
        for shift in (0, 5):
            buf = raw[shift:shift + n * stride]
            for pat in [b"foo(bar|baz)", b"f+o", b"^f", b"r$", b"a*", b"[fz]o+"]:
                monkeypatch.setenv("FX_SPARSE", "1")
                p = fx.Pattern(pat, "in")
                got = p.in_fixed(buf, n, stride)
                assert p.info()["sparse_used"] == p.info()["sparse"]
                exp = oracle_bool(pat, "in", np.ascontiguousarray(buf), n=n, stride=stride)
                assert np.array_equal(got, exp), (stride, shift, pat, np.nonzero(got != exp)[0][:10])
                monkeypatch.setenv("FX_SPARSE", "0")
                assert np.array_equal(p.in_fixed(buf, n, stride), exp), (stride, shift, pat, "K1")


@pytest.mark.parametrize("seed", range(6))
def test_generated_patterns_on_gpu(seed, monkeypatch):
    """random patterns (the generator of the CPU fuzz) through every batch kernel and the buffer path, against the
    oracle: whatever kernel the host picks for a pattern -- sparse starts, tile walk, linear spans, emulation, sparse
    or LUT buffer scan, prefix candidates -- must give the oracle's answer"""
    import random
    from tests.test_host_tables import gen_pattern, gen_text
    monkeypatch.setenv("FX_SPARSE_MAX_FIRST", "128")
    rng = random.Random(9000 + seed)
    texts = [gen_text(rng) for _ in range(700)] + [b"", b" ", b"", b"a" * 300, gen_text(rng) * 40]
    buf, off = pack(texts)
    stride = 12
    nfix = len(buf) // stride
    joined = b"\n".join(texts[:300])
    jarr = np.frombuffer(joined, dtype=np.uint8)
    tried = {"in": 0, "match": 0, "regex": 0, "buffer": 0, "sparse": 0, "unsupported": 0}
    for _ in range(70):
        pat = gen_pattern(rng).encode()
        for op in ("in", "match", "regex"):
            p = fx.Pattern(pat, op)
            if p.status != 0:
                continue
            c = O.Compiled(pat, 1 if op == "match" else 0)
            if op == "regex":
                f, t = p.regex_batch(buf, off)
                ef, et = c.regex_batch(buf, off)
                assert np.array_equal(f, ef) and np.array_equal(t, et), (pat, np.nonzero((f != ef) | (t != et))[0][:5])
                tried["regex"] += 1
                assert p.regex_buffer(jarr) == c.regex_buffer(jarr), (pat, "buffer")      # every pattern is accepted on the buffer path
                tried["buffer"] += 1
            else:
                o = 1 if op == "match" else 0
                got = p.in_batch(buf, off) if op == "in" else p.match_batch(buf, off)
                assert np.array_equal(got, c.bool_batch(o, buf, off)), (pat, op, np.nonzero(got != c.bool_batch(o, buf, off))[0][:5])
                gotf = p.in_fixed(buf, nfix, stride) if op == "in" else p.match_fixed(buf, nfix, stride)
                assert np.array_equal(gotf, c.bool_fixed(o, buf, nfix, stride)), (pat, op, "fixed")
                tried[op] += 1
                tried["sparse"] += p.info()["sparse_used"] if op == "in" else 0
    assert tried["in"] > 30 and tried["regex"] > 30 and tried["buffer"] > 20 and tried["sparse"] > 5, tried


def test_span_kernel_degenerate_strings_behind_a_long_one():
    """a "" or " " that shares a tile with an over-long string is not staged (its end lies past the staged bytes) and
    takes the global-memory walk: the blank-text rule (api_internal_m.F90:68-74) must hold there too"""
    strings = [b"y" * 70000, b"", b" ", b"a", b" ", b"", b"x" * 40000 + b" ", b" ", b""] + [b" ", b""] * 20
    buf, off = pack(strings)
    for pat in [b"^$", rb"\s", b".", b"[ a]", b"a*", b" *", rb"\s*$"]:
        p = fx.Pattern(pat, "regex")
        f, t = p.regex_batch(buf, off)
        ef, et = O.Compiled(pat, 0).regex_batch(buf, off)
        assert np.array_equal(f, ef) and np.array_equal(t, et), (pat, f[:9], ef[:9], t[:9], et[:9])


def test_literal_patterns_on_the_buffer_and_window_paths():
    """a pattern that is one literal never consults the automaton: regex() = index(text, literal), plain bytes
    (forgex.F90:281-307).  On the long-buffer path that is a parallel sweep (k_buffer_literal), also over windows."""
    import torch
    from forgex_b200 import dist as fxd
    rng = np.random.default_rng(41)
    filler = bytes(rng.integers(0x20, 0x7F, size=300000, dtype=np.uint8)).replace(b"ERR", b"E_R").replace(b"fo", b"f0")
    texts = [filler + b"ERROR" + filler + b"ERROR", b"ERROR", b"ERRO", b"", b" ", filler, b"xERROR", filler[:70001] + b"foo" + filler[:5],
             b"\xc0\xaf/", b"a{1,7}aaa", b"aaa"]
    for pat in [b"ERROR", b"foo", b"/", b"a{1,7}", b"[/]", rb"\x41", b"o"]:
        p = fx.Pattern(pat, "regex")
        assert p.info()["literal_only"] == 1
        c = O.Compiled(pat, 0)
        for text in texts:
            for shift in (0, 5):
                arr = np.frombuffer(b"#" * shift + text, dtype=np.uint8)[shift:]
                assert p.regex_buffer(arr) == c.regex_buffer(np.ascontiguousarray(arr)), (pat, len(text), shift)
    # windows: two "GPUs", literal in the second slab / across the cut / nowhere
    p = fx.Pattern(b"ERROR", "regex")
    c = O.Compiled(b"ERROR", 0)
    cut_text = filler[:100014] + b"ERROR" + filler[:99984]           # straddles the 2-rank cut at 100016
    for text in [filler + b"ERROR" + filler[:1000], cut_text, filler, b"ERROR" + filler]:
        text = np.frombuffer(text, dtype=np.uint8)
        nbytes = len(text)
        exp = c.regex_buffer(text)
        d_text = torch.from_numpy(text.copy()).cuda()
        for world in (2, 3):
            keys, und = [], 0
            for rank in range(world):
                lo, hi = fxd.slab_bounds(nbytes, world, rank)
                w_lo, w_hi = fxd.window_for_slab(nbytes, lo, hi, 64)
                win = d_text[w_lo:w_hi].clone()
                best = torch.tensor([-1, 0, 0], dtype=torch.int64, device="cuda")
                p.buffer_scan_dev(win, w_hi - w_lo, lo - w_lo, hi - w_lo, w_lo, w_lo == 0, w_hi == nbytes, best)
                b = best.cpu().numpy().view(np.uint64)
                keys.append(int(b[0])); und += int(b[1])
            assert und == 0
            key = min(keys)
            if key == fxd.NO_START:
                assert exp == (0, 0)
                continue
            owner = keys.index(key)
            lo, hi = fxd.slab_bounds(nbytes, world, owner)
            w_lo, w_hi = fxd.window_for_slab(nbytes, lo, hi, 64)
            win = d_text[w_lo:w_hi].clone()
            ft = torch.zeros(2, dtype=torch.int64, device="cuda")
            p.buffer_finish_dev(win, w_hi - w_lo, w_lo, w_hi == nbytes, torch.tensor([key], dtype=torch.int64, device="cuda"), ft)
            assert tuple(ft.cpu().tolist()) == exp, (nbytes, world)


def test_c4_buffer_beyond_4_gib():
    """the reason the long-buffer path is 64-bit (SURVEY H7): a 4.5 GiB text whose only match starts past offset 2^32.
    The span is known by construction (planted line + the LF consumed by `^` + the LF consumed by `$`, SURVEY Q1) and is
    cross-checked against the oracle on the slice that ends behind the planted line."""
    import torch
    nbytes = (4 << 30) + (512 << 20)
    hb = synth.gen_c4_block(64 << 20, seed_stream=3)
    last_nl = int(np.nonzero(hb == 10)[0][-1]) + 1
    d_block = torch.from_numpy(hb[:last_nl]).cuda()
    buf = d_block.repeat((nbytes + last_nl - 1) // last_nl)[:nbytes].contiguous()
    pos = (1 << 32) + (100 << 20) + 12345
    nls = np.nonzero(hb[:last_nl] == 10)[0]
    tpos = pos % last_nl
    k = int(np.searchsorted(nls, tpos, side="left")) - 1
    start = (pos - tpos) + int(nls[k]) + 1
    assert start > (1 << 32)
    line = synth.C4_MATCH_LINE + b"\n"
    buf[start:start + len(line) + 5] = torch.from_numpy(np.frombuffer(line + b"INFO ", dtype=np.uint8).copy()).cuda()
    crlf_before = int(hb[(start - 1) % last_nl - 1]) == 13
    expect = (start - (1 if crlf_before else 0), start + len(line))
    p = fx.Pattern(synth.PATTERNS["c4"], "regex")
    ft = torch.zeros(2, dtype=torch.int64, device="cuda")
    work = torch.zeros(p.buffer_work_bytes(nbytes), dtype=torch.uint8, device="cuda")
    p.regex_buffer_dev(buf, nbytes, ft, work)
    got = tuple(ft.cpu().tolist())
    assert got == expect and got[0] > (1 << 32), (got, expect)
    # oracle on the last 24 MiB up to just behind the planted line: same span, shifted
    a, b = start - (24 << 20), start + 1000
    sl = buf[a:b].contiguous()
    exp = O.Compiled(synth.PATTERNS["c4"], 0).regex_buffer(sl.cpu().numpy())
    assert exp[0] > 0 and (exp[0] + a, exp[1] + a) == got
    p.regex_buffer_dev(sl, b - a, ft, work)
    assert tuple(ft.cpu().tolist()) == exp
    # the same text without the planted line: no match anywhere
    buf[start:start + 5] = torch.from_numpy(np.frombuffer(b"WARN ", dtype=np.uint8).copy()).cuda()
    p.regex_buffer_dev(buf, nbytes, ft, work)
    assert tuple(ft.cpu().tolist()) == (0, 0)


def test_statemap_scan_against_the_oracle(monkeypatch):
    """K5, the chunked state-map scan of the long-buffer path, forced for every pattern that has the span path
    (FX_STATEMAP=2): same spans as the oracle on texts that cross sub-chunk (512 B), segment (16 KB) and region cuts,
    with multi-byte sequences and invalid bytes on the cuts"""
    import random
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
    used = 0
    for pat in pats:
        p = fx.Pattern(pat, "regex")
        if p.status != 0 or not p.info()["statemap"] or p.info()["literal_only"] or p.info()["literal_prefix_len"]:
            continue
        c = O.Compiled(pat, 0)
        for text in texts:
            if len(text) > 6000 and pat not in pats[:2]:
                continue                       # (the oracle is quadratic in the worst case: long texts only for the two config patterns,
                                               #  whose attempts end at the next line end / separator)
            arr = np.frombuffer(b"#" + text, dtype=np.uint8)[1:]       # odd address: the sub-chunk grid is address-aligned
            exp = c.regex_buffer(np.ascontiguousarray(arr))
            monkeypatch.setenv("FX_STATEMAP", "2")
            got = p.regex_buffer(arr)
            assert p.info()["statemap_used"] == (1 if len(text) >= 2 else 0), pat
            assert got == exp, (pat, len(text), got, exp)
            monkeypatch.setenv("FX_STATEMAP", "1")
            assert p.regex_buffer(arr) == exp, (pat, len(text), "default flow")
        used += 1
    assert used >= 25, used


def test_long_attempts_are_linear_time():
    """`[ab].*c` over 64 MiB of `a` without a newline: every byte is a candidate start and every attempt runs to the end
    of the text -- the reference's loop (and K4) is quadratic here.  The work budget stops K4 and the state-map scan
    answers: no `c`, no match.  With a `c` at the end of 4 MiB the match is the whole text."""
    import time
    import torch
    p = fx.Pattern(b"[ab].*c", "regex")
    assert p.info()["statemap"] == 1 and p.info()["sparse"] == 1
    n = 64 << 20
    buf = torch.full((n,), ord("a"), dtype=torch.uint8, device="cuda")
    ft = torch.zeros(2, dtype=torch.int64, device="cuda")
    work = torch.zeros(p.buffer_work_bytes(n), dtype=torch.uint8, device="cuda")
    p.regex_buffer_dev(buf, n, ft, work)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    p.regex_buffer_dev(buf, n, ft, work)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    assert tuple(ft.cpu().tolist()) == (0, 0)
    assert dt < 0.25, "%.3f s for 64 MiB" % dt
    assert p.info()["statemap_used"] == 2
    m = 4 << 20
    buf[m - 1] = ord("c")
    p.regex_buffer_dev(buf, m, ft, work)
    assert tuple(ft.cpu().tolist()) == (1, m)
    small = np.frombuffer(b"a" * 3000 + b"c" + b"a" * 100, dtype=np.uint8)
    assert p.regex_buffer(small) == O.Compiled(b"[ab].*c", 0).regex_buffer(small) == (1, 3001)


def oracle_all(c, text):
    """the caller's loop: regex(), then regex() again on text(to+1:), each call framed afresh"""
    out, pos = [], 0
    arr = np.frombuffer(text, dtype=np.uint8)
    while True:
        f, t = c.regex_buffer(np.ascontiguousarray(arr[pos:]))
        if f <= 0 or t <= 0:
            return out
        out.append((pos + f, pos + t))
        pos += t


def test_all_matches_and_counts():
    """fx_regex_buffer_all / fx_regex_count_batch against the oracle's loop (README.md:197-222): dense and sparse
    matches, anchors that re-match at every restart (fresh leading NUL), literals, prefix literals, UTF-8"""
    import random
    from tests.test_host_tables import gen_pattern, gen_text
    rng = random.Random(99)
    log = bytes(synth.gen_c4(60000, 0.3)) + synth.C4_MATCH_LINE + b"\n" + bytes(synth.gen_c4_block(30000, 5)) + synth.C4_MATCH_LINE
    texts = [b"foobar foobaz fooba foobarfoobaz", b"abc\nabc\r\nabc", b"aaa", b"", b" ", b"x y  z", log,
             "あいう えお かきく".encode() * 50, b"\n".join(gen_text(rng) for _ in range(300)), b"a" * 5000, b"ab" * 3000 + b"\n" + b"ba" * 200]
    pats = [b"foo(bar|baz)", b"^abc", b"abc$", b"a", b"[a-z]+", rb"\s", synth.PATTERNS["c4"], "[ぁ-ん]+".encode(), b"a{1,7}", b"(ab)+", b"^", b".",
            b"[ab]{2,3}", b"ERROR", rb"\w+\s"]
    pats += [gen_pattern(rng).encode() for _ in range(25)]
    used = 0
    for pat in pats:
        p = fx.Pattern(pat, "regex")
        if p.status != 0:
            continue
        c = O.Compiled(pat, 0)
        for text in texts:
            if len(text) > 20000 and pat not in pats[:15]:
                continue
            exp = oracle_all(c, text)
            f, t, cnt = p.regex_buffer_all(np.frombuffer(text, dtype=np.uint8), capacity=max(1, len(exp) + 3))
            assert cnt == len(exp) and list(zip(f.tolist(), t.tolist())) == exp, (pat, len(text), cnt, len(exp), exp[:3], list(zip(f, t))[:3])
            if exp:
                f2, t2, cnt2 = p.regex_buffer_all(np.frombuffer(text, dtype=np.uint8), capacity=1)
                assert cnt2 == len(exp) and (f2[0], t2[0]) == exp[0]
        buf, off = pack(texts)
        counts = p.regex_count_batch(buf, off)
        assert counts.tolist() == [len(oracle_all(c, x)) for x in texts], (pat, counts.tolist())
        used += 1
    assert used >= 25


def test_c_abi_from_compiled_c():
    """tests/c/cabi_smoke.c, built by the CMake target (`__graft_entry__.build()`), calls the C ABI from compiled C:
    on a GPU box it runs the matching entry points and compares with the reference's documented answers"""
    import subprocess
    exe = os.path.join(os.path.dirname(os.path.abspath(__file__)), "c", "cabi_smoke")
    if not os.path.exists(exe):
        pytest.skip("cabi_smoke has not been built (cmake --build build)")
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "device checks ok" in r.stdout, r.stdout


def test_prefix_literal_patterns_under_the_budget_and_the_statemap_scan(monkeypatch):
    """`a.*[bc]` over 64 MiB of `a`: the pattern has the prefix literal `a`, Forgex's candidates are its occurrences --
    every byte -- and every attempt runs to the end of the text.  The candidate scan (K4, PREFIX form) runs under the work
    budget; past it the state-map scan answers (every match provably begins with the literal, so "every boundary" and
    "every occurrence" pick the same winner unless the winner is an overlong encoding -- then the candidate scan decides).
    `a.*b` itself also has the SUFFIX literal `b`: its candidate list is sequential (one thread replays it), but two
    parallel literal sweeps come first -- the prefix occurs, the suffix occurs nowhere: no match, at once."""
    import time
    import torch
    n = 64 << 20
    buf = torch.full((n,), ord("a"), dtype=torch.uint8, device="cuda")
    ft = torch.zeros(2, dtype=torch.int64, device="cuda")
    for pat, scan in ((b"a.*[bc]", 1), (b"a.*b", 0)):
        p = fx.Pattern(pat, "regex")
        inf = p.info()
        assert inf["literal_prefix_len"] == 1 and inf["prefix_scan"] == scan and inf["statemap"] == 1
        work = torch.zeros(p.buffer_work_bytes(n), dtype=torch.uint8, device="cuda")
        p.regex_buffer_dev(buf, n, ft, work)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        p.regex_buffer_dev(buf, n, ft, work)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        assert tuple(ft.cpu().tolist()) == (0, 0), pat
        assert dt < 0.25, "%r: %.3f s for 64 MiB" % (pat, dt)
        m = 2 << 20
        buf[m - 1] = ord("b")
        p.regex_buffer_dev(buf, m, ft, work)
        assert tuple(ft.cpu().tolist()) == (1, m), pat
        buf[m - 1] = ord("a")
    # parity, the state-map scan forced (FX_STATEMAP=2) and the default flow, incl. overlong starts with / without the literal elsewhere
    rng = np.random.default_rng(61)
    filler = bytes(rng.integers(0x20, 0x7F, size=150000, dtype=np.uint8)).replace(b"foo", b"f0o").replace(b"ERR", b"E_R").replace(b"key", b"k3y")
    texts = [b"xx foobar foobaz", b"fooba foobar", b"\xc1\xa6oobar", b"x\xc1\xa6oobar foobaz", b"x\xc1\xa6oobar fooba!", b"zzz", b"", b" ", b"fooba",
             filler + b"foobaz" + filler, filler + b"\xc1\xa6oobar" + filler, filler + b"\xc1\xa6oobar" + filler + b"fooba", filler,
             b"ERROR x timeout=12 ERROR timeout=5", filler + b"ERROR a timeout=777\n" + filler, b"a key=12 key=", b"aaab", b"ab", b"a\nb ab", b"aaa\nxxc"]
    for pat in [b"foo(bar|baz)", rb"ERROR.*timeout=\d+", b"key=[0-9]*", b"a.*[bc]", b"ab*", b"a.*b"]:
        q = fx.Pattern(pat, "regex")
        c = O.Compiled(pat, 0)
        for text in texts:
            if pat in (b"a.*[bc]", b"a.*b") and len(text) > 5000:
                continue                      # (quadratic for the oracle)
            arr = np.frombuffer(b"#" + text, dtype=np.uint8)[1:]
            exp = c.regex_buffer(np.ascontiguousarray(arr))
            for mode in ("2", "1"):
                monkeypatch.setenv("FX_STATEMAP", mode)
                assert q.regex_buffer(arr) == exp, (pat, text[:40], len(text), mode)


def test_work_budget_is_an_error_where_no_linear_stand_in_exists():
    """Patterns whose candidate list must be replayed in order (a bordered prefix literal such as `aa`, or a suffix
    literal) and patterns whose prefix literal is not provably neutral (a non-ASCII prefix) have no linear-time
    stand-in.  Forgex's loop is quadratic on `aa.*[xy]` over a run of `a`: the reference would grind for hours; the
    library stops after 16 byte steps per text byte and says so -- FX_ERR_WORK_BUDGET from the host forms, (-2, -2) from the
    _dev forms -- instead of holding the GPU.  Ordinary texts are untouched (parity with the oracle below)."""
    import time
    import torch
    from forgex_b200 import _lib as L
    n = 1 << 20
    cases = [(b"aa.*[xy]", b"a" * n, 0), ("é.*[xy]".encode(), "é".encode() * (n // 2), 1),
             (b"ab[^c]*cd", b"ab" * (n // 2) + b"ccd", 0)]
    for pat, text, scan in cases:
        p = fx.Pattern(pat, "regex")
        assert p.info()["prefix_scan"] == scan, pat
        arr = np.frombuffer(text, dtype=np.uint8)
        t0 = time.perf_counter()
        with pytest.raises(fx.ForgexError) as e:
            p.regex_buffer(arr)
        assert e.value.status == L.FX_ERR_WORK_BUDGET, pat
        assert time.perf_counter() - t0 < 20.0, pat
        with pytest.raises(fx.ForgexError) as e:
            p.regex_buffer_all(arr, capacity=4)
        assert e.value.status == L.FX_ERR_WORK_BUDGET, pat
        dev = torch.from_numpy(arr.copy()).cuda()
        ft = torch.zeros(2, dtype=torch.int64, device="cuda")
        work = torch.zeros(p.buffer_work_bytes(len(text)), dtype=torch.uint8, device="cuda")
        p.regex_buffer_dev(dev, len(text), ft, work)
        assert tuple(ft.cpu().tolist()) == (-2, -2), pat
        # the same handle right afterwards, on texts within the budget
        c = O.Compiled(pat, 0)
        for small in (text[:3000] + b"x", text[:2001], b"zz " + text[:40] + b" y cd", b"", b" "):
            s = np.frombuffer(b"#" + small, dtype=np.uint8)[1:]
            assert p.regex_buffer(s) == c.regex_buffer(np.ascontiguousarray(s)), (pat, small[:20])


def test_match_with_a_literal_that_is_blank_but_not_empty():
    """` +x`: the extracted prefix literal is one blank.  Fortran's `prefix /= ''` treats it as absent, but the gates
    of do_matching_exactly also compare LENGTHS (api_internal_m.F90:199-233): a text equal to the literal matches, a text
    shorter than it does not -- `' ' .match. ' +ab'` is true.  Such patterns must take the gated path for every string
    (found by the extended GPU fuzz, seed 14: the fast path walked the automaton and said false)."""
    texts = [b" ", b"", b"  ", b" ab", b"  ab.", b"ab", b" a", b"x ", b" ab ", b"ab ", b"ab  ", b"   ", b"a", b" abc.de"]
    buf, off = pack(texts)
    for pat in [rb" +(\w{2,3}\.?){1,}", b" +ab", b"ab +", b"  +", rb" \w+ ", b"a* ", b" a*", b" ", b"  ", b" ?", b"( |ab)"]:
        for op in ("match", "in"):
            p = fx.Pattern(pat, op)
            assert p.status == 0, pat
            o = 1 if op == "match" else 0
            c = O.Compiled(pat, o)
            got = p.match_batch(buf, off) if op == "match" else p.in_batch(buf, off)
            assert np.array_equal(got, c.bool_batch(o, buf, off)), (pat, op, got.tolist())
            for stride in (1, 2, 3):
                fb = np.frombuffer(b" a  b ab  a   aab ba", dtype=np.uint8)
                n = len(fb) // stride
                gotf = p.match_fixed(fb, n, stride) if op == "match" else p.in_fixed(fb, n, stride)
                assert np.array_equal(gotf, c.bool_fixed(o, fb, n, stride)), (pat, op, stride)


def test_value_forms_for_pure_callers_on_gpu():
    """fx_in_value / fx_match_value / fx_regex_sub (what a `pure` Fortran operator binds) against the oracle"""
    import ctypes as C
    lib = _lib.lib()
    cases = [(b"foo(bar|baz)", b"xx foobaz"), (b"ab+c", b"abbc"), (b"ab+c", b"abbd"), (b"^a", b"b\na"), (b" +ab", b" "), (b"(", b"abc"),
             ("[ぁ-ん]+".encode(), "xあいy".encode()), (b"a*", b""), (b"a", b" ")]
    for pat, text in cases:
        assert lib.fx_in_value(pat, len(pat), text, len(text)) == max(0, O.op_in(pat, text)), (pat, text)
        assert lib.fx_match_value(pat, len(pat), text, len(text)) == max(0, O.op_match(pat, text)), (pat, text)
        f, t, ln, st, rc = C.c_int64(7), C.c_int64(7), C.c_int64(7), C.c_int(7), C.c_int(7)
        lib.fx_regex_sub(pat, len(pat), text, len(text), C.byref(f), C.byref(t), C.byref(ln), C.byref(st), C.byref(rc))
        res, eln, ef, et, est = O.regex(pat, text)
        assert rc.value == 0 and st.value == est and ln.value == eln, (pat, text)
        if est == 0:
            assert (f.value, t.value) == (ef, et), (pat, text)
