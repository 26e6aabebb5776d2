"""Batch kernels at the shapes where 32-bit arithmetic breaks, and the span kernels' table forms forced on purpose.

Part 1: ragged and fixed-stride batches past 2^31 and 2^32 bytes, and `n` on both sides of 2^31.  The oracle cannot
walk 4.5 GiB, but the strings of a batch are independent: a seeded BLOCK (a prime number of strings, an odd byte
length) is answered once by the oracle and tiled on the device, behind a leading PAD string whose length places chosen
strings across byte 2^31 and byte 2^32.  Every string of the batch then has an exact expected answer, compared on the
device.  `test_tiled_construction_on_the_cpu` checks that premise with the oracle alone.

Part 2: the span kernels' template forms -- the forward table from global memory (FK 2), the classed table forced
(FK 1), the reverse tables in global memory (rs false) -- and pattern pairs on both sides of each host size threshold,
every side asserted, so that a change of the automata cannot quietly move a pair off its edge.

Every GPU test frees its device memory and skips (naming the size) when the shared device has too little free.
"""
import gc
import os
import random
import time

import numpy as np
import pytest

from tests import oracle_lib as O
from tools import synth

GiB = 1 << 30
B31, B32 = 1 << 31, 1 << 32
BLOCK_STRINGS = 10007                    # prime: copies of the block fall on different tile and warp cuts
PAD_BYTE = ord("7")                      # every attempt of the config patterns dies on it: the oracle is linear there
C1, C2, C3 = synth.PATTERNS["c1"], synth.PATTERNS["c2"], synth.PATTERNS["c3"]
UTF8_PIECES = [b"a", b"z", b" ", "あ".encode(), "ん".encode(), "α".encode(), "　".encode(), b"\x80", b"\xbf", b"\xc3", b"\xe3\x81",
               b"\xf0\x9f\x98", b"\xff", b"\xc0\x80", b"\xc1\xa1", b"\xe0\x81\xa1", b"\xef\xbf\xbf", b"\xf4\x90\x80\x81", b"\n", b"\r\n",
               b"_", b"7"]

SPAN_REV_SMEM_BYTES = 24 * 1024          # fx_cabi.cu: reverse tables staged in shared memory up to this size
SPAN_DIRECT_MAX_STATES = 127
SPAN_CLASSED_SMEM_BYTES = 96 * 1024
DIRECT_LIMIT_BYTES = 40 * 1024
SMEM_TABLE_LIMIT_BYTES = 160 * 1024
SPARSE_STATE_CAP = 2048


# ---- the block, the pad and the tiled batch (host side) -------------------------------------------------------
def pack(strings):
    offsets = np.zeros(len(strings) + 1, dtype=np.int64)
    np.cumsum([len(s) for s in strings], out=offsets[1:])
    return np.frombuffer(b"".join(strings), dtype=np.uint8).copy(), offsets


def make_block(nstrings=BLOCK_STRINGS, seed=1, long_strings=6):
    """a seeded ragged block of `nstrings` strings and an odd byte length: C2 / C3 / C1 lines, the UTF-8 / invalid /
    CRLF / overlong pieces, empty strings and lone blanks, HIT strings (true for `.in.` C2 and a C3 span), and a few
    strings of 6-40 KB, longer than a warp's tile, built so that every failing attempt of the config patterns dies at
    its first byte"""
    rng = np.random.default_rng(seed)
    k = nstrings // 6
    c2b, c2o = synth.gen_c2(k, seed_stream=seed)
    c3b, c3o = synth.gen_c3(k, seed_stream=seed)
    c1b, _, _ = synth.gen_c1(k, seed_stream=seed)
    strings = [bytes(c2b[c2o[i]:c2o[i + 1]]) for i in range(k)] + [bytes(c3b[c3o[i]:c3o[i + 1]]) for i in range(k)]
    strings += [bytes(c1b[8 * i:8 * i + 8]) for i in range(k)]
    strings += [b"".join(UTF8_PIECES[i] for i in rng.integers(0, len(UTF8_PIECES), size=int(m))) for m in rng.integers(0, 24, size=k)]
    words = ["αβγ", "ωψ", "あいう", "ぁ"]
    for i in range(k):
        pre = bytes(rng.integers(0x20, 0x7F, size=int(rng.integers(0, 60)), dtype=np.uint8)).replace(b"foo", b"f0o")
        strings.append(pre + b"foobar " + words[i % 4].encode() + b" w%d tail" % i)
    for i in range(long_strings):
        n = int(rng.integers(6000, 40000))
        body = b"7" * n
        if i % 2 == 0:
            body = body[:n // 2] + b"foobaz " + "ωψ".encode() + b" ab" + body[n // 2:]
        strings.append(body)
    while len(strings) < nstrings:
        strings.append([b"", b" ", b"", b"  ", b"\n"][len(strings) % 5])
    strings = strings[:nstrings]
    order = rng.permutation(nstrings)
    strings = [strings[i] for i in order]
    if sum(len(s) for s in strings) % 2 == 0:
        strings[int(np.argmax([len(s) for s in strings]))] += b"7"
    return pack(strings)


def oracle_counts(c, buf, offsets):
    """matches per string, the caller's loop: regex(), then regex() again on text(to+1:)"""
    out = np.zeros(len(offsets) - 1, dtype=np.int64)
    for i in range(len(offsets) - 1):
        pos, end = int(offsets[i]), int(offsets[i + 1])
        while True:
            f, t = c.regex_buffer(buf[pos:end])
            if f <= 0 or t <= 0:
                break
            out[i] += 1
            pos += t
    return out


def block_answers(buf, off):
    """the oracle's answers of every string of a block (also of the pad, passed as a one-string block)"""
    f, t = O.Compiled(C3, 0).regex_batch(buf, off)
    return {"in": O.Compiled(C2, 0).bool_batch(0, buf, off), "match": O.Compiled(C1, 1).bool_batch(1, buf, off),
            "from": f, "to": t, "count": oracle_counts(O.Compiled(C3, 0), buf, off)}


def locate(pos, pad, off):
    """(copy, string of the block) that holds byte `pos` of the tiled batch; (-1, 0) for the pad"""
    if pos < pad:
        return -1, 0
    L = int(off[-1])
    c, r = divmod(pos - pad, L)
    return c, int(np.searchsorted(off, r, side="right")) - 1


def straddles(boundary, pad, off, j):
    """does some copy of block string j hold both byte boundary-1 and byte boundary?"""
    c, jj = locate(boundary, pad, off)
    L = int(off[-1])
    return c >= 0 and jj == j and pad + c * L + int(off[j]) < boundary


def choose_pad(off, good, targets=(B32, B31), min_pad=1):
    """the shortest pad length >= min_pad for which a `good` string straddles every target byte.  Each (string, split)
    pair for the first target fixes the pad modulo the block length; the other targets are checked."""
    L = int(off[-1])
    lens = np.diff(off)
    best = None
    for j in np.nonzero(good & (lens >= 2))[0]:
        for s in range(1, int(lens[j])):
            pad = (targets[0] - int(off[j]) - s) % L
            while pad < min_pad:
                pad += L
            if best is not None and pad >= best:
                continue
            if all(good[locate(t, pad, off)[1]] and straddles(t, pad, off, locate(t, pad, off)[1]) for t in targets):
                best = pad
    assert best is not None, "no pad places good strings across every target"
    return best


def tiled_host(buf, off, pad, copies):
    """the tiled batch on the host (small sizes only): pad string, then `copies` copies of the block"""
    L = int(off[-1])
    tb = np.concatenate([np.full(pad, PAD_BYTE, dtype=np.uint8), np.tile(buf, copies)])
    toff = np.concatenate([[0, pad], (pad + np.arange(copies, dtype=np.int64)[:, None] * L + off[None, 1:]).reshape(-1)])
    return tb, toff.astype(np.int64)


def pad_answers(pad):
    return block_answers(np.full(pad, PAD_BYTE, dtype=np.uint8), np.array([0, pad], dtype=np.int64))


# ---- part 3: the construction, checked by the oracle alone ------------------------------------------------------
def test_tiled_construction_on_the_cpu():
    """the oracle run on a whole small tiled batch equals the tiled oracle answers of the block (strings are
    independent), for `.in.`, `.match.`, spans and counts; and the pad arithmetic places chosen strings across chosen
    bytes"""
    buf, off = make_block(101, seed=3, long_strings=2)
    L = int(off[-1])
    assert L % 2 == 1 and len(off) - 1 == 101
    ans = block_answers(buf, off)
    good = (ans["in"] == 1) & (ans["from"] > 0)
    assert good.sum() >= 5
    copies = 4
    targets = (3 * L + L // 3, L + L // 2)        # two bytes inside the batch, like 2^32 and 2^31 at full size
    pad = choose_pad(off, good, targets)
    assert 0 < pad < 2 * L
    for t in targets:
        c, j = locate(t, pad, off)
        assert 0 <= c < copies and good[j] and straddles(t, pad, off, j)
        assert pad + c * L + off[j] < t < pad + c * L + off[j + 1]
    tb, toff = tiled_host(buf, off, pad, copies)
    assert len(toff) == 2 + copies * 101 and toff[-1] == len(tb) == pad + copies * L
    whole = block_answers(tb, toff)
    pa = pad_answers(pad)
    for k in ("in", "match", "from", "to", "count"):
        exp = np.concatenate([pa[k], np.tile(ans[k], copies)])
        assert np.array_equal(whole[k], exp), k
    # the straddling strings are the ones the arithmetic named
    for t in targets:
        i = int(np.searchsorted(toff, t, side="right")) - 1
        assert toff[i] < t < toff[i + 1] and good[(i - 1) % 101]
    assert locate(pad - 1, pad, off) == (-1, 0) and locate(pad, pad, off) == (0, 0)


# ---- device helpers ---------------------------------------------------------------------------------------------
@pytest.fixture
def device():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    yield torch
    gc.collect()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def need_free(torch, nbytes):
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip("needs %.1f GiB of free device memory, %.1f GiB free" % (nbytes / GiB, free / GiB))


def tile_into(dst, src):
    """fill `dst` with copies of `src` (device tensors, one dimension), the last one cut short"""
    L = src.numel()
    full = dst.numel() // L
    if full:
        dst[:full * L].view(full, L).copy_(src.unsqueeze(0).expand(full, L))
    rest = dst.numel() - full * L
    if rest:
        dst[full * L:].copy_(src[:rest])
    return dst


def tiled_expect(torch, pad_val, block_vals, n, dtype):
    e = torch.empty(n, dtype=dtype, device="cuda")
    e[0] = int(pad_val)
    tile_into(e[1:], torch.from_numpy(np.ascontiguousarray(block_vals).astype(np.int64 if dtype == torch.int64 else np.uint8)).cuda())
    return e


class Ragged:
    """pad + whole copies of the block, on the device, at least `min_bytes` long"""

    def __init__(self, torch, min_bytes):
        buf, off = make_block()
        self.hbuf, self.hoff = buf, off
        self.L, self.m = int(off[-1]), len(off) - 1
        self.ans = block_answers(buf, off)
        self.good = (self.ans["in"] == 1) & (self.ans["from"] > 0)
        self.pad = choose_pad(off, self.good)
        self.pans = pad_answers(self.pad)
        self.reps = -(-(min_bytes - self.pad) // self.L)
        self.total = self.pad + self.reps * self.L
        self.n = 1 + self.reps * self.m
        self.buf = torch.empty(self.total, dtype=torch.uint8, device="cuda")
        self.buf[:self.pad].fill_(PAD_BYTE)
        tile_into(self.buf[self.pad:], torch.from_numpy(buf).cuda())
        self.off = torch.empty(self.n + 1, dtype=torch.int64, device="cuda")
        self.off[0] = 0
        self.off[1] = self.pad
        base = self.pad + torch.arange(self.reps, dtype=torch.int64, device="cuda")[:, None] * self.L
        self.off[2:].view(self.reps, self.m).copy_(base + torch.from_numpy(off[1:]).cuda()[None, :])
        self.torch = torch

    def expect(self, key):
        t = self.torch
        return tiled_expect(t, self.pans[key][0], self.ans[key], self.n, t.uint8 if key in ("in", "match") else t.int64)

    def index_at(self, pos):
        """batch index of the string that holds byte `pos`"""
        c, j = locate(pos, self.pad, self.hoff)
        return 0 if c < 0 else 1 + c * self.m + j


# ---- part 1: ragged batches past 2^32 bytes ---------------------------------------------------------------------
@pytest.mark.gpu
def test_ragged_batch_past_4_gib(device, monkeypatch):
    """4.5 GiB of tiled strings: every batch kernel against the oracle's tiled answers, on every string"""
    import forgex_b200 as fx
    torch = device
    need_free(torch, 20 * GiB)
    R = Ragged(torch, (4 << 30) + (512 << 20))
    n, total = R.n, R.total
    assert total >= 4.5 * GiB and total > B32
    # the straddles: good strings (`.in.` true, a span) hold bytes on both sides of 2^31 and of 2^32
    straddle = {}
    for t in (B31, B32):
        i = R.index_at(t)
        o0, o1 = int(R.off[i].item()), int(R.off[i + 1].item())
        assert o0 < t < o1 and o1 - o0 >= 2, (t, o0, o1)
        straddle[t] = i
    exp_in, exp_match = R.expect("in"), R.expect("match")
    exp_f, exp_t = R.expect("from"), R.expect("to")
    for t, i in straddle.items():
        assert int(exp_in[i].item()) == 1 and int(exp_f[i].item()) > 0, t
    out = torch.empty(n, dtype=torch.uint8, device="cuda")

    p = fx.Pattern(C2, "in")
    p.in_batch_dev(R.buf, R.off, n, total, out)
    assert p.info()["sparse_used"] == 1                              # K2c
    assert torch.equal(out, exp_in), torch.nonzero(out != exp_in)[:8].tolist()
    monkeypatch.setenv("FX_SPARSE", "0")
    out.fill_(7)
    p.in_batch_dev(R.buf, R.off, n, total, out)
    assert p.info()["sparse_used"] == 0                              # K2
    assert torch.equal(out, exp_in), torch.nonzero(out != exp_in)[:8].tolist()
    monkeypatch.delenv("FX_SPARSE")

    q = fx.Pattern(C1, "match")
    out.fill_(7)
    q.match_batch_dev(R.buf, R.off, n, total, out)
    assert q.info()["sparse_used"] == 0                              # K2
    assert torch.equal(out, exp_match), torch.nonzero(out != exp_match)[:8].tolist()
    assert int(exp_match.sum().item()) > 0

    r = fx.Pattern(C3, "regex")
    assert r.info()["statemap"] == 1 and r.span_tables() is not None
    f = torch.empty(n, dtype=torch.int64, device="cuda")
    to = torch.empty(n, dtype=torch.int64, device="cuda")
    for linear in ("1", "0"):                                        # K3f, then K3
        monkeypatch.setenv("FX_SPAN_LINEAR", linear)
        f.fill_(-7); to.fill_(-7)
        r.regex_batch_dev(R.buf, R.off, n, total, f, to)
        assert torch.equal(f, exp_f) and torch.equal(to, exp_t), (linear, torch.nonzero((f != exp_f) | (to != exp_t))[:8].tolist())
    monkeypatch.delenv("FX_SPAN_LINEAR")
    del f, to
    counts = torch.full((n,), -7, dtype=torch.int64, device="cuda")
    r.regex_count_batch_dev(R.buf, R.off, n, total, counts)
    exp_c = R.expect("count")
    assert torch.equal(counts, exp_c), torch.nonzero(counts != exp_c)[:8].tolist()
    del counts, exp_c, exp_f, exp_t

    # the host-pointer form a Fortran caller uses: numpy in, numpy out (the library stages the batch itself)
    hbuf, hoff = R.buf.cpu().numpy(), R.off.cpu().numpy()
    h = fx.Pattern(C2, "in")
    got = h.in_batch(hbuf, hoff)
    assert h.info()["sparse_used"] == 1
    assert np.array_equal(got, exp_in.cpu().numpy())
    h.close()
    del hbuf, hoff, got

    # a sub-batch at large offsets: a slice of the offsets with the whole buffer (offsets are absolute positions)
    # for the NFA engine, too slow for the whole batch
    lo = straddle[B32] - 1500
    sub = R.off[lo:lo + 3001]
    ns = 3000
    assert int(sub[0].item()) < B32 < int(sub[-1].item())
    so = torch.empty(ns, dtype=torch.uint8, device="cuda")
    monkeypatch.setenv("FX_STATE_CAP", "3")                          # the NFA engine
    for pat, op, exp in ((C2, "in", exp_in), (C1, "match", exp_match)):
        e = fx.Pattern(pat, op)
        assert e.info()["nfa_engine"] == 1
        so.fill_(7)
        getattr(e, op + "_batch_dev")(R.buf, sub, ns, total, so)
        assert torch.equal(so, exp[lo:lo + ns]), ("nfa", op)
    e = fx.Pattern(C3, "regex")
    assert e.info()["nfa_engine"] == 1
    sf = torch.empty(ns, dtype=torch.int64, device="cuda")
    st = torch.empty(ns, dtype=torch.int64, device="cuda")
    e.regex_batch_dev(R.buf, sub, ns, total, sf, st)
    ef = torch.from_numpy(np.concatenate([R.pans["from"], np.tile(R.ans["from"], 2 + (lo + ns) // R.m)])[lo:lo + ns]).cuda()
    et = torch.from_numpy(np.concatenate([R.pans["to"], np.tile(R.ans["to"], 2 + (lo + ns) // R.m)])[lo:lo + ns]).cuda()
    assert torch.equal(sf, ef) and torch.equal(st, et), "nfa regex"
    assert int((ef > 0).sum().item()) > 100


# ---- part 1: fixed-stride batches --------------------------------------------------------------------------------
def fixed_block(kind, m=BLOCK_STRINGS):
    """m rows of a fixed-stride block (host) and the stride"""
    rng = np.random.default_rng(21)
    if kind == "c1":
        b, _, stride = synth.gen_c1(m, seed_stream=5)
        return b.copy(), stride
    if kind == "c5":
        b, _, stride = synth.gen_c5(m, seed_stream=5)
        b = b.copy()
        b[5 * 64 + 7:5 * 64 + 9] = (0xC3, 0xA9)
        b[11 * 64 + 3:11 * 64 + 5] = (0xC1, 0xA1)
        return b, stride
    if kind == "c2f":
        stride = 160
        b = rng.integers(0x20, 0x7F, size=m * stride, dtype=np.uint8)
        for k in rng.integers(0, m * stride - 8, size=m // 4):
            b[k:k + 6] = np.frombuffer(b"foobar" if k & 1 else b"fooba!", dtype=np.uint8)
        b[rng.random(b.size) < 0.002] = 0xC1
        return b, stride
    stride = 2                                   # kind == "ab"
    alphabet = np.frombuffer(b"abc x\xc3", dtype=np.uint8)
    b = alphabet[rng.choice(len(alphabet), size=m * stride, p=[0.2, 0.2, 0.2, 0.15, 0.15, 0.1])]
    return b.copy(), stride


def plant_across(block, stride, m, boundary, text):
    """write `text` into the block row that lands on `boundary` in the tiled batch, across the boundary"""
    row, inrow = divmod(boundary, stride)
    at = (row % m) * stride + inrow - len(text) // 2
    assert (row % m) * stride <= at and at + len(text) <= (row % m + 1) * stride
    block[at:at + len(text)] = np.frombuffer(text, dtype=np.uint8)


def run_fixed(torch, fx, pattern, op, block, stride, n, residency="auto"):
    m = len(block) // stride
    exp_h = O.Compiled(pattern, 1 if op == "match" else 0).bool_fixed(1 if op == "match" else 0, block, m, stride)
    d_block = torch.from_numpy(block).cuda()
    buf = tile_into(torch.empty(n * stride, dtype=torch.uint8, device="cuda"), d_block)
    exp = tile_into(torch.empty(n, dtype=torch.uint8, device="cuda"), torch.from_numpy(exp_h).cuda())
    out = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
    p = fx.Pattern(pattern, op, residency=residency)
    getattr(p, op + "_fixed_dev")(buf, n, stride, out)
    ok = torch.equal(out, exp)
    bad = [] if ok else torch.nonzero(out != exp)[:8].flatten().tolist()
    info = p.info()
    del buf, out
    return ok, bad, info, exp_h


@pytest.mark.gpu
def test_fixed_stride_past_4_gib(device):
    """K1 (C1's shape, the four-strings-per-thread VEC=8 branch), K2c's fixed form (stride 160) and K1c from global
    memory (the C5 pattern, stride 64), each over more than 2^32 bytes"""
    import forgex_b200 as fx
    torch = device
    need_free(torch, 7 * GiB)
    block, stride = fixed_block("c1")
    m = len(block) // stride
    n = (B32 // stride) + 12345
    for b in (B31, B32):                                             # rows starting exactly at 2^31 / 2^32, and before them
        r = b // stride
        block[(r % m) * stride:(r % m + 1) * stride] = np.frombuffer(b"123-4567", dtype=np.uint8)
        block[((r - 1) % m) * stride:((r - 1) % m + 1) * stride] = np.frombuffer(b"987-6543", dtype=np.uint8)
    ok, bad, info, exp_h = run_fixed(torch, fx, C1, "match", block, stride, n)
    assert ok, ("K1 stride 8", bad)
    assert info["sparse_used"] == 0 and info["compact_used"] == 0 and n * stride > B32 and 0 < exp_h.mean() < 1

    block, stride = fixed_block("c2f")
    m = len(block) // stride
    n = B32 // stride + 40000
    for b in (B31, B32):
        plant_across(block, stride, m, b, b"foobar")
    ok, bad, info, exp_h = run_fixed(torch, fx, C2, "in", block, stride, n)
    assert ok, ("K2c stride 160", bad)
    assert info["sparse_used"] == 1 and n * stride > B32
    for b in (B31, B32):
        assert exp_h[(b // stride) % m] == 1

    block, stride = fixed_block("c5")
    n = B32 // stride + 777
    ok, bad, info, exp_h = run_fixed(torch, fx, synth.PATTERNS["c5"], "in", block, stride, n, residency="global")
    assert ok, ("K1c stride 64", bad)
    assert info["compact_used"] == 2 and n * stride > B32 and 0 < exp_h.mean() < 1


@pytest.mark.gpu
def test_fixed_stride_count_on_both_sides_of_2_31(device):
    """stride 2 `.in.`: K2c takes fixed-stride batches of fewer than 2^31 strings, K1 the rest"""
    import forgex_b200 as fx
    torch = device
    need_free(torch, 9 * GiB)
    block, stride = fixed_block("ab")
    pat = b"[ab][bc]"
    for n, sparse in ((B31 - 1, 1), (B31 + 4097, 0)):
        ok, bad, info, exp_h = run_fixed(torch, fx, pat, "in", block, stride, n)
        assert info["sparse"] == 1 and info["sparse_used"] == sparse, (n, info["sparse_used"])
        assert ok, (n, bad)
        assert 0 < exp_h.mean() < 1
        gc.collect()
        torch.cuda.empty_cache()


# ---- part 1: one string of more than 2 GiB ----------------------------------------------------------------------
@pytest.mark.gpu
def test_one_string_past_2_gib(device, monkeypatch):
    """a string of 2^31 + 2^20 bytes inside a small ragged batch, its only match planted past 2^31 within it.  K3f walks
    a string of 2 GiB or more with the anchored emulation (64-bit positions); `.in.` with FX_SPARSE=0 with K2's walk
    from global memory.  Both are one thread over the whole string; their times are printed."""
    import forgex_b200 as fx
    torch = device
    need_free(torch, 3 * GiB)
    big = B31 + (1 << 20)
    plant = b"foobar " + "αβγ".encode() + b" xy"
    at = big - 4096                                                  # past 2^31 within the string
    assert at > B31
    head = [b"foobar \xce\xb1\xce\xb2 ab", b"", b" ", b"7" * 9000]
    tail = [b"x foobaz", b"", "ωψ aa".encode()]
    lens = [len(s) for s in head] + [big] + [len(s) for s in tail]
    off = np.zeros(len(lens) + 1, dtype=np.int64)
    np.cumsum(lens, out=off[1:])
    total = int(off[-1])
    buf = torch.full((total,), PAD_BYTE, dtype=torch.uint8, device="cuda")
    hb = b"".join(head)
    buf[:len(hb)] = torch.from_numpy(np.frombuffer(hb, dtype=np.uint8).copy()).cuda()
    tb = b"".join(tail)
    buf[total - len(tb):] = torch.from_numpy(np.frombuffer(tb, dtype=np.uint8).copy()).cuda()
    o_big = int(off[len(head)])
    buf[o_big + at:o_big + at + len(plant)] = torch.from_numpy(np.frombuffer(plant, dtype=np.uint8).copy()).cuda()
    # expected: the same strings with the long one cut to a short analog (same bytes around the plant), span shifted
    short_pre = 100
    short = b"7" * short_pre + plant + b"7" * (big - at - len(plant))
    strings = head + [short] + tail
    sbuf, soff = pack(strings)
    ef, et = O.Compiled(C3, 0).regex_batch(sbuf, soff)
    ein = O.Compiled(C2, 0).bool_batch(0, sbuf, soff)
    k = len(head)
    assert ef[k] == short_pre + 7 + 1 and et[k] > ef[k] and ein[k] == 1
    ef[k] += at - short_pre
    et[k] += at - short_pre
    assert ef[k] > B31
    d_off = torch.from_numpy(off).cuda()
    n = len(lens)
    times = {}

    r = fx.Pattern(C3, "regex")
    f = torch.full((n,), -7, dtype=torch.int64, device="cuda")
    t = torch.full((n,), -7, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r.regex_batch_dev(buf, d_off, n, total, f, t)
    torch.cuda.synchronize()
    times["regex K3f emulation"] = time.perf_counter() - t0
    assert f.cpu().tolist() == ef.tolist() and t.cpu().tolist() == et.tolist(), (f.cpu().tolist(), ef.tolist(), t.cpu().tolist(), et.tolist())

    monkeypatch.setenv("FX_SPARSE", "0")
    p = fx.Pattern(C2, "in")
    out = torch.full((n,), 7, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    p.in_batch_dev(buf, d_off, n, total, out)
    torch.cuda.synchronize()
    times[".in. K2 global walk"] = time.perf_counter() - t0
    assert p.info()["sparse_used"] == 0
    assert out.cpu().tolist() == ein.tolist()
    print("\none string of %d bytes: %s" % (big, ", ".join("%s %.2f s" % kv for kv in times.items())))


# ---- part 2: the span table forms -------------------------------------------------------------------------------
def span_fk(sp):
    """(forward-table bytes of the classed form, reverse-table bytes as launch_regex_ragged counts them, rs)"""
    d = sp["direct"]
    ncls = len({d[:, b].tobytes() for b in range(256)})
    shift = 0
    while (1 << shift) < ncls:
        shift += 1
    classed = (d.shape[0] << shift) * 2
    rbytes = sp["rdelta"].nbytes + 1024 + (0 if sp["rmixed"] is None else sp["rmixed"].nbytes)
    return classed, rbytes, sp["rpage"] is not None and rbytes <= SPAN_REV_SMEM_BYTES


def corpus_texts():
    from tests.test_host_tables import gen_text
    rng = random.Random(77)
    nrng = np.random.default_rng(78)
    texts = [gen_text(rng) for _ in range(600)]
    texts += [b"".join(UTF8_PIECES[i] for i in nrng.integers(0, len(UTF8_PIECES), size=int(k))) for k in nrng.integers(0, 24, size=600)]
    c3b, c3o = synth.gen_c3(300, seed_stream=9)
    texts += [bytes(c3b[c3o[i]:c3o[i + 1]]) for i in range(300)]
    texts += [b"", b" ", b"", b"abc\r\n", b"abc\n", b"\r\n", b"a\r\nb", b"ab\r", "αβ\r\n".encode(), b"x" * 300, b"ab" * 200 + b"\r\n"]
    return texts


def corpus_patterns():
    from tests.test_host_tables import gen_pattern
    rng = random.Random(4711)
    pats = [C3, synth.PATTERNS["c4"], C2, C1, synth.PATTERNS["c5"],
            b"^abc", b"abc$", b"^abc$", b"^$", b"^", b"$", rb"\s\S+$", rb"[^a]{2,3}$", rb"^\w", b"(|^)a", b"ab\r?$",
            "[ぁ-ん]+a".encode(), "[α-ω]+".encode(), b".+", rb"\S+", b"[a-z]+r", b"(a|b)*a(a|b){3}", b"a{1,7}", b"(ab)+", b"[ab]{2,3}"]
    return pats + [gen_pattern(rng).encode() for _ in range(40)]


@pytest.mark.gpu
def test_span_forms_forced_against_the_oracle(device, monkeypatch):
    """residency="global" on `regex` handles forces the forward table into global memory: K3f FK 2 (regex_batch and the
    count kernel), K5 FK 2 (FX_STATEMAP=2) and K4 KIND 3 (the default flow); FX_SPAN_FK=1 forces the classed table
    wherever it fits 96 KB"""
    import forgex_b200 as fx
    from forgex_b200 import _lib
    texts = corpus_texts()
    buf, off = pack(texts)
    joined = np.frombuffer(b"\n".join(texts[:300]), dtype=np.uint8)
    used = {"span": 0, "fk1": 0, "statemap": 0}
    for pat in corpus_patterns():
        p = fx.Pattern(pat, "regex", residency="global")
        if p.status != 0:
            continue
        c = O.Compiled(pat, 0)
        ef, et = c.regex_batch(buf, off)
        f, t = p.regex_batch(buf, off)
        assert np.array_equal(f, ef) and np.array_equal(t, et), (pat, np.nonzero((f != ef) | (t != et))[0][:5])
        info = p.info()
        assert info["residency"] == _lib.FX_TABLE_GLOBAL, pat
        assert np.array_equal(p.regex_count_batch(buf, off), oracle_counts(c, buf, off)), (pat, "counts")
        exp = c.regex_buffer(joined)
        if info["statemap"] and not info["literal_only"] and not info["literal_prefix_len"]:
            monkeypatch.setenv("FX_STATEMAP", "2")
            assert p.regex_buffer(joined) == exp, (pat, "statemap")
            assert p.info()["statemap_used"] == 1
            used["statemap"] += 1
        monkeypatch.delenv("FX_STATEMAP", raising=False)
        assert p.regex_buffer(joined) == exp, (pat, "buffer")
        sp = p.span_tables()
        if sp is None:
            continue
        used["span"] += 1
        if span_fk(sp)[0] <= SPAN_CLASSED_SMEM_BYTES:
            monkeypatch.setenv("FX_SPAN_FK", "1")
            q = fx.Pattern(pat, "regex")
            f, t = q.regex_batch(buf, off)
            assert np.array_equal(f, ef) and np.array_equal(t, et), (pat, "FK 1")
            monkeypatch.delenv("FX_SPAN_FK")
            used["fk1"] += 1
    assert used["span"] >= 30 and used["fk1"] >= 30 and used["statemap"] >= 20, used


def ab_texts(seed, n=2500, maxlen=300, extra=b"c "):
    """texts over [ab] (some `c` / blank cuts, so matches start inside strings), a few longer than a warp's tile"""
    rng = np.random.default_rng(seed)
    alphabet = np.frombuffer(b"ab" + extra, dtype=np.uint8)
    p = np.array([0.47, 0.47] + [0.06 / len(extra)] * len(extra))
    texts = [bytes(alphabet[rng.choice(len(alphabet), size=int(k), p=p)]) for k in rng.integers(0, maxlen, size=n)]
    texts += [b"", b" ", b"a", b"b" * 40 + b"a" * 3, bytes(alphabet[rng.choice(len(alphabet), size=7000, p=p)]),
              bytes(alphabet[rng.choice(len(alphabet), size=9001, p=p)])]
    return pack(texts)


@pytest.mark.gpu
def test_reverse_tables_in_global_memory(device):
    """(a|b){k}a(a|b)*: k = 10 keeps the reverse tables in shared memory (rs true), k = 11 does not (rs false, the
    reverse walk reads them from global memory); a second pattern past 24 KB as well"""
    import forgex_b200 as fx
    buf, off = ab_texts(5)
    sides = []
    for pat in (b"(a|b){10}a(a|b)*", b"(a|b){11}a(a|b)*", b"[abc]{11}[ab][abc]*"):
        p = fx.Pattern(pat, "regex")
        sp = p.span_tables()
        classed, rbytes, rs = span_fk(sp)
        sides.append(rs)
        f, t = p.regex_batch(buf, off)
        ef, et = O.Compiled(pat, 0).regex_batch(buf, off)
        assert np.array_equal(f, ef) and np.array_equal(t, et), (pat, rbytes, np.nonzero((f != ef) | (t != et))[0][:5])
        assert 0.2 < (ef > 0).mean() < 1 and (ef > 1).sum() > 100, pat
    assert sides == [True, False, False], sides


@pytest.mark.gpu
def test_size_threshold_pairs(device, monkeypatch):
    """a pattern pair on each side of every host size threshold, the side asserted, both against the oracle"""
    import forgex_b200 as fx
    from forgex_b200 import _lib
    buf, off = ab_texts(9, n=3000, maxlen=80, extra=b"c")

    def check_bool(p, pat, op):
        got = p.match_batch(buf, off) if op == "match" else p.in_batch(buf, off)
        o = 1 if op == "match" else 0
        exp = O.Compiled(pat, o).bool_batch(o, buf, off)
        assert np.array_equal(got, exp), (pat, op)
        return exp

    def check_regex(p, pat):
        f, t = p.regex_batch(buf, off)
        ef, et = O.Compiled(pat, 0).regex_batch(buf, off)
        assert np.array_equal(f, ef) and np.array_equal(t, et), pat
        assert (ef > 0).sum() > 10, pat

    # 255 / 256 byte states: the one-byte 256-column table (u8) or the classed table in shared memory
    monkeypatch.setenv("FX_SPARSE", "0")
    for pat, op, small in ((b"[ab]{62}c", "match", True), (b"[ab]{63}c", "match", False),
                           (b"[ab]{60}c", "in", True), (b"[ab]{61}c", "in", False)):
        p = fx.Pattern(pat, op)
        states = p.info()["byte_states"]
        assert (states <= 255) == small and 250 <= states <= 260, (pat, states)
        check_bool(p, pat, op)
        assert p.info()["direct"] == (1 if small else 0) and p.info()["residency"] == _lib.FX_TABLE_SMEM, pat
    monkeypatch.delenv("FX_SPARSE")
    # 127 / 128 span states: forward table as 256-column rows (FK 0) or classed (FK 1)
    for pat, small in ((b"[ab]{29}c", True), (b"[ab]{30}c", False)):
        p = fx.Pattern(pat, "regex")
        ns = p.span_tables()["direct"].shape[0]
        assert (ns <= SPAN_DIRECT_MAX_STATES) == small and 120 <= ns <= 135, (pat, ns)
        check_regex(p, pat)
    # 40 KB: the 256-column flag-bit table in shared memory (K3 walks it) or the classed one
    monkeypatch.setenv("FX_SPAN_LINEAR", "0")
    for pat, small in ((b"[ab]{18}c", True), (b"[ab]{19}c", False)):
        p = fx.Pattern(pat, "regex")
        db = p.info()["direct_bytes"]
        assert (db <= DIRECT_LIMIT_BYTES) == small and abs(db - DIRECT_LIMIT_BYTES) < 2048, (pat, db)
        check_regex(p, pat)
        assert p.info()["direct"] == (1 if small else 0), pat
    monkeypatch.delenv("FX_SPAN_LINEAR")
    # 160 KB: the classed table in shared memory or in global memory
    for pat, small in ((b"(a|b)*a(a|b){9}", True), (b"(a|b)*a(a|b){10}", False)):
        p = fx.Pattern(pat, "match")
        tb = p.info()["table_bytes"]
        assert (tb <= SMEM_TABLE_LIMIT_BYTES) == small and p.info()["byte_states"] > 255, (pat, tb)
        assert 0 < check_bool(p, pat, "match").mean() < 1
        assert p.info()["residency"] == (_lib.FX_TABLE_SMEM if small else _lib.FX_TABLE_GLOBAL), pat
    # 2048 anchored states: a prefix-less `.in.` pattern takes K2c only when its anchored automaton fits
    for pat, small in ((b"(a|b)*a(a|b){9}", True), (b"(a|b)*a(a|b){10}", False)):
        cp = fx.Pattern(pat, "regex").info()["cp_states"]
        assert (cp <= SPARSE_STATE_CAP) == small and abs(cp - SPARSE_STATE_CAP) < 1100, (pat, cp)
        p = fx.Pattern(pat, "in")
        assert p.info()["sparse"] == (1 if small else 0), pat
        check_bool(p, pat, "in")
        assert p.info()["sparse_used"] == (1 if small else 0), pat
