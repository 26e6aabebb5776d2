"""K2c's two-byte sweep filter at the edges of its units, rows, groups, segments and tiles, against the oracle and
against the kernel chosen with the sparse path switched off (FX_SPARSE=0).

The sweep reads 32-byte units (unit k of a tile starts at the tile's first byte rounded down to 32, plus 32 k); 32
lanes take 32 consecutive units per row, a group is 4 rows, a segment 1024 units.  The pair test of a unit's last
byte looks at the next unit's first byte in another lane or row, or assumes a match where that unit is not loaded.
These batches put first bytes and pairs on exactly those cuts: every byte offset 0..63 of a unit pair, after every
base misalignment 0..31 of the batch, with winners, near misses and a string ending in the first byte followed by a
string that starts with the rest of a winner (which must not win).

Every pattern here with a sparse sweep takes the HIGH form (its first byte's overlong encodings are lead bytes), and
`f[oé]` also lets lead bytes follow the first byte.  The !HIGH pair form is reached by no pattern of the reference's
syntax; tests/test_sparse_pair_filter.py checks it on a model.
"""
import numpy as np
import pytest

import forgex_b200 as fx
from tests import oracle_lib as O

pytestmark = pytest.mark.gpu

PATTERNS = [b"foo(bar|baz)", "f[oé]".encode(), "f(o|é)(bar|baz)".encode()]
PLANTS = [b"foobar", b"foobaz", b"foobax", b"fooba", b"fo", b"f", "fé".encode(), "féba".encode(), b"fx", b"ffoobar",
          b"fobar", "fébaz".encode(), b"fobax"]
BACKGROUND = np.array([c for c in range(0x20, 0x7F) if c not in b"fo"], dtype=np.uint8)


def pack(strings):
    offsets = np.zeros(len(strings) + 1, dtype=np.int64)
    np.cumsum([len(s) for s in strings], out=offsets[1:])
    return np.frombuffer(b"".join(strings), dtype=np.uint8).copy(), offsets


def background(rng, n):
    return bytes(BACKGROUND[rng.integers(0, BACKGROUND.size, size=n)])


def plant(s, pos, lit):
    pos = max(0, min(pos, len(s) - len(lit)))
    return s[:pos] + lit + s[pos + len(lit):]


def make_edge_batches():
    """(name, buf, offsets): seeded ragged batches with pairs on the sweep's cuts"""
    rng = np.random.default_rng(2024)
    out = []
    # every byte offset 0..63 relative to a 32-byte unit, after a pad of 0..31 bytes; strings of 72 bytes
    for mis in range(32):
        strings = [background(rng, mis)]
        for i in range(256):
            s = background(rng, 72)
            lit = PLANTS[i % len(PLANTS)]
            j = (i * 7) % 64
            strings.append(plant(s, j, lit) if j + len(lit) <= 72 else s[:j] + lit[:72 - j])
        strings[-1] = strings[-1][:-6] + b"foobar" if mis % 2 else strings[-1][:-1] + b"f"   # the end of the buffer
        out.append(("offsets/mis=%d" % mis, *pack(strings)))
    # a string ending in "f" followed by one starting with "oobar" (must not win), at every offset of the cut
    strings = []
    for j in range(64):
        strings.append(background(rng, 40 + j) + b"f")
        strings.append(b"oobar" + background(rng, 20))
        strings.append(background(rng, 32 - (j % 32)) + "f".encode())
        strings.append("é".encode() + background(rng, 9))
    out.append(("split-string", *pack(strings)))
    # strings of 2048 bytes: 32 strings (64 KB) per tile, so a tile holds two segments of 1024 units; one pair per
    # string across a unit cut (lane 30 -> 31, lane 31 -> the next row, a group's last row -> the next group, the
    # segment's last unit -> the next segment, the tile's last unit -> the next tile)
    for mis in (0, 1, 17, 31):
        strings = [background(rng, mis)] if mis else []
        for i in range(640):
            s = background(rng, 2048)
            lit = PLANTS[rng.integers(0, len(PLANTS))]
            start = sum(len(x) for x in strings)
            kind = i % 4
            if kind == 0:
                u = int(rng.integers(0, 64))                   # any unit cut of the string
            elif kind == 1:
                u = 63 if i % 8 == 1 else 31                   # the string's middle and last unit cuts
            elif kind == 2:
                u = int(rng.integers(0, 16)) * 4 + 3           # a group's last row boundary (mis = 0)
            else:
                u = -1
            if u >= 0:
                pos = (start // 32 + u) * 32 + 31 - start - int(rng.integers(0, 2))   # 'f' on a unit's last bytes
                if 0 <= pos < 2048:
                    s = s[:pos] + lit[:2048 - pos] + s[pos + len(lit[:2048 - pos]):]
            strings.append(s[:2048])
        out.append(("tiles/mis=%d" % mis, *pack(strings)))
    # one string per tile, longer than a segment: cuts at 1024-unit boundaries inside a string
    strings = []
    for i in range(12):
        n = 1024 * 32 * (1 + i % 3) + int(rng.integers(0, 64))
        s = bytearray(background(rng, n))
        cut = 1024 * 32 * (1 + int(rng.integers(0, 1 + i % 3))) - 1 - (i % 2) - len(strings[-1] if strings else b"") % 32
        cut = max(0, min(cut, n - 6))
        lit = [b"foobar", b"foobax", b"fooba "][i % 3]
        s[cut:cut + len(lit)] = lit
        strings.append(bytes(s))
    out.append(("long", *pack(strings)))
    return out


@pytest.fixture(scope="module")
def edge_batches():
    return make_edge_batches()


def check_ragged(monkeypatch, pat, buf, off, name):
    exp = O.Compiled(pat, 0).bool_batch(0, buf, off)
    monkeypatch.setenv("FX_SPARSE", "1")
    p = fx.Pattern(pat, "in")
    got = p.in_batch(buf, off)
    assert p.info()["sparse_used"] == 1
    assert np.array_equal(got, exp), (name, pat, np.nonzero(got != exp)[0][:10])
    monkeypatch.setenv("FX_SPARSE", "0")
    ref = p.in_batch(buf, off)
    assert p.info()["sparse_used"] == 0
    assert np.array_equal(ref, exp), (name, pat, "FX_SPARSE=0")
    return int(exp.sum())


@pytest.mark.parametrize("pat", PATTERNS)
def test_pairs_on_sweep_cuts(pat, edge_batches, monkeypatch):
    info = fx.Pattern(pat, "in").info()
    assert info["sparse"] == 1 and info["sparse_second"] == ord("o") and info["sparse_high"] == 1
    wins = 0
    for name, buf, off in edge_batches:
        wins += check_ragged(monkeypatch, pat, buf, off, name)
    assert wins > 100                                        # winners are there to be lost


def test_split_string_does_not_win(monkeypatch):
    buf, off = pack([b"xf", b"oobar", b"f", b"oobaz", b"foobar", b"zzf"])
    exp = np.array([0, 0, 0, 0, 1, 0], dtype=np.uint8)
    assert np.array_equal(O.Compiled(b"foo(bar|baz)", 0).bool_batch(0, buf, off), exp)
    assert check_ragged(monkeypatch, b"foo(bar|baz)", buf, off, "split") == 1


@pytest.mark.parametrize("pat", PATTERNS)
def test_fixed_strides_1_to_64(pat, monkeypatch):
    rng = np.random.default_rng(7)
    for stride in range(1, 65):
        n = max(64, 6000 // stride)
        raw = bytearray(background(rng, n * stride + 31))
        for k in rng.integers(0, len(raw) - 8, size=max(8, n // 4)):
            lit = PLANTS[int(k) % len(PLANTS)]
            raw[k:k + len(lit)] = lit
        for k in range(31, len(raw) - 8, 32 * 7):               # pairs across unit cuts
            raw[k:k + 6] = b"foobar" if k & 64 else b"fooba!"
        for shift in (0, 1, 13, 31):
            buf = np.frombuffer(bytes(raw[shift:shift + n * stride]), dtype=np.uint8).copy()
            exp = O.Compiled(pat, 0).bool_fixed(0, buf, n, stride)
            monkeypatch.setenv("FX_SPARSE", "1")
            p = fx.Pattern(pat, "in")
            got = p.in_fixed(buf, n, stride)
            assert np.array_equal(got, exp), (stride, shift, pat, np.nonzero(got != exp)[0][:10])
            monkeypatch.setenv("FX_SPARSE", "0")
            assert np.array_equal(p.in_fixed(buf, n, stride), exp), (stride, shift, pat, "FX_SPARSE=0")
