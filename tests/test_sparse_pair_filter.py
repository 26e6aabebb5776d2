"""A NumPy model of K2c's two-byte sweep filter (fx_kernels.cuh: second_zero, pair_mask, unit_any with TWO,
sweep_group's successor exchange, the candidate mask of sparse_run_units), fuzzed on random and adversarial words.

The filter may over-approximate (every candidate is confirmed by the table) but must never lose a pair: byte j
is a candidate when it is the first byte F and byte j + 1 is the second byte S, or a byte >= 0x80 when lead bytes may
follow (second_high).  Extra flags are allowed only as borrow neighbours of the zero-byte test (above a true pair in
the same word).  A unit's last byte looks at the next unit's first byte, or counts as followed by S where the next
unit is not loaded.
"""
import numpy as np
import pytest

F, S = ord("f"), ord("o")
ROWS = 4                     # SPARSE_ROWS


def rep(b):
    return b * 0x01010101


def second_zero(w, lead):
    z = w ^ np.uint32(rep(S))
    if lead:                 # PRMT 0xBA98: each byte's bit 7 replicated over the byte
        b = (w >> np.uint32(7)) & np.uint32(0x01010101)
        z &= ~(b * np.uint32(0xFF))
    return z


def pair_mask(w, z, z_next):
    t = (w ^ np.uint32(rep(F))) | (z >> np.uint32(8)) | (z_next << np.uint32(24))
    return ((t - np.uint32(0x01010101)) & ~t) & np.uint32(0x80808080)


def words_of(units):
    """units: (n, 32) uint8 -> (n, 8) uint32 little-endian words"""
    return np.ascontiguousarray(units).view("<u4").astype(np.uint32)


def unit_flags(units, z_next, high, second_high, in_unit_lead):
    """per-byte flag masks (n, 8) words of the pair test over each unit; z_next (n,) uint32"""
    w = words_of(units)
    out = np.zeros_like(w)
    zn = z_next.astype(np.uint32)
    for k in range(7, -1, -1):
        z = second_zero(w[:, k], second_high and in_unit_lead)
        out[:, k] = pair_mask(w[:, k], z, zn)
        zn = z
    return out


def unit_any(units, z_next, high, second_high):
    """the sweep's unit test: lead bytes inside the unit need no test with HIGH (every byte >= 0x80 passes)"""
    m = unit_flags(units, z_next, high, second_high, in_unit_lead=not high)
    anyw = np.bitwise_or.reduce(m, axis=1)
    if high:
        anyw |= np.bitwise_or.reduce(words_of(units), axis=1) & np.uint32(0x80808080)
    return anyw != 0


def flags_to_bytes(m):
    """(n, 8) flag words -> (n, 32) bool"""
    b = np.ascontiguousarray(m).view(np.uint8).reshape(m.shape[0], 32)
    return (b & 0x80) != 0


def true_pairs(text, nunits, second_high, loaded_next):
    """(nunits, 32) bool: byte is F and the following byte may follow it; the byte after a unit whose next unit is
    not loaded counts as S"""
    nxt = text[1:nunits * 32 + 1].astype(np.int32)
    last = np.arange(31, nunits * 32, 32)
    nxt[last] = np.where(loaded_next, nxt[last], S)
    ok = (nxt == S) | (second_high & (nxt >= 0x80))
    return ((text[:nunits * 32] == F) & ok).reshape(nunits, 32)


def gen_text(rng, n, kind):
    if kind == "random":
        return rng.integers(0, 256, size=n, dtype=np.uint8)
    if kind == "ascii":
        return rng.integers(0x20, 0x7F, size=n, dtype=np.uint8)
    # adversarial: F, S, 0x00, 0x01, F ^ 1, S ^ 1, lead and continuation bytes, densely
    alphabet = np.array([F, S, 0, 1, F ^ 1, S ^ 1, 0x80, 0xC3, 0xFF, F | 0x80, S | 0x80, 0x20], dtype=np.uint8)
    return alphabet[rng.integers(0, alphabet.size, size=n)]


def check_flags(flags, truth):
    """every true pair flagged; an extra flag only above a true pair of the same 4-byte word"""
    assert not (truth & ~flags).any()
    extra = flags & ~truth
    t4 = truth.reshape(truth.shape[0], 8, 4)
    below = np.cumsum(t4, axis=2) > 0
    below = np.concatenate([np.zeros_like(below[:, :, :1]), below[:, :, :-1]], axis=2).reshape(truth.shape)
    assert not (extra & ~below).any()


@pytest.mark.parametrize("kind", ["random", "ascii", "adversarial"])
@pytest.mark.parametrize("second_high", [False, True])
@pytest.mark.parametrize("high", [False, True])
def test_unit_filter_keeps_every_pair(kind, second_high, high):
    rng = np.random.default_rng(hash((kind, second_high, high)) & 0xFFFF)
    for _ in range(20):
        nunits = 257
        text = gen_text(rng, nunits * 32 + 32, kind)
        units = text[:nunits * 32].reshape(nunits, 32)
        loaded = rng.random(nunits) < 0.8                    # the next unit is loaded (else assumed to match)
        first_next = words_of(text[32:nunits * 32 + 32].reshape(nunits, 32))[:, 0]
        z_next = np.where(loaded, second_zero(first_next, second_high), np.uint32(0))
        truth = true_pairs(text, nunits, second_high, loaded)
        # the unit phase's candidates: the lead test in every word
        check_flags(flags_to_bytes(unit_flags(units, z_next, high, second_high, in_unit_lead=True)), truth)
        # the sweep: exact per unit, up to bytes >= 0x80 with HIGH
        want = truth.any(axis=1)
        if high:
            want |= (units >= 0x80).any(axis=1)
        assert np.array_equal(unit_any(units, z_next, high, second_high), want)


@pytest.mark.parametrize("second_high", [False, True])
def test_successor_rule_at_the_last_byte(second_high):
    """the last byte of a unit is flagged only if the next unit starts with S (or a lead byte, with second_high), or
    the next unit is not loaded"""
    units = np.full((6, 32), 0x20, dtype=np.uint8)
    units[:, 31] = F
    nxt = np.array([S, 0x20, 0xC3, 0, S ^ 1, S], dtype=np.uint8)
    loaded = np.array([True, True, True, True, True, False])
    first_next = nxt.astype(np.uint32) | np.uint32(0x20202000)
    z_next = np.where(loaded, second_zero(first_next, second_high), np.uint32(0))
    got = flags_to_bytes(unit_flags(units, z_next, False, second_high, in_unit_lead=True))[:, 31]
    assert got.tolist() == [True, False, second_high, False, False, True]
    assert unit_any(units, z_next, False, second_high).tolist() == [True, False, second_high, False, False, True]


@pytest.mark.parametrize("lim", [1, 31, 32, 33, 127, 128, 129, 500, 1023, 1024])
def test_sweep_successor_exchange(lim):
    """sweep_group's shuffle: lane L reads lane L + 1 of its row, lane 31 reads lane 0 of the next row (lane 0 gives
    the next row's word); after a group's last row and after the segment's last unit the successor is assumed.  The
    model follows the kernel's expressions and must give unit u + 1's word exactly where that unit is loaded."""
    nrows = (lim + 31) // 32
    word = np.arange(1, 1025, dtype=np.int64) * 1000003          # stands for second_zero of unit u's first word
    for r in range(0, nrows, ROWS):
        whole = (r + ROWS) * 32 <= lim
        for k in range(ROWS):
            z0 = lambda kk, lane: (word[(r + kk) * 32 + lane] if (whole or (r + kk) * 32 + lane < lim) else -1)
            for lane in range(32):
                src = (lane + 1) & 31
                give = z0(k, src) if src != 0 else (z0(k + 1, 0) if k + 1 < ROWS else 0)
                u = (r + k) * 32 + lane
                zn = 0 if (not whole and u + 1 >= lim) else give
                if u >= lim:
                    continue
                loaded = u + 1 < lim and (u + 1) % (32 * ROWS) != 0
                assert zn == (word[u + 1] if loaded else 0), (lim, r, k, lane)
