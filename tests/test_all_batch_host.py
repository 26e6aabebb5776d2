"""fx_regex_all_batch* without a device: the scratch size is host arithmetic over the scan's grid, and the status codes
come in fx_regex_count_batch*'s order (handle, pattern status, entry point, then the device)."""
import numpy as np
import pytest

import forgex_b200 as fx
from forgex_b200 import _lib as L
from tests.test_gpu_parity import pack

SCAN_TILE, SCAN_MAX_BLOCKS = 1024, 1024          # include/forgex_b200.h: one scan block per 1024 strings, at most 1024


def scan_blocks(n):
    return min(SCAN_MAX_BLOCKS, max(1, -(-n // SCAN_TILE)))


def test_work_bytes_cover_the_scan_grid_without_a_device():
    """8 bytes per block of the scan, for every n up past 2^31 and 2^40 strings; the same through the Python binding"""
    sizes = [0, 1, 2, 1023, 1024, 1025, 2048, 2049, SCAN_TILE * SCAN_MAX_BLOCKS - 1, SCAN_TILE * SCAN_MAX_BLOCKS,
             SCAN_TILE * SCAN_MAX_BLOCKS + 1, 20_000_000, (1 << 31) + 5, 1 << 40]
    got = [L.lib().fx_regex_all_batch_work_bytes(n) for n in sizes]
    assert got == [8 * scan_blocks(n) for n in sizes]
    assert got == sorted(got) and max(got) == 8 * SCAN_MAX_BLOCKS
    assert L.lib().fx_regex_all_batch_work_bytes(-3) == L.lib().fx_regex_all_batch_work_bytes(0)
    assert fx.Pattern.all_batch_work_bytes(5000) == 8 * 5


def statuses(p):
    """(host form, _dev form) status of one small batch.  The _dev form gets host addresses: only for calls that return
    before they touch the device."""
    lib = L.lib()
    buf, off = pack([b"ab aab", b"", b"c"])
    n = len(off) - 1
    rows, f, t = np.zeros(n + 1, np.int64), np.zeros(8, np.int64), np.zeros(8, np.int64)
    work = np.zeros(L.lib().fx_regex_all_batch_work_bytes(n), np.uint8)
    h = p.h if p is not None else None
    host = lib.fx_regex_all_batch(h, buf.ctypes.data, off.ctypes.data, n, rows.ctypes.data, f.ctypes.data, t.ctypes.data, 8)
    dev = lib.fx_regex_all_batch_dev(h, buf.ctypes.data, off.ctypes.data, n, len(buf), rows.ctypes.data, f.ctypes.data,
                                     t.ctypes.data, 8, work.ctypes.data, None)
    return host, dev


def test_status_codes_before_the_device():
    """a NULL handle and a handle compiled for `.in.` answer FX_ERR_BAD_ARGUMENT, an invalid pattern its SYNTAX_* code"""
    assert statuses(None) == (L.FX_ERR_BAD_ARGUMENT,) * 2
    p = fx.Pattern(b"a+", "in")
    assert p.status == 0 and statuses(p) == (L.FX_ERR_BAD_ARGUMENT,) * 2
    for pat in (b"(", b"a{2,1}", b"[b-a]"):
        p = fx.Pattern(pat, "regex")
        assert 1 <= p.status <= 24, pat
        assert statuses(p) == (p.status,) * 2, pat
        with pytest.raises(fx.ForgexError) as e:
            p.regex_all_batch(*pack([b"a"]))
        assert e.value.status == p.status


def test_no_device_answers_no_device():
    """without a CUDA device both matching forms answer FX_ERR_NO_DEVICE (there is no CPU fallback)"""
    import torch
    if torch.cuda.is_available():
        pytest.skip("checks the answer without a device")
    p = fx.Pattern(rb"a+", "regex")
    assert p.status == 0 and statuses(p) == (L.FX_ERR_NO_DEVICE,) * 2
    with pytest.raises(fx.ForgexError) as e:
        p.regex_all_batch(*pack([b"a", b"ba"]))
    assert e.value.status == L.FX_ERR_NO_DEVICE
