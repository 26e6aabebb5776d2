"""Host-side mirror of Forgex's public interface (reference: src/forgex.F90:24-54) over the C ABI.

    reference                              here
    -------------------------------------  ---------------------------------------------
    pattern .in. text                      op_in(pattern, text)
    pattern .match. text                   op_match(pattern, text)
    call regex(pattern, text, res, length, from, to, status, err_msg)
                                           regex(pattern, text) -> RegexResult
    regex_f(pattern, text)                 regex_f(pattern, text)
    is_valid_regex(pattern)                is_valid_regex(pattern)
    (new) one pattern against N strings    Pattern(...).match_fixed / in_fixed / match_batch / in_batch / regex_batch
    (new) one pattern, one huge buffer     Pattern(...).regex_buffer

Same argument meaning and error behaviour as the reference: an invalid pattern makes the operators
return False, and makes regex return res=b'', length=0, from=to=-9999 with the SYNTAX_* status and
its message (src/forgex.F90:101-104, :197-200, :266-274).  Byte strings in, byte strings out; indices
are 1-based inclusive like Fortran's.  All matching runs on the GPU through libforgex_b200.so.
"""
import ctypes as C
from collections import namedtuple

import numpy as np

from . import _lib as L

INVALID_CHAR_INDEX = -9999

RegexResult = namedtuple("RegexResult", "res length from_ to status err_msg")


class ForgexError(RuntimeError):
    def __init__(self, status, where=""):
        self.status = status
        super().__init__("%s: status %d: %s" % (where, status, status_message(status)))


def status_message(status):
    return L.lib().fx_status_message(status).decode()


def _b(x):
    if isinstance(x, str):
        return x.encode("utf-8")
    return bytes(x)


def _check(rc, where):
    if rc != 0:
        raise ForgexError(rc, where)


def _is_torch(x):
    return type(x).__module__.startswith("torch")


def _ptr(x):
    """data pointer of a numpy array or a torch tensor"""
    if _is_torch(x):
        return x.data_ptr()
    return x.ctypes.data


class Pattern:
    """A pattern compiled once for one entry point (op = 'match' | 'in' | 'regex')."""

    OPS = {"match": L.FX_OP_MATCH, "in": L.FX_OP_IN, "regex": L.FX_OP_REGEX}

    def __init__(self, pattern, op, residency="auto"):
        self.pattern = _b(pattern)
        self.op = self.OPS[op] if isinstance(op, str) else op
        h = C.c_void_p()
        self.status = L.lib().fx_compile(self.pattern, len(self.pattern), self.op, C.byref(h))
        self.h = h
        if residency != "auto":
            self.set_residency(residency)

    @classmethod
    def from_dfa(cls, op, cuts, delta, accept, q0, literals=(b"", b"", b""), pattern=b""):
        """the Fortran-side route: a handle built from an anchored code-point DFA (fx_compile_from_dfa)"""
        self = cls.__new__(cls)
        self.pattern = _b(pattern)
        self.op = cls.OPS[op] if isinstance(op, str) else op
        cuts = np.ascontiguousarray(cuts, dtype=np.int32)
        delta = np.ascontiguousarray(delta, dtype=np.int32)
        accept = np.ascontiguousarray(accept, dtype=np.uint8)
        nstates, ncls = delta.shape
        assert len(cuts) == ncls + 1 and len(accept) == nstates
        a, pre, suf = (_b(x) for x in literals)
        h = C.c_void_p()
        self.status = L.lib().fx_compile_from_dfa(self.op, _ptr(cuts), ncls, _ptr(delta), nstates, _ptr(accept), int(q0),
                                                  a, len(a), pre, len(pre), suf, len(suf), C.byref(h))
        self.h = h
        return self

    def cp_automaton(self):
        """the anchored code-point DFA of a 'regex' handle: dict(cuts, delta[states, classes], accept, q0, start_nul)"""
        ptrs = [C.c_void_p() for _ in range(3)]
        sc = (C.c_int32 * 4)()
        _check(L.lib().fx_pattern_cp_automaton(self.h, C.byref(ptrs[0]), C.byref(ptrs[1]), C.byref(ptrs[2]), C.byref(sc)),
               "fx_pattern_cp_automaton")

        def arr(p, n, dt):
            return np.ctypeslib.as_array(C.cast(p, C.POINTER(dt)), shape=(n,)).copy()
        ns, nc = sc[0], sc[1]
        return {"cuts": arr(ptrs[0], nc + 1, C.c_int32), "delta": arr(ptrs[1], ns * nc, C.c_int32).reshape(ns, nc),
                "accept": arr(ptrs[2], ns, C.c_uint8), "q0": sc[2], "start_nul": sc[3]}

    def close(self):
        if getattr(self, "h", None):
            L.lib().fx_pattern_free(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def valid(self):
        return self.status == 0

    def set_residency(self, mode):
        m = {"auto": L.FX_TABLE_AUTO, "smem": L.FX_TABLE_SMEM, "global": L.FX_TABLE_GLOBAL}[mode]
        _check(L.lib().fx_pattern_set_residency(self.h, m), "fx_pattern_set_residency")

    def info(self):
        inf = L.PatternInfo()
        _check(L.lib().fx_pattern_get_info(self.h, C.byref(inf)), "fx_pattern_get_info")
        out = {n: getattr(inf, n) for n, _ in inf._fields_}
        for k in ("sparse_lo", "sparse_hi"):
            out[k] = list(out[k])[:out["sparse_ranges"]]
        return out

    def literals(self):
        inf = self.info()
        bufs = [C.create_string_buffer(max(1, inf[k])) for k in
                ("literal_all_len", "literal_prefix_len", "literal_suffix_len")]
        _check(L.lib().fx_pattern_literals(self.h, *bufs), "fx_pattern_literals")
        return tuple(b.raw[:inf[k]] for b, k in zip(bufs, ("literal_all_len", "literal_prefix_len",
                                                           "literal_suffix_len")))

    def tables(self):
        """host copies of the device tables as numpy arrays (tests / tools)"""
        inf = self.info()
        ptrs = [C.c_void_p() for _ in range(4)]
        sc = (C.c_int32 * 6)()
        _check(L.lib().fx_pattern_tables(self.h, *[C.byref(p) for p in ptrs], C.byref(sc)), "fx_pattern_tables")
        ns, rs = inf["byte_states"], inf["row_shift"]

        def arr(p, n, dt):
            return np.ctypeslib.as_array(C.cast(p, C.POINTER(dt)), shape=(n,)).copy()
        return {
            "table": arr(ptrs[0], ns << rs, C.c_uint16).reshape(ns, 1 << rs),
            "direct": arr(ptrs[1], ns * 256, C.c_uint16).reshape(ns, 256),
            "classmap": arr(ptrs[2], 256, C.c_uint8),
            "flags": arr(ptrs[3], ns, C.c_uint8),
            "start": sc[0], "start_nul": sc[1], "q0": sc[2], "matched": sc[3], "q0_accepting": bool(sc[4]), "result_threshold": sc[5],
            "row_shift": rs,
        }

    def span_tables(self):
        """tables of the linear-time span path (None if the pattern has none)"""
        ptrs = [C.c_void_p() for _ in range(6)]
        sc, rsc = (C.c_int32 * 4)(), (C.c_int32 * 4)()
        rc = L.lib().fx_pattern_span_tables(self.h, C.byref(ptrs[0]), C.byref(ptrs[1]), C.byref(sc), C.byref(ptrs[2]),
                                            C.byref(ptrs[3]), C.byref(ptrs[4]), C.byref(ptrs[5]), C.byref(rsc))
        if rc == 1:
            return None
        _check(rc, "fx_pattern_span_tables")

        def arr(p, n, dt):
            return np.ctypeslib.as_array(C.cast(p, C.POINTER(dt)), shape=(n,)).copy()
        ns, nr, nc, nm = sc[0], rsc[0], rsc[1], rsc[3]
        return {"direct": arr(ptrs[0], ns * 256, C.c_uint16).reshape(ns, 256), "endinfo": arr(ptrs[1], ns, C.c_uint8),
                "start": sc[1], "start_acc": bool(sc[2]), "rdelta": arr(ptrs[2], nr * nc, C.c_uint16).reshape(nr, nc),
                "rpage": arr(ptrs[3], 1024, C.c_uint8) if ptrs[3].value else None,
                "rmixed": arr(ptrs[4], nm * 64, C.c_uint8) if ptrs[4].value and nm else None,
                "cuts": arr(ptrs[5], nc + 1, C.c_int32), "rstart": rsc[2]}

    def nfa_tables(self):
        """tables of the NFA engine (None for a table-engine handle)"""
        ptrs = [C.c_void_p() for _ in range(3)]
        sc = (C.c_int32 * 5)()
        rc = L.lib().fx_pattern_nfa_tables(self.h, C.byref(ptrs[0]), C.byref(ptrs[1]), C.byref(ptrs[2]), C.byref(sc))
        if rc == 1:
            return None
        _check(rc, "fx_pattern_nfa_tables")

        def arr(p, n, dt):
            return np.ctypeslib.as_array(C.cast(p, C.POINTER(dt)), shape=(n,)).copy()
        ns, w, nc = sc[0], sc[1], sc[2]
        return {"trans": arr(ptrs[0], (ns + 1) * nc * w, C.c_uint64).reshape(ns + 1, nc, w), "q0": arr(ptrs[1], w, C.c_uint64),
                "cuts": arr(ptrs[2], nc + 1, C.c_int32), "exit": sc[3], "q0_accepting": bool(sc[4])}

    # ---- host-buffer batch calls (numpy in, numpy out; copies happen inside the library) ----
    # `out=`: caller-provided result arrays (e.g. pinned host memory: the device-to-host copy then runs at PCIe speed)
    @staticmethod
    def _out(out, n, dtype):
        if out is None:
            return np.empty(n, dtype=dtype)
        assert out.dtype == dtype and out.size >= n and out.flags["C_CONTIGUOUS"]
        return out

    def _bool_fixed(self, fn, buf, n, stride, out=None):
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        assert buf.size >= n * stride
        out = self._out(out, n, np.uint8)
        _check(fn(self.h, _ptr(buf), n, stride, _ptr(out)), fn.__name__)
        return out[:n]

    def match_fixed(self, buf, n, stride, out=None):
        return self._bool_fixed(L.lib().fx_match_fixed, buf, n, stride, out)

    def in_fixed(self, buf, n, stride, out=None):
        return self._bool_fixed(L.lib().fx_in_fixed, buf, n, stride, out)

    def _bool_batch(self, fn, buf, offsets, out=None):
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n = len(offsets) - 1
        out = self._out(out, n, np.uint8)
        _check(fn(self.h, _ptr(buf), _ptr(offsets), n, _ptr(out)), fn.__name__)
        return out[:n]

    def match_batch(self, buf, offsets, out=None):
        return self._bool_batch(L.lib().fx_match_batch, buf, offsets, out)

    def in_batch(self, buf, offsets, out=None):
        return self._bool_batch(L.lib().fx_in_batch, buf, offsets, out)

    def regex_batch(self, buf, offsets, out=None):
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n = len(offsets) - 1
        f = self._out(None if out is None else out[0], n, np.int64)
        t = self._out(None if out is None else out[1], n, np.int64)
        _check(L.lib().fx_regex_batch(self.h, _ptr(buf), _ptr(offsets), n, _ptr(f), _ptr(t)), "fx_regex_batch")
        return f[:n], t[:n]

    def regex_buffer(self, buf):
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        f, t = C.c_int64(0), C.c_int64(0)
        _check(L.lib().fx_regex_buffer(self.h, _ptr(buf), buf.size, C.byref(f), C.byref(t)), "fx_regex_buffer")
        return f.value, t.value

    def regex_count_batch(self, buf, offsets):
        """matches per string, counted the way a caller loops regex() on text(to+1:)"""
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        n = len(offsets) - 1
        counts = np.zeros(n, dtype=np.int64)
        _check(L.lib().fx_regex_count_batch(self.h, _ptr(buf), _ptr(offsets), n, _ptr(counts)), "fx_regex_count_batch")
        return counts

    def regex_buffer_all(self, buf, capacity=1 << 20):
        """every match of the buffer in order: (from[], to[], count); at most `capacity` spans are returned"""
        buf = np.ascontiguousarray(buf, dtype=np.uint8)
        f = np.zeros(max(capacity, 1), dtype=np.int64)
        t = np.zeros(max(capacity, 1), dtype=np.int64)
        cnt = C.c_int64(0)
        _check(L.lib().fx_regex_buffer_all(self.h, _ptr(buf), buf.size, _ptr(f), _ptr(t), capacity, C.byref(cnt)), "fx_regex_buffer_all")
        k = min(cnt.value, capacity)
        return f[:k], t[:k], cnt.value

    # ---- device-resident calls (torch CUDA tensors; nothing is copied; runs on torch's current stream) ----
    @staticmethod
    def _stream():
        import torch
        return torch.cuda.current_stream().cuda_stream

    def match_fixed_dev(self, d_buf, n, stride, d_out):
        _check(L.lib().fx_match_fixed_dev(self.h, _ptr(d_buf), n, stride, _ptr(d_out), self._stream()),
               "fx_match_fixed_dev")

    def in_fixed_dev(self, d_buf, n, stride, d_out):
        _check(L.lib().fx_in_fixed_dev(self.h, _ptr(d_buf), n, stride, _ptr(d_out), self._stream()),
               "fx_in_fixed_dev")

    def match_batch_dev(self, d_buf, d_offsets, n, total, d_out):
        _check(L.lib().fx_match_batch_dev(self.h, _ptr(d_buf), _ptr(d_offsets), n, total, _ptr(d_out),
                                          self._stream()), "fx_match_batch_dev")

    def in_batch_dev(self, d_buf, d_offsets, n, total, d_out):
        _check(L.lib().fx_in_batch_dev(self.h, _ptr(d_buf), _ptr(d_offsets), n, total, _ptr(d_out),
                                       self._stream()), "fx_in_batch_dev")

    def regex_batch_dev(self, d_buf, d_offsets, n, total, d_from, d_to):
        _check(L.lib().fx_regex_batch_dev(self.h, _ptr(d_buf), _ptr(d_offsets), n, total, _ptr(d_from), _ptr(d_to),
                                          self._stream()), "fx_regex_batch_dev")

    @staticmethod
    def buffer_work_bytes(length):
        """size of the device scratch fx_regex_buffer_dev needs for a text of `length` bytes"""
        return int(L.lib().fx_regex_buffer_work_bytes(length))

    def regex_buffer_dev(self, d_buf, length, d_from_to, d_work):
        assert d_work.numel() * d_work.element_size() >= self.buffer_work_bytes(length), "d_work is too small"

        _check(L.lib().fx_regex_buffer_dev(self.h, _ptr(d_buf), length, _ptr(d_from_to), _ptr(d_work),
                                           self._stream()), "fx_regex_buffer_dev")


    def regex_count_batch_dev(self, d_buf, d_offsets, n, total, d_counts):
        _check(L.lib().fx_regex_count_batch_dev(self.h, _ptr(d_buf), _ptr(d_offsets), n, total, _ptr(d_counts),
                                                self._stream()), "fx_regex_count_batch_dev")

    def regex_buffer_all_dev(self, d_buf, length, d_from, d_to, capacity, d_work):
        cnt = C.c_int64(0)
        _check(L.lib().fx_regex_buffer_all_dev(self.h, _ptr(d_buf), length, _ptr(d_from), _ptr(d_to), capacity, C.byref(cnt),
                                               _ptr(d_work), self._stream()), "fx_regex_buffer_all_dev")
        return cnt.value

    def buffer_scan_dev(self, d_window, window_len, start_lo, start_hi, origin, is_first, is_last, d_best):
        _check(L.lib().fx_buffer_scan_dev(self.h, _ptr(d_window), window_len, start_lo, start_hi, origin,
                                          int(is_first), int(is_last), _ptr(d_best), self._stream()), "fx_buffer_scan_dev")

    def buffer_scan_all_dev(self, d_window, window_len, start_lo, start_hi, origin, is_first, is_last, d_best):
        _check(L.lib().fx_buffer_scan_all_dev(self.h, _ptr(d_window), window_len, start_lo, start_hi, origin,
                                              int(is_first), int(is_last), _ptr(d_best), self._stream()),
               "fx_buffer_scan_all_dev")

    def buffer_finish_dev(self, d_window, window_len, origin, is_last, d_key, d_from_to):
        _check(L.lib().fx_buffer_finish_dev(self.h, _ptr(d_window), window_len, origin, int(is_last), _ptr(d_key),
                                            _ptr(d_from_to), self._stream()), "fx_buffer_finish_dev")

    # ---- linear-time window form (include/forgex_b200.h: fx_statemap_*) ----
    def statemap_window_dev(self, d_window, window_len, slab_lo, slab_hi, origin, d_map, d_work):
        """slab map of window bytes [slab_lo, slab_hi) into d_map (FX_STATEMAP_MAP_WORDS int64)"""
        assert d_map.numel() >= L.FX_STATEMAP_MAP_WORDS, "d_map is too small"
        assert d_work.numel() * d_work.element_size() >= self.buffer_work_bytes(slab_hi - slab_lo), "d_work is too small"
        _check(L.lib().fx_statemap_window_dev(self.h, _ptr(d_window), window_len, slab_lo, slab_hi, origin, _ptr(d_map),
                                              _ptr(d_work), self._stream()), "fx_statemap_window_dev")

    def statemap_combine(self, maps, text_len):
        """slab maps (nmaps x FX_STATEMAP_MAP_WORDS, text order) -> int64[2] = (end of the match, declined); host-only"""
        maps = np.ascontiguousarray(maps, dtype=np.int64).reshape(-1, L.FX_STATEMAP_MAP_WORDS)
        out = np.zeros(2, dtype=np.int64)
        _check(L.lib().fx_statemap_combine(self.h, _ptr(maps), maps.shape[0], text_len, _ptr(out)), "fx_statemap_combine")
        return out

    def statemap_back_dev(self, d_window, window_len, origin, text_len, d_walk):
        """advance the backward walk d_walk (FX_STATEMAP_WALK_WORDS int64) over this window"""
        assert d_walk.numel() >= L.FX_STATEMAP_WALK_WORDS, "d_walk is too small"
        _check(L.lib().fx_statemap_back_dev(self.h, _ptr(d_window), window_len, origin, text_len, _ptr(d_walk),
                                            self._stream()), "fx_statemap_back_dev")


# ---- the reference's public API: one pattern, one text, compiled per call -----------------------
def is_valid_regex(pattern):
    p = _b(pattern)
    st = C.c_int(0)
    return bool(L.lib().fx_is_valid_regex(p, len(p), C.byref(st)))


def is_valid_regex_batch(patterns):
    """is_valid_regex over a list of patterns (elemental in the reference): returns (valid uint8[n], status int32[n])"""
    pats = [_b(x) for x in patterns]
    n = len(pats)
    off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum([len(x) for x in pats], out=off[1:])
    buf = np.frombuffer(b"".join(pats) + b"\0", dtype=np.uint8)
    valid, status = np.zeros(n, dtype=np.uint8), np.zeros(n, dtype=np.int32)
    _check(L.lib().fx_is_valid_regex_batch(_ptr(buf), _ptr(off), n, _ptr(valid), _ptr(status)), "fx_is_valid_regex_batch")
    return valid, status


def op_in(pattern, text):
    """`pattern .in. text` (src/forgex.F90:74)"""
    p, t = _b(pattern), _b(text)
    r = C.c_int(0)
    _check(L.lib().fx_in(p, len(p), t, len(t), C.byref(r)), "fx_in")
    return bool(r.value)


def op_match(pattern, text):
    """`pattern .match. text` (src/forgex.F90:163)"""
    p, t = _b(pattern), _b(text)
    r = C.c_int(0)
    _check(L.lib().fx_match(p, len(p), t, len(t), C.byref(r)), "fx_match")
    return bool(r.value)


def regex(pattern, text):
    """`call regex(pattern, text, res, length, from, to, status, err_msg)` (src/forgex.F90:235)"""
    p, t = _b(pattern), _b(text)
    f, to, ln, st = C.c_int64(0), C.c_int64(0), C.c_int64(0), C.c_int(0)
    _check(L.lib().fx_regex(p, len(p), t, len(t), C.byref(f), C.byref(to), C.byref(ln), C.byref(st)), "fx_regex")
    res = t[f.value - 1:to.value] if f.value > 0 and to.value > 0 else b""
    return RegexResult(res, ln.value, f.value, to.value, st.value, status_message(st.value))


def regex_f(pattern, text):
    """`regex_f(pattern, text)` (src/forgex.F90:351)"""
    return regex(pattern, text).res


def launch_count():
    return L.lib().fx_launch_count()
