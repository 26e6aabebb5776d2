"""Times the linear-time window form (fx_statemap_*) on one GPU, the slabs of a split text run one after another.

    python tools/statemap_windows_bench.py [--c4-bytes N] [--slabs 1,2,4,8] [--reps R] [--out DIR]

Prints one JSON line; with --out it also writes DIR/statemap_windows_bench.json.

1. The C4 text (bench.py's construction, 32 GiB by default): K5 over the whole buffer (FX_STATEMAP=2) next to the window
   form over 1 / 2 / 4 / 8 slabs.  Reported per slab count: the sum of the slab-map times (CUDA events around each
   fx_statemap_window_dev), the host combine (fx_statemap_combine, after one copy of the maps), the backward walk, and
   the end-to-end time of the whole split search.  Every answer is checked against the span known by construction.
2. `[ab].*c` over 64 MiB, 256 MiB and 1 GiB of `a` in 4 slabs, end to end: the time grows with the text, linearly.
The card's name, power limit and SM clock limit are read in the same run and written next to the numbers.
Times are medians over --reps runs after two warm-up runs; the texts are larger than the L2.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def median(xs):
    return float(np.median(np.array(xs)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c4-bytes", type=int, default=32 << 30)
    ap.add_argument("--slabs", default="1,2,4,8")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="directory for statemap_windows_bench.json (default: print only)")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    import bench
    import forgex_b200 as fx
    from forgex_b200 import _lib
    from forgex_b200 import dist as fxd
    os.environ["FX_STATEMAP"] = "2"                     # the whole-buffer reference: K5 forced
    rec = {"card": card(), "reps": args.reps}

    def events_ms(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b)

    def split(p, buf, n, k, parts=None):
        """one split search, slabs in turn; returns ((from, to), declined, hops) and per-phase times in ms"""
        slabs = [fxd.slab_bounds(n, k, r) for r in range(k)]
        windows = [fxd.window_for_statemap_slab(n, lo, hi) for lo, hi in slabs]
        maps = torch.empty((k, _lib.FX_STATEMAP_MAP_WORDS), dtype=torch.int64, device="cuda")
        t_map = 0.0
        for i, ((lo, hi), (w_lo, w_hi)) in enumerate(zip(slabs, windows)):
            t_map += events_ms(lambda: p.statemap_window_dev(buf[w_lo:w_hi], w_hi - w_lo, lo - w_lo, hi - w_lo, w_lo, maps[i], work))
        t0 = time.perf_counter()
        end, declined = (int(x) for x in p.statemap_combine(maps.cpu().numpy(), n))
        t_comb = (time.perf_counter() - t0) * 1e3
        t0 = time.perf_counter()
        span, hops = (0, 0), 0
        if not declined and end > 0:
            owner = lambda b: next(i for i, (a, z) in enumerate(slabs) if a <= b < z)     # noqa: E731
            w = owner(end - 1) if end <= n else k - 1
            walk = torch.tensor([0, 0, _lib.FX_STATEMAP_WALK_NEW, end], dtype=torch.int64, device="cuda")
            while True:
                w_lo, w_hi = windows[w]
                p.statemap_back_dev(buf[w_lo:w_hi], w_hi - w_lo, w_lo, n, walk)
                pos, best, state, _ = walk.cpu().tolist()
                if state == _lib.FX_STATEMAP_WALK_DONE:
                    span = (pos, best)
                    break
                w, hops = owner(pos - 1), hops + 1
        t_back = (time.perf_counter() - t0) * 1e3
        if parts is not None:
            parts.append((t_map, t_comb, t_back))
        return span, bool(declined), hops

    def timed_split(p, buf, n, k):
        parts, e2e = [], []
        for r in range(2 + args.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = split(p, buf, n, k, parts if r >= 2 else None)
            e2e.append((time.perf_counter() - t0) * 1e3)
        e2e = e2e[2:]
        return res, {"slab_maps_sum_ms": median([x[0] for x in parts]), "combine_ms": median([x[1] for x in parts]),
                     "backward_walk_ms": median([x[2] for x in parts]), "end_to_end_ms": median(e2e),
                     "slab_maps_gb_per_s": n / median([x[0] for x in parts]) / 1e6}

    # ---- 1. C4 ----
    n = args.c4_bytes
    w = bench.build_workload(torch, "c4", n, 0, 1)
    p, buf, expect = w["pattern_obj"], w["buf"], tuple(w["expect_span"])
    work = torch.empty(p.buffer_work_bytes(n), dtype=torch.uint8, device="cuda")
    ft = torch.zeros(2, dtype=torch.int64, device="cuda")
    whole = []
    for r in range(2 + args.reps):
        ms = events_ms(lambda: p.regex_buffer_dev(buf, n, ft, work))
        if r >= 2:
            whole.append(ms)
    c4 = {"bytes": n, "expected_span": list(expect), "k5_whole_buffer": {"ms": median(whole), "gb_per_s": n / median(whole) / 1e6,
                                                                           "span": ft.cpu().tolist()}}
    assert tuple(c4["k5_whole_buffer"]["span"]) == expect
    for k in [int(x) for x in args.slabs.split(",")]:
        (span, declined, hops), t = timed_split(p, buf, n, k)
        assert span == expect and not declined, (k, span, expect)
        c4["slabs_%d" % k] = dict(t, hops=hops, span=list(span))
    rec["c4"] = c4
    del buf, work, w
    torch.cuda.empty_cache()

    # ---- 2. `[ab].*c` over `a` only: linear growth ----
    p = fx.Pattern(b"[ab].*c", "regex")
    lin = {}
    for n in (64 << 20, 256 << 20, 1 << 30):
        buf = torch.full((n,), ord("a"), dtype=torch.uint8, device="cuda")
        work = torch.empty(p.buffer_work_bytes(n), dtype=torch.uint8, device="cuda")
        (span, declined, hops), t = timed_split(p, buf, n, 4)
        assert span == (0, 0) and not declined
        lin["%d_MiB" % (n >> 20)] = t
        del buf, work
    rec["ab_dot_star_c_4_slabs"] = lin
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "statemap_windows_bench.json"), "w") as fh:
            json.dump(rec, fh, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
