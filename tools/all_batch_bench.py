"""Times the all-matches batch form (fx_regex_all_batch_dev) against the count it is built on (fx_regex_count_batch_dev).

    python tools/all_batch_bench.py [--c3-lines N] [--c2-lines N] [--reps R] [--sample S] [--out DIR]

Prints one JSON line; with --out it also writes DIR/all_batch_bench.json.

Two workloads, generated on the device the way bench.py does it (tools/synth.py's generators and seeds):
  c3     C3's strings (20 M by default) with C3's pattern: a few matches per string.
  c2_w   `\\w+` on C2's lines (100 M by default): dense matches, about one per five bytes.  When the spans of every line
         do not fit in the free device memory, the first lines whose spans fit are used (`lines` says how many).
Per workload, three calls on the same batch: the count (fx_regex_count_batch_dev); the batch form with capacity 0 (count +
scan of the rows); the batch form with room for every span (count + scan + span pass).  Each is timed with CUDA events,
the median of --reps runs after two warm-up runs; the texts are larger than the L2.  Reported: ms, GB/s of text,
matches/s, and all / count ratios.  The rows are checked against the counts, and the spans of a seeded sample of strings
against the oracle's loop.  The card's name, power limit and SM clock limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

GiB = 1 << 30


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--c3-lines", type=int, default=20_000_000)
    ap.add_argument("--c2-lines", type=int, default=100_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sample", type=int, default=300, help="strings per workload checked against the oracle")
    ap.add_argument("--out", default=None, help="directory for all_batch_bench.json (default: print only)")
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    import bench
    import forgex_b200 as fx
    from tests import oracle_lib as O
    from tests.test_gpu_parity import oracle_all
    from tools import synth
    rec = {"card": card(), "reps": args.reps}

    def timed(fn):
        ts = []
        for r in range(2 + args.reps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            if r >= 2:
                ts.append(a.elapsed_time(b))
        return float(np.median(ts))

    def measure(name, pat, buf, off, n):
        p = fx.Pattern(pat, "regex")
        work = torch.empty(p.all_batch_work_bytes(n), dtype=torch.uint8, device="cuda")
        rows = torch.empty(n + 1, dtype=torch.int64, device="cuda")
        p.regex_all_batch_dev(buf, off, n, int(off[n]), rows, None, None, 0, work)
        torch.cuda.synchronize()
        # the spans of the first m lines must fit next to what is allocated already
        budget = torch.cuda.mem_get_info()[0] - 4 * GiB
        cap = torch.tensor([budget // 16], dtype=torch.int64, device="cuda")
        m = min(n, int(torch.searchsorted(rows, cap, right=True)[0]) - 1)
        if m < n:
            off = off[:m + 1]
            n = m
            del rows, work
            work = torch.empty(p.all_batch_work_bytes(n), dtype=torch.uint8, device="cuda")
            rows = torch.empty(n + 1, dtype=torch.int64, device="cuda")
        total_bytes = int(off[n])
        counts = torch.empty(n, dtype=torch.int64, device="cuda")
        t_count = timed(lambda: p.regex_count_batch_dev(buf, off, n, total_bytes, counts))
        t_rows = timed(lambda: p.regex_all_batch_dev(buf, off, n, total_bytes, rows, None, None, 0, work))
        matches = int(rows[n])
        assert int(rows[0]) == 0 and torch.equal(rows[1:], torch.cumsum(counts, 0)), name
        d_from = torch.empty(matches, dtype=torch.int64, device="cuda")
        d_to = torch.empty(matches, dtype=torch.int64, device="cuda")
        t_all = timed(lambda: p.regex_all_batch_dev(buf, off, n, total_bytes, rows, d_from, d_to, matches, work))
        assert int(rows[n]) == matches and torch.equal(rows[1:], torch.cumsum(counts, 0)), name
        # a seeded sample of strings against the oracle's loop
        c = O.Compiled(pat, 0)
        rows_h, off_h = rows.cpu().numpy(), off.cpu().numpy()
        for i in np.random.default_rng(17).choice(n, size=min(n, args.sample), replace=False):
            s = bytes(buf[int(off_h[i]):int(off_h[i + 1])].cpu().numpy())
            r0, r1 = int(rows_h[i]), int(rows_h[i + 1])
            got = list(zip(d_from[r0:r1].tolist(), d_to[r0:r1].tolist()))
            assert got == oracle_all(c, s), (name, int(i))
        del d_from, d_to, counts, rows, work
        torch.cuda.empty_cache()

        def leg(ms):
            return {"ms": ms, "text_gb_per_s": total_bytes / ms / 1e6, "matches_per_s": matches / ms * 1e3}
        return {"pattern": pat.decode("utf-8"), "lines": n, "text_bytes": total_bytes, "matches": matches,
                "count": leg(t_count), "all_rows_only": leg(t_rows), "all_full": leg(t_all),
                "ratio_all_over_count": t_all / t_count, "ratio_rows_only_over_count": t_rows / t_count,
                "sample_checked": min(n, args.sample)}

    # C3's strings and pattern (bench.py's construction: a seeded block tiled on the device)
    w = bench.build_workload(torch, "c3", args.c3_lines, 0)
    rec["c3"] = measure("c3", synth.PATTERNS["c3"], w["buf"], w["off"], w["units"])
    del w
    torch.cuda.empty_cache()
    # `\w+` on C2's lines
    buf, off, _ = bench.make_c2_device(torch, args.c2_lines, synth.SEEDS["c2"])
    rec["c2_w"] = measure("c2_w", rb"\w+", buf, off, args.c2_lines)
    del buf, off
    torch.cuda.empty_cache()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "all_batch_bench.json"), "w") as fh:
            json.dump(rec, fh, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
