"""One-off extended GPU fuzz of the long-buffer paths (not part of the -m gpu suite): random patterns over a text of a few
hundred KB -- large enough for the state-map scan to work with many regions and for the candidate scan to run many
CTAs -- in the default flow, with K5 forced (FX_STATEMAP=2) and with K4 alone (FX_STATEMAP=0), against the oracle; and
the all-matches loop against the oracle's loop on the first few hundred matches."""
import os
import random
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import forgex_b200 as fx  # noqa: E402
from tests import oracle_lib as O  # noqa: E402
from tests.test_host_tables import gen_pattern, gen_text  # noqa: E402


def main():
    budget = float(sys.argv[1]) if len(sys.argv) > 1 else 150.0
    seed = int(sys.argv[2]) if len(sys.argv) > 2 else 0
    t0 = time.time()
    tried = skipped = nall = 0
    while time.time() - t0 < budget:
        rng = random.Random(77000 + seed)
        pieces = [gen_text(rng) for _ in range(rng.choice((40000, 120000, 250000)))]
        text = (b"\n" if seed % 3 else b" ").join(pieces)
        arr = np.frombuffer(b"#" * (seed % 5) + text, dtype=np.uint8)[seed % 5:]          # unaligned views too
        for _ in range(12):
            pat = gen_pattern(rng).encode()
            p = fx.Pattern(pat, "regex")
            if p.status != 0:
                continue
            c = O.Compiled(pat, 0)
            t1 = time.time()
            exp = c.regex_buffer(np.ascontiguousarray(arr))
            if time.time() - t1 > 5.0:
                skipped += 1          # (the oracle itself is quadratic on this one: once is enough)
            for mode in ("1", "2", "0"):
                os.environ["FX_STATEMAP"] = mode
                try:
                    got = p.regex_buffer(arr)
                except fx.ForgexError as e:
                    assert e.status == 106, (pat, mode, e.status)      # work budget: only where no stand-in exists
                    assert not p.info()["statemap"] or p.info()["literal_prefix_len"] > 0, (pat, mode)
                    continue
                assert got == exp, (seed, pat, mode, got, exp, len(arr))
            tried += 1
            # all matches: the first 300 of the oracle's loop
            os.environ["FX_STATEMAP"] = "1"
            if p.info()["nfa_engine"]:
                continue
            pos, want = 0, []
            t1 = time.time()
            while len(want) < 300 and time.time() - t1 < 3.0:
                f, t = c.regex_buffer(np.ascontiguousarray(arr[pos:]))
                if f <= 0 or t <= 0:
                    break
                want.append((pos + f, pos + t))
                pos += t
            complete = len(want) < 300 and time.time() - t1 < 3.0
            try:
                f, t, cnt = p.regex_buffer_all(arr, capacity=300)
            except fx.ForgexError as e:
                assert e.status == 106, (pat, e.status)                 # work budget: only where no stand-in exists
                assert not p.info()["statemap"] or p.info()["literal_prefix_len"] > 0, (seed, pat, "all matches")
                continue
            got = list(zip(f.tolist(), t.tolist()))
            assert got[:len(want)] == want[:len(got)] and len(got) >= min(len(want), 300), (seed, pat, got[:3], want[:3], cnt, len(want))
            if complete:
                assert cnt == len(want), (seed, pat, cnt, len(want))
            nall += 1
        print("seed", seed, "text", len(arr), "patterns", tried, "all-matches", nall, "slow-oracle", skipped, flush=True)
        seed += 1
    print("extended buffer fuzz ok: %d patterns, %d all-matches loops, in %.0f s" % (tried, nall, time.time() - t0))


if __name__ == "__main__":
    main()
