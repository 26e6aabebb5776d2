#!/usr/bin/env python3
"""bench.py -- throughput of the Forgex matching hot path on B200 (contract: see the task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2] [--lines L] [--impl reference] [--dump-outputs DIR]

Headline workload = BASELINE.json configs[1] ("c2"): `foo(bar|baz)` .in. over 100 M random ASCII lines of
64-256 bytes, one pattern against N strings (flat buffer + int64 offsets).  A step = one pass of the
hot path over that batch.  `value` = input GB/s with the batch resident in HBM; `e2e` = the same through
the host-pointer C-ABI call (pinned host buffers, H2D + kernel + D2H inside the timed region).
Without --config the run measures ALL FIVE BASELINE configs at their full sizes, one after the other, and
puts them into `per_config` (each with its own roofline, e2e, oracle cross-check and by-construction
checks); the top-level keys are c2's.  `--config cX` measures that one config only.
Multi-GPU: one process per GPU (torchrun).  Batches (c1, c2, c3, c5): strings sharded across ranks, no
data-path collective, weak scaling (every rank holds a full-size batch).  The long buffer (c4): ONE 32 GiB
text is cut into N slabs (forgex_b200.dist), every rank scans its slab, the ranks agree on the winner
with one all-gather of 3 integers and one 16-byte all-reduce INSIDE the timed region: strong scaling.

`--impl reference` times the CPU restatement of Forgex's own loop (oracle/, kind "port": the Fortran
reference cannot be built in this image) on all host cores, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

from tools import synth  # noqa: E402

WORKLOADS = {
    "c1": "c1: '\\d{3}-\\d{4}' .match. over fixed 8-byte ASCII strings",
    "c2": "c2: 'foo(bar|baz)' .in. over random ASCII lines of 64-256 bytes (flat buffer + int64 offsets)",
    "c3": "c3: '[α-ωぁ-ん]+\\s\\w{2,8}' regex() spans over mixed Greek/Japanese/ASCII strings incl. invalid bytes",
    "c4": "c4: '^ERROR.*timeout=\\d+$' regex() over one synthetic log buffer",
    "c5": "c5: '(a|b)*a(a|b){12}' .in. over fixed 64-byte strings, table in global memory (L2)",
    "c2f": "c2f (experiment): 'foo(bar|baz)' .in. over FIXED 160-byte random ASCII strings (per-lane 16-byte global loads)",
}
DEFAULT_UNITS = {"c2f": 20_000_000, "c1": 1 << 30, "c2": 100_000_000, "c3": 16_000_000, "c4": 32 << 30, "c5": 10_000_000}
# algorithmic bytes per unit besides the text itself (SURVEY 8d): offsets read + result written
EXTRA_BYTES = {"c2f": 1, "c1": 1, "c2": 8 + 1, "c3": 8 + 16, "c4": 0, "c5": 1}


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def known_traffic(cfg, algo_bytes):
    """dram bytes per launch of the dominant kernel from the committed ncu capture (profiles/traffic.json) -- only when
    that capture was taken on a workload of the same size as this run's (same algorithmic bytes, within 2 %)"""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
            e = json.load(fh).get(cfg)
        if isinstance(e, dict) and abs(e["algorithmic_bytes"] - algo_bytes) <= 0.02 * algo_bytes:
            return int(e["bytes"])
    except Exception:
        pass
    return None


DUMP_MAX_ELEMS = 1 << 20     # per array; at most seven arrays of 8-byte elements keep a dump under 64 MB


def dump_index(n):
    """the elements of an n-element output that --dump-outputs keeps: all of them up to DUMP_MAX_ELEMS, else a fixed
    seeded sample (sorted, distinct), so that two runs with the same arguments write the same elements"""
    if n <= DUMP_MAX_ELEMS:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_MAX_ELEMS, replace=False))


def dump_output(torch, d, name, t):
    """device tensor t -> d/<name>.npy (the elements dump_index picks): int64 spans as float64, which holds them exactly,
    everything else as float32"""
    a = t.reshape(-1)[torch.from_numpy(dump_index(t.numel())).to(t.device)].cpu().numpy()
    np.save(os.path.join(d, name + ".npy"), a.astype(np.float64 if a.dtype == np.int64 else np.float32))


class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.samples = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            parts = [x.strip() for x in s.split(",")]
            try:
                sm.append(float(parts[0]))
                mx = max(mx, float(parts[1]))
                for nm, v in zip(names, parts[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---- device-side synthetic data (torch; same shapes as tools/synth.py) ----------------------------
def make_c2_device(torch, n, seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    lens = torch.randint(64, 257, (n,), device="cuda", generator=g, dtype=torch.int64)
    offsets = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    torch.cumsum(lens, 0, out=offsets[1:])
    total = int(offsets[-1].item())
    buf = torch.empty(total, dtype=torch.uint8, device="cuda")
    chunk = 1 << 30
    for a in range(0, total, chunk):
        b = min(total, a + chunk)
        buf[a:b] = torch.randint(0x20, 0x7F, (b - a,), device="cuda", generator=g, dtype=torch.uint8)
    kind = torch.randint(0, 16, (n,), device="cuda", generator=g)
    where = (torch.rand(n, device="cuda", generator=g) * (lens - 6).float()).long().clamp_(min=0)
    which = torch.randint(0, 2, (n,), device="cuda", generator=g)
    words = [b"foobar", b"foobaz", b"foobax", b"fooba "]
    ar = torch.arange(6, device="cuda")
    for k, base in ((0, 0), (1, 2)):
        for w in (0, 1):
            rows = torch.nonzero((kind == k) & (which == w)).squeeze(1)
            lit = torch.tensor(list(words[base + w]), dtype=torch.uint8, device="cuda")
            idx = (offsets[rows] + where[rows])[:, None] + ar[None, :]
            buf[idx.reshape(-1)] = lit.repeat(rows.numel())
    del lens, kind, where, which
    return buf, offsets, total


def tile_ragged_device(torch, buf_np, off_np, n):
    """replicate a host-generated ragged batch on the device until it holds n strings"""
    m = len(off_np) - 1
    reps = (n + m - 1) // m
    d_buf = torch.from_numpy(buf_np).cuda().repeat(reps)
    lens = torch.from_numpy(np.diff(off_np)).cuda().repeat(reps)[:n]
    offsets = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    torch.cumsum(lens, 0, out=offsets[1:])
    total = int(offsets[-1].item())
    return d_buf[:total].contiguous(), offsets, total


def build_workload(torch, cfg, units, rank, world=1):
    """returns dict(run=callable, text_bytes, units, verify=callable or None, host=(...) for e2e/cpu legs)"""
    import forgex_b200 as fx
    pat = synth.PATTERNS.get(cfg, synth.PATTERNS["c2"])
    op = synth.OPS.get(cfg, "in")
    w = {"cfg": cfg, "pattern": pat, "op": op}
    if cfg == "c2":
        p = fx.Pattern(pat, "in")
        buf, off, total = make_c2_device(torch, units, synth.SEEDS[cfg] + rank)
        out = torch.empty(units, dtype=torch.uint8, device="cuda")
        w.update(run=lambda: p.in_batch_dev(buf, off, units, total, out), text_bytes=total, units=units, out=out,
                 buf=buf, off=off, pattern_obj=p)
    elif cfg == "c2f":
        p = fx.Pattern(synth.PATTERNS["c2"], "in")
        g = torch.Generator(device="cuda")
        g.manual_seed(1234 + rank)
        stride = int(os.environ.get("FX_C2F_STRIDE", "160"))
        buf = torch.randint(0x20, 0x7F, (units * stride,), device="cuda", generator=g, dtype=torch.uint8)
        out = torch.empty(units, dtype=torch.uint8, device="cuda")
        w.update(run=lambda: p.in_fixed_dev(buf, units, stride, out), text_bytes=units * stride, units=units, out=out,
                 buf=buf, stride=stride, pattern_obj=p)
    elif cfg in ("c1", "c5"):
        gen = synth.gen_c1 if cfg == "c1" else synth.gen_c5
        block_n = min(units, 1 << 20)
        hb, _, stride = gen(block_n, seed_stream=rank)
        reps = (units + block_n - 1) // block_n
        buf = torch.from_numpy(hb).cuda().repeat(reps)[: units * stride].contiguous()
        out = torch.empty(units, dtype=torch.uint8, device="cuda")
        # c5: BASELINE states the config as the L2/HBM table path, so the table stays in global memory (FX_C5_AUTO=1: let
        # the library choose -- it then keeps the compact table in shared memory; reported beside it in the README)
        p = fx.Pattern(pat, op, residency="global" if cfg == "c5" and not os.environ.get("FX_C5_AUTO") else "auto")
        fn = p.match_fixed_dev if op == "match" else p.in_fixed_dev
        w.update(run=lambda: fn(buf, units, stride, out), text_bytes=units * stride, units=units, out=out, buf=buf,
                 stride=stride, pattern_obj=p)
    elif cfg == "c3":
        block_n = min(units, 1 << 17)
        hb, ho = synth.gen_c3(block_n, seed_stream=rank)
        buf, off, total = tile_ragged_device(torch, hb, ho, units)
        f = torch.empty(units, dtype=torch.int64, device="cuda")
        t = torch.empty(units, dtype=torch.int64, device="cuda")
        p = fx.Pattern(pat, "regex")
        w.update(run=lambda: p.regex_batch_dev(buf, off, units, total, f, t), text_bytes=total, units=units, out=f,
                 out2=t, buf=buf, off=off, pattern_obj=p)
    elif cfg == "c4":
        # ONE text of `units` bytes: a 256 MiB block of seeded log lines, cut at its last line end and tiled, with
        # exactly one fully matching line planted at byte fraction 0.999.  With world > 1 the text is cut into
        # slabs (forgex_b200.dist.slab_bounds) and this rank materialises only its slab + look-back + halo.
        from forgex_b200 import dist as fxd
        block = min(units, 256 << 20)
        hb = synth.gen_c4_block(block, seed_stream=0)
        last_nl = int(np.nonzero(hb == 10)[0][-1]) + 1
        d_block = torch.from_numpy(hb[:last_nl]).cuda()
        lo, hi = fxd.slab_bounds(units, world, rank)
        w_lo, w_hi = fxd.window_for_slab(units, lo, hi, 1 << 20) if world > 1 else (0, units)
        phase = w_lo % last_nl
        reps = (w_hi - w_lo + phase + last_nl - 1) // last_nl
        buf = d_block.repeat(reps)[phase:phase + (w_hi - w_lo)].contiguous()
        line = synth.C4_MATCH_LINE + b"\n"
        pos = int(units * 0.999)
        # the planted line starts at the last line start at or before `pos` of the TILED text (same on every rank)
        nls = np.nonzero(hb[:last_nl] == 10)[0]
        tpos = pos % last_nl
        k = int(np.searchsorted(nls, tpos, side="left")) - 1
        start = (pos - tpos) + (int(nls[k]) + 1 if k >= 0 else 0)
        plant = np.frombuffer(line + b"INFO ", dtype=np.uint8)
        a, b = max(start, w_lo), min(start + len(plant), w_hi)
        if b > a:
            buf[a - w_lo:b - w_lo] = torch.from_numpy(plant[a - start:b - start].copy()).cuda()
        ft = torch.zeros(2, dtype=torch.int64, device="cuda")
        p = fx.Pattern(pat, "regex")
        work = torch.zeros(p.buffer_work_bytes(units), dtype=torch.uint8, device="cuda")
        # by construction (SURVEY Q1): the span holds the LF that `^` consumed and the LF that `$` consumed
        crlf_before = start >= 2 and int(hb[(start - 1) % last_nl - 1]) == 13     # `^` = LF | CR LF | NUL: the CR is part of the match
        expect = (start - (1 if crlf_before else 0), start + len(line)) if start > 0 else (1, len(line))
        if world > 1:
            stats = {}

            def run_split():
                f, t, und = fxd.gpu_buffer_search(p, buf, w_lo, units, rank, world, (lo, hi), stats=stats)
                ft[0], ft[1] = f, t
                stats["undecided"] = und
            w.update(run=run_split, split=dict(slab=[lo, hi], window=[w_lo, w_hi], halo=1 << 20), stats=stats)
        else:
            w.update(run=lambda: p.regex_buffer_dev(buf, units, ft, work))
        w.update(text_bytes=units, units=1, out=ft, buf=buf, pattern_obj=p, expect_span=expect, planted_at=start,
                 window_lo=w_lo)
    else:
        raise SystemExit("unknown config " + cfg)
    return w


# ---- CPU legs (oracle; the only place bench.py executes oracle/) ------------------------------------
def _oracle_worker(args):
    cfg, buf, off, stride = args
    from tests import oracle_lib as O
    pat = synth.PATTERNS[cfg]
    op = synth.OPS[cfg]
    c = O.Compiled(pat, 1 if op == "match" else 0)
    t0 = time.perf_counter()
    if op == "regex":
        if off is None:
            r = c.regex_buffer(buf)
        else:
            r = c.regex_batch(buf, off)
    elif off is None:
        r = c.bool_fixed(1 if op == "match" else 0, buf, len(buf) // stride, stride)
    else:
        r = c.bool_batch(1 if op == "match" else 0, buf, off)
    return time.perf_counter() - t0, r


_REF_SHARDS = None


def _ref_step(i):
    return _oracle_worker(_REF_SHARDS[i])[0]


def host_sample(cfg, w, torch, nunits):
    """first nunits units of this rank's device data, on the host"""
    if cfg in ("c2", "c3"):
        off = w["off"][: nunits + 1].cpu().numpy().copy()
        buf = w["buf"][: int(off[-1])].cpu().numpy()
        return buf, off, None
    if cfg in ("c1", "c5"):
        return w["buf"][: nunits * w["stride"]].cpu().numpy(), None, w["stride"]
    return w["buf"][:nunits].cpu().numpy(), None, None


def cpu_baseline_leg(cfg, w, torch, target_seconds=12.0):
    """single-threaded oracle on a bounded prefix of the same data; also cross-checks the GPU results"""
    probe = {"c1": 20000, "c2": 4000, "c3": 3000, "c4": 1 << 20, "c5": 300}[cfg]
    buf, off, stride = host_sample(cfg, w, torch, probe)
    dt, _ = _oracle_worker((cfg, buf, off, stride))
    n = int(min(w["units"] if cfg != "c4" else w["text_bytes"], max(probe, probe * target_seconds / max(dt, 1e-6))))
    buf, off, stride = host_sample(cfg, w, torch, n)
    dt, res = _oracle_worker((cfg, buf, off, stride))
    nbytes = int(off[-1]) if off is not None else len(buf)
    ok = None
    if cfg in ("c1", "c2", "c5"):
        ok = bool(np.array_equal(w["out"][:n].cpu().numpy(), res))
    elif cfg == "c3":
        ok = bool(np.array_equal(w["out"][:n].cpu().numpy(), res[0]) and np.array_equal(w["out2"][:n].cpu().numpy(), res[1]))
    return {"value": nbytes / dt / 1e9, "unit": "GB/s", "cores": 1, "kind": "port",
            "sample": "first %d %s of rank 0's batch (%d bytes), oracle/forgex_oracle.cpp single thread, pattern compiled once"
                      % (n, "bytes" if cfg == "c4" else "strings", nbytes),
            "strings_per_s": (n / dt) if cfg != "c4" else None, "seconds": dt, "gpu_results_equal_oracle": ok}


def reference_arm(args):
    """--impl reference: the CPU restatement on all host cores, bounded sample per step"""
    import multiprocessing as mp
    cfg = args.config
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    per_core = {"c1": 400000, "c2": 40000, "c3": 30000, "c4": 4 << 20, "c5": 2500}[cfg]
    shards = []
    for c in range(cores):
        if cfg == "c2":
            b, o = synth.gen_c2(per_core, seed_stream=1000 + c)
            shards.append((cfg, b, o, None))
        elif cfg == "c3":
            b, o = synth.gen_c3(min(per_core, 8000), seed_stream=1000 + c)
            shards.append((cfg, b, o, None))
        elif cfg in ("c1", "c5"):
            b, _, s = (synth.gen_c1 if cfg == "c1" else synth.gen_c5)(per_core, seed_stream=1000 + c)
            shards.append((cfg, b, None, s))
        else:
            shards.append((cfg, synth.gen_c4(per_core, None, seed_stream=1000 + c), None, None))
    nbytes = sum(int(s[2][-1]) if s[2] is not None else len(s[1]) for s in shards)
    nunits = sum((len(s[2]) - 1) if s[2] is not None else (len(s[1]) // s[3] if s[3] else 1) for s in shards)
    from tests import oracle_lib as O
    O.build()
    global _REF_SHARDS
    _REF_SHARDS = shards          # inherited by the forked workers: a step only ships shard indices and timings
    times = []
    with mp.get_context("fork").Pool(cores) as pool:
        for it in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            pool.map(_ref_step, range(len(shards)), chunksize=1)
            dt = time.perf_counter() - t0
            if it >= args.warmup:
                times.append(dt)
    ms = 1000.0 * sum(times) / len(times)
    val = nbytes / (ms / 1000.0) / 1e9
    line = {
        "impl": "reference", "metric": "input_GBps", "value": val, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": WORKLOADS[cfg], "sample_strings_per_step": nunits, "sample_bytes_per_step": nbytes},
        "strings_per_s": nunits / (ms / 1000.0),
        "cpu_baseline": {"value": val, "unit": "GB/s", "cores": cores, "kind": "port",
                         "sample": "%d strings (%d bytes) per step, one oracle process per host core (fork pool), "
                                   "pattern compiled once per process per step" % (nunits, nbytes)},
        "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CPU restatement of Forgex's own per-character subset-step loop (oracle/); the Fortran original cannot "
                "be compiled in this image and carries extra allocation / formatted-I/O overhead (SURVEY 3.4)",
    }
    print(json.dumps(line))
    return 0



def numa_pin(local):
    """bind this rank to the host cores (and, by first touch, the memory) of its GPU's NUMA node: with 8 ranks copying
    4 GB each to their GPUs at once, unpinned ranks share whatever socket the scheduler put them on"""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        bus = bus.lower()
        if len(bus.split(":")[0]) == 8:
            bus = bus[4:]
        path = "/sys/bus/pci/devices/%s/local_cpulist" % bus
        cpus = set()
        for part in open(path).read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            node = open("/sys/bus/pci/devices/%s/numa_node" % bus).read().strip()
            return {"numa_node": int(node), "cpus": len(cpus)}
    except Exception as e:      # not fatal: the run is just not pinned
        return {"error": str(e)[:80]}
    return None


def verify_c4(torch, w, fx):
    """C4 parity at BASELINE size: (1) the span found in the full text equals the span known by construction (the
    planted line + the LF / CR LF consumed by `^` and the LF consumed by `$`, SURVEY Q1; offsets beyond 2^31 / 2^32);
    (2) the oracle and the GPU agree on a bounded slice of the same text that ends just behind the planted line."""
    got = tuple(int(x) for x in w["out"].cpu().tolist())
    rec = {"span": list(got), "expected_by_construction": list(w["expect_span"]), "span_equals_construction": got == tuple(w["expect_span"]),
           "offsets_beyond_2_31": got[0] > (1 << 31), "offsets_beyond_2_32": got[0] > (1 << 32)}
    return rec


def c4_oracle_slice(torch, w, nbytes=96 << 20):
    """oracle vs GPU on the last `nbytes` of the text up to just behind the planted line (single GPU only)"""
    from tests import oracle_lib as O
    end = min(w["text_bytes"], w["planted_at"] + 4096)
    a = max(0, end - nbytes)
    sl = w["buf"][a:end]
    host = sl.cpu().numpy()
    t0 = time.perf_counter()
    exp = O.Compiled(w["pattern"], 0).regex_buffer(host)
    dt = time.perf_counter() - t0
    ft = torch.zeros(2, dtype=torch.int64, device="cuda")
    work = torch.zeros(w["pattern_obj"].buffer_work_bytes(end - a), dtype=torch.uint8, device="cuda")
    w["pattern_obj"].regex_buffer_dev(sl.contiguous(), end - a, ft, work)
    got = tuple(int(x) for x in ft.cpu().tolist())
    full = tuple(int(x) for x in w["out"].cpu().tolist())
    return {"slice": [a, end], "oracle_span": list(exp), "gpu_span": list(got), "equal": got == tuple(exp),
            "full_text_span_is_slice_span_plus_offset": exp[0] > 0 and full == (exp[0] + a, exp[1] + a),
            "oracle_seconds": dt, "oracle_GBps": (end - a) / dt / 1e9}


def measure_config(cfg, args, env):
    """one BASELINE config at full size on this rank's GPU: device-timed steps, e2e through the host-pointer ABI, CPU leg"""
    torch, dist, fx = env["torch"], env["dist"], env["fx"]
    world, rank, local = env["world"], env["rank"], env["local"]
    units = (args.lines if args.config == cfg else 0) or DEFAULT_UNITS[cfg]
    w = build_workload(torch, cfg, units, rank, world)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        w["run"]()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = fx.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        w["run"]()
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = fx.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    if args.dump_outputs and rank == 0:
        # what the last timed step handed its caller (every step overwrites the same output tensors)
        if cfg == "c3":
            dump_output(torch, args.dump_outputs, "c3_from", w["out"])
            dump_output(torch, args.dump_outputs, "c3_to", w["out2"])
        else:
            dump_output(torch, args.dump_outputs, cfg + "_span" if cfg == "c4" else cfg, w["out"])

    split = cfg == "c4" and world > 1
    # match counts: the only cross-GPU exchange of a sharded batch (8 bytes per rank), outside the timed region
    if cfg == "c4":
        count = torch.tensor([int(w["out"][0].item() > 0)], dtype=torch.int64, device="cuda")
    elif cfg == "c3":
        count = (w["out"] > 0).sum().to(torch.int64).reshape(1)
    else:
        count = w["out"].sum(dtype=torch.int64).reshape(1)
    if world > 1 and not split:
        dist.all_reduce(count)
    text_bytes_all = w["text_bytes"] * (1 if split else world)
    units_all = (w["units"] if cfg != "c4" else 1) * (1 if split else world)
    value = text_bytes_all / (ms_step / 1000.0) / 1e9

    verified = {}
    general = None
    if cfg == "c2" and not os.environ.get("FX_BENCH_NO_GENERAL"):
        # the same batch through the GENERAL walker (K2): `\w+@\w+` has a dense first-byte set, so it cannot take the
        # sparse-start kernel the headline pattern runs on -- it is what most patterns get
        gp = fx.Pattern(rb"\w+@\w+", "in")
        gout = torch.empty(w["units"], dtype=torch.uint8, device="cuda")
        grun = lambda: gp.in_batch_dev(w["buf"], w["off"], w["units"], w["text_bytes"], gout)
        for _ in range(args.warmup):
            grun()
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(args.steps):
            grun()
        g1.record()
        barrier()
        gt = torch.tensor([g0.elapsed_time(g1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(gt, op=dist.ReduceOp.MAX)
        gms = float(gt.item()) / args.steps
        if args.dump_outputs and rank == 0:
            dump_output(torch, args.dump_outputs, "c2_general", gout)
        general = {"pattern": "\\w+@\\w+", "op": ".in.", "ms_per_step": gms, "value": w["text_bytes"] * world / (gms / 1000.0) / 1e9, "unit": "GB/s",
                   "sparse_used": gp.info()["sparse_used"], "matches_rank0": int(gout.sum(dtype=torch.int64).item())}
        if rank == 0 and world == 1 and not args.no_cpu:
            from tests import oracle_lib as O
            ns = 60000
            off = w["off"][: ns + 1].cpu().numpy().copy()
            hb = w["buf"][: int(off[-1])].cpu().numpy()
            general["gpu_results_equal_oracle"] = bool(np.array_equal(gout[:ns].cpu().numpy(), O.Compiled(rb"\w+@\w+", 0).bool_batch(0, hb, off)))
            general["oracle_sample_strings"] = ns
        del gout
    if cfg == "c4":
        verified.update(verify_c4(torch, w, fx))
        if split:
            verified["undecided_attempts"] = w["stats"].get("undecided")
            verified["halo_widenings"] = w["stats"].get("widenings")

    # ---- e2e: host-pointer C-ABI call, pinned host buffers, H2D + kernel + D2H inside the timed region ----
    e2e = None
    if not args.no_e2e:
        p = w["pattern_obj"]
        n_e = min(w["units"], args.e2e_lines or {"c1": 1 << 27, "c2": 25_000_000, "c3": 8_000_000, "c5": 10_000_000}.get(cfg, 0))
        if cfg == "c4":
            nb = min(w["buf"].numel(), 4 << 30)
            hbuf = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
            hbuf.copy_(w["buf"][:nb])
            call = lambda: p.regex_buffer(hbuf.numpy())
            h2d, d2h, ebytes, eunits = nb, 16, nb, 1
        elif cfg in ("c2", "c3"):
            off = w["off"][: n_e + 1]
            nb = int(off[-1].item())
            hbuf = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
            hbuf.copy_(w["buf"][:nb])
            hoff = torch.empty(n_e + 1, dtype=torch.int64, pin_memory=True)
            hoff.copy_(off)
            hb, ho = hbuf.numpy(), hoff.numpy()
            # results land in caller-provided pinned buffers (what a host program that cares about throughput passes)
            if cfg == "c2":
                hout = torch.empty(n_e, dtype=torch.uint8, pin_memory=True).numpy()
                call = lambda: p.in_batch(hb, ho, out=hout)
            else:
                hf = torch.empty(n_e, dtype=torch.int64, pin_memory=True).numpy()
                ht = torch.empty(n_e, dtype=torch.int64, pin_memory=True).numpy()
                call = lambda: p.regex_batch(hb, ho, out=(hf, ht))
            h2d, d2h, ebytes, eunits = nb + 8 * (n_e + 1), n_e * (1 if cfg == "c2" else 16), nb, n_e
        else:
            nb = n_e * w["stride"]
            hbuf = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
            hbuf.copy_(w["buf"][:nb])
            hb = hbuf.numpy()
            fn = p.match_fixed if cfg == "c1" else p.in_fixed
            hout = torch.empty(n_e, dtype=torch.uint8, pin_memory=True).numpy()
            call = lambda: fn(hb, n_e, w["stride"], out=hout)
            h2d, d2h, ebytes, eunits = nb, n_e, nb, n_e
        call()  # warm-up (grows the library's device scratch)
        barrier()
        # the platform's ceiling beside it: the bare pinned H2D copy of the same bytes, all ranks at once
        dscratch = torch.empty(nb, dtype=torch.uint8, device="cuda")
        dscratch.copy_(hbuf, non_blocking=True)
        barrier()
        t0 = time.perf_counter()
        dscratch.copy_(hbuf, non_blocking=True)
        torch.cuda.synchronize()
        dt_copy = time.perf_counter() - t0
        del dscratch
        barrier()
        reps = 3
        t0 = time.perf_counter()
        for _ in range(reps):
            res = call()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / reps
        tt = torch.tensor([dt, dt_copy], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt, dt_copy = (float(x) for x in tt.tolist())
        e2e = {"value": ebytes * world / dt / 1e9, "unit": "GB/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "strings_per_step_per_gpu": int(eunits), "ms_per_step": dt * 1000.0, "strings_per_s": eunits * world / dt,
               "bare_pinned_h2d_GBps_all_ranks": nb * world / dt_copy / 1e9,
               "api": "forgex_b200.Pattern.%s (fx_*_batch / fx_*_fixed host-pointer entry points)" %
                      {"c1": "match_fixed", "c2": "in_batch", "c3": "regex_batch", "c4": "regex_buffer", "c5": "in_fixed"}[cfg]}
        if cfg == "c4" and world == 1:
            e2e["note"] = "first 4 GiB of the text (no match in it): one host buffer, one call"
        del hbuf

    rec = None
    if rank == 0:
        peak, peak_src = measured_peak()
        algo_bytes = w["text_bytes"] + EXTRA_BYTES[cfg] * (w["units"] if cfg != "c4" else 0)
        if split:
            algo_bytes = w["split"]["slab"][1] - w["split"]["slab"][0]
        kernel_ms = ms_step
        achieved = algo_bytes / (kernel_ms / 1000.0) / 1e9
        rec = {
            "metric": "input_GBps", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if split else "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": WORKLOADS[cfg], "strings_per_gpu": w["units"] if cfg != "c4" else 1,
                       "text_bytes_per_gpu": int(w["buf"].numel()) if split else w["text_bytes"],
                       "pattern": synth.PATTERNS.get(cfg, synth.PATTERNS["c2"]).decode("utf-8"),
                       "l2": "inputs larger than L2 (no flush needed)" if w["text_bytes"] > (256 << 20) else "input fits L2: latency-bound case",
                       "table": w["pattern_obj"].info()},
            "strings_per_s": units_all / (ms_step / 1000.0),
            "matches": int(count.item()),
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": known_traffic(cfg, algo_bytes), "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": int(algo_bytes), "kernel_ms": kernel_ms},
            "e2e": e2e,
        }
        if split:
            rec["config"]["split"] = ("ONE text of %d bytes cut into %d slabs (forgex_b200.dist.slab_bounds), 1 MiB look-ahead halo, "
                                      "one all-gather of 3 int64 + one 16-byte all-reduce per search, inside the timed region"
                                      % (w["text_bytes"], world))
            rec["roofline"]["note"] = "per GPU: this rank's slab bytes / step time (the step includes the two collectives and their host syncs)"
            # what the collectives cost: the same search on the same slabs minus the local scan alone
            stats = w["stats"]
            rec["collectives"] = {"per_search": "all_gather(3 x int64) + all_reduce(2 x int64)", "scan_rounds": stats.get("scan_rounds", 0) // max(1, args.steps + args.warmup)}
        if general is not None:
            peak_g, _ = measured_peak()
            ab = w["text_bytes"] + EXTRA_BYTES[cfg] * w["units"]
            general["roofline_frac"] = ab / (general["ms_per_step"] / 1000.0) / 1e9 / peak_g
            rec["general_walker"] = general
        if verified:
            rec["verified"] = verified
        if not args.no_cpu and world == 1:
            rec["cpu_baseline"] = cpu_baseline_leg(cfg, w, torch, target_seconds=args.cpu_seconds if cfg != "c2" else max(args.cpu_seconds, 12.0))
            if cfg == "c4":
                rec["verified"]["oracle_slice"] = c4_oracle_slice(torch, w)
                rec["cpu_baseline"]["gpu_results_equal_oracle"] = bool(rec["verified"]["oracle_slice"]["equal"] and
                                                                       rec["verified"]["span_equals_construction"])
    if split:
        # time of the collectives alone (same tensors, no scan), max over ranks: named in microseconds
        from forgex_b200 import dist as fxd
        span = torch.zeros(2, dtype=torch.int64, device="cuda")
        for _ in range(3):
            fxd.gather_ints((1, 0, 0), None, span.device)
            dist.all_reduce(span)
        barrier()
        t0 = time.perf_counter()
        for _ in range(20):
            fxd.gather_ints((1, 0, 0), None, span.device)
            dist.all_reduce(span)
            span.cpu()
        dtc = (time.perf_counter() - t0) / 20
        tc = torch.tensor([dtc], dtype=torch.float64, device="cuda")
        dist.all_reduce(tc, op=dist.ReduceOp.MAX)
        if rec is not None:
            rec["collectives"]["us_per_search"] = float(tc.item()) * 1e6
    del w
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="all", choices=sorted(WORKLOADS) + ["all"])
    ap.add_argument("--lines", type=int, default=0, help="units per GPU (strings; bytes for c4); default = BASELINE size")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--e2e-lines", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=6.0, help="target length of each cpu_baseline leg (c2: at least 12 s)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-pin", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step of each measured config computed (rank 0) as DIR/<name>.npy, "
                         "float32 (float64 for int64 spans); outputs longer than %d elements as a fixed seeded sample"
                         % DUMP_MAX_ELEMS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        if args.impl == "reference":
            ap.error("--dump-outputs records the GPU path's outputs; the reference arm runs other inputs")
        os.makedirs(args.dump_outputs, exist_ok=True)
    if args.warmup < 3 and args.impl == "b200" and not os.environ.get("FX_BENCH_ALLOW_SHORT_WARMUP"):
        args.warmup = 3
    if args.impl == "reference":
        if args.config == "all":
            args.config = "c2"
        return reference_arm(args)

    import torch
    import torch.distributed as dist
    import forgex_b200 as fx

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the matching path has no CPU fallback")
    pin = None if args.no_pin else numa_pin(local)
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    env = {"torch": torch, "dist": dist, "fx": fx, "world": world, "rank": rank, "local": local}
    if args.config != "all":
        line = measure_config(args.config, args, env)
    else:
        # the headline is c2 (BASELINE.json configs[1]); every BASELINE config is measured in the same run
        recs = {}
        for cfg in ("c2", "c1", "c3", "c4", "c5"):
            t0 = time.perf_counter()
            recs[cfg] = measure_config(cfg, args, env)
            if rank == 0:
                recs[cfg]["wall_seconds_incl_setup"] = time.perf_counter() - t0
        line = None
        if rank == 0:
            line = dict(recs["c2"])
            keep = ("value", "unit", "ms_per_step", "scaling", "strings_per_s", "matches", "gpu_launches", "roofline", "e2e",
                    "cpu_baseline", "verified", "collectives", "clocks", "config", "wall_seconds_incl_setup", "general_walker")
            line["per_config"] = {c: {k: r[k] for k in keep if k in r} for c, r in recs.items()}
            for c, r in line["per_config"].items():
                r["config"] = {k: v for k, v in r["config"].items() if k != "table"} | {"kernel_path": {
                    k: recs[c]["config"]["table"].get(k) for k in ("byte_states", "residency", "direct", "sparse_used", "prefix_mode")}}
    if rank == 0:
        if pin:
            line["numa_pin"] = pin
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
