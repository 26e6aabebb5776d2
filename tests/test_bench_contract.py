"""Checks of bench.py.  On the CPU: the committed DRAM-traffic figures it reports, the reference arm's JSON line, and the
product arm's refusal to run without a device (no CPU fallback).  On the GPU: the outputs --dump-outputs writes."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_traffic_figures_are_tied_to_the_workload_they_were_captured_on():
    import bench
    with open(os.path.join(ROOT, "profiles", "traffic.json")) as fh:
        t = json.load(fh)
    for cfg in ("c1", "c2", "c3", "c4", "c5"):
        e = t[cfg]
        assert os.path.exists(os.path.join(ROOT, e["source"])), e["source"]
        assert e["bytes"] >= e["algorithmic_bytes"] > 0                       # a kernel cannot read less than its input
        assert bench.known_traffic(cfg, e["algorithmic_bytes"]) == e["bytes"]
        assert bench.known_traffic(cfg, e["algorithmic_bytes"] // 2) is None   # another size: no figure rather than a wrong one
    assert bench.known_traffic("nope", 1) is None


def test_reference_arm_prints_the_contract_line_and_product_arm_needs_a_device():
    import torch
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--cpu-seconds", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-500:]
    line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "input_GBps" and line["unit"] == "GB/s" and line["higher_is_better"] is True
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["value"] > 0
    assert line["e2e"] == {"value": line["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    if not torch.cuda.is_available():
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert r.returncode != 0 and "no CPU fallback" in (r.stdout + r.stderr)


@pytest.mark.gpu
def test_dump_outputs_are_what_the_timed_steps_computed(tmp_path):
    """--dump-outputs writes the last timed step's results: a whole c3 span batch, and the seeded sample of a c1 batch
    longer than the dump keeps, each against the oracle on the same strings; --steps is the number of timed steps"""
    import bench
    from tests import oracle_lib as O
    from tools import synth
    for cfg, n in (("c3", 3000), ("c1", bench.DUMP_MAX_ELEMS + 12345)):
        d = tmp_path / cfg
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", cfg, "--lines", str(n), "--steps", "2",
                            "--warmup", "3", "--no-cpu", "--no-e2e", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == 2
        if cfg == "c3":
            assert sorted(os.listdir(d)) == ["c3_from.npy", "c3_to.npy"]
            f, t = np.load(d / "c3_from.npy"), np.load(d / "c3_to.npy")
            assert f.dtype == t.dtype == np.float64
            ef, et = O.Compiled(synth.PATTERNS["c3"], 0).regex_batch(*synth.gen_c3(n))
            assert np.array_equal(f, ef) and np.array_equal(t, et)
        else:
            assert os.listdir(d) == ["c1.npy"]
            got = np.load(d / "c1.npy")
            assert got.dtype == np.float32 and len(got) == bench.DUMP_MAX_ELEMS
            block, _, stride = synth.gen_c1(1 << 20)      # bench.py tiles a block of 2^20 strings
            rows = block.reshape(-1, stride)[bench.dump_index(n) % (1 << 20)].reshape(-1)
            exp = O.Compiled(synth.PATTERNS["c1"], 1).bool_fixed(1, rows, len(got), stride)
            assert np.array_equal(got, exp)
