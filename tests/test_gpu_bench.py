"""bench.py's GPU arm with --dump-outputs: the proofs its last timed steps returned are written as float32 arrays, equal
to the oracle prover's bytes for the same configuration (cfg2, which the CPU oracle proves in seconds)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_are_the_proof(oracle, tmp_path):
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--config", "cfg2", "--steps", "2", "--warmup", "1", "--no-cpu-baseline",
           "--no-sub-record", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 2
    assert sorted(os.listdir(out)) == ["proof.npy", "proof_e2e.npy"]
    res, e2e = np.load(out / "proof.npy"), np.load(out / "proof_e2e.npy")
    assert res.dtype == e2e.dtype == np.float32 and res.size == line["proof_bytes"]
    assert (res == e2e).all()

    import bench
    pairs, log_n, ext = bench.CONFIGS["cfg2"]
    trace, results = oracle.build_fib_trace(pairs, 1 << log_n)
    want = oracle.prove_fib(trace, results, bench.proof_opts(ext))
    assert (res == np.frombuffer(want, dtype=np.uint8)).all()
