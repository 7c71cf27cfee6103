"""wf_prove_air_sharded: one proof of an AIR description over several ranks must be byte-identical to wf_prove_air on one
GPU (which the other GPU tests pin to the oracle), the same on every rank, and leave no device buffer behind; arguments one
rank refuses must make every rank return an error. The ranks share GPU 0 and use gloo through host staging
(tests/sharded_air_worker.py runs a list of cases per launch); the NCCL path is the same library code with device-to-device
transfers (tools/bench_air_sharded.py)."""
import json
import os
import socket
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FRI5 = {"WF_SHARD_FRI_MIN_LOG": 5}   # FRI layers folded on shards down to tiny ranges


def _run(world, cases):
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "sharded_air_worker.py"), json.dumps(cases)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ))
    assert r.returncode == 0, r.stdout[-6000:] + r.stderr[-4000:]
    assert r.stdout.count(": ok ") == len(cases), r.stdout[-6000:]


# narrow AIRs: one rank owns every column, the others none (they still take part in every collective)
NARROW = [{"air": "mulfib2", "ext": 1, "env": FRI5},
          {"air": "periodic_mix", "ext": 2, "env": FRI5},                  # periodic columns, 2 exemptions, periodic assertion
          {"air": "sequence_mix", "ext": 3, "log_n": 13, "env": FRI5}]     # sequence-assertion tables
# degree 7 (constraint-evaluation blowup 8), several composition columns: interpreter and NVRTC kernel
RESCUE = [{"air": "rescue_like", "arg": 6, "ext": 2, "jit": 0, "env": FRI5},
          {"air": "rescue_like", "arg": 6, "ext": 3, "jit": 1, "env": FRI5}]
# 24 columns = 3 segments: an uneven split, at 4 ranks one rank owns nothing
WIDE = [{"air": "fib_small_x", "arg": 12, "ext": 1, "env": FRI5}]


def test_sharded_air_two_ranks():
    _run(2, NARROW + RESCUE + WIDE + [
        {"air": "fib_small_x", "arg": 6, "ext": 2, "env": FRI5},           # 12 columns: one full and one partial segment
        {"air": "fib_small_x", "arg": 8, "ext": 3, "fib": 1, "env": FRI5},  # also equal to wf_prove_fib_sharded's bytes
        {"air": "rescue_like", "arg": 6, "ext": 2, "oracle": 1, "env": FRI5},   # the oracle prover's bytes, accepted by its verifier
    ])


def test_sharded_air_four_ranks():
    _run(4, NARROW + RESCUE + WIDE)


def test_sharded_air_options_and_transports():
    # the same proof with every other option and transport: Rp64_256, PartitionOptions(2, 8), columns resident in HBM,
    # Montgomery input, the communicator's exchange (WF_PEER_PUSH=0), the LDE's fused scatter (WF_FUSED_SCATTER=1: taken for an
    # even split of whole segments, the copy-engine push otherwise), the default FRI sharding threshold
    _run(2, [
        {"air": "periodic_mix", "ext": 1, "hash": 1, "env": {"WF_SHARD_FRI_MIN_LOG": 6}},
        {"air": "fib_small_x", "arg": 6, "ext": 3, "parts": 2, "rate": 8, "env": FRI5},
        {"air": "rescue_like", "arg": 6, "ext": 2, "resident": 1, "log_n": 13},
        {"air": "fib_small_x", "arg": 12, "ext": 2, "resident": 1, "env": FRI5},
        {"air": "fib_small_x", "arg": 6, "ext": 1, "mont": 1, "env": FRI5},
        {"air": "fib_small_x", "arg": 12, "ext": 3, "env": {"WF_PEER_PUSH": 0, "WF_SHARD_FRI_MIN_LOG": 5}, "peer_push": 0},
        {"air": "sequence_mix", "ext": 2, "env": {"WF_PEER_PUSH": 0}, "peer_push": 0},
        {"air": "fib_small_x", "arg": 8, "ext": 3, "env": {"WF_FUSED_SCATTER": 1}, "peer_push": 2},
        {"air": "fib_small_x", "arg": 6, "ext": 2, "env": {"WF_FUSED_SCATTER": 1}, "peer_push": 1},
    ])


def test_sharded_air_refusals():
    # each refused on every rank with an error (and no device buffer left); -3 = WF_ERR_UNSUPPORTED, -2 = WF_ERR_INVALID
    _run(2, [
        {"air": "mulfib2", "refuse": "aux", "code": -3},                # auxiliary segment
        {"air": "rescue_like", "arg": 6, "refuse": "short", "code": -3},  # too few rows for the world
        {"air": "fib_small_x", "arg": 6, "refuse": "opts", "code": -2},   # one rank passes other options
        {"air": "fib_small_x", "arg": 6, "refuse": "cols", "code": -2},   # one rank passes a wrong number of columns
        {"air": "mulfib2", "refuse": "cols", "code": -2},
        {"air": "mulfib2", "ext": 2, "env": FRI5},                       # and the context still proves afterwards
    ])


def test_sharded_air_refuses_world_three():
    _run(3, [{"air": "mulfib2", "refuse": "world", "code": -2}, {"air": "fib_small_x", "arg": 12, "refuse": "world", "code": -2}])
