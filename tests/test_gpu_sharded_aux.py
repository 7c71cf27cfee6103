"""wf_prove_air_aux_sharded: one proof of a two-segment AIR over several ranks must be byte-identical to wf_prove_air_aux (or
wf_prove_air_aux_dyn) on one GPU, the same on every rank, leave no device buffer behind, and call each rank's aux builder once
with exactly the E columns covering its aux base columns; a refusal or a failing callback on one rank must make every rank
return an error. The ranks share GPU 0 and use gloo through host staging (tests/sharded_aux_worker.py runs a list of cases
per launch)."""
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
           "--master-port", str(port), os.path.join(ROOT, "tests", "sharded_aux_worker.py"), json.dumps(cases)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ))
    assert r.returncode == 0, r.stdout[-6000:] + r.stderr[-4000:]
    assert r.stdout.count(": ok ") == len(cases), r.stdout[-6000:]


# perm_rap: 3 main columns (one rank owns them all), aux 3 E columns = 3, 6 or 9 base columns; at ext 3 the 9 base columns
# are 2 segments, so at 2 ranks E column 2 straddles them and rank 1 owns aux columns but no main column
PERM_RAP = [{"air": "perm_rap", "ext": 1, "env": FRI5},
            {"air": "perm_rap", "ext": 2, "env": FRI5},
            {"air": "perm_rap", "ext": 3, "env": FRI5}]
# perm_rap_lanes: 9 main columns (2 segments), 9 E aux columns = 18 or 27 base columns: uneven splits, and at 4 ranks a rank
# that owns nothing; interpreter (jit 0) and NVRTC kernel (jit 1) with the aux program on row shards
LANES = [{"air": "perm_rap_lanes", "ext": 2, "jit": 0, "env": FRI5},
         {"air": "perm_rap_lanes", "ext": 3, "jit": 1, "env": FRI5},
         {"air": "perm_rap_lanes", "ext": 2, "jit": 1, "env": FRI5},
         {"air": "perm_rap_lanes", "ext": 3, "jit": 0, "env": FRI5}]
# aux assertion values computed from the random elements (values_fn on every rank)
DYN = [{"air": "perm_rap", "dyn": 1, "ext": 3, "env": FRI5}]


def test_sharded_aux_two_ranks():
    _run(2, PERM_RAP + LANES + DYN + [
        {"air": "perm_rap", "ext": 2, "oracle": 1, "env": FRI5},                 # the oracle prover's bytes, its verifier accepts
        {"air": "perm_rap", "dyn": 1, "ext": 2, "oracle": 1, "env": FRI5},
    ])


def test_sharded_aux_four_ranks():
    _run(4, PERM_RAP + LANES + DYN)


def test_sharded_aux_options_and_transports():
    # Rp64_256, PartitionOptions(2, 8) on all three commitments, main columns resident in HBM, Montgomery input (random
    # elements and builder output too), the communicator's exchange (WF_PEER_PUSH=0), the fused LDE scatter (WF_FUSED_SCATTER=1)
    # where both segments split evenly (rap_sums at ext 2: 16 + 16 base columns) and where they do not (perm_rap_lanes at
    # ext 3: 9 + 27, which takes the copy-engine push), the default FRI sharding threshold
    _run(2, [
        {"air": "perm_rap", "ext": 2, "hash": 1, "env": {"WF_SHARD_FRI_MIN_LOG": 6}},
        {"air": "perm_rap_lanes", "ext": 3, "parts": 2, "rate": 8, "env": FRI5},
        {"air": "perm_rap_lanes", "ext": 2, "resident": 1, "log_n": 13},
        {"air": "perm_rap", "ext": 3, "mont": 1, "env": FRI5},
        {"air": "perm_rap_lanes", "ext": 3, "env": {"WF_PEER_PUSH": 0, "WF_SHARD_FRI_MIN_LOG": 5}, "peer_push": 0},
        {"air": "rap_sums", "ext": 2, "env": {"WF_FUSED_SCATTER": 1}, "peer_push": 2},
        {"air": "perm_rap_lanes", "ext": 3, "env": {"WF_FUSED_SCATTER": 1}, "peer_push": 1},
    ])


def test_sharded_aux_refusals():
    # each refused on every rank with an error (and no device buffer left), then the context proves again; -3 =
    # WF_ERR_UNSUPPORTED, -2 = WF_ERR_INVALID
    _run(2, [
        {"air": "perm_rap", "refuse": "single", "code": -2},                    # a single-segment description
        {"air": "perm_rap", "ext": 2, "refuse": "builder", "code": -2},         # the builder fails on one rank only
        {"air": "perm_rap", "dyn": 1, "ext": 2, "refuse": "values", "code": -2},   # values_fn differs on one rank
        {"air": "perm_rap", "refuse": "null_builder", "code": -2},              # no builder on one rank
        {"air": "perm_rap_lanes", "ext": 2, "refuse": "short", "code": -3},     # too few rows for the world
        {"air": "perm_rap", "ext": 3, "env": FRI5},                             # and the context still proves afterwards
    ])


def test_sharded_aux_refuses_world_three():
    _run(3, [{"air": "perm_rap", "refuse": "world", "code": -2}, {"air": "perm_rap_lanes", "ext": 2, "refuse": "world", "code": -2}])
