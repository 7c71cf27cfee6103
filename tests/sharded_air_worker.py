"""One rank of the sharded-AIR GPU test (tests/test_gpu_sharded_air.py): `world` processes share GPU 0 and talk over gloo
(TorchComm's host-staged mode). One process runs a list of cases (argv[1]: JSON), so the torch import is paid once per launch.

Proof case: every rank proves its columns (wf.shard_columns) with wf_prove_air_sharded; rank 0 compares the bytes with
ctx.prove_air on the whole trace (and, on request, with wd.prove_fib_sharded and the oracle prover / verifier); every rank
must hold the same bytes and no live device buffer afterwards.
Refusal case: every rank must get an error and keep no live device buffer."""
import hashlib
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

ENV_KEYS = ("WF_SHARD_FRI_MIN_LOG", "WF_PEER_PUSH", "WF_FUSED_SCATTER")


def build_air(name, arg, n):
    import airs
    if name == "fib_small_x":
        return airs.fib_small_x(arg, n)
    if name == "rescue_like":
        return airs.rescue_like(n, arg)
    return getattr(airs, name)(n)[:2]


def all_ranks_agree(flag):
    t = torch.tensor([1 if flag else 0], dtype=torch.int64)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(t.item())


def same_bytes_everywhere(proof, world):
    digest = torch.frombuffer(bytearray(hashlib.sha256(proof).digest()), dtype=torch.uint8)
    all_d = [torch.empty_like(digest) for _ in range(world)]
    dist.all_gather(all_d, digest)
    return all(bool((d == all_d[0]).all()) for d in all_d)


def run_case(case, ctx, comm, rank, world):
    import winterfell_b200 as wf
    from winterfell_b200 import dist as wd
    from oracle import oracle as O
    for k in ENV_KEYS:
        os.environ.pop(k, None)
    os.environ.update({k: str(v) for k, v in case.get("env", {}).items()})
    log_n = case.get("log_n", 12)
    n = 1 << log_n
    desc, trace = build_air(case["air"], case.get("arg"), n)
    opts = O.make_opts(num_queries=24, blowup=8, grinding=6, ext=case.get("ext", 1), folding=4, rem_max_deg=31,
                       hash_id=case.get("hash", 0), num_partitions=case.get("parts", 1), hash_rate=case.get("rate", 1))
    ctx.set_jit(case.get("jit", 1))
    try:
        first, count = wf.shard_columns(trace.shape[0], world, rank)
    except wf.WfError:   # a world the library refuses: rank 0 passes everything
        first, count = 0, trace.shape[0] if rank == 0 else 0
    local = np.ascontiguousarray(trace[first:first + count])
    refuse = case.get("refuse")
    if refuse:
        lg = log_n
        if refuse == "aux":
            import airs
            desc, trace, _ = airs.perm_rap(n)
        elif refuse == "short":
            lg = 6
            local = np.ascontiguousarray(local[:, : 1 << lg])
        elif refuse == "opts" and rank == world - 1:
            opts = opts.copy()
            opts[0] += 1
        elif refuse == "cols" and rank == world - 1:
            local = np.ascontiguousarray(local[:-1])
        try:
            wd.prove_air_sharded(ctx, comm, desc, local, lg, opts)
            err = None
        except wf.WfError as e:
            err = str(e)
        live = ctx.mem_stats()[0]
        want = case.get("code")
        ok = err is not None and (want is None or err.startswith(f"error {want}:")) and live == 0
        return all_ranks_agree(ok), f"refusal {refuse}: {err} live={live}"
    mont = case.get("mont", 0)
    if mont:
        local = np.vectorize(lambda v: O.to_mont(int(v)), otypes=[np.uint64])(local) if count else local
    stats = {}
    if case.get("resident") and count:
        dev = torch.from_numpy(local.view(np.int64)).cuda()
        proof = wd.prove_air_sharded(ctx, comm, desc, None, log_n, opts, mont=mont, device_ptr=dev.data_ptr(), stats=stats)
        del dev
    else:
        proof = wd.prove_air_sharded(ctx, comm, desc, local, log_n, opts, mont=mont, stats=stats)
    ok, note = True, ""
    if rank == 0:
        want = ctx.prove_air(desc, trace, opts)
        ok = proof == want
        note = f"sharded {len(proof)} bytes, single-GPU {len(want)}, equal={ok}, stats={stats}"
        if case.get("oracle"):
            ok = ok and proof == O.prove_air(desc, trace, opts) and O.verify_air(desc, proof, int(opts[8]) & 0xff) == 0
            note += f", oracle={ok}"
    if case.get("fib"):   # the same trace through the FibSmall entry point (its own kernel): the same bytes
        k = trace.shape[0] // 2
        res = np.array([int(trace[2 * j + 1, n - 1]) for j in range(k)], dtype=np.uint64)
        fproof = wd.prove_fib_sharded(ctx, comm, local, k, log_n, res, opts)
        ok = ok and fproof == proof
    if "peer_push" in case:
        ok = ok and stats.get("peer_push") == case["peer_push"]
    ctx.sync()
    ok = ok and same_bytes_everywhere(proof, world) and ctx.mem_stats()[0] == 0
    return all_ranks_agree(ok), note


def main():
    cases = json.loads(sys.argv[1])
    dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    import winterfell_b200 as wf
    from winterfell_b200 import dist as wd
    torch.cuda.set_device(0)
    stream = torch.cuda.Stream()
    ctx = wf.Context(0, stream.cuda_stream)
    comm = wd.TorchComm(stream)
    failed = 0
    with torch.cuda.stream(stream):
        for case in cases:
            ok, note = run_case(case, ctx, comm, rank, world)
            if rank == 0:
                print(f"case {json.dumps(case)}: {'ok' if ok else 'FAILED'} {note}", flush=True)
            failed += 0 if ok else 1
    ctx.close()
    dist.destroy_process_group()
    sys.exit(1 if failed else 0)


if __name__ == "__main__":
    main()
