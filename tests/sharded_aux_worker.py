"""One rank of the sharded two-segment AIR GPU test (tests/test_gpu_sharded_aux.py): `world` processes share GPU 0 and talk
over gloo (TorchComm's host-staged mode). One process runs a list of cases (argv[1]: JSON), so the torch import is paid once
per launch.

Proof case: every rank proves its main columns (wf.shard_columns) with wf_prove_air_aux_sharded and builds only the aux
columns it owns; rank 0 compares the bytes with ctx.prove_air_aux (or prove_air_aux_dyn) on the whole trace (and, on request,
with the oracle prover and verifier); every rank must hold the same bytes and no live device buffer afterwards, and each
rank's builder must have been called with exactly the E columns covering its aux base columns (or not at all).
Refusal case: every rank must get an error and keep no live device buffer, and the context must prove afterwards."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from sharded_air_worker import ENV_KEYS, all_ranks_agree, same_bytes_everywhere  # noqa: E402


def build_air(case, n):
    """(description, trace, full builder(rand), builder of a column range (rand, first_col, num_cols), values_fn or None)."""
    import airs
    import airs_aux
    if case["air"] in ("perm_rap_lanes", "rap_sums"):
        desc, trace, full = getattr(airs_aux, case["air"])(n)
        return desc, trace, full, full.columns, None
    desc, trace, full = airs.perm_rap(n, dyn_last_q=bool(case.get("dyn")))
    return desc, trace, full, lambda rand, f, c: full(rand)[f:f + c], (full.values_fn if case.get("dyn") else None)


def expected_call(aw, d, world, rank):
    """The E columns wf_prove_air_aux_sharded asks this rank's builder for: those covering its aux base columns, or None."""
    import winterfell_b200 as wf
    first, count = wf.shard_columns(aw * d, world, rank)
    if not count:
        return None
    return first // d, -(-(first + count) // d) - first // d


def mont_map(fn, a):
    return np.frompyfunc(lambda v: fn(int(v)), 1, 1)(a).astype(np.uint64)


def run_case(case, ctx, comm, rank, world):
    import winterfell_b200 as wf
    from winterfell_b200 import dist as wd
    from oracle import oracle as O
    for k in ENV_KEYS:
        os.environ.pop(k, None)
    os.environ.update({k: str(v) for k, v in case.get("env", {}).items()})
    log_n = case.get("log_n", 12)
    n = 1 << log_n
    ext = case.get("ext", 1)
    desc, trace, full, cols_fn, values_fn = build_air(case, n)
    aw, nr, nv = wf.aux_shape(desc)
    opts = O.make_opts(num_queries=24, blowup=8, grinding=6, ext=ext, folding=4, rem_max_deg=31,
                       hash_id=case.get("hash", 0), num_partitions=case.get("parts", 1), hash_rate=case.get("rate", 1))
    ctx.set_jit(case.get("jit", 1))
    try:
        first, count = wf.shard_columns(trace.shape[0], world, rank)
    except wf.WfError:   # a world the library refuses: rank 0 passes everything
        first, count = 0, trace.shape[0] if rank == 0 else 0
    local = np.ascontiguousarray(trace[first:first + count])
    mont = case.get("mont", 0)
    calls = []

    def builder(rand, f, c):
        calls.append((int(f), int(c)))
        if mont:   # random elements arrive in Montgomery form and the columns must leave in it
            return mont_map(O.to_mont, cols_fn(mont_map(O.from_mont, rand), f, c))
        return cols_fn(rand, f, c)

    refuse = case.get("refuse")
    if refuse:
        lg, vf, bf = log_n, values_fn, builder
        if refuse == "single":
            import airs
            desc, trace = airs.mulfib2(n)
            first, count = wf.shard_columns(trace.shape[0], world, rank)
            local = np.ascontiguousarray(trace[first:first + count])
        elif refuse == "short":
            lg = 6
            local = np.ascontiguousarray(local[:, : 1 << lg])
        elif refuse == "builder" and rank == world - 1:
            def bf(rand, f, c):
                raise RuntimeError("builder failed on purpose")
        elif refuse == "values" and rank == world - 1:
            def vf(rand, values):
                out = values_fn(rand, values)
                out[0, 0] = (int(out[0, 0]) + 1) % O.P
                return out
        elif refuse == "null_builder" and rank == world - 1:
            bf = None
        try:
            wd.prove_air_aux_sharded(ctx, comm, desc, local, lg, opts, bf, values_fn=vf)
            err = None
        except wf.WfError as e:
            err = str(e)
        except RuntimeError as e:   # the rank whose builder raised gets its own exception back
            err = f"error {case.get('code')}: {e}" if refuse == "builder" and rank == world - 1 else None
        live = ctx.mem_stats()[0]
        want = case.get("code")
        ok = err is not None and (want is None or err.startswith(f"error {want}:")) and live == 0
        return all_ranks_agree(ok), f"refusal {refuse}: {err} live={live}"
    if mont and count:
        local = mont_map(O.to_mont, local)
    stats = {}
    if case.get("resident") and count:
        dev = torch.from_numpy(local.view(np.int64)).cuda()
        proof = wd.prove_air_aux_sharded(ctx, comm, desc, None, log_n, opts, builder, values_fn=values_fn, mont=mont,
                                         device_ptr=dev.data_ptr(), stats=stats)
        del dev
    else:
        proof = wd.prove_air_aux_sharded(ctx, comm, desc, local, log_n, opts, builder, values_fn=values_fn, mont=mont, stats=stats)
    want_call = expected_call(aw, ext, world, rank)
    ok = calls == ([want_call] if want_call else [])
    note = f"rank 0 builder calls {calls}"
    if rank == 0:
        if values_fn is None:
            want = ctx.prove_air_aux(desc, trace, opts, full, aw, nr)
        else:
            want = ctx.prove_air_aux_dyn(desc, trace, opts, full, values_fn, aw, nr, nv)
        ok = ok and proof == want
        note += f", sharded {len(proof)} bytes, single-GPU {len(want)}, equal={proof == want}, stats={stats}"
        if case.get("oracle"):
            if values_fn is None:
                same = proof == O.prove_air_aux(desc, trace, opts, full, aw, nr)
                accepted = O.verify_air(desc, proof, int(opts[8]) & 0xff) == 0
            else:
                same = proof == O.prove_air_aux_dyn(desc, trace, opts, full, values_fn, aw, nr, nv)
                accepted = O.verify_air_dyn(desc, proof, int(opts[8]) & 0xff, values_fn, nr, nv, ext) == 0
            ok = ok and same and accepted
            note += f", oracle bytes {same}, oracle verifier {accepted}"
    if "peer_push" in case:
        ok = ok and stats.get("peer_push") == case["peer_push"]
    ok = ok and stats.get("callback_ms", -1) >= 0
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
