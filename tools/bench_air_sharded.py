"""Strong scaling of wf_prove_air_sharded / wf_prove_air_aux_sharded: one proof of an AIR description over N GPUs of a node
(NCCL), against the one-GPU proof. Start with torchrun, one process per GPU:

    torchrun --nproc-per-node=N tools/bench_air_sharded.py [--cases fib16,rescue6,rap] [--steps 5] [--warmup 2] [--out FILE]

Cases: `fib16` = FibSmall x 16 (32 columns) at 2^22 rows described generically (the bytecode evaluator / its NVRTC kernel),
next to wf_prove_fib_sharded (the specialised kernel) on the same trace where its whole-segment rule allows; `rescue6` =
rescue_like(6) at 2^20 rows (degree 7), the widest Rescue-like AIR a description can express; `rap` (opt-in, not in the default
list) = perm_rap_lanes(3) at 2^20 rows, a two-segment AIR whose aux columns a host callback builds (each rank builds only the
lanes covering its aux columns; the line's "callback_ms" is the time spent in the callbacks per proof, max over ranks). N = 1
times wf_prove_air (wf_prove_air_aux for `rap`) on one GPU (host columns: the one-GPU AIR entry points take no device trace)
and wf_prove_fib_dev. Per case rank 0 prints one JSON
line: ms per proof (CUDA events on the context stream, max over ranks of the per-rank mean, 256 MiB L2 flush before every
step), the library's stage times and stats, byte identity against the one-GPU proof (checked once, before timing), and the
card's name, power limit and SM clock read in the same run. Traces are built once and cached in a temporary directory."""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np
import torch
import torch.distributed as dist

import airs
import airs_aux
import winterfell_b200 as wf
from oracle import oracle as O
from winterfell_b200 import dist as wd

OPTS = dict(num_queries=32, blowup=8, grinding=16, ext=3, folding=4, rem_max_deg=31)   # bench.py's ProofOptions


def fib_desc(k, n, results):
    """airs.fib_small_x's description for a trace built by wf.build_fib_trace (the same trace, built in C)."""
    A = airs.AirBuilder(2 * k)
    A.pub = [int(v) for v in results]
    for j in range(k):
        A.constraint(A.sub(A.nxt(2 * j), A.add(A.cur(2 * j), A.cur(2 * j + 1))), 1)
        A.constraint(A.sub(A.nxt(2 * j + 1), A.add(A.cur(2 * j + 1), A.nxt(2 * j))), 1)
        A.assert_single(2 * j, 0, j + 1)
        A.assert_single(2 * j + 1, 0, j + 1)
        A.assert_single(2 * j + 1, n - 1, int(results[j]))
    return A.build()


def load_case(name, cache):
    if name == "rap":   # returns the aux builder in place of FibSmall results
        log_n = 20
        desc, trace, builder = airs_aux.perm_rap_lanes(1 << log_n)
        return log_n, desc, trace, builder
    if name == "fib16":
        log_n = 22
        trace, results = wf.build_fib_trace(16, 1 << log_n)
        return log_n, fib_desc(16, 1 << log_n, results), trace, results
    log_n = 20
    path = os.path.join(cache, f"rescue6_{log_n}.npz")
    if not os.path.exists(path):   # a Python loop over 2^20 rows: built once, shared by the ranks and later launches
        if dist.get_rank() == 0:
            desc, trace = airs.rescue_like(1 << log_n, 6)
            np.savez(path + ".tmp.npz", desc=desc, trace=trace)
            os.replace(path + ".tmp.npz", path)
        dist.barrier()
    z = np.load(path)
    return log_n, z["desc"], z["trace"], None


def card(local_rank):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", str(local_rank)], capture_output=True, text=True).stdout
    return dict(zip(q.split(","), [x.strip() for x in out.strip().split(",")]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default="fib16,rescue6")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    ap.add_argument("--cache", default=os.path.join(tempfile.gettempdir(), "wf_bench_air_sharded"))
    a = ap.parse_args()
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl" if torch.cuda.device_count() > 1 else "gloo", device_id=torch.device("cuda", local_rank))
    rank, world = dist.get_rank(), dist.get_world_size()
    os.makedirs(a.cache, exist_ok=True)
    stream = torch.cuda.Stream()
    ctx = wf.Context(local_rank, stream.cuda_stream)
    comm = wd.TorchComm(stream) if world > 1 else None
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    out_buf = np.zeros(1 << 23, dtype=np.uint8)

    def timed(fn):
        per = []
        for _ in range(a.steps):
            flush.zero_()
            torch.cuda.synchronize()
            dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            per.append(e0.elapsed_time(e1))
        mine = torch.tensor([sum(per) / len(per)], dtype=torch.float64, device="cuda")
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        return round(max(float(t) for t in allr), 3), [round(x, 3) for x in per]

    def breakdown(fn):
        flush.zero_()
        torch.cuda.synchronize()
        dist.barrier()
        ctx.set_profiling(True)
        fn()
        ctx.set_profiling(False)
        return {k: round(v, 3) for k, v in ctx.stage_times()}

    for name in a.cases.split(","):
        log_n, desc, trace, results = load_case(name, a.cache)
        opts = O.make_opts(**OPTS)
        width = trace.shape[0]
        variants = {}
        cb_ms = []   # one-GPU `rap`: time inside the aux builder, per proof
        if name == "rap":
            builder, results = results, None
            aw, nr, _ = wf.aux_shape(desc)

            def one_gpu_builder(rand):
                t0 = time.perf_counter()
                aux = builder(rand)
                cb_ms.append((time.perf_counter() - t0) * 1e3)
                return aux
        if name == "rap" and world == 1:
            pinned = torch.from_numpy(trace.view(np.int64)).pin_memory().numpy().view(np.uint64)
            variants["air_aux"] = (lambda: ctx.prove_air_aux(desc, pinned, opts, one_gpu_builder, aw, nr), "host columns (pinned)")
        elif name == "rap":
            first, count = wf.shard_columns(width, world, rank)
            local = torch.from_numpy(np.ascontiguousarray(trace[first:first + count]).view(np.int64)).cuda()
            ptr = local.data_ptr() if count else None
            stats = {}
            variants["air_aux"] = (lambda: wd.prove_air_aux_sharded(ctx, comm, desc, None, log_n, opts, builder.columns, device_ptr=ptr,
                                                                    stats=stats, out_buf=out_buf), "resident main columns")
        elif world == 1:
            pinned = torch.from_numpy(trace.view(np.int64)).pin_memory().numpy().view(np.uint64)
            variants["air"] = (lambda: ctx.prove_air(desc, pinned, opts), "host columns (pinned)")
            if results is not None:
                dev = torch.from_numpy(trace.view(np.int64)).cuda()
                variants["fib_specialised"] = (lambda: ctx.prove_fib_dev(dev.data_ptr(), width // 2, log_n, results, opts, out_buf=out_buf),
                                               "resident")
        else:
            first, count = wf.shard_columns(width, world, rank)
            local = torch.from_numpy(np.ascontiguousarray(trace[first:first + count]).view(np.int64)).cuda()
            ptr = local.data_ptr() if count else None
            stats = {}
            variants["air"] = (lambda: wd.prove_air_sharded(ctx, comm, desc, None, log_n, opts, device_ptr=ptr, stats=stats, out_buf=out_buf),
                               "resident")
            if results is not None and width % (8 * world) == 0:
                variants["fib_specialised"] = (lambda: wd.prove_fib_sharded(ctx, comm, None, width // 2, log_n, results, opts, out_buf=out_buf,
                                                                            device_ptr=local.data_ptr(), stats=stats), "resident")
        with torch.cuda.stream(stream):
            if rank != 0:
                want = None
            elif name == "rap":
                want = ctx.prove_air_aux(desc, trace, opts, builder, aw, nr)
            else:
                want = ctx.prove_air(desc, trace, opts)   # the one-GPU proof, untimed
            for vname, (fn, inp) in variants.items():
                t0 = time.perf_counter()
                first_proof = fn()
                first_s = time.perf_counter() - t0      # ranks other than 0 compile the AIR's kernel (NVRTC) here
                for _ in range(a.warmup):
                    fn()
                identical = (first_proof == want) if rank == 0 else None
                before = card(local_rank)
                cb_ms.clear()
                ms, per = timed(fn)
                after = card(local_rank)
                callback = None
                if name == "rap":   # this rank's callback time per proof (the last timed step), max over the ranks
                    mine = cb_ms[-1] if world == 1 else stats["callback_ms"]
                    t = torch.tensor([mine], dtype=torch.float64, device="cuda")
                    allr = [torch.empty_like(t) for _ in range(world)]
                    dist.all_gather(allr, t)
                    callback = round(max(float(x) for x in allr), 3)
                bd = breakdown(fn)
                rec = {"tool": "bench_air_sharded", "case": name, "variant": vname, "gpus": world, "log_n": log_n, "width": width,
                       "opts": {k: int(v) for k, v in OPTS.items()}, "input": inp, "ms_per_proof": ms, "rank_steps_ms": per,
                       "first_call_s": round(first_s, 3), "byte_identical_to_one_gpu": identical, "callback_ms": callback, "breakdown": bd,
                       "stats": dict(stats) if world > 1 else None, "columns": [wf.shard_columns(width, world, q) for q in range(world)] if world > 1 else None,
                       "jit": ctx.jit_stats(), "card_before": before, "card_after": after,
                       "l2": "256 MiB memset before every timed step", "steps": a.steps, "warmup": a.warmup}
                if rank == 0:
                    line = json.dumps(rec)
                    print(line, flush=True)
                    if a.out:
                        with open(a.out, "a") as f:
                            f.write(line + "\n")
        del variants
        torch.cuda.synchronize()
        dist.barrier()
    ctx.close()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
