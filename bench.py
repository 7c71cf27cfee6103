#!/usr/bin/env python3
"""bench.py — one "step" = one complete STARK proof (Prover::prove, prover/src/lib.rs:250-492) of
BASELINE.json configs[2], the configuration north_star's targets are quoted on:

    cfg3: "FibSmall x 32" (32 copies of examples/src/fibonacci/fib_small/air.rs side by side = 64 columns) on a
    2^22-row Goldilocks trace, blowup 8, Blake3_256, CUBIC extension, 32 queries, FRI folding 4 / remainder max
    degree 31, grinding 16 — trace interpolation + LDE + row hashing + Merkle commitment, constraint evaluation,
    composition polynomial LDE + commitment, OOD frames, DEEP composition, FRI commit phase, PoW grinding, query
    openings and proof serialisation.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config cfg3|cfg2] [--dump-outputs DIR]

Prints ONE JSON line (rank 0). `value` = ms per proof with the trace already resident in HBM; `e2e` = ms per proof
through the C ABI with HOST buffers (pinned trace columns copied H2D inside the timed region, proof bytes returned
to the host). N = 1: one GPU. N > 1: ONE proof sharded over the N GPUs (strong scaling; winterfell_b200/dist.py),
byte-identical to the single-GPU proof. A short cfg2 (2^20 x 8, base field) record rides along as `cfg2`.

`--dump-outputs DIR` writes the proofs the last timed step of each arm returned, `proof.npy` (resident) and
`proof_e2e.npy` (e2e), one float32 per proof byte. The trace is a fixed function of the configuration, so two builds run
with the same arguments can be compared output for output.

`--impl reference` times the CPU arm: the oracle (C++ restatement of the reference's `concurrent` prover — the
reference is Rust and cannot be built in this image) at the FULL configuration, for as many steps as fit the wall
budget (WF_REF_BUDGET_S, default 170 s; at least one); the line reports the steps actually run, never a scaled sample.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (which may be read-only)

P = 0xFFFFFFFF00000001
METRIC = "prover_ms"
FOLDING, REM_MAX_DEG, LOG_BLOWUP, NUM_QUERIES, GRINDING = 4, 31, 3, 32, 16
CONFIGS = {
    # name: (pairs, log_n, ext)
    "cfg3": (32, 22, 3),   # BASELINE.json configs[2]: 2^22 x 64, cubic extension
    "cfg2": (4, 20, 1),    # BASELINE.json configs[1]: 2^20 x 8, base field
}
# dram__bytes_read.sum + dram__bytes_write.sum of the NTT launches of the trace interpolate + LDE of one proof, from the
# committed `ncu --set full` capture of the same command (profiles/, per config); None = not captured for this build
NCU_NTT_TRAFFIC = {"cfg3": None, "cfg2": None}
try:
    NCU_NTT_TRAFFIC.update(json.load(open(os.path.join(ROOT, "profiles", "ntt_traffic.json"))))
except Exception:
    pass


class ClockSampler(threading.Thread):
    """Samples SM clocks and throttle reasons during the timed region (NVML in-process: no process spawn inside the
    timed region — a cold `nvidia-smi` start takes a driver lock for several ms)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False
        self.nv, self.h = self._nvml()

    def _nvml(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)
        except Exception:
            return None, None

    def run(self):
        nv, h = self.nv, self.h
        while not self.stop_flag:
            try:
                if nv is not None:
                    sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                    mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                        else nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                    bit = lambda name: "Active" if r & getattr(nv, name, 0) else "Not Active"
                    self.samples.append([str(sm), str(mx), bit("nvmlClocksThrottleReasonHwSlowdown"),
                                         bit("nvmlClocksThrottleReasonHwThermalSlowdown"), bit("nvmlClocksThrottleReasonSwThermalSlowdown"),
                                         bit("nvmlClocksThrottleReasonSwPowerCap")])
                    time.sleep(0.2)
                    continue
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        mx = max((int(s[1]) for s in self.samples if s[1].isdigit()), default=None)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples if len(s) > 2 + i)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons, "samples": len(self.samples)}


def workload_name(cfg):
    pairs, log_n, ext = CONFIGS[cfg]
    field = {1: "base field", 2: "quadratic extension", 3: "cubic extension"}[ext]
    return (f"{cfg}: full STARK proof of FibSmall x {pairs} ({2 * pairs} columns) on a 2^{log_n}-row Goldilocks trace, blowup 8, "
            f"Blake3_256, {field}, {NUM_QUERIES} queries, FRI folding {FOLDING}, remainder max degree {REM_MAX_DEG}, grinding {GRINDING}: "
            "trace LDE+commit, constraint evaluation, composition LDE+commit, OOD, DEEP, FRI, grinding, openings")


def proof_opts(ext):
    return np.array([NUM_QUERIES, 1 << LOG_BLOWUP, GRINDING, ext, FOLDING, REM_MAX_DEG, 0, 0, 0], dtype=np.uint32)


def host_cores():
    """Usable host cores: CPU affinity, capped by the cgroup CPU quota."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = max(1, min(n, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


# --------------------------------------------------------------------------------------------------
# CPU arm: the oracle = C++ restatement of the reference's prover with the `concurrent` build's parallel
# decomposition (split-radix FFT fft/concurrent.rs:131-171, cosets x segments segments.rs:127-141, columns
# col_matrix.rs:194, row batches row_matrix.rs:195, Merkle levels merkle/concurrent.rs:26-75).
# --------------------------------------------------------------------------------------------------
ORACLE_DESC = ("oracle prover (C++ restatement of winterfell v0.13.1 generate_proof with the `concurrent` decomposition, OpenMP {cores} "
               "threads, scalar BLAKE3; the reference itself is Rust and cannot be built in this image)")


def cpu_prove(pairs, log_n, ext, max_steps, warmup, budget_s):
    """Runs the oracle prover at exactly this size: `warmup` untimed proofs (skipped when one proof alone takes > 20 s),
    then up to max_steps timed proofs within budget_s. Returns (ms per proof, steps run, warmup run, cores)."""
    os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")
    from oracle import oracle as o
    o.lib()
    cores = host_cores()
    o.set_threads(cores)
    tr, res = o.build_fib_trace(pairs, 1 << log_n)
    opts = proof_opts(ext)
    t_start = time.perf_counter()
    times, warm_run = [], 0
    for _ in range(warmup):
        t0 = time.perf_counter()
        o.prove_fib(tr, res, opts)
        dt = time.perf_counter() - t0
        warm_run += 1
        if dt > 20.0:           # a multi-second proof has no cold-start effect worth a second untimed run: count it
            times.append(dt)
            warm_run -= 1
            break
    while len(times) < max_steps:
        if times and (time.perf_counter() - t_start) + times[-1] > budget_s:
            break
        t0 = time.perf_counter()
        o.prove_fib(tr, res, opts)
        times.append(time.perf_counter() - t0)
    return sum(times) / len(times) * 1e3, len(times), warm_run, cores


def run_reference(args, rank, world):
    if rank != 0:
        return
    pairs, log_n, ext = CONFIGS[args.config]
    budget = float(os.environ.get("WF_REF_BUDGET_S", "170"))
    ms, steps_run, warm_run, cores = cpu_prove(pairs, log_n, ext, args.steps, min(args.warmup, 1), budget)
    sample = (ORACLE_DESC.format(cores=cores) + f"; FULL configuration (2^{log_n} rows x {2 * pairs} columns), {steps_run} timed proof(s) "
              f"actually run inside a {budget:.0f} s wall budget ({args.steps} requested), no scaling")
    # how the port's parallel decomposition scales on this host: the same AIR at 2^16 rows with 1 thread and with all of them
    scaling = None
    try:
        from oracle import oracle as o
        s_log = min(16, log_n)
        tr, res = o.build_fib_trace(pairs, 1 << s_log)
        opts = proof_opts(ext)
        tms = {}
        for th in (1, cores):
            o.set_threads(th)
            t0 = time.perf_counter()
            o.prove_fib(tr, res, opts)
            tms[th] = (time.perf_counter() - t0) * 1e3
        scaling = {"rows_log2": s_log, "ms_1_thread": round(tms[1], 1), f"ms_{cores}_threads": round(tms[cores], 1),
                   "speedup": round(tms[1] / tms[cores], 2)}
    except Exception as e:  # never take the line down
        scaling = {"failed": str(e)}
    line = {
        "impl": "reference", "metric": METRIC, "value": round(ms, 3), "unit": "ms", "n_gpus": args.gpus, "steps": steps_run,
        "warmup": warm_run, "steps_requested": args.steps, "warmup_requested": args.warmup,
        "ms_per_step": round(ms, 3), "higher_is_better": False, "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None,
        "dtype": "u64", "data": "synthetic", "config": {"workload": workload_name(args.config)},
        "cpu_baseline": {"value": round(ms, 3), "unit": "ms", "cores": cores, "kind": "port", "sample": sample, "thread_scaling": scaling},
        "e2e": {"value": round(ms, 3), "unit": "ms", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# roofline arithmetic (SURVEY.md 8d; DESIGN.md 4)
# --------------------------------------------------------------------------------------------------
def fri_algorithmic_bytes(N, d):
    """sum over layers of e*L*1.25 + 32*L (read layer, write folded layer, leaf digests + tree), e = 8d bytes,
    L = N, N/4, ... while the next layer stays above the remainder bound (fri/src/options.rs:85-93)."""
    total, L, e = 0.0, N, 8 * d
    while (L // FOLDING) >= (REM_MAX_DEG + 1) * (1 << LOG_BLOWUP) and L > FOLDING:
        total += e * L * 1.25 + 32 * L
        L //= FOLDING
    return total


def sharded_records(bd, log_n, pairs, world, hbm, peak_src, sm_mhz=None):
    """Roofline and throughput keys of an N > 1 line (one proof sharded over `world` GPUs) from rank 0's stage times. The
    `trace_lde` stage covers this rank's column block: layout, interpolation, extension of every coset (the copy-engine
    pushes of the finished cosets run under it). Per-GPU algorithmic bytes 8n(2+b) x cols / world; the aggregate is what
    BASELINE's "NTT Gelem/s at 1/2/4/8 GPUs" asks for."""
    n_, cols_ = 1 << log_n, 2 * pairs
    N = n_ << LOG_BLOWUP
    alg = 8.0 * n_ * (2 + (1 << LOG_BLOWUP)) * cols_ / world
    t = bd["trace_lde"] * 1e-3
    ach = alg / t / 1e9
    alu = None
    try:  # the ALU-pipe roofline of the instruction mix (profiles/ntt_alu_model.json), per GPU
        m = json.load(open(os.path.join(ROOT, "profiles", "ntt_alu_model.json")))
        per = m["alu_instr_per_element_pass"]
        mean_instr = (per["contiguous_2p11"] + per["strided_2p11"]) / 2.0
        ceil_passes = m["sms"] * m["alu_lanes_per_clk_per_sm"] * (sm_mhz or 1965) * 1e6 / mean_instr
        passes = 2.0 * (n_ + N) * cols_ / world / t
        alu = {"bound": "alu_pipe", "achieved": round(passes / 1e9, 2), "peak": round(ceil_passes / 1e9, 2), "unit": "G element-passes/s per GPU",
               "frac": round(passes / ceil_passes, 4), "alu_instr_per_element_pass": mean_instr, "sm_mhz": sm_mhz or 1965}
    except Exception:
        pass
    out = {"roofline": {"bound": "hbm", "kernel": "ntt_pass (per GPU: layout + interpolate + LDE of this rank's column block, the exchange of the "
                                                  "finished cosets running under it on the copy engines)",
                        "achieved": round(ach, 1), "peak": hbm, "unit": "GB/s", "alu_pipe": alu, "frac": round(ach / hbm, 4), "traffic": None,
                        "peak_source": peak_src, "algorithmic_bytes": int(alg), "kernel_ms": round(bd["trace_lde"], 4),
                        "aggregate_GBps": round(ach * world, 1),
                        "note": "rank 0's stage time; includes the segment layout kernel; integer-ALU-bound (DESIGN.md 4)"},
           "ntt_gelem_per_s": round(N * cols_ / t / 1e9, 3),
           "merkle_leaves_per_s": round(N / (bd["trace_commit"] * 1e-3), 1) if bd.get("trace_commit") else None,
           "lde_commit_fri_ms": round(sum(bd.get(k, 0.0) for k in ("trace_lde", "trace_exchange", "trace_commit", "composition_lde",
                                                                     "composition_commit", "fri_layers")), 4)}
    return out


def rooflines(breakdown, cfg, hbm, peak_src, compress_gps, sm_mhz=None):
    pairs, log_n, ext = CONFIGS[cfg]
    n, cols = 1 << log_n, 2 * pairs
    N = n << LOG_BLOWUP
    out = []
    # 1. NTT (K1 + K2 = trace interpolate + LDE): 8n(2 + b) bytes per base column
    ntt_ms = breakdown["trace_interpolate"] + breakdown["trace_lde"]
    alg = 8.0 * n * (2 + (1 << LOG_BLOWUP)) * cols
    ach = alg / (ntt_ms * 1e-3) / 1e9
    # the ALU-pipe roofline of the kernel's own instruction mix (DESIGN.md 4 / 10): ALU-pipe instructions per element and pass
    # from the committed ncu capture, 64 ALU lanes per clock per SM
    alu = None
    try:
        m = json.load(open(os.path.join(ROOT, "profiles", "ntt_alu_model.json")))
        per = m["alu_instr_per_element_pass"]
        mean_instr = (per["contiguous_2p11"] + per["strided_2p11"]) / 2.0        # every transform is one strided + one contiguous pass
        clk = (sm_mhz or 1965) * 1e6
        ceil_passes = m["sms"] * m["alu_lanes_per_clk_per_sm"] * clk / mean_instr
        passes = 2.0 * (n + N) * cols / (ntt_ms * 1e-3)
        alu = {"bound": "alu_pipe", "achieved": round(passes / 1e9, 2), "peak": round(ceil_passes / 1e9, 2), "unit": "G element-passes/s",
               "frac": round(passes / ceil_passes, 4), "alu_instr_per_element_pass": mean_instr, "sm_mhz": sm_mhz or 1965}
    except Exception:
        pass
    out.append({"bound": "hbm", "kernel": "ntt_pass (trace interpolate + LDE launches)", "achieved": round(ach, 1), "peak": hbm, "unit": "GB/s", "alu_pipe": alu,
                "frac": round(ach / hbm, 4), "traffic": NCU_NTT_TRAFFIC.get(cfg), "peak_source": peak_src, "algorithmic_bytes": int(alg),
                "kernel_ms": round(ntt_ms, 4), "elements_per_s": round(N * cols / (ntt_ms * 1e-3), 1),
                "note": "algorithmic bytes = 8n(2+b) per column (read trace, write polys, write LDE); the kernel is integer-ALU-bound "
                        "(64-bit modular arithmetic on 32-bit pipes), see DESIGN.md 4 for the ALU roofline beside this one"})
    # 2. leaf hashing + Merkle tree of the trace commitment: 8c (row) + 32 (digest) + 96 (tree node) bytes per leaf
    mk_ms = breakdown["trace_commit"]
    per_leaf = 8 * cols + 32 + 96
    ach = per_leaf * N / (mk_ms * 1e-3) / 1e9
    comp_per_leaf = (8 * cols + 63) // 64 + 1
    int_ceiling = compress_gps * 1e9 / comp_per_leaf * per_leaf / 1e9   # GB/s equivalent of the INT32 compression ceiling
    out.append({"bound": "hbm", "kernel": "hash_rows_blake3 + merkle (trace commitment)", "achieved": round(ach, 1), "peak": hbm, "unit": "GB/s",
                "frac": round(ach / hbm, 4), "traffic": None, "peak_source": peak_src, "algorithmic_bytes": int(per_leaf * N),
                "kernel_ms": round(mk_ms, 4), "leaves_per_s": round(N / (mk_ms * 1e-3), 1),
                "int32_ceiling_GBps": round(int_ceiling, 1), "frac_of_min_hbm_int32": round(ach / min(hbm, int_ceiling), 4),
                "note": f"{comp_per_leaf} BLAKE3 compressions per leaf (row + its tree node); INT32 ceiling from {compress_gps} G compressions/s"})
    # 3. FRI commit phase (fold + leaf hash + tree, all layers)
    fri_ms = breakdown["fri_layers"]
    alg = fri_algorithmic_bytes(N, ext)
    ach = alg / (fri_ms * 1e-3) / 1e9
    out.append({"bound": "hbm", "kernel": "fri_hash + fri_fold + merkle (all FRI layers)", "achieved": round(ach, 1), "peak": hbm, "unit": "GB/s",
                "frac": round(ach / hbm, 4), "traffic": None, "peak_source": peak_src, "algorithmic_bytes": int(alg), "kernel_ms": round(fri_ms, 4),
                "note": "sum over layers of e*L*1.25 + 32*L bytes (SURVEY.md 8d); tail layers are launch-bound"})
    return out


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="cfg3", choices=sorted(CONFIGS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub-record", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the proofs the last timed step returned as DIR/<name>.npy (float32, one value per byte)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)   # fail on an unusable DIR before the timed run, not after it
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist

    import winterfell_b200 as wf

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    stream = torch.cuda.Stream()
    ctx = wf.Context(local_rank, stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")     # > L2 (126 MB)
    warmup = max(args.warmup, 3)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def ev():
        return torch.cuda.Event(enable_timing=True)

    def timed(fn, steps):
        """Mean ms per step over `steps` calls of fn, and what the last call returned."""
        total, out = 0.0, None
        for _ in range(steps):
            flush.zero_()
            a, b = ev(), ev()
            a.record(stream)
            out = fn()
            b.record(stream)
            b.synchronize()
            total += a.elapsed_time(b)
        return total / steps, out

    def run_config(cfg, steps, warm, sample_clocks):
        """Resident and e2e arms of one configuration on this rank's GPU. Returns a dict."""
        pairs, log_n, ext = CONFIGS[cfg]
        cols, n = 2 * pairs, 1 << log_n
        opts = proof_opts(ext)
        host = torch.empty((cols, n), dtype=torch.int64).pin_memory()       # pinned host trace (ColMatrix columns)
        host_np = host.numpy().view(np.uint64)
        _, results = wf.build_fib_trace(pairs, n, out=host_np)               # FibSmallProver::build_trace, k copies
        dev = host.cuda(non_blocking=False)                                  # resident copy for the kernel-only arm
        out_buf = np.zeros(1 << 23, dtype=np.uint8)
        e2e_buf = np.zeros(1 << 23, dtype=np.uint8)

        def step_resident():
            return ctx.prove_fib_dev(dev.data_ptr(), pairs, log_n, results, opts, out_buf)

        def step_e2e():
            return ctx.prove_fib(host_np, results, opts, out_buf=e2e_buf)     # H2D of the trace and D2H of the proof inside

        with torch.cuda.stream(stream):
            for _ in range(warm):
                p_res = step_resident()
            p_e2e = step_e2e()
            assert p_res == p_e2e, "resident and e2e arms produced different proofs"
            sampler = None
            if sample_clocks:
                sampler = ClockSampler(local_rank)
                sampler.start()
            barrier()
            l0 = ctx.launches
            t_wall0 = time.perf_counter()
            ms_step, last_res = timed(step_resident, steps)
            barrier()
            wall_ms = (time.perf_counter() - t_wall0) * 1e3
            launches = int(ctx.launches - l0) // max(steps, 1)
            e2e_step, last_e2e = timed(step_e2e, steps)
            barrier()
            if sampler:
                sampler.stop_flag = True
                sampler.join(timeout=2)
            # stage breakdown: one extra proof with the library's stage events on
            flush.zero_()
            ctx.set_profiling(True)
            step_resident()
            breakdown = {k: round(v, 4) for k, v in ctx.stage_times()}
            ctx.set_profiling(False)
        del dev
        return {"ms": ms_step, "e2e_ms": e2e_step, "launches": launches, "breakdown": breakdown, "proof": p_e2e, "h2d": int(host_np.nbytes),
                "wall_ms": wall_ms / steps, "clocks": sampler.summary() if sampler else None,
                "last_outputs": {"proof": last_res, "proof_e2e": last_e2e}}

    def fri_compressions(L):
        """BLAKE3 compressions of the FRI commit phase on an L-point base-field codeword (folding 4): every layer of n points
        hashes n/4 leaves of 32 bytes (one compression each) and n/4 - 1 tree nodes; layers until the remainder's domain."""
        tot, n = 0, L
        while n > (REM_MAX_DEG + 1) << LOG_BLOWUP:
            tot += n // FOLDING + n // FOLDING - 1
            n //= FOLDING
        return tot

    def fri_sweep():
        """BASELINE.json configs[4]: FRI commit phase alone (fold + leaf hash + Merkle tree of every layer, device-side coin) on
        2^20 .. 2^26-point base-field codewords (LDE, blowup 8, of random polynomials), folding 4, remainder max degree 31,
        Blake3_256. Every rank folds its own codeword (independent objects: weak scaling, no data-path collective); CUDA
        events on the context stream, max over ranks; GB/s over SURVEY.md 8d's algorithmic bytes."""
        rng = np.random.default_rng(100 + rank)
        recs = []
        for log_len in (20, 22, 24, 26):
            L = 1 << log_len
            with torch.cuda.stream(stream):
                m = ctx.mat_from_host_columns(rng.integers(0, P, size=(1, L >> LOG_BLOWUP), dtype=np.uint64))
                cw = m.lde(LOG_BLOWUP)
                for _ in range(3):
                    f, _ = ctx.fri_build_layers_default(wf.HASH_BLAKE3_256, cw, 1, FOLDING, REM_MAX_DEG, 1 << LOG_BLOWUP)
                    f.free()
                barrier()
                reps, tot = 5, 0.0
                for _ in range(reps):
                    flush.zero_()
                    a, b = ev(), ev()
                    a.record(stream)
                    f, _ = ctx.fri_build_layers_default(wf.HASH_BLAKE3_256, cw, 1, FOLDING, REM_MAX_DEG, 1 << LOG_BLOWUP)
                    b.record(stream)
                    b.synchronize()
                    tot += a.elapsed_time(b)
                    f.free()
                m.free(); cw.free()
            ms = tot / reps
            if world > 1:
                t = torch.tensor([ms], device="cuda", dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t[0])
            recs.append((log_len, ms))
        return recs

    import gc
    gc.collect()
    gc.disable()  # no collector pauses inside the timed regions
    from winterfell_b200 import dist as wfdist
    if world > 1 and hasattr(wfdist, "bench_sharded"):
        main_rec = wfdist.bench_sharded(ctx, stream, args.config, args.steps, warmup, CONFIGS, proof_opts, flush, ClockSampler, local_rank)
    else:
        main_rec = run_config(args.config, args.steps, warmup, True)
        if world > 1:
            main_rec["parallelism"] = f"{world} independent replicas of the proof, one per GPU (no data-path collective)"
    sub = None
    if world == 1 and args.config == "cfg3" and not args.no_sub_record:
        sub = run_config("cfg2", args.steps, 3, False)
    sweep = None if args.no_sub_record else fri_sweep()
    gc.enable()

    ms_step, e2e_step = main_rec["ms"], main_rec["e2e_ms"]
    if world > 1:
        t = torch.tensor([ms_step, e2e_step], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step, e2e_step = float(t[0]), float(t[1])

    if rank == 0:
        if args.dump_outputs:
            # the serialized proof is what a caller of the timed path receives; its bytes are exact in float32. The proof buffer
            # holds at most 8 MiB, so the two files stay within 64 MiB.
            for name, proof in main_rec["last_outputs"].items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), np.frombuffer(proof, dtype=np.uint8).astype(np.float32))
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        compress_gps = 46.0   # BLAKE3 compressions/s ceiling in G/s: INT32 issue estimate of SURVEY.md 8d (see profiles/ for the measured figure)
        try:
            compress_gps = float(json.load(open(os.path.join(ROOT, "profiles", "blake3_compress_peak.json")))["gcompress_per_s"])
        except Exception:
            pass
        bd = main_rec["breakdown"]
        pairs, log_n, ext = CONFIGS[args.config]
        N = (1 << log_n) << LOG_BLOWUP
        line = {
            "metric": METRIC, "value": round(ms_step, 4), "unit": "ms", "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": round(ms_step, 4), "higher_is_better": False, "scaling": "strong" if world > 1 else "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": {"workload": workload_name(args.config), "l2": "256 MiB memset between timed steps (L2 flush); inputs (2 GiB trace) exceed L2",
                       "parallelism": main_rec.get("parallelism", "single GPU")},
            "e2e": {"value": round(e2e_step, 4), "unit": "ms", "h2d_bytes_per_step": main_rec["h2d"], "d2h_bytes_per_step": len(main_rec["proof"])},
            "gpu_launches": main_rec["launches"],
            "clocks": main_rec["clocks"],
            "stage_ms": bd,
            "proof_bytes": len(main_rec["proof"]),
            "wall_ms_per_step_incl_flush": round(main_rec["wall_ms"], 3),
        }
        if "trace_interpolate" in bd:
            rl = rooflines(bd, args.config, hbm, peak_src, compress_gps, (main_rec.get("clocks") or {}).get("sm_mhz"))
            line["roofline"] = dict(rl[0], kernels=rl)   # dominant kernel first; all three listed under `kernels`
            line["lde_commit_fri_ms"] = round(sum(bd.get(k, 0.0) for k in ("trace_interpolate", "trace_lde", "trace_commit", "composition_lde",
                                                                                "composition_commit", "fri_layers")), 4)
            line["ntt_gelem_per_s"] = round(rl[0]["elements_per_s"] / 1e9, 3)
            line["merkle_leaves_per_s"] = rl[1]["leaves_per_s"]
        elif "trace_lde" in bd and world > 1:
            line.update(sharded_records(bd, log_n, pairs, world, hbm, peak_src, (main_rec.get("clocks") or {}).get("sm_mhz")))
        for k in ("comm", "roofline", "ntt_gelem_per_s", "merkle_leaves_per_s", "lde_commit_fri_ms"):
            if k in main_rec:
                line[k] = main_rec[k]
        if sub:
            srl = rooflines(sub["breakdown"], "cfg2", hbm, peak_src, compress_gps)
            line["cfg2"] = {"workload": workload_name("cfg2"), "value": round(sub["ms"], 4), "e2e": round(sub["e2e_ms"], 4), "unit": "ms",
                            "gpu_launches": sub["launches"], "stage_ms": sub["breakdown"], "roofline": dict(srl[0], kernels=srl)}
        if sweep:
            line["fri_sweep"] = {"workload": "cfg5: FRI commit phase only, 2^20..2^26-point base-field codewords, folding 4, remainder max degree 31, "
                                             "Blake3_256; one codeword per GPU (weak scaling, no data-path collective), max over ranks",
                                 "points": [{"log2_len": ll, "ms": round(ms, 4),
                                             "GBps_per_gpu": round(fri_algorithmic_bytes(1 << ll, 1) / (ms * 1e-3) / 1e9, 1),
                                             "frac_of_hbm": round(fri_algorithmic_bytes(1 << ll, 1) / (ms * 1e-3) / 1e9 / hbm, 4),
                                             "aggregate_GBps": round(world * fri_algorithmic_bytes(1 << ll, 1) / (ms * 1e-3) / 1e9, 1),
                                             # the layers' leaf hashes and trees are BLAKE3 compressions on the INT32 pipes: the bound that
                                             # applies before HBM does (one per 32-byte leaf of 4 evaluations + one per tree node)
                                             "blake3_compressions": fri_compressions(1 << ll),
                                             "frac_of_compress_ceiling": round(fri_compressions(1 << ll) / (ms * 1e-3) / 1e9 / compress_gps, 4)}
                                            for ll, ms in sweep],
                                 "compress_ceiling_G_per_s": compress_gps}
        if not args.no_cpu_baseline:
            # bounded sample of the same workload in a fresh process (torch has already initialised libgomp here with the
            # spinning wait policy): the same AIR / columns / extension on 1/16 of the rows; the value is the SAMPLE's own
            # time, never scaled — the full-size CPU number is the `--impl reference` arm's
            try:
                s_log_n = max(log_n - 4, 10)
                code = ("import json,sys; sys.path.insert(0, %r); import bench; ms, steps, warm, cores = bench.cpu_prove(%d, %d, %d, 1, 0, 120.0); "
                        "print(json.dumps({'ms': ms, 'cores': cores}))" % (ROOT, pairs, s_log_n, ext))
                out = subprocess.run([sys.executable, "-B", "-c", code], capture_output=True, text=True, timeout=600,
                                     env={**os.environ, "OMP_WAIT_POLICY": "PASSIVE"}).stdout.strip().splitlines()[-1]
                r = json.loads(out)
                line["cpu_baseline"] = {"value": round(r["ms"], 3), "unit": "ms", "cores": r["cores"], "kind": "port", "rows_log2": s_log_n,
                                        "sample": ORACLE_DESC.format(cores=r["cores"]) + f"; ONE proof of the same AIR at 2^{s_log_n} rows x {2 * pairs} "
                                        f"columns (1/{1 << (log_n - s_log_n)} of the workload's rows), value = that sample's own time, NOT scaled; "
                                        "the full-size CPU time is the --impl reference arm's"}
            except Exception as e:  # the reported baseline must never take the GPU line down
                line["cpu_baseline"] = {"value": None, "unit": "ms", "cores": host_cores(), "kind": "port", "sample": f"failed: {e}"}
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
