"""Multi-GPU plumbing for the column-sharded trace commitment (SURVEY.md §8e, option 1).

One process per GPU (`torch.distributed`, backend "nccl"; the host-logic tests run the same code over
"gloo" on CPU with a test backend). The reference has no distributed code at all — its only
distribution-aware feature is `PartitionOptions` (air/src/options.rs:405-445) — so the decomposition
is new, but the result is bit-identical to the single-device commitment (`DefaultTraceLde::new`,
prover/src/trace/trace_lde/default/mod.rs:63, :245-282):

  1. rank g owns columns [g*c/G, (g+1)*c/G): interpolate + LDE locally (no communication; K1/K2 are
     independent per column).
  2. ONE all-to-all turns column shards into row shards: rank r receives rows [r*N/G, (r+1)*N/G) of
     every column block (each rank sends (G-1)/G of its LDE slice).
  3. rank r hashes its rows and builds the Merkle subtree over them — rows [r*N/G, (r+1)*N/G) are
     exactly one depth-log2(G) subtree of the reference's heap layout (crypto/src/merkle/mod.rs:344-368).
  4. ONE all-gather of the G subtree roots (32 bytes each); every rank computes the top log2(G) levels
     redundantly on the host (H::merge, crypto/src/hash/mod.rs:45).

This module contains no arithmetic: local compute goes through a backend (the CUDA context in the
product; the tests substitute a CPU backend), collectives through torch.distributed.
"""
import os

import numpy as np
import torch
import torch.distributed as dist

import winterfell_b200 as wf


def column_range(ncols, world, rank):
    """Contiguous column block of `rank`; the first (ncols % world) ranks get one extra column."""
    base, extra = divmod(ncols, world)
    lo = rank * base + min(rank, extra)
    return lo, lo + base + (1 if rank < extra else 0)


def top_levels(hash_id, roots):
    """Root of the tree whose depth-log2(G) nodes are `roots` (list of 32-byte digests, in order).
    Same heap rule as build_merkle_nodes: parent(i) = merge(child 2i, child 2i+1)."""
    level = list(roots)
    assert len(level) & (len(level) - 1) == 0 and len(level) >= 1
    while len(level) > 1:
        level = [wf.host_merge(hash_id, level[2 * i], level[2 * i + 1]) for i in range(len(level) // 2)]
    return level[0]


class CudaBackend:
    """Local compute on this rank's GPU through the C ABI.

    Exchange format (when the rank owns a multiple of 8 columns, i.e. whole segments): the LDE is written
    by the library straight into a torch buffer in segment layout [local segment][N rows][8]; the send
    buffer is that tensor regrouped by destination, [dest][local segment][rows_per][8] (one device copy);
    what arrives, [source][local segment][rows_per][8], IS the segment layout of the rank's
    rows_per x ncols_total row shard (global segment = source * local_segments + local segment), so the
    commitment kernels run on the receive buffer in place. Other widths take a row-major exchange."""

    def __init__(self, ctx):
        self.ctx = ctx
        self.device = torch.device("cuda", torch.cuda.current_device())

    def pack(self, cols_dev, ncols, n, log_blowup, world):
        """cols_dev: int64 CUDA tensor [ncols, n]. Returns the all-to-all send tensor [world, chunk]."""
        N = n << log_blowup
        m = self.ctx.mat_from_device_columns(cols_dev.data_ptr(), ncols, n)
        polys = m.interpolate()
        if ncols % 8 == 0:
            nsl = ncols // 8
            seg = torch.empty((nsl, N, 8), dtype=torch.int64, device=self.device)
            out = self.ctx.mat_wrap_device(seg.data_ptr(), N, ncols)
            polys.lde_into(log_blowup, out)
            self.ctx.sync()
            for h in (m, polys, out):
                h.free()
            rp = N // world
            return seg.view(nsl, world, rp * 8).permute(1, 0, 2).contiguous().view(world, nsl * rp * 8)
        lde = polys.lde(log_blowup)
        rows = torch.empty((N, ncols), dtype=torch.int64, device=self.device)
        lde.to_device_rows(rows.data_ptr())
        self.ctx.sync()
        for h in (m, polys, lde):
            h.free()
        return rows.view(world, (N // world) * ncols)

    def commit(self, hash_id, recv, rows_per, ncols_total, cl):
        """recv: [world, chunk] as received. Returns (subtree root bytes, row shard tensor, leaf digests, nodes)."""
        world = recv.shape[0]
        if cl % 8 == 0:
            shard = self.ctx.mat_wrap_device(recv.data_ptr(), rows_per, ncols_total)
            tree = self.ctx.commit_rows(hash_id, shard)
            root = tree.root()
            leaves, nodes = tree.to_host() if rows_per <= (1 << 16) else (None, None)
            shard.free()
            tree.free()
            return root, recv, leaves, nodes
        rows = recv.view(world, rows_per, cl).permute(1, 0, 2).reshape(rows_per, ncols_total).contiguous()
        digests = torch.empty(rows_per * 32, dtype=torch.uint8, device=self.device)
        nodes = torch.empty(rows_per * 32, dtype=torch.uint8, device=self.device)
        self.ctx.hash_rows_dev(hash_id, rows.data_ptr(), rows_per, ncols_total, digests.data_ptr())
        self.ctx.merkle_dev(hash_id, digests.data_ptr(), rows_per, nodes.data_ptr())
        self.ctx.sync()
        return bytes(nodes[32:64].cpu().numpy()), rows, digests, nodes


def sharded_trace_commit(backend, hash_id, local_cols, ncols_total, log_n, log_blowup, group=None):
    """Column-sharded trace commitment. `local_cols`: this rank's column block [c_local, n] as a
    torch int64 tensor on the backend's device. All ranks must own the same number of columns
    (ncols_total % world == 0). Returns (root, row shard, subtree leaf digests, subtree nodes)."""
    world = dist.get_world_size(group)
    n = 1 << log_n
    N = n << log_blowup
    assert ncols_total % world == 0, "columns must divide evenly across ranks"
    assert N % world == 0 and world & (world - 1) == 0, "world size must be a power of two"
    cl = ncols_total // world
    assert tuple(local_cols.shape) == (cl, n)
    rows_per = N // world
    # 1. local LDE of the owned columns, regrouped by destination rank
    send = backend.pack(local_cols, cl, n, log_blowup, world)
    # 2. ONE all-to-all: row range r of every column block goes to rank r
    recv = torch.empty_like(send)
    dist.all_to_all_single(recv.view(-1), send.view(-1), group=group)
    # 3. leaves + subtree over my rows
    root_local, rows, digests, nodes = backend.commit(hash_id, recv, rows_per, ncols_total, cl)
    # 4. all-gather the subtree roots, finish the top of the tree on every rank
    mine = torch.frombuffer(bytearray(root_local), dtype=torch.uint8).to(send.device)
    gathered = [torch.empty_like(mine) for _ in range(world)]
    dist.all_gather(gathered, mine, group=group)
    roots = [bytes(g.cpu().numpy()) for g in gathered]
    return top_levels(hash_id, roots), rows, digests, nodes


# --------------------------------------------------------------------------------------------------
# One proof sharded over the ranks of a torch.distributed group (wf_prove_fib_sharded, wf_prove_air_sharded,
# wf_prove_air_aux_sharded, include/winterfell_b200.h).
# The library does all arithmetic and orchestration; this module only supplies the three collectives of `wf_comm`.
# --------------------------------------------------------------------------------------------------
import ctypes as C
import time

_EXCHANGE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_void_p), C.c_size_t, C.POINTER(C.c_int),
                           C.POINTER(C.c_void_p), C.c_size_t)
_GATHER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t)
_REDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t)
_FORK_FN = C.CFUNCTYPE(C.c_int, C.c_void_p)


class WfComm(C.Structure):
    _fields_ = [("user", C.c_void_p), ("rank", C.c_int), ("world", C.c_int), ("exchange", _EXCHANGE_FN), ("all_gather_host", _GATHER_FN),
                ("all_reduce_sum", _REDUCE_FN), ("fork", _FORK_FN), ("join", _FORK_FN)]


class _DevBuf:
    """Raw device memory as a CUDA-array-interface object (torch.as_tensor wraps it without a copy)."""

    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (int(ptr), False), "version": 2}


def _dev_tensor(ptr, nbytes, device):
    return torch.as_tensor(_DevBuf(ptr, nbytes), device=device)


class TorchComm:
    """wf_comm over torch.distributed. backend "nccl": device buffers go straight into NCCL send/recv on the context's
    stream (NVLink / NVSwitch peer copies). backend "gloo": staged through host memory — the CPU-side test double of the
    same call sequence (lets two ranks share one GPU in the tests)."""

    def __init__(self, stream=None, group=None, device=None):
        self.group = group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.nccl = dist.get_backend(group) == "nccl"
        self.stream = stream
        self.device = device if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.error = None
        self.side = torch.cuda.Stream(device=self.device) if self.nccl else None   # exchanges overlapped with compute (fork / join)
        self._forked = False
        # gloo (host-staged test double): no overlap, the callbacks stay NULL and every exchange is ordered on the ctx stream
        # WF_COMM_NO_FORK=1: NCCL exchanges stay on the context stream (blocking in stream order; the measured alternative)
        overlap = self.nccl and os.environ.get("WF_COMM_NO_FORK", "0") in ("", "0")
        fork = _FORK_FN(self._fork) if overlap else _FORK_FN()
        join = _FORK_FN(self._join) if overlap else _FORK_FN()
        self._keep = (_EXCHANGE_FN(self._exchange), _GATHER_FN(self._gather), _REDUCE_FN(self._reduce), fork, join)
        self.struct = WfComm(None, self.rank, self.world, *self._keep)

    def _main(self):
        return self.stream if self.stream is not None else torch.cuda.current_stream()

    def _ctx(self):
        return torch.cuda.stream(self.side if self._forked else self._main())

    def _fork(self, _user):
        def run():
            ev = torch.cuda.Event()
            ev.record(self._main())
            self.side.wait_event(ev)
            self._forked = True
        return self._guard(run)

    def _join(self, _user):
        def run():
            if self._forked:
                ev = torch.cuda.Event()
                ev.record(self.side)
                self._main().wait_event(ev)
            self._forked = False
        return self._guard(run)

    def _guard(self, fn):
        try:
            fn()
            return 0
        except Exception as e:  # must not unwind through the C caller
            import traceback
            traceback.print_exc()
            self.error = e
            return 1

    def _exchange(self, _user, nsend, send_peer, send_ptr, nrecv, recv_peer, recv_ptr, nbytes):
        def run():
            with self._ctx():
                sends = [(send_peer[i], _dev_tensor(send_ptr[i], nbytes, self.device)) for i in range(nsend)]
                recvs = [(recv_peer[i], _dev_tensor(recv_ptr[i], nbytes, self.device)) for i in range(nrecv)]
                if self.nccl:
                    ops = [dist.P2POp(dist.isend, t, p, self.group) for p, t in sends] + [dist.P2POp(dist.irecv, t, p, self.group) for p, t in recvs]
                    if ops:
                        for req in dist.batch_isend_irecv(ops):
                            req.wait()   # stream-ordered on the current (= context) stream, not a host wait
                else:
                    if self.stream is not None:
                        self.stream.synchronize()
                    host_in = [torch.empty(nbytes, dtype=torch.uint8) for _ in recvs]
                    reqs = [dist.isend(t.cpu(), p, group=self.group) for p, t in sends]
                    reqs += [dist.irecv(h, p, group=self.group) for (p, _), h in zip(recvs, host_in)]
                    for q in reqs:
                        q.wait()
                    for (_, t), h in zip(recvs, host_in):
                        t.copy_(h)
        return self._guard(run)

    def _gather(self, _user, send, recv, nbytes):
        def run():
            mine = torch.frombuffer((C.c_uint8 * nbytes).from_address(send), dtype=torch.uint8).clone()
            out = torch.frombuffer((C.c_uint8 * (nbytes * self.world)).from_address(recv), dtype=torch.uint8)
            if self.nccl:
                with self._ctx():
                    d_all = torch.empty(nbytes * self.world, dtype=torch.uint8, device=self.device)
                    dist.all_gather_into_tensor(d_all, mine.to(self.device), group=self.group)
                    out.copy_(d_all.cpu())
            else:
                parts = [torch.empty(nbytes, dtype=torch.uint8) for _ in range(self.world)]
                dist.all_gather(parts, mine, group=self.group)
                out.copy_(torch.cat(parts))
        return self._guard(run)

    def _reduce(self, _user, d_buf, words):
        def run():
            with self._ctx():
                t = _dev_tensor(d_buf, words * 8, self.device).view(torch.int64)
                if self.nccl:
                    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
                else:
                    if self.stream is not None:
                        self.stream.synchronize()
                    h = t.cpu()
                    dist.all_reduce(h, op=dist.ReduceOp.SUM, group=self.group)
                    t.copy_(h)
        return self._guard(run)


def prove_fib_sharded(ctx, comm, local_trace, k, log_n, results, opts, out_buf=None, device_ptr=None, stats=None):
    """One FibSmall x k proof over comm.world GPUs. local_trace: this rank's [2k / world, n] uint64 columns (host), or
    device_ptr = raw pointer to the same block column-major in HBM. Returns the proof bytes (identical on every rank)."""
    L = wf.lib()
    r_ = np.ascontiguousarray(results, dtype=np.uint64)
    o_ = np.ascontiguousarray(opts, dtype=np.uint32)
    buf = out_buf if out_buf is not None else np.zeros(1 << 23, dtype=np.uint8)
    ln = C.c_size_t(buf.size)
    st = (C.c_double * 8)()
    if device_ptr is None:
        a = np.ascontiguousarray(local_trace, dtype=np.uint64)
        ptrs = (wf.u64p * a.shape[0])(*[a[j].ctypes.data_as(wf.u64p) for j in range(a.shape[0])])
        dptr = None
    else:
        ptrs, dptr = None, C.c_void_p(device_ptr)
    ctx.check(L.wf_prove_fib_sharded(ctx.h, C.byref(comm.struct), ptrs, dptr, 0, k, log_n, r_.ctypes.data_as(wf.u64p),
                                     o_.ctypes.data_as(C.POINTER(C.c_uint32)), buf.ctypes.data_as(wf.u8p), C.byref(ln), st))
    if comm.error is not None:
        raise comm.error
    if stats is not None:
        stats.update(_sharded_stats(st))
    return buf[: ln.value].tobytes()


def _local_columns(comm, d_, local_trace, log_n, device_ptr):
    """This rank's main columns for wf_prove_air[_aux]_sharded: (column pointers, device pointer, what is wrong with the block
    or None, the array the pointers point into)."""
    ptrs, dptr, wrong, a = None, None, None, None
    if device_ptr is not None:
        dptr = C.c_void_p(device_ptr)
    elif local_trace is not None and len(local_trace):
        a = np.ascontiguousarray(local_trace, dtype=np.uint64)
        ptrs = (wf.u64p * a.shape[0])(*[a[j].ctypes.data_as(wf.u64p) for j in range(a.shape[0])])
        try:
            _, count = wf.shard_columns(int(d_[0]) if d_.size else 0, comm.world, comm.rank)
        except wf.WfError:   # no ownership to compare against: the library refuses the description or the world size itself
            count = a.shape[0]
        if a.shape[0] != count or a.shape[1] != 1 << log_n:
            # the library cannot see the length of a column list: this rank passes no columns, which the library refuses for a
            # rank that owns some (and columns, which it refuses for one that owns none), so the refusal goes through its
            # agreement step and every rank returns the error instead of waiting on this one
            wrong = f"rank {comm.rank} passed a [{a.shape[0]}, {a.shape[1]}] block, owns {count} columns of {1 << log_n} rows"
            ptrs = None if count else ptrs
    return ptrs, dptr, wrong, a


def _sharded_stats(st):
    return {"bytes_sent": st[0], "exchange_ms": st[1], "collectives": st[2], "small_collective_ms": st[3], "sharded_fri_layers": st[4],
            "bytes_overlapped": st[5], "peer_push": st[6]}


def prove_air_sharded(ctx, comm, desc, local_trace, log_n, opts, mont=False, device_ptr=None, stats=None, out_buf=None):
    """One proof of a single-segment AIR description (as Context.prove_air) over comm.world GPUs. local_trace: this rank's
    columns (wf.shard_columns(width, world, rank)) as a [count, n] uint64 host array, or device_ptr = raw pointer to the same
    block column-major in HBM; a rank that owns no column passes an empty array or None. desc, log_n and opts are the whole
    proof's. Returns the proof bytes (identical on every rank). Every rank raises when any rank refuses the arguments."""
    L = wf.lib()
    d_ = np.ascontiguousarray(desc, dtype=np.uint64)
    o_ = np.ascontiguousarray(opts, dtype=np.uint32)
    buf = out_buf if out_buf is not None else np.zeros(1 << 23, dtype=np.uint8)
    ln = C.c_size_t(buf.size)
    st = (C.c_double * 8)()
    ptrs, dptr, wrong, _keep = _local_columns(comm, d_, local_trace, log_n, device_ptr)
    r = L.wf_prove_air_sharded(ctx.h, C.byref(comm.struct), d_.ctypes.data_as(wf.u64p), d_.size, ptrs, dptr, int(mont), log_n,
                               o_.ctypes.data_as(C.POINTER(C.c_uint32)), buf.ctypes.data_as(wf.u8p), C.byref(ln), st)
    if comm.error is not None:
        raise comm.error
    if r != wf.WF_OK and wrong:
        raise wf.WfError(f"error {r}: {wrong}")
    ctx.check(r)
    if stats is not None:
        stats.update(_sharded_stats(st))
    return buf[: ln.value].tobytes()


def prove_air_aux_sharded(ctx, comm, desc, local_trace, log_n, opts, builder, values_fn=None, mont=False, device_ptr=None, stats=None,
                          out_buf=None):
    """One proof of a two-segment AIR description (as Context.prove_air_aux, or prove_air_aux_dyn with values_fn) over
    comm.world GPUs. The main columns are passed as in prove_air_sharded. builder(rand [nr, d], first_col, num_cols) ->
    [num_cols, n, d]: the aux E columns [first_col, first_col + num_cols) this rank owns components of (wf_prove_air_aux_sharded;
    not called on a rank that owns no aux column; must be deterministic: an E column split between two ranks is built by
    both). values_fn(rand, values [nv, d]) -> values: the aux assertion values (Air::get_aux_assertions), called on every
    rank, which must all return the same. An exception inside a callback makes every rank fail: the rank it happened on
    re-raises it, the others raise WfError. Returns the proof bytes (identical on every rank); stats also gets "callback_ms",
    the time this rank spent in the two callbacks."""
    L = wf.lib()
    d_ = np.ascontiguousarray(desc, dtype=np.uint64)
    o_ = np.ascontiguousarray(opts, dtype=np.uint32)
    buf = out_buf if out_buf is not None else np.zeros(1 << 23, dtype=np.uint8)
    ln = C.c_size_t(buf.size)
    st = (C.c_double * 8)()
    ptrs, dptr, wrong, _keep = _local_columns(comm, d_, local_trace, log_n, device_ptr)
    _, nr, nv = wf.aux_shape(d_)
    d, n = int(o_[3]) if o_.size > 3 else 1, 1 << log_n
    raised = []

    def guard(fn):
        def wrapped(*args):
            try:
                fn(*args)
                return 0
            except Exception as e:  # must not unwind through the C caller; the library's agreement step fails every rank
                raised.append(e)
                return 1
        return wrapped

    def cb_build(_user, rand_p, first_col, num_cols, out_p):
        rand = np.ctypeslib.as_array(rand_p, shape=(nr, d)).copy() if nr else np.zeros((0, d), dtype=np.uint64)
        aux = np.ascontiguousarray(builder(rand, first_col, num_cols), dtype=np.uint64).reshape(num_cols, n, d)
        np.ctypeslib.as_array(out_p, shape=(num_cols, n, d))[:] = aux

    def cb_values(_user, rand_p, val_p):
        rand = np.ctypeslib.as_array(rand_p, shape=(nr, d)).copy() if nr else np.zeros((0, d), dtype=np.uint64)
        vals = np.ctypeslib.as_array(val_p, shape=(nv, d))
        vals[:] = np.ascontiguousarray(values_fn(rand, vals.copy()), dtype=np.uint64).reshape(nv, d)

    fb = wf.AUX_SHARD_BUILDER(guard(cb_build)) if builder is not None else wf.AUX_SHARD_BUILDER()   # (NULL: refused)
    fv = wf.AUX_BUILDER(guard(cb_values)) if values_fn is not None else wf.AUX_BUILDER()
    r = L.wf_prove_air_aux_sharded(ctx.h, C.byref(comm.struct), d_.ctypes.data_as(wf.u64p), d_.size, ptrs, dptr, int(mont), log_n,
                                   o_.ctypes.data_as(C.POINTER(C.c_uint32)), fb, fv, None, buf.ctypes.data_as(wf.u8p), C.byref(ln), st)
    if comm.error is not None:
        raise comm.error
    if raised:
        raise raised[0]
    if r != wf.WF_OK and wrong:
        raise wf.WfError(f"error {r}: {wrong}")
    ctx.check(r)
    if stats is not None:
        stats.update(_sharded_stats(st))
        stats["callback_ms"] = st[7]
    return buf[: ln.value].tobytes()


def bench_sharded(ctx, stream, cfg, steps, warmup, configs, proof_opts, flush, clock_sampler_cls, local_rank):
    """bench.py's N > 1 arm: ONE proof of `cfg` sharded over the ranks (strong scaling). Returns bench.py's record:
    ms per proof with this rank's column block resident in HBM, e2e ms from pinned host columns, stage times, the
    communication volume, and the byte-identity check against the single-GPU proof (rank 0 proves the whole trace once,
    untimed)."""
    pairs, log_n, ext = configs[cfg]
    rank, world = dist.get_rank(), dist.get_world_size()
    cols, n = 2 * pairs, 1 << log_n
    cl = cols // world
    opts = proof_opts(ext)
    full, results = wf.build_fib_trace(pairs, n)                       # every rank derives the public inputs
    host = torch.empty((cl, n), dtype=torch.int64).pin_memory()
    host_np = host.numpy().view(np.uint64)
    host_np[:] = full[rank * cl:(rank + 1) * cl]
    if rank != 0:
        del full
    dev = host.cuda()
    comm = TorchComm(stream)
    out_buf = np.zeros(1 << 23, dtype=np.uint8)
    stats = {}

    def step_resident():
        return prove_fib_sharded(ctx, comm, None, pairs, log_n, results, opts, out_buf=out_buf, device_ptr=dev.data_ptr(), stats=stats)

    def step_e2e():
        return prove_fib_sharded(ctx, comm, host_np, pairs, log_n, results, opts, out_buf=out_buf, stats=stats)

    def barrier():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()

    step_log, last_outputs = {}, {}

    def timed(fn, k, name):
        total, per = 0.0, []
        for _ in range(k):
            flush.zero_()
            barrier()                                                    # ranks start a proof together
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            out = fn()
            b.record(stream)
            b.synchronize()
            per.append(a.elapsed_time(b))
            total += per[-1]
        step_log[name] = per
        last_outputs[name] = out
        return total / k

    with torch.cuda.stream(stream):
        for _ in range(warmup):
            proof = step_resident()
        p2 = step_e2e()
        assert proof == p2, "resident and e2e arms produced different proofs"
        identical = None
        if rank == 0:                                                    # single-GPU proof of the whole trace, untimed
            want = ctx.prove_fib(full, results, opts)
            identical = proof == want
            del full
        barrier()
        # rank 0's single-GPU proof re-shuffled its buffer pool: the staging buffer of its next sharded proof is a different
        # allocation, which every peer has to map once (cudaIpcOpenMemHandle, ~7 ms on all ranks). One more untimed proof puts
        # the pools back into their steady state before the timed region.
        proof = step_resident()
        barrier()
        sampler = clock_sampler_cls(local_rank)
        sampler.start()
        l0 = ctx.launches
        t0 = time.perf_counter()
        ms = timed(step_resident, steps, "resident")
        wall = (time.perf_counter() - t0) * 1e3 / steps
        launches = int(ctx.launches - l0) // max(steps, 1)
        res_stats = dict(stats)
        e2e = timed(step_e2e, steps, "e2e")
        sampler.stop_flag = True
        sampler.join(timeout=2)
        flush.zero_()
        barrier()
        ctx.set_profiling(True)
        step_resident()
        breakdown = {k: round(v, 4) for k, v in ctx.stage_times()}
        ctx.set_profiling(False)
    # every rank's device time of every timed step (ms): the reported value is the max over ranks of the per-rank means
    per_rank = torch.tensor([step_log["resident"], step_log["e2e"]], device="cuda", dtype=torch.float64)
    gathered = [torch.empty_like(per_rank) for _ in range(world)]
    dist.all_gather(gathered, per_rank)
    step_ms_by_rank = {"resident": [[round(float(x), 3) for x in g[0]] for g in gathered],
                       "e2e": [[round(float(x), 3) for x in g[1]] for g in gathered]}
    gbps = res_stats["bytes_sent"] / max(res_stats["exchange_ms"], 1e-9) / 1e6
    bd_ex = breakdown.get("trace_exchange", 0.0)
    return {"ms": ms, "e2e_ms": e2e, "launches": launches, "breakdown": breakdown, "proof": proof, "h2d": int(host_np.nbytes) * world,
            "wall_ms": wall, "clocks": sampler.summary(),
            "last_outputs": {"proof": last_outputs["resident"], "proof_e2e": last_outputs["e2e"]},
            "parallelism": f"one proof sharded over {world} GPUs: column-sharded interpolate + LDE, exchange into row shards, row-sharded "
                           "commitments / constraints / DEEP / first FRI layers, subtree-root all-gathers (winterfell_b200/dist.py)",
            "comm": {"limiting_collective": ("column shards -> row shards of the trace LDE fused into the LDE: the last pass of every coset's transform stores each "
                                             "row (and the halo rows) straight into its owner's shard, peer memory mapped through CUDA IPC, over NVLink; closed "
                                             "by one host barrier; no NCCL call on the data path"
                                             if res_stats.get("peer_push") == 2 else
                                             "column shards -> row shards of the trace LDE, per coset, as peer copies (copy engines over NVLink) into the other "
                                             "ranks' buffers mapped through CUDA IPC, overlapped with the extension of the next coset; closed by one host barrier"
                                             if res_stats.get("peer_push") else
                                             "exchange (NCCL send/recv all-to-all: column shards -> row shards of the trace LDE), issued per coset on the "
                                             "communicator's stream and overlapped with the extension of the next coset"),
                     "overlapped_bytes_sent_per_rank": int(res_stats.get("bytes_overlapped", 0)),
                     "exposed_trace_exchange_ms_rank0": round(bd_ex, 3),
                     "effective_GBps_per_rank_if_not_overlapped": round(res_stats.get("bytes_overlapped", 0) / max(bd_ex, 1e-9) / 1e6, 1),
                     "blocking_bytes_sent_per_rank": int(res_stats["bytes_sent"]), "blocking_exchange_ms_rank0": round(res_stats["exchange_ms"], 3),
                     "blocking_exchange_GBps_per_rank": round(gbps, 1), "collectives_per_proof": int(res_stats["collectives"]),
                     "host_collective_ms": round(res_stats["small_collective_ms"], 3), "sharded_fri_layers": int(res_stats["sharded_fri_layers"]),
                     "byte_identical_to_single_gpu": identical, "step_ms_by_rank": step_ms_by_rank}}
