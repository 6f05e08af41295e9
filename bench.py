#!/usr/bin/env python
"""bench.py -- Allreduce(float32, sum) bus bandwidth, the metric BASELINE.json names.

    python bench.py --gpus N --steps K --warmup W            (N>1: one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N ...            (restated reference TCP path, host cores)

One JSON line on stdout (rank 0).  A "step" is one Allreduce of S bytes per rank (default
S = 256 MiB, the headline point) on synthetic uniform[0,1) buffers; out of place, so the input
is identical every step.  Send+recv buffers (2 x 256 MiB) exceed the 126 MB L2, so no flush is
needed between steps.

  value     N >= 2: bus bandwidth, nccl-tests convention: S/t * 2(N-1)/N, GB = 1e9 B, device
            resident buffers, t = CUDA-event time over K back-to-back steps / K, max over ranks.
            N == 1: the collective degenerates to a local copy; the bus factor is 0 there, so the
            line reports algorithm bandwidth S/t and says so in config.note.
  e2e       the same quantity through the blocking public call with HOST (pinned, NUMA-local)
            buffers: H2D of the input and D2H of the result inside every step.  e2e.roofline is the
            measured bound of that path on this box: all ranks copying S up and S down at the same
            time with no collective (b200mpi_pcie_probe).  e2e_pageable: the same call on plain
            numpy (pageable) arrays, what an unmodified Go caller passes.
  parity    N >= 2: before anything is timed every collective is checked against the CPU oracle
            over the WHOLE buffer on every rank (block by block): Allreduce f32 S bytes with the
            algorithm that is then timed, an odd count (tail path), i64 through the switch, LL,
            Bcast S from the first and the last rank, Allgather i64 1 Mi per rank, ReduceScatter,
            a 1 MiB float64 ping-pong.  Any mismatch: the flag is false and the exit code is 1.
  secondary N >= 2: Bcast S busbw, Allgather (1 Mi int64 per rank) busbw, 1 MiB float64 bounce
            round trip, 1 KiB / 32 KiB / 1 MiB Allreduce latency, the link ceilings measured in the
            same job (b200mpi_link_probe: one direction busy, both directions busy), NCCL's allreduce
            on the same buffers (comparison line only, run last and under a deadline; NCCL is never
            on the product path).  roofline.nvlink_counters: hardware link byte counts
            (nvidia-smi nvlink) around 50 more steps of the timed call, when the tool exposes them.
  roofline  N == 1: HBM (read S + write S per launch) against MEASURED_PEAKS.json hbm_gbs;
            N >= 2: NVLink, busbw against 900 GB/s nominal (measured peer copy ~770 GB/s) plus the
            HBM side ((3 - 1/N) * S per launch).
  cpu_baseline / --impl reference: oracle/ref_tcp.c, the restated gob-over-TCP-loopback path of
            the reference (it has no Allreduce; composed as a ring over Send/Receive), SAME
            config: S bytes per rank, N ranks, same steps/warm-up unless that exceeds ~90 s (then
            capped, and config.steps_capped says so).  The only uses of oracle/ here are that
            baseline, the input generator and the parity checks -- never the measured path.

  --dump-outputs DIR  after the timed steps every rank writes the Allreduce result its last timed step
            delivered, DIR/allreduce_recv_rank<r>.npy (float32), so that two builds can be compared output
            for output on the same seeded inputs.  Above DUMP_ELEMS elements over all ranks each rank writes
            a stratified sample instead: with k = DUMP_ELEMS // N and stride = count // k, element
            i * stride + o_i for i < k, o_i = np.random.default_rng(SEED).integers(0, stride, k)[i].
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SEED = 0xB2000000
NVLINK_NOMINAL_GBS = 900.0   # per direction per GPU (B200_PROFILING.md)
NVLINK_MEASURED_GBS = 770.0  # peer copy measured on this pool (B200_PROFILING.md)
HBM_FALLBACK_GBS = 6650.0
BLOCK = 1 << 22              # elements per parity block
DUMP_ELEMS = 1 << 23         # --dump-outputs: float32 elements over all ranks (32 MiB)


def world_from_env(args):
    """torchrun env (RANK/LOCAL_RANK/WORLD_SIZE/MASTER_*) or a single rank."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    if world == 1:
        return rank, world, local, "", []
    mport = int(os.environ.get("MASTER_PORT", "29500"))
    base = 20000 + (mport * 7 + 13) % 30000  # 5 digits for every rank: sorted order == rank order
    addrs = ["127.0.0.1:%d" % (base + r) for r in range(world)]
    return rank, world, local, addrs[rank], addrs


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu = gpu
        self.rows = []
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([c.strip() for c in line.split(",")])
        except Exception:  # noqa: BLE001
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        self.join(timeout=2)
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for k, nm in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:  # noqa: BLE001
                continue
        # the sampler also sees idle samples around the region: "under load" = top half
        sm.sort()
        load = sm[len(sm) // 2:] if sm else []
        return {"sm_mhz": (load[len(load) // 2] if load else None), "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:  # noqa: BLE001
        return {"hbm_gbs": HBM_FALLBACK_GBS}, "fallback"


def measured_traffic(n, nbytes, kernel):
    """dram read+write bytes per launch from the committed ncu captures (profiles/traffic.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            for e in json.load(f)["entries"]:
                if e["n"] == n and e["bytes"] == nbytes and e["kernel"] == kernel:
                    return e["traffic_bytes"], e["source"]
    except Exception:  # noqa: BLE001
        pass
    return None, None


def nvlink_counters(gpu):
    """Sum of the per-link NVLink data counters of one GPU (`nvidia-smi nvlink -gt d`), in bytes:
    (tx, rx), or None when the tool or the counters are not there.  ncu cannot read the NVLink
    counters on this pool, so this is the only hardware count of link bytes."""
    import re
    try:
        out = subprocess.run(["nvidia-smi", "nvlink", "-gt", "d", "-i", str(gpu)], capture_output=True, text=True, timeout=20).stdout
        tx = rx = 0
        seen = False
        for m in re.finditer(r"Data\s+(Tx|Rx)\s*:\s*(\d+)\s*(KiB|KB|MiB|B)?", out):
            mult = {"KiB": 1024, "KB": 1000, "MiB": 1 << 20, "B": 1, None: 1024}[m.group(3)]
            if m.group(1) == "Tx":
                tx += int(m.group(2)) * mult
            else:
                rx += int(m.group(2)) * mult
            seen = True
        return (tx, rx) if seen else None
    except Exception:  # noqa: BLE001
        return None


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:  # noqa: BLE001
        return os.cpu_count() or 1


def reference_arm(n, count, dtype, steps, warmup, budget_s=90.0, processes=True):
    """Times oracle/ref_tcp.c (restated reference) on this host with n ranks, one OS process per rank
    as gompirun starts them (2 threads each: Send runs beside Receive): the same S, n, steps and warm-up
    as the GPU arm unless a one-step probe says that takes longer than budget_s, in which case
    steps/warm-up are cut (and reported)."""
    from oracle import oracle as O
    t0 = time.time()
    procs = processes
    if procs:
        try:
            probe, _ = O.ref_bench(O.COLL_ALLREDUCE, dtype, n, count, iters=1, warmup=0, seed=SEED, processes=True)
        except RuntimeError:  # fork not possible here: ranks as threads of one process
            procs = False
    if not procs:
        probe, _ = O.ref_bench(O.COLL_ALLREDUCE, dtype, n, count, iters=1, warmup=0, seed=SEED)
    k, w = steps, warmup
    if probe * (k + w) > budget_s:
        w = 1
        k = int(max(1, min(steps, (budget_s - probe) // max(probe, 1e-9))))
    secs, out = O.ref_bench(O.COLL_ALLREDUCE, dtype, n, count, iters=k, warmup=w, seed=SEED, processes=procs)
    ok = True
    for lo in range(0, count, BLOCK):  # whole-buffer check, block by block
        m = min(BLOCK, count - lo)
        want = O.allreduce([O.fill_at(dtype, SEED + r, lo, m) for r in range(n)], order=O.ORDER_F64)
        ok = ok and bool(np.allclose(out[lo:lo + m], want, rtol=1e-6, atol=0))
    return {"secs": secs, "ok": ok, "steps": k, "warmup": w, "capped": (k, w) != (steps, warmup), "probe_s": probe, "wall_s": time.time() - t0,
            "cores": min(2 * n, host_cores()), "ranks_as": "processes" if procs else "threads"}


# ------------------------------------------------------------------------------------------------
def nccl_comparison(lib, L, mpi, rank, n, local, sizes, send_ptr, recv_ptr, cross_check=None):
    """NCCL's own allreduce (float32 sum) on the same device buffers and stream, timed with the same
    event stopwatch.  Comparison line only: loaded with ctypes after every product measurement."""
    out = {}
    try:
        cands = ["libnccl.so.2"]
        try:
            import importlib.util
            spec = importlib.util.find_spec("nvidia.nccl")
            if spec and spec.submodule_search_locations:
                cands.append(os.path.join(list(spec.submodule_search_locations)[0], "lib", "libnccl.so.2"))
        except Exception:  # noqa: BLE001
            pass
        nccl = None
        for c in cands:
            try:
                nccl = ctypes.CDLL(c)
                break
            except OSError:
                continue
        if nccl is None:
            return {"unavailable": "libnccl.so.2 not found"}
        ver = ctypes.c_int(0)
        nccl.ncclGetVersion(ctypes.byref(ver))

        class UniqueId(ctypes.Structure):
            _fields_ = [("internal", ctypes.c_byte * 128)]

        nccl.ncclCommInitRank.argtypes = [ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, UniqueId, ctypes.c_int]
        nccl.ncclCommDestroy.argtypes = [ctypes.c_void_p]

        def agree(flag):
            a = np.array([1 if flag else 0], dtype=np.int64)
            o = np.zeros(1, dtype=np.int64)
            mpi.Allreduce(a, o, mpi.MIN)
            return bool(o[0])

        comm, note = None, None
        for attempt in range(2):
            uid = UniqueId()
            if rank == 0 and nccl.ncclGetUniqueId(ctypes.byref(uid)) != 0:
                return {"unavailable": "ncclGetUniqueId failed"}
            raw = np.frombuffer(bytes(uid), dtype=np.uint8).copy()
            mpi.Bcast(raw, 0)  # the id travels over this library's own Bcast
            ctypes.memmove(ctypes.byref(uid), raw.ctypes.data, 128)
            c = ctypes.c_void_p()
            rc = nccl.ncclCommInitRank(ctypes.byref(c), n, uid, rank)
            if agree(rc == 0):
                comm = c
                break
            if rc == 0:
                nccl.ncclCommDestroy(c)
            note = "first ncclCommInitRank failed on some rank (rc=%d here); retried with NCCL_NVLS_ENABLE=0" % rc
            os.environ["NCCL_NVLS_ENABLE"] = "0"
        if comm is None:
            return {"unavailable": "ncclCommInitRank failed twice", "note": note}
        nccl.ncclAllReduce.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        stream = ctypes.c_void_p()
        lib.b200mpi_get_stream(ctypes.byref(stream))
        out = {"version": ver.value, "sizes": {}}
        if note:
            out["note"] = note
        for nbytes in sizes:
            cnt = nbytes // 4
            iters, warm = (200, 20) if nbytes <= (1 << 20) else (20, 5)
            for _ in range(warm):
                nccl.ncclAllReduce(send_ptr, recv_ptr, cnt, 7, 0, comm, stream)
            lib.b200mpi_stream_sync()
            mpi.Barrier()
            ms = ctypes.c_float()
            lib.b200mpi_timer_start()
            for _ in range(iters):
                nccl.ncclAllReduce(send_ptr, recv_ptr, cnt, 7, 0, comm, stream)
            lib.b200mpi_timer_stop(ctypes.byref(ms))
            a = np.array([ms.value / iters], dtype=np.float64)
            o = np.zeros(1)
            mpi.Allreduce(a, o, mpi.MAX)
            t = float(o[0]) * 1e-3
            out["sizes"][str(nbytes)] = {"us": t * 1e6, "busbw_gbs": nbytes / t / 1e9 * 2 * (n - 1) / n}
        lib.b200mpi_stream_sync()
        # an independent implementation of the same semantics: NCCL's result for the last (largest) size,
        # held to the same tolerance against the CPU oracle as this library's own switch path
        if cross_check is not None:
            try:
                out["result_agrees_with_oracle"] = bool(cross_check())
            except Exception as e:  # noqa: BLE001
                out["result_agrees_with_oracle"] = "check failed: %s" % e
        nccl.ncclCommDestroy(comm)
        return out
    except Exception as e:  # noqa: BLE001
        out["error"] = "%s: %s" % (type(e).__name__, e)
        return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--bytes", type=int, default=256 << 20, help="message size S per rank")
    ap.add_argument("--algo", default="auto")
    ap.add_argument("--params", default="", help="name=value;... passed to b200mpi_set_param")
    ap.add_argument("--cpu-sample-bytes", type=int, default=64 << 20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-nccl", action="store_true")
    ap.add_argument("--deadline", type=int, default=300, help="seconds after which a partial contract line is printed and the run ends")
    ap.add_argument("--nccl-deadline", type=int, default=60, help="seconds the NCCL comparison may take before it is abandoned")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write each rank's Allreduce result of the last timed step to DIR (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what this library's timed path computed; it does not apply to --impl reference")
    if args.warmup < 3:
        args.warmup = 3
    rank, world, local, addr, addrs = world_from_env(args)
    n = world
    dtype = np.float32
    count = args.bytes // 4
    S = count * 4
    bus = (2.0 * (n - 1) / n) if n > 1 else 1.0
    metric = "allreduce_f32_sum_busbw" if n > 1 else "allreduce_f32_sum_algbw"
    workload = "Allreduce float32 sum, %d MiB per rank, %d GPU(s)" % (S >> 20, n)

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        rn = max(args.gpus, 1)
        r = reference_arm(rn, count, dtype, args.steps, args.warmup)
        rbus = (2.0 * (rn - 1) / rn) if rn > 1 else 1.0
        val = S / r["secs"] * rbus / 1e9
        line = {
            "impl": "reference", "metric": "allreduce_f32_sum_busbw" if rn > 1 else "allreduce_f32_sum_algbw",
            "value": val, "unit": "GB/s", "n_gpus": rn, "steps": r["steps"], "warmup": r["warmup"],
            "ms_per_step": r["secs"] * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "Allreduce float32 sum, %d MiB per rank, %d host rank(s) over TCP loopback" % (S >> 20, rn), "bytes_per_rank": S,
                       "steps_capped": r["capped"], "steps_requested": args.steps, "warmup_requested": args.warmup,
                       "note": "restated reference path (oracle/ref_tcp.c): gob encode/decode + 2 TCP conns per pair + ack, ring allreduce composed from Send/Receive; same bytes per rank and rank count as the GPU arm"
                               + ("; steps/warm-up cut to keep the run near 90 s (one step takes %.2f s)" % r["probe_s"] if r["capped"] else "")},
            "cpu_baseline": {"value": val, "unit": "GB/s", "cores": r["cores"], "kind": "port",
                             "sample": "%d MiB per rank, %d timed iterations, %d rank %s x 2 threads" % (S >> 20, r["steps"], rn, r["ranks_as"]), "parity_ok": r["ok"]},
            "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "host_cores": host_cores(), "wall_s": r["wall_s"],
        }
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm
    t_start = time.time()
    os.environ.setdefault("B200MPI_HEAP_BYTES", str(4 * S + (768 << 20)))
    import mpi_b200 as mpi
    from mpi_b200 import _lib as L
    lib = L.load()
    mpi.api._reset_for_tests(mpi.Cuda(Addr=addr, Addrs=addrs, Timeout=120 * 10**9, Gpu=local))
    mpi.Init()
    algo_ids = {"auto": 0, "oneshot": 1, "twoshot": 2, "ring": 3, "nvls": 4, "smem": 5, "ll": 6, "hybrid": 7}
    for kv in [x for x in args.params.split(";") if x]:
        k, v = kv.split("=")
        if lib.b200mpi_set_param(k.encode(), int(v)):
            raise RuntimeError(L.last_error())
    lib.b200mpi_set_algo(L.COLL_ALLREDUCE, algo_ids[args.algo])
    from oracle import oracle as O  # input generator + parity checks only

    info = (ctypes.c_size_t(), ctypes.c_size_t(), ctypes.c_int())
    lib.b200mpi_heap_info(ctypes.byref(info[0]), ctypes.byref(info[1]), ctypes.byref(info[2]))
    nvls = bool(info[2].value)

    send = mpi.Alloc(count, dtype)
    recv = mpi.Alloc(count, dtype)
    for lo in range(0, count, BLOCK):  # inputs generated and uploaded block by block
        m = min(BLOCK, count - lo)
        send[lo:lo + m].copy_from_host(O.fill_at(dtype, SEED + rank, lo, m))
    algo_used = lib.b200mpi_get_algo(L.COLL_ALLREDUCE, count, L.F32) if n > 1 else 0

    def run_steps(k):
        for _ in range(k):
            rc = lib.b200mpi_allreduce_async(send.ptr, recv.ptr, count, L.F32, L.SUM)
            if rc:
                raise RuntimeError(L.last_error())

    def max_over_ranks(v):
        a = np.array([v], dtype=np.float64)
        o = np.zeros(1, dtype=np.float64)
        mpi.Allreduce(a, o, mpi.MAX)
        return float(o[0])

    def all_ranks(flag):
        a = np.array([1 if flag else 0], dtype=np.int64)
        o = np.zeros(1, dtype=np.int64)
        mpi.Allreduce(a, o, mpi.MIN)
        return bool(o[0])

    def close(got, want, ins):
        """SURVEY 8(c): exact for integers; floats within 1e-6 of sum |x_r| (order is the switch's)."""
        if got.dtype.kind != "f":
            return bool(np.array_equal(got, want))
        scale = np.sum([np.abs(x.astype(np.float64)) for x in ins], axis=0)
        return bool(np.all(np.abs(got.astype(np.float64) - want.astype(np.float64)) <= 1e-6 * scale + 1e-300))

    def ring_expect(ins, dt, cnt, lo, m):
        """allreduce_ring_kernel's order for elements [lo, lo+m) of a cnt-element message: chunk c (of
        ceil(groups/n) 16-byte groups) is summed cyclically from rank c; the count % EPV tail in rank order."""
        epv = 16 // np.dtype(dt).itemsize
        groups = cnt // epv
        per = -(-groups // n) if groups else 0
        want = np.empty(m, dtype=dt)
        e = lo
        while e < lo + m:
            if e < groups * epv and per > 0:
                c = (e // epv) // per
                hi = min(lo + m, min((c + 1) * per, groups) * epv)
                rot = [ins[(c + k) % n][e - lo:hi - lo] for k in range(n)]
            else:
                hi = lo + m
                rot = [x[e - lo:hi - lo] for x in ins]
            want[e - lo:hi - lo] = O.allreduce(rot, order=O.ORDER_RANK)
            e = hi
        return want

    def check_allreduce_blocks(dev, dt, cnt, seed, exact_order=None):
        ok = True
        for lo in range(0, cnt, BLOCK):
            m = min(BLOCK, cnt - lo)
            ins = [O.fill_at(dt, seed + r, lo, m) for r in range(n)]
            got = dev[lo:lo + m].to_host()
            if exact_order == O.ORDER_RING:  # chunk boundaries are global: restate them per block
                ok = ok and bool(np.array_equal(got, ring_expect(ins, dt, cnt, lo, m)))
            elif exact_order is not None:
                ok = ok and bool(np.array_equal(got, O.allreduce(ins, order=exact_order)))
            else:
                ok = ok and close(got, O.allreduce(ins, order=O.ORDER_F64), ins)
        return ok

    parity, parity_algos = {}, {}
    t_par = time.time()
    run_steps(args.warmup)
    if lib.b200mpi_stream_sync():
        raise RuntimeError(L.last_error())
    if not args.no_parity:
        # (1) the timed call itself: whole buffer, every rank
        order = None if algo_used in (L.ALGO_NVLS, L.ALGO_HYBRID) else (O.ORDER_RING if algo_used == L.ALGO_RING else O.ORDER_RANK)
        parity["allreduce_f32_full_buffer"] = check_allreduce_blocks(recv, dtype, count, SEED, order) if n > 1 else \
            all(np.array_equal(recv[lo:lo + min(BLOCK, count - lo)].to_host(), O.fill_at(dtype, SEED, lo, min(BLOCK, count - lo))) for lo in range(0, count, BLOCK))
        parity_algos["allreduce_f32_full_buffer"] = L.ALGO_NAMES.get(algo_used, "copy") if n > 1 else "copy"
    if n > 1 and not args.no_parity:
        def fresh(dt, cnt, seed):
            buf = mpi.Alloc(cnt, dt)
            for lo in range(0, cnt, BLOCK):
                m = min(BLOCK, cnt - lo)
                buf[lo:lo + m].copy_from_host(O.fill_at(dt, seed + rank, lo, m))
            return buf
        # (2) odd count: the tail elements and the partial last ownership block, in place
        odd = (1 << 20) + 3
        b = fresh(np.float32, odd, SEED + 100)
        used = lib.b200mpi_get_algo(L.COLL_ALLREDUCE, odd, L.F32)
        mpi.Allreduce(b, b)
        parity["allreduce_f32_odd_count_in_place"] = check_allreduce_blocks(b, np.float32, odd, SEED + 100, None if used in (L.ALGO_NVLS, L.ALGO_HYBRID) else O.ORDER_RANK)
        parity_algos["allreduce_f32_odd_count_in_place"] = L.ALGO_NAMES.get(used)
        b.free()
        # (3) int64 sum, 64 MiB, switch reduction when there is one: bit-exact (wrap-around adds)
        cnt64 = 8 << 20
        b = fresh(np.int64, cnt64, SEED + 200)
        lib.b200mpi_set_algo(L.COLL_ALLREDUCE, L.ALGO_NVLS if nvls else 0)
        used = lib.b200mpi_get_algo(L.COLL_ALLREDUCE, cnt64, L.I64)
        mpi.Allreduce(b, b)
        parity["allreduce_i64_%s" % L.ALGO_NAMES.get(used)] = check_allreduce_blocks(b, np.int64, cnt64, SEED + 200, O.ORDER_RANK)
        b.free()
        # (4) every other allreduce algorithm on 16 Mi elements (64 MiB), exact in its own order
        mid = 16 << 20
        hyb_default = L.get_param("hybrid_p2p_permille")
        b = fresh(np.float32, mid, SEED + 300)
        r2 = mpi.Alloc(mid, np.float32)
        for name, aid, order in (("twoshot", L.ALGO_TWOSHOT, O.ORDER_RANK), ("twoshot_smem", L.ALGO_TWOSHOT_SMEM, O.ORDER_RANK), ("ring", L.ALGO_RING, O.ORDER_RING),
                                 ("nvls", L.ALGO_NVLS, None), ("hybrid", L.ALGO_HYBRID, None)):
            if name in ("nvls", "hybrid") and not nvls:
                continue
            if name == "hybrid" and hyb_default == 0:
                lib.b200mpi_set_param(b"hybrid_p2p_permille", 200)
            lib.b200mpi_set_algo(L.COLL_ALLREDUCE, aid)
            if lib.b200mpi_get_algo(L.COLL_ALLREDUCE, mid, L.F32) != aid:
                continue
            mpi.Allreduce(b, r2)
            parity["allreduce_f32_64MiB_%s" % name] = check_allreduce_blocks(r2, np.float32, mid, SEED + 300, order)
        b.free()
        r2.free()
        # (5) LL (barrier-free small-message path), 1 KiB and 24 KiB, rank order, bit-exact
        lib.b200mpi_set_algo(L.COLL_ALLREDUCE, L.ALGO_LL)
        okll = True
        for c in (256, 6144):
            x = [O.fill(np.float32, SEED + 400 + r, c) for r in range(n)]
            d = mpi.Alloc(c, np.float32).copy_from_host(x[rank])
            for _ in range(3):  # both parities of the cell lanes
                d.copy_from_host(x[rank])
                mpi.Allreduce(d, d)
                okll = okll and bool(np.array_equal(d.to_host(), O.allreduce(x)))
            h = np.array(x[rank])
            mpi.Allreduce(h, h)  # host slice: mapped pinned bounce, one kernel
            okll = okll and bool(np.array_equal(h, O.allreduce(x)))
            d.free()
        parity["allreduce_ll_small"] = okll
        lib.b200mpi_set_algo(L.COLL_ALLREDUCE, algo_ids[args.algo])
        lib.b200mpi_set_param(b"hybrid_p2p_permille", hyb_default)
        # (6) Bcast S bytes from the first and the last rank (AUTO), whole buffer
        for root in (0, n - 1):
            if rank != root:
                for lo in range(0, count, BLOCK):
                    recv[lo:lo + min(BLOCK, count - lo)].copy_from_host(np.full(min(BLOCK, count - lo), -1, dtype=dtype))
            else:
                for lo in range(0, count, BLOCK):
                    m = min(BLOCK, count - lo)
                    recv[lo:lo + m].copy_from_host(O.fill_at(dtype, SEED + 500 + root, lo, m))
            mpi.Bcast(recv, root)
            ok = True
            for lo in range(0, count, BLOCK):
                m = min(BLOCK, count - lo)
                ok = ok and bool(np.array_equal(recv[lo:lo + m].to_host(), O.fill_at(dtype, SEED + 500 + root, lo, m)))
            parity["bcast_f32_root%d" % root] = ok
        parity_algos["bcast"] = L.ALGO_NAMES.get(lib.b200mpi_get_algo(L.COLL_BCAST, count, L.F32))
        # (7) Allgather int64, 1 Mi indices per rank (BASELINE.json configs[4]) with every algorithm
        ag = 1 << 20
        mine = O.fill(np.int64, SEED + 600 + rank, ag)
        gs = mpi.Alloc(ag, np.int64).copy_from_host(mine)
        gr = mpi.Alloc(ag * n, np.int64)
        for name, aid in (("auto", 0), ("push", L.ALGO_ONESHOT), ("ring", L.ALGO_RING), ("nvls", L.ALGO_NVLS)):
            if name == "nvls" and not nvls:
                continue
            lib.b200mpi_set_algo(L.COLL_ALLGATHER, aid)
            gr.copy_from_host(np.zeros(ag * n, dtype=np.int64))
            mpi.Allgather(gs, gr)
            got = gr.to_host()
            parity["allgather_i64_1Mi_%s" % name] = all(np.array_equal(got[r * ag:(r + 1) * ag], O.fill(np.int64, SEED + 600 + r, ag)) for r in range(n))
        lib.b200mpi_set_algo(L.COLL_ALLGATHER, 0)
        parity_algos["allgather"] = L.ALGO_NAMES.get(lib.b200mpi_get_algo(L.COLL_ALLGATHER, ag, L.I64))
        # (8) ReduceScatter int64 (exact) over the gathered buffer
        rs = mpi.Alloc(ag // n * 1, np.int64)
        mpi.ReduceScatter(gr[: (ag // n) * n], rs)
        full = np.concatenate([O.fill(np.int64, SEED + 600 + r, ag) for r in range(n)])[: (ag // n) * n]
        parity["reduce_scatter_i64"] = bool(np.array_equal(rs.to_host(), O.reduce_scatter([full] * n, rank)))
        rs.free()
        gs.free()
        gr.free()
        # (9) bounce: 1 MiB float64 ping-pong between rank pairs (BASELINE.json configs[1]), device and host buffers
        pc = 131072
        ok = True
        if n % 2 == 0:
            msg = O.fill(np.float64, SEED + 700 + (rank & ~1), pc)
            for kind in ("device", "host"):
                # the same two allocations on every rank: the heaps stay laid out identically
                b1 = mpi.Alloc(pc, np.float64) if kind == "device" else np.zeros(pc)
                b2 = mpi.Alloc(pc, np.float64) if kind == "device" else np.zeros(pc)
                if rank % 2 == 0:
                    if kind == "device":
                        b1.copy_from_host(msg)
                    else:
                        b1[:] = msg
                    mpi.Send(b1, rank + 1, 3)
                    back = mpi.Receive(b2, rank + 1, 3)
                    got = back.to_host() if kind == "device" else back
                    ok = ok and bool(np.array_equal(got, msg))
                else:
                    tmp = mpi.Receive(b1, rank - 1, 3)
                    mpi.Send(tmp, rank - 1, 3)
                if kind == "device":
                    b1.free()
                    b2.free()
        parity["bounce_f64_1MiB"] = ok
        # every rank must agree that every check passed on every rank
        for k in list(parity):
            parity[k] = all_ranks(parity[k])
    elif not args.no_parity:
        for k in list(parity):
            parity[k] = bool(parity[k])
    parity_s = time.time() - t_par
    parity_ok = all(parity.values()) if parity else None

    # ------------------------------------------------------------------ timed region (device buffers)
    run_steps(args.warmup)
    if lib.b200mpi_stream_sync():
        raise RuntimeError(L.last_error())
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    mpi.Barrier()
    l0 = lib.b200mpi_launch_count()
    ms = ctypes.c_float(0)
    lib.b200mpi_timer_start()
    run_steps(args.steps)
    if lib.b200mpi_timer_stop(ctypes.byref(ms)):
        raise RuntimeError(L.last_error())
    launches = int(lib.b200mpi_launch_count() - l0)
    mpi.Barrier()
    t_step = max_over_ranks(ms.value / 1e3 / args.steps)
    if args.dump_outputs:  # before anything later in the run writes into recv
        k = min(count, DUMP_ELEMS // n)
        idx = np.arange(count, dtype=np.int64)
        if k < count:
            stride = count // k
            idx = np.arange(k, dtype=np.int64) * stride + np.random.default_rng(SEED).integers(0, stride, k)
        dump = np.empty(idx.size, dtype=dtype)
        for lo in range(0, count, BLOCK):
            m = min(BLOCK, count - lo)
            a, b = np.searchsorted(idx, [lo, lo + m])
            if b > a:
                dump[a:b] = recv[lo:lo + m].to_host()[idx[a:b] - lo]
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "allreduce_recv_rank%d.npy" % rank), dump)

    algbw = S / t_step / 1e9
    value = algbw * bus

    # Everything below adds to the line (end-to-end, secondary, comparison); none of it may cost the run
    # its result.  If the whole bench is still running at the deadline, rank 0 prints what it has.
    core = {"metric": metric, "value": value, "unit": "GB/s", "n_gpus": n, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": t_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload, "bytes_per_rank": S, "algo": L.ALGO_NAMES.get(algo_used, "copy") if n > 1 else "local copy (world of 1)", "nvls": nvls,
                       "note": "partial line: a later section of bench.py did not finish before --deadline"},
            "algbw_gbs": algbw, "e2e": None, "gpu_launches": launches, "clocks": None,
            "roofline": {"bound": "hbm" if n == 1 else "nvlink", "achieved": (2 * S / t_step / 1e9) if n == 1 else value,
                         "peak": HBM_FALLBACK_GBS if n == 1 else NVLINK_NOMINAL_GBS, "unit": "GB/s",
                         "frac": ((2 * S / t_step / 1e9) / HBM_FALLBACK_GBS) if n == 1 else value / NVLINK_NOMINAL_GBS, "traffic": None},
            "parity": dict(parity), "parity_ok": parity_ok}

    def deadline_bail():
        if rank == 0:
            print(json.dumps(core), flush=True)
        os._exit(0 if parity_ok in (True, None) else 1)
    deadline = threading.Timer(max(1.0, args.deadline - (time.time() - t_start)), deadline_bail)
    deadline.daemon = True
    deadline.start()

    # ---- end to end: blocking public call, HOST buffers, H2D + D2H inside every step
    e2e = None
    e2e_pageable = None
    if not args.no_e2e:
        # measured bound of the path: every rank copies S up and S down at once, no collective
        up, down, both = ctypes.c_double(), ctypes.c_double(), ctypes.c_double()
        mpi.Barrier()
        if lib.b200mpi_pcie_probe(S, 3, ctypes.byref(up), ctypes.byref(down), ctypes.byref(both)):
            raise RuntimeError(L.last_error())
        bound = -max_over_ranks(-both.value)  # slowest rank
        roof = {"bound": "pcie", "h2d_gbs": -max_over_ranks(-up.value), "d2h_gbs": -max_over_ranks(-down.value), "bidir_gbs_per_direction": bound,
                "value": bound * bus, "unit": "GB/s", "how": "all %d ranks copy S pinned->device and S device->pinned concurrently, no collective, slowest rank" % n}
        hs, hr = ctypes.c_void_p(), ctypes.c_void_p()
        lib.b200mpi_host_alloc(S, ctypes.byref(hs))
        lib.b200mpi_host_alloc(S, ctypes.byref(hr))
        for lo in range(0, count, BLOCK):
            m = min(BLOCK, count - lo)
            blk = O.fill_at(dtype, SEED + rank, lo, m)
            ctypes.memmove(hs.value + lo * 4, blk.ctypes.data, m * 4)
        k_e2e = max(3, min(args.steps, 10))

        def timed_host(sp, rp):
            for _ in range(2):
                if lib.b200mpi_allreduce(sp, rp, count, L.F32, L.SUM, L.HOST):
                    raise RuntimeError(L.last_error())
            mpi.Barrier()
            t0 = time.perf_counter()
            for _ in range(k_e2e):
                if lib.b200mpi_allreduce(sp, rp, count, L.F32, L.SUM, L.HOST):
                    raise RuntimeError(L.last_error())
            t = max_over_ranks((time.perf_counter() - t0) / k_e2e)
            mpi.Barrier()
            return t
        t_e2e = timed_host(hs, hr)
        e2e = {"value": S / t_e2e / 1e9 * bus, "unit": "GB/s", "h2d_bytes_per_step": S, "d2h_bytes_per_step": S,
               "ms_per_step": t_e2e * 1e3, "steps": k_e2e, "host_memory": "pinned (b200mpi_host_alloc), NUMA node %d" % lib.b200mpi_numa_node(),
               "roofline": roof, "frac_of_roofline": (S / t_e2e / 1e9) / bound if bound > 0 else None}
        core["e2e"] = dict(e2e)
        # result check of the host path (first block + last block)
        res = np.frombuffer((ctypes.c_char * S).from_address(hr.value), dtype=dtype)
        for lo in (0, max(0, count - BLOCK)):
            m = min(BLOCK, count - lo)
            ins = [O.fill_at(dtype, SEED + r, lo, m) for r in range(n)]
            parity["e2e_host_result"] = parity.get("e2e_host_result", True) and close(res[lo:lo + m], O.allreduce(ins, order=O.ORDER_F64), ins)
        lib.b200mpi_host_free(hs)
        lib.b200mpi_host_free(hr)
        # pageable: plain numpy arrays, what an unmodified caller passes (bounce ring + helper threads)
        ps = np.empty(count, dtype=dtype)
        for lo in range(0, count, BLOCK):
            m = min(BLOCK, count - lo)
            ps[lo:lo + m] = O.fill_at(dtype, SEED + rank, lo, m)
        pr = np.zeros(count, dtype=dtype)
        t_pg = timed_host(ps.ctypes.data, pr.ctypes.data)
        lo = max(0, count - BLOCK)
        ins = [O.fill_at(dtype, SEED + r, lo, count - lo) for r in range(n)]
        parity["e2e_pageable_result"] = close(pr[lo:], O.allreduce(ins, order=O.ORDER_F64), ins)
        e2e_pageable = {"value": S / t_pg / 1e9 * bus, "unit": "GB/s", "ms_per_step": t_pg * 1e3, "steps": k_e2e,
                        "host_memory": "pageable numpy arrays through a pinned bounce ring", "vs_pinned": t_pg / t_e2e}
        # opt-in mode for callers whose buffers stay mapped: pin them in place once (cudaHostRegister, cached)
        lib.b200mpi_set_param(b"host_register", 1)
        t_first0 = time.perf_counter()
        if lib.b200mpi_allreduce(ps.ctypes.data, pr.ctypes.data, count, L.F32, L.SUM, L.HOST):
            raise RuntimeError(L.last_error())
        t_first = max_over_ranks(time.perf_counter() - t_first0)
        t_reg = timed_host(ps.ctypes.data, pr.ctypes.data)
        lib.b200mpi_set_param(b"host_register", 0)
        parity["e2e_pageable_result"] = parity["e2e_pageable_result"] and close(pr[lo:], O.allreduce(ins, order=O.ORDER_F64), ins)
        e2e_pageable["registered"] = {"value": S / t_reg / 1e9 * bus, "unit": "GB/s", "ms_per_step": t_reg * 1e3, "vs_pinned": t_reg / t_e2e, "first_call_ms": t_first * 1e3,
                                      "note": "opt-in B200MPI_HOST_REGISTER=1: the caller's arrays are pinned in place on first use (cached by address range), then DMA'd directly"}
        for k in ("e2e_host_result", "e2e_pageable_result"):
            parity[k] = all_ranks(parity[k]) if n > 1 else bool(parity[k])
        parity_ok = all(parity.values())
        del ps, pr

    # ------------------------------------------------------------------ secondary measurements
    secondary = None
    if n > 1 and not args.no_secondary:
        secondary = {}

        def timed_async(fn, iters, warm):
            for _ in range(warm):
                fn()
            if lib.b200mpi_stream_sync():
                raise RuntimeError(L.last_error())
            mpi.Barrier()
            m2 = ctypes.c_float()
            lib.b200mpi_timer_start()
            for _ in range(iters):
                fn()
            if lib.b200mpi_timer_stop(ctypes.byref(m2)):
                raise RuntimeError(L.last_error())
            return max_over_ranks(m2.value * 1e-3 / iters)

        def chk(rc):
            if rc:
                raise RuntimeError(L.last_error())
        t = timed_async(lambda: chk(lib.b200mpi_bcast_async(recv.ptr, count, L.F32, 0)), 10, 3)
        secondary["bcast_%dMiB_busbw_gbs" % (S >> 20)] = S / t / 1e9
        secondary["bcast_algo"] = L.ALGO_NAMES.get(lib.b200mpi_get_algo(L.COLL_BCAST, count, L.F32))
        ag = 1 << 20
        gs = mpi.Alloc(ag, np.int64)
        gr = mpi.Alloc(ag * n, np.int64)
        t = timed_async(lambda: chk(lib.b200mpi_allgather_async(gs.ptr, gr.ptr, ag, L.I64)), 50, 10)
        secondary["allgather_1Mi_i64_busbw_gbs"] = ag * 8 * n / t / 1e9 * (n - 1) / n
        secondary["allgather_1Mi_i64_us"] = t * 1e6
        secondary["allgather_algo"] = L.ALGO_NAMES.get(lib.b200mpi_get_algo(L.COLL_ALLGATHER, ag, L.I64))
        gs.free()
        gr.free()
        # small-message latency: device time per call, back to back on the stream
        for nb in (1024, 32768, 1 << 20):
            c = nb // 4
            t = timed_async(lambda: chk(lib.b200mpi_allreduce_async(send.ptr, recv.ptr, c, L.F32, L.SUM)), 200, 20)
            secondary["allreduce_%dB_us" % nb] = t * 1e6
            secondary["allreduce_%dB_algo" % nb] = L.ALGO_NAMES.get(lib.b200mpi_get_algo(L.COLL_ALLREDUCE, c, L.F32))
        # bounce: 1 MiB float64 round trip (bounce.go:85-138), device buffers then host slices
        if n % 2 == 0:
            pc = 131072
            for kind in ("device", "host"):
                a_ = mpi.Alloc(pc, np.float64) if kind == "device" else np.zeros(pc)
                b_ = mpi.Alloc(pc, np.float64) if kind == "device" else np.zeros(pc)
                reps = 30
                mpi.Barrier()
                t0 = 0.0
                for i in range(reps + 5):
                    if i == 5:
                        t0 = time.perf_counter()
                    if rank % 2 == 0:
                        mpi.Send(a_, rank + 1, 1)
                        mpi.Receive(b_, rank + 1, 1)
                    else:
                        mpi.Receive(b_, rank - 1, 1)
                        mpi.Send(b_, rank - 1, 1)
                rt = max_over_ranks((time.perf_counter() - t0) / reps)
                secondary["bounce_1MiB_f64_rt_us_%s" % kind] = rt * 1e6
                if kind == "device":
                    a_.free()
                    b_.free()

    # what the links deliver to this library's plain copy kernel, measured in the same job: the ceilings
    # the busbw above is held against (one direction busy / both directions busy)
    if secondary is not None:
        tot, used = ctypes.c_size_t(), ctypes.c_size_t()
        lib.b200mpi_heap_info(ctypes.byref(tot), ctypes.byref(used), None)
        if all_ranks(tot.value - used.value >= 2 * S + (64 << 20)):
            probe = {}
            for mode, name in ((2, "rank0_pulls_other_direction_idle"), (3, "rank0_pushes_other_direction_idle"), (0, "all_ranks_pull"),
                               (1, "all_ranks_push"), (4, "all_ranks_pull_and_push")):
                pm = ctypes.c_float()
                if lib.b200mpi_link_probe(S, mode, 5, ctypes.byref(pm)):
                    probe = {"error": L.last_error()}
                    break
                tp = max_over_ranks(pm.value * 1e-3)
                probe[name] = ((2 if mode == 4 else 1) * S / tp / 1e9) if tp > 0 else None
            secondary["link_probe_gbs_per_direction"] = probe
            secondary["link_probe_note"] = "b200mpi_link_probe: copy_bytes_kernel between rank r and r+1, %d MiB, 5 iterations, slowest rank" % (S >> 20)

    # hardware count of link bytes for the timed call (rank 0's GPU): counters before / after 50 more steps
    nvl = None
    if n > 1:
        mpi.Barrier()
        c0 = nvlink_counters(local) if rank == 0 else None
        mpi.Barrier()
        run_steps(50)
        if lib.b200mpi_stream_sync():
            raise RuntimeError(L.last_error())
        mpi.Barrier()
        c1 = nvlink_counters(local) if rank == 0 else None
        if c0 and c1:
            nvl = {"tx_bytes_per_step": (c1[0] - c0[0]) / 50.0, "rx_bytes_per_step": (c1[1] - c0[1]) / 50.0,
                   "tx_gbs": (c1[0] - c0[0]) / 50.0 / t_step / 1e9, "rx_gbs": (c1[1] - c0[1]) / 50.0 / t_step / 1e9,
                   "source": "nvidia-smi nvlink -gt d on rank 0's GPU around 50 more steps of the timed call (includes protocol overhead the counters see)"}

    # keep the GPU under the same load a little longer so nvidia-smi (100 ms period) sees it:
    # the timed region itself is only K x ~0.1-0.7 ms
    n_load = int(min(max(0.6 / t_step, 10), 20000))  # same count on every rank (t_step is the max over ranks)
    run_steps(n_load)
    if lib.b200mpi_stream_sync():
        raise RuntimeError(L.last_error())
    clocks = sampler.stop()
    clocks["window"] = "timed region + e2e region + secondary + 0.6 s of the same launches (sampler period 100 ms)"
    peaks, peak_kind = measured_peaks()
    hbm_peak = float(peaks.get("hbm_gbs", HBM_FALLBACK_GBS))
    if n == 1:
        roof = {"bound": "hbm", "achieved": 2 * S / t_step / 1e9, "peak": hbm_peak, "unit": "GB/s",
                "frac": 2 * S / t_step / 1e9 / hbm_peak, "traffic": None, "peak_source": peak_kind,
                "kernel": "copy_bytes_kernel", "algorithmic_bytes_per_launch": 2 * S}
    else:
        hbm_bytes = (3.0 - 1.0 / n) * S
        aname = L.ALGO_NAMES.get(algo_used, "?")
        roof = {"bound": "nvlink", "achieved": value, "peak": NVLINK_NOMINAL_GBS, "unit": "GB/s",
                "frac": value / NVLINK_NOMINAL_GBS, "frac_of_measured_peer_copy": value / NVLINK_MEASURED_GBS,
                "traffic": None, "peak_source": "nominal NVLink 5 per direction per GPU; measured peer copy %.0f GB/s" % NVLINK_MEASURED_GBS,
                "kernel": "allreduce_%s_kernel" % aname,
                "nvls_link_bytes_per_launch": (1.0 + 1.0 / n) * S if aname == "nvls" else None,
                "algorithmic_bytes_per_launch": 2.0 * (n - 1) / n * S,
                "hbm": {"achieved": hbm_bytes / t_step / 1e9, "peak": hbm_peak, "frac": hbm_bytes / t_step / 1e9 / hbm_peak, "peak_source": peak_kind}}

    if n > 1:
        roof["nvlink_counters"] = nvl
    traffic, tsrc = measured_traffic(n, S, roof["kernel"])
    if traffic is not None:
        roof["traffic"] = traffic
        roof["traffic_source"] = tsrc

    cpu = None
    if rank == 0 and n == 1 and not args.no_cpu_baseline:
        sample = min(args.cpu_sample_bytes, S)
        r = reference_arm(1, sample // 4, dtype, 3, 1, budget_s=30.0, processes=False)  # no fork from a process that holds a CUDA context
        cpu = {"value": sample / r["secs"] / 1e9, "unit": "GB/s", "cores": r["cores"], "kind": "port",
               "sample": "%d MiB, %d iterations, world of 1 = Send/Receive to self (gob encode + decode); the full-size run is `--impl reference`" % (sample >> 20, r["steps"]), "parity_ok": r["ok"]}

    rc_exit = 0 if parity_ok in (True, None) else 1
    line = {
        "metric": metric, "value": value, "unit": "GB/s", "n_gpus": n, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": t_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload, "bytes_per_rank": S, "algo": L.ALGO_NAMES.get(algo_used, "copy") if n > 1 else "local copy (world of 1)",
                   "nvls": nvls, "l2": "inputs+outputs (%d MiB) exceed L2, no flush" % (2 * S >> 20), "params": args.params,
                   "note": ("world of 1: Allreduce degenerates to a device copy, busbw factor 2(N-1)/N is 0, value is algbw S/t" if n == 1
                            else "busbw = S/t * 2(N-1)/N (nccl-tests convention)")},
        "algbw_gbs": algbw, "aggregate_gbs": algbw * n,
        "e2e": e2e, "e2e_pageable": e2e_pageable, "gpu_launches": launches, "clocks": clocks, "roofline": roof,
        "parity": parity, "parity_ok": parity_ok, "parity_algos": parity_algos, "parity_seconds": parity_s,
    }
    if secondary is not None:
        line["secondary"] = secondary
    if cpu is not None:
        line["cpu_baseline"] = cpu

    # NCCL's allreduce on the same buffers: comparison line only, after every product measurement.
    # A foreign library must not be able to cost the run its result: if it has not returned within
    # the deadline, every rank prints what it has (rank 0: the contract line) and leaves.
    if n > 1 and secondary is not None and not args.no_nccl:
        def bail():
            if rank == 0:
                secondary["nccl_allreduce_comparison"] = {"unavailable": "NCCL did not return within %d s; abandoned" % args.nccl_deadline}
                print(json.dumps(line), flush=True)
            os._exit(rc_exit)
        guard = threading.Timer(args.nccl_deadline, bail)
        guard.daemon = True
        guard.start()
        def nccl_cross_check():  # recv now holds NCCL's sum of the same inputs (first and last block)
            ok = True
            for lo in sorted({0, max(0, count - BLOCK)}):
                m = min(BLOCK, count - lo)
                ins = [O.fill_at(dtype, SEED + r, lo, m) for r in range(n)]
                ok = ok and close(recv[lo:lo + m].to_host(), O.allreduce(ins, order=O.ORDER_F64), ins)
            return all_ranks(ok)
        secondary["nccl_allreduce_comparison"] = nccl_comparison(lib, L, mpi, rank, n, local, [1024, 1 << 20, S], send.ptr, recv.ptr, nccl_cross_check)
        guard.cancel()

    deadline.cancel()
    send.free()
    recv.free()
    mpi.Finalize()
    if rank != 0:
        return rc_exit
    print(json.dumps(line))
    return rc_exit


if __name__ == "__main__":
    sys.exit(main())
