"""One rank of a test world.  Usage: _worker.py <scenario> --out FILE [scenario args] -mpi-* flags.
Every scenario drives the product through the public mpi_b200 API / C ABI and checks results
against the CPU oracle (oracle/), which is test infrastructure only."""
import argparse
import json
import os
import sys
import threading
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import mpi_b200 as mpi  # noqa: E402
from mpi_b200 import _lib as L  # noqa: E402
from oracle import oracle as O  # noqa: E402
import _exact as X  # noqa: E402  (tests/, this script's directory)

SEED = 0xB2000000
DTYPES = {"f32": np.float32, "f64": np.float64, "i64": np.int64}
ALGOS = {"auto": 0, "oneshot": 1, "twoshot": 2, "ring": 3, "nvls": 4, "smem": 5, "ll": 6, "hybrid": 7}


def inputs_for(dtype, n, count, salt=0):
    return [O.fill(dtype, SEED + salt * 1000 + r, count) for r in range(n)]


def expect_allreduce(ins, op, algo_used, n, count, dtype):
    """The oracle order that matches the kernel the library ran."""
    nvec = -(-count // (16 // np.dtype(dtype).itemsize))
    if algo_used == L.ALGO_ONESHOT:
        order = O.ORDER_TREE if (n in (2, 4, 8) and nvec <= 4096) else O.ORDER_RANK
    elif algo_used == L.ALGO_RING:
        order = O.ORDER_RING
    elif algo_used in (L.ALGO_NVLS, L.ALGO_HYBRID):
        order = O.ORDER_F64
    else:
        order = O.ORDER_RANK
    return O.allreduce(ins, op=op, order=order), order


TRACE = os.environ.get("B200MPI_TEST_TRACE")
_T0 = None


def trace(msg):
    global _T0
    if not TRACE:
        return
    import time
    if _T0 is None:
        _T0 = time.time()
    with open("%s.rank%d" % (TRACE, mpi.Rank()), "a") as f:
        f.write("%8.3f %s\n" % (time.time() - _T0, msg))


def check_equal(got, want, what, exact=True, ins=None):
    trace(what)
    if exact:
        same = np.array_equal(got.view(np.uint8), want.view(np.uint8))
        if not same and got.dtype.kind == "f":
            # NaN payloads may differ; compare values with NaN == NaN
            same = np.array_equal(got, want, equal_nan=True)
        if not same:
            bad = np.flatnonzero(got != want)[:5]
            raise AssertionError("%s: mismatch at %s got %s want %s" % (what, bad, got[bad], want[bad]))
    else:
        # SURVEY 8(c): |gpu - ref| <= 1e-6 * sum_r |x_r[i]|
        scale = np.sum([np.abs(x.astype(np.float64)) for x in ins], axis=0)
        err = np.abs(got.astype(np.float64) - want.astype(np.float64))
        if not np.all(err <= 1e-6 * scale + 1e-300):
            i = int(np.argmax(err - 1e-6 * scale))
            raise AssertionError("%s: |err| %g > 1e-6*%g at %d" % (what, err[i], scale[i], i))


def make_buffer(kind, arr):
    """kind: 'heap' (DeviceSlice), 'host' (numpy)."""
    if kind == "heap":
        return mpi.Alloc(arr.size, arr.dtype).copy_from_host(arr)
    return np.array(arr, copy=True)


def read_buffer(buf):
    return buf.to_host() if isinstance(buf, mpi.DeviceSlice) else buf


def free_buffer(buf):
    if isinstance(buf, mpi.DeviceSlice):
        buf.free()


# ------------------------------------------------------------------------------------------------
def scenario_collectives(a):
    lib = L.load()
    rank, n = mpi.Rank(), mpi.Size()
    sizes = [int(s) for s in a.sizes.split(",")]
    dtypes = a.dtypes.split(",")
    kinds = a.kinds.split(",")
    info = (L.ctypes.c_size_t(), L.ctypes.c_size_t(), L.ctypes.c_int())
    lib.b200mpi_heap_info(L.ctypes.byref(info[0]), L.ctypes.byref(info[1]), L.ctypes.byref(info[2]))
    nvls = bool(info[2].value)
    # an explicit request for a switch algorithm that cannot run is REPORTED (the test then skips
    # or fails visibly); the default list only names what this world can run
    explicit = a.algos != "default"
    algos = a.algos.split(",") if explicit else ["oneshot", "twoshot", "ring", "smem"] + (["nvls", "hybrid"] if nvls else [])
    done = 0
    skipped = set()
    if "hybrid" in algos:
        lib.b200mpi_set_param(b"hybrid_p2p_permille", 250)
        lib.b200mpi_set_param(b"hybrid_min_bytes", 0)
    for kind in kinds:
        for dn in dtypes:
            dt = DTYPES[dn]
            for count in sizes:
                ins = inputs_for(dt, n, count, salt=count % 97)
                for algo in algos:
                    if algo in ("nvls", "hybrid") and not nvls:
                        skipped.add("allreduce:" + algo)  # reported, never silently passed
                        continue
                    if algo in ("ring", "smem") and n == 1:
                        continue
                    lib.b200mpi_set_algo(L.COLL_ALLREDUCE, ALGOS[algo])
                    used = lib.b200mpi_get_algo(L.COLL_ALLREDUCE, count, O.NP2DT[np.dtype(dt)]) if n > 1 else L.ALGO_TWOSHOT
                    for inplace in (False, True):
                        send = make_buffer(kind, ins[rank])
                        recv = send if inplace else make_buffer(kind, np.zeros(count, dtype=dt))
                        mpi.Allreduce(send, recv, mpi.SUM)
                        got = read_buffer(recv)
                        want, order = expect_allreduce(ins, O.SUM, used, n, count, dt)
                        exact = dt == np.int64 or order != O.ORDER_F64
                        check_equal(got, want, "allreduce %s %s n=%d count=%d algo=%s(%d) inplace=%s" % (kind, dn, n, count, algo, used, inplace), exact=exact, ins=ins)
                        if not inplace:
                            check_equal(read_buffer(send), ins[rank], "allreduce send buffer untouched")
                            free_buffer(recv)
                        free_buffer(send)
                        done += 1
                lib.b200mpi_set_algo(L.COLL_ALLREDUCE, 0)
                # max / min once per dtype and size (default algorithm)
                for op, oop in ((mpi.MAX, O.MAX), (mpi.MIN, O.MIN)):
                    send = make_buffer(kind, ins[rank])
                    recv = make_buffer(kind, np.zeros(count, dtype=dt))
                    mpi.Allreduce(send, recv, op)
                    check_equal(read_buffer(recv), O.allreduce(ins, op=oop), "allreduce op=%d %s count=%d" % (op, dn, count))
                    free_buffer(send)
                    free_buffer(recv)
                    done += 1
                # allgather: push, ring and the switch form
                for algo in ("oneshot", "ring", "nvls"):
                    if algo == "nvls" and not nvls:
                        if explicit and "nvls" in algos:
                            skipped.add("allgather:nvls")
                        continue
                    lib.b200mpi_set_algo(L.COLL_ALLGATHER, ALGOS[algo])
                    send = make_buffer(kind, ins[rank])
                    recv = make_buffer(kind, np.full(count * n, -1, dtype=dt))
                    mpi.Allgather(send, recv)
                    check_equal(read_buffer(recv), O.allgather(ins), "allgather %s %s count=%d algo=%s" % (kind, dn, count, algo))
                    free_buffer(send)
                    free_buffer(recv)
                    done += 1
                lib.b200mpi_set_algo(L.COLL_ALLGATHER, 0)
                # bcast from every root with every algorithm (root 0 and last only for big sizes)
                roots = range(n) if count <= 4096 else sorted({0, n - 1})
                for algo in ("oneshot", "twoshot", "nvls", "nvls_root"):
                    if algo.startswith("nvls") and not nvls:
                        if explicit and "nvls" in algos:
                            skipped.add("bcast:" + algo)
                        continue
                    lib.b200mpi_set_param(b"bcast_nvls2", 0 if algo == "nvls_root" else 1)
                    lib.b200mpi_set_algo(L.COLL_BCAST, ALGOS["nvls" if algo == "nvls_root" else algo])
                    for root in roots:
                        buf = make_buffer(kind, ins[root] if rank == root else np.full(count, -1, dtype=dt).astype(dt))
                        mpi.Bcast(buf, root)
                        check_equal(read_buffer(buf), O.bcast(ins[root]), "bcast %s %s count=%d root=%d algo=%s" % (kind, dn, count, root, algo))
                        free_buffer(buf)
                        done += 1
                lib.b200mpi_set_algo(L.COLL_BCAST, 0)
    mpi.Barrier()
    return {"checked": done, "nvls": nvls, "nvls_skipped": bool(skipped), "skipped": sorted(skipped)}


def pinned_array(count, dtype):
    """numpy view of pinned host memory from b200mpi_host_alloc (on the GPU's NUMA node)."""
    import ctypes
    dt = np.dtype(dtype)
    p = ctypes.c_void_p()
    if L.load().b200mpi_host_alloc(max(count * dt.itemsize, 1), ctypes.byref(p)):
        raise RuntimeError(L.last_error())
    buf = (ctypes.c_char * max(count * dt.itemsize, 1)).from_address(p.value)
    return np.frombuffer(buf, dtype=dt, count=count), p


def scenario_newcolls(a):
    """ReduceScatter, Reduce, Alltoall (API added along the reference's conventions) against the oracle."""
    lib = L.load()
    rank, n = mpi.Rank(), mpi.Size()
    sizes = [int(s) for s in a.sizes.split(",")]
    info = (L.ctypes.c_size_t(), L.ctypes.c_size_t(), L.ctypes.c_int())
    lib.b200mpi_heap_info(L.ctypes.byref(info[0]), L.ctypes.byref(info[1]), L.ctypes.byref(info[2]))
    nvls = bool(info[2].value)
    done, skipped = 0, set()
    for kind in a.kinds.split(","):
        for dn in a.dtypes.split(","):
            dt = DTYPES[dn]
            for count in sizes:
                ins = inputs_for(dt, n, count * n, salt=count % 89 + 3)  # n blocks of `count` per rank
                # ---- ReduceScatter
                for algo in ("twoshot", "nvls"):
                    if algo == "nvls" and not nvls:
                        skipped.add("reduce_scatter:nvls")
                        continue
                    lib.b200mpi_set_algo(L.COLL_REDUCE_SCATTER, ALGOS[algo])
                    for op, oop in ((mpi.SUM, O.SUM), (mpi.MAX, O.MAX)):
                        send = make_buffer(kind, ins[rank])
                        recv = make_buffer(kind, np.zeros(count, dtype=dt))
                        mpi.ReduceScatter(send, recv, op)
                        exact = dt == np.int64 or algo != "nvls" or op != mpi.SUM
                        want = O.reduce_scatter(ins, rank, op=oop, order=O.ORDER_RANK if exact else O.ORDER_F64)
                        blocks = [x[rank * count:(rank + 1) * count] for x in ins]
                        check_equal(read_buffer(recv), want, "reduce_scatter %s %s count=%d algo=%s op=%d" % (kind, dn, count, algo, op), exact=exact, ins=blocks)
                        check_equal(read_buffer(send), ins[rank], "reduce_scatter send untouched")
                        free_buffer(send)
                        free_buffer(recv)
                        done += 1
                    if kind == "heap":  # in place: recv is the caller's own block of send
                        send = make_buffer(kind, ins[rank])
                        mpi.ReduceScatter(send, send[rank * count:(rank + 1) * count], mpi.SUM)
                        exact = dt == np.int64 or algo != "nvls"
                        want = O.reduce_scatter(ins, rank, order=O.ORDER_RANK if exact else O.ORDER_F64)
                        check_equal(send.to_host()[rank * count:(rank + 1) * count], want, "reduce_scatter in place %s count=%d algo=%s" % (dn, count, algo), exact=exact,
                                    ins=[x[rank * count:(rank + 1) * count] for x in ins])
                        free_buffer(send)
                        done += 1
                lib.b200mpi_set_algo(L.COLL_REDUCE_SCATTER, 0)
                # ---- Reduce to every root (small) or to {0, n-1}
                red = [x[:count] for x in ins]
                roots = range(n) if count <= 4096 else sorted({0, n - 1})
                for algo in ("twoshot", "auto"):
                    lib.b200mpi_set_algo(L.COLL_ALLREDUCE, ALGOS[algo])
                    for root in roots:
                        send = make_buffer(kind, red[rank])
                        recv = make_buffer(kind, np.full(count, -7, dtype=dt))
                        mpi.Reduce(send, recv, mpi.SUM, root)
                        got = read_buffer(recv)
                        if rank == root:
                            exact = dt == np.int64 or algo == "twoshot" or not nvls or n < 4
                            check_equal(got, O.allreduce(red, order=O.ORDER_RANK if exact else O.ORDER_F64), "reduce %s %s count=%d root=%d algo=%s" % (kind, dn, count, root, algo), exact=exact, ins=red)
                        else:
                            check_equal(got, np.full(count, -7, dtype=dt), "reduce: non-root recv untouched")
                        free_buffer(send)
                        free_buffer(recv)
                        done += 1
                lib.b200mpi_set_algo(L.COLL_ALLREDUCE, 0)
                # ---- Alltoall
                send = make_buffer(kind, ins[rank])
                recv = make_buffer(kind, np.full(count * n, -1, dtype=dt))
                mpi.Alltoall(send, recv)
                check_equal(read_buffer(recv), O.alltoall(ins, rank), "alltoall %s %s count=%d" % (kind, dn, count))
                free_buffer(send)
                free_buffer(recv)
                done += 1
    mpi.Barrier()
    return {"checked": done, "nvls": nvls, "nvls_skipped": bool(skipped), "skipped": sorted(skipped)}


def scenario_hostpipe(a):
    """Host slices through the chunked H2D | collective | D2H pipeline: pageable memory (pinned
    bounce ring + helper threads) and pinned memory (direct DMA), several chunks per call."""
    lib = L.load()
    rank, n = mpi.Rank(), mpi.Size()
    for k, v in (("pipe_min_bytes", 65536), ("pipe_chunk_bytes", 65536), ("bounce_chunk_bytes", 65536)):
        if lib.b200mpi_set_param(k.encode(), v):
            raise RuntimeError(L.last_error())
    done = 0
    frees = []
    for dn in a.dtypes.split(","):
        dt = DTYPES[dn]
        for count in [int(s) for s in a.sizes.split(",")]:
            ins = inputs_for(dt, n, count, salt=count % 83 + 11)
            for mem in ("pageable", "pinned"):
                def host(arr):
                    if mem == "pageable":
                        return np.array(arr, copy=True)
                    v, p = pinned_array(arr.size, arr.dtype)
                    frees.append(p)
                    v[:] = arr
                    return v
                # allreduce, out of place and in place
                send, recv = host(ins[rank]), host(np.zeros(count, dtype=dt))
                mpi.Allreduce(send, recv)
                used = lib.b200mpi_get_algo(L.COLL_ALLREDUCE, min(count, 65536 // dt().itemsize), O.NP2DT[np.dtype(dt)]) if n > 1 else L.ALGO_TWOSHOT
                exact = dt == np.int64 or used not in (L.ALGO_NVLS, L.ALGO_HYBRID)
                want = O.allreduce(ins, order=O.ORDER_F64) if not exact else None
                if exact:  # chunks of 64 KiB: small-message algorithms, tree order below 4096 vectors
                    want = np.empty(count, dtype=dt)
                    ce = max(65536 // dt().itemsize, 4096) // 4096 * 4096
                    for lo in range(0, count, ce):
                        part = [x[lo:lo + ce] for x in ins]
                        want[lo:lo + ce], _ = expect_allreduce(part, O.SUM, lib.b200mpi_get_algo(L.COLL_ALLREDUCE, len(part[0]), O.NP2DT[np.dtype(dt)]) if n > 1 else L.ALGO_TWOSHOT, n, len(part[0]), dt)
                check_equal(recv, want, "hostpipe allreduce %s %s count=%d" % (mem, dn, count), exact=exact, ins=ins)
                check_equal(send, ins[rank], "hostpipe allreduce send untouched")
                mpi.Allreduce(send, send)
                check_equal(send, want, "hostpipe allreduce in place %s %s count=%d" % (mem, dn, count), exact=exact, ins=ins)
                done += 2
                # bcast from first and last rank
                for root in sorted({0, n - 1}):
                    buf = host(ins[root] if rank == root else np.full(count, -3, dtype=dt))
                    mpi.Bcast(buf, root)
                    check_equal(buf, ins[root], "hostpipe bcast %s %s count=%d root=%d" % (mem, dn, count, root))
                    done += 1
                # allgather
                send, recv = host(ins[rank]), host(np.full(count * n, -1, dtype=dt))
                mpi.Allgather(send, recv)
                check_equal(recv, O.allgather(ins), "hostpipe allgather %s %s count=%d" % (mem, dn, count))
                done += 1
    for p in frees:
        lib.b200mpi_host_free(p)
    mpi.Barrier()
    return {"checked": done, "numa_node": lib.b200mpi_numa_node()}


def scenario_isend(a):
    """Isend/Wait (mpi.go:132-152): the buffer is reusable right after Isend; Wait frees the tag."""
    rank, n = mpi.Rank(), mpi.Size()
    peer = rank ^ 1
    done = 0
    for kind in ("host", "heap"):
        for count in (0, 1, 1000, 300000):
            x = O.fill(np.float64, SEED + rank + count, count)
            buf = make_buffer(kind, x)
            if rank % 2 == 0:
                mpi.Isend(buf, peer, 4)
                # the data left the buffer: scribble over it before the peer has received
                if kind == "host":
                    buf[:] = -1.0
                else:
                    buf.copy_from_host(np.full(count, -1.0))
                try:
                    mpi.Isend(x, peer, 4)
                    raise AssertionError("tag reusable before Wait")
                except mpi.TagExists:
                    pass
                mpi.Send(np.arange(3, dtype=np.int64), peer, 5)  # a second message overtakes nothing: tags differ
                mpi.Wait(peer, 4)
                mpi.Isend(x, peer, 4)  # pair is free again
                mpi.Wait(peer, 4)
            else:
                mpi.Receive(np.zeros(3, dtype=np.int64), peer, 5)
                got = mpi.Receive(make_buffer(kind, np.zeros(count)), peer, 4)
                check_equal(read_buffer(got), O.fill(np.float64, SEED + peer + count, count), "isend %s count=%d" % (kind, count))
                got2 = mpi.Receive(np.zeros(count), peer, 4)
                check_equal(got2, O.fill(np.float64, SEED + peer + count, count), "isend again %s count=%d" % (kind, count))
            free_buffer(buf)
            done += 1
    try:
        mpi.Wait(peer, 77)
        raise AssertionError("Wait without Isend succeeded")
    except mpi.MpiError as e:
        if e.code != L.ERR_ARG:
            raise
    mpi.Barrier()
    return {"checked": done}


def scenario_sendtimeout(a):
    """A Send that times out withdraws its post: a late Receive must not match it, the staging block
    and the mailbox slot are reusable (run with a short B200MPI_WATCHDOG_S)."""
    import time
    rank, n = mpi.Rank(), mpi.Size()
    lib = L.load()
    x = O.fill(np.int64, SEED + 9, 5000)
    used0 = L.ctypes.c_size_t()
    lib.b200mpi_heap_info(None, L.ctypes.byref(used0), None)
    if rank == 0:
        lib.b200mpi_set_param(b"watchdog_ms", 700)
        for _ in range(3):
            try:
                mpi.Send(x, 1, 21)
                raise AssertionError("send without receiver succeeded")
            except mpi.MpiError as e:
                if e.code != L.ERR_TIMEOUT:
                    raise
        used1 = L.ctypes.c_size_t()
        lib.b200mpi_heap_info(None, L.ctypes.byref(used1), None)
        if used1.value != used0.value:
            raise AssertionError("staging leaked after timeouts: %d -> %d" % (used0.value, used1.value))
        lib.b200mpi_set_param(b"watchdog_ms", 120000)
        mpi.Send(np.arange(2, dtype=np.int64), 1, 22)  # go
        for i in range(40):  # more than the 16 slots of the pair
            mpi.Send(x + i, 1, 21)
    elif rank == 1:
        mpi.Receive(np.zeros(2, dtype=np.int64), 0, 22)
        for i in range(40):
            got = mpi.Receive(np.zeros(5000, dtype=np.int64), 0, 21)
            check_equal(got, x + i, "message %d after withdrawn posts" % i)
    mpi.Barrier()
    return {"checked": 41}


def scenario_edge_values(a):
    """f32 edge set {+-0, +-Inf, NaN, subnormal, 1e38} and i64 wrap-around (SURVEY 8(c))."""
    lib = L.load()
    rank, n = mpi.Rank(), mpi.Size()
    edge = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e-45, -1e-45, 1e38, -1e38, 1.0, 3.4e38, 1.17549435e-38], dtype=np.float32)
    count = edge.size * 8
    ins = []
    for r in range(n):
        x = np.tile(edge, 8)
        x = np.roll(x, r * 5)  # different pairings per rank: inf + -inf, 1e38 + 1e38 ...
        ins.append(x.astype(np.float32))
    done = 0
    for algo in ("oneshot", "twoshot", "ring", "smem"):
        if algo == "ring" and n == 1:
            continue
        lib.b200mpi_set_algo(L.COLL_ALLREDUCE, ALGOS[algo])
        used = lib.b200mpi_get_algo(L.COLL_ALLREDUCE, count, L.F32) if n > 1 else L.ALGO_TWOSHOT
        send = mpi.Alloc(count, np.float32).copy_from_host(ins[rank])
        recv = mpi.Alloc(count, np.float32)
        mpi.Allreduce(send, recv)
        want, _ = expect_allreduce(ins, O.SUM, used, n, count, np.float32)
        got = recv.to_host()
        # NaN positions must agree, everything else bit-exact
        if not np.array_equal(np.isnan(got), np.isnan(want)):
            raise AssertionError("edge f32 %s: NaN pattern differs" % algo)
        m = ~np.isnan(want)
        check_equal(got[m], want[m], "edge f32 algo=%s" % algo)
        send.free()
        recv.free()
        done += 1
    lib.b200mpi_set_algo(L.COLL_ALLREDUCE, 0)
    big = np.array([2**63 - 1, -2**63, 2**62, -1, 1, 0x7FFFFFFFFFFFFFF0, 123456789012345678, -987654321098765432], dtype=np.int64)
    ins = [np.roll(np.tile(big, 33), r * 3) for r in range(n)]
    for algo in ("oneshot", "twoshot", "ring", "nvls"):
        if algo == "ring" and n == 1:
            continue
        lib.b200mpi_set_algo(L.COLL_ALLREDUCE, ALGOS[algo])
        buf = mpi.Alloc(ins[0].size, np.int64).copy_from_host(ins[rank])
        mpi.Allreduce(buf, buf)
        check_equal(buf.to_host(), O.allreduce(ins), "i64 wrap algo=%s" % algo)
        buf.free()
        done += 1
    lib.b200mpi_set_algo(L.COLL_ALLREDUCE, 0)
    # all ranks must hold bit-identical floating results: gather everyone's result and compare
    x = [O.fill(np.float32, SEED + 77 + r, 1000) for r in range(n)]
    for algo in ("oneshot", "twoshot", "ring", "nvls"):
        if algo == "ring" and n == 1:
            continue
        lib.b200mpi_set_algo(L.COLL_ALLREDUCE, ALGOS[algo])
        res = np.zeros(1000, dtype=np.float32)
        mpi.Allreduce(np.array(x[rank]), res)
        allres = np.zeros(1000 * n, dtype=np.float32)
        mpi.Allgather(res, allres)
        for r in range(n):
            check_equal(allres[r * 1000:(r + 1) * 1000], res, "rank %d result identical to mine (algo %s)" % (r, algo))
        done += 1
    lib.b200mpi_set_algo(L.COLL_ALLREDUCE, 0)
    return {"checked": done}


def scenario_unaligned(a):
    """Offsets that are not 16-byte aligned and differ between ranks."""
    lib = L.load()
    rank, n = mpi.Rank(), mpi.Size()
    done = 0
    count = 1003
    for dn, dt in DTYPES.items():
        ins = inputs_for(dt, n, count, salt=5)
        big = mpi.Alloc(count + 16, dt)
        out = mpi.Alloc(count + 16, dt)
        so = 1 + (rank % 3)  # element offsets: 4/8 byte granularity, rank dependent
        ro = 1 + ((rank + 1) % 2)
        send = big[so:so + count].copy_from_host(ins[rank])
        recv = out[ro:ro + count]
        for algo in ("oneshot", "twoshot", "ring", "smem"):
            if algo == "ring" and n == 1:
                continue
            lib.b200mpi_set_algo(L.COLL_ALLREDUCE, ALGOS[algo])
            used = lib.b200mpi_get_algo(L.COLL_ALLREDUCE, count, O.NP2DT[np.dtype(dt)]) if n > 1 else L.ALGO_TWOSHOT
            mpi.Allreduce(send, recv)
            want, _ = expect_allreduce(ins, O.SUM, used, n, count, dt)
            if used == L.ALGO_ONESHOT and n in (2, 4, 8):
                want = O.allreduce(ins, order=O.ORDER_TREE)
            check_equal(recv.to_host(), want, "unaligned allreduce %s algo=%s" % (dn, algo))
            done += 1
        lib.b200mpi_set_algo(L.COLL_ALLREDUCE, 0)
        gath = mpi.Alloc(count * n + 16, dt)
        g = gath[ro:ro + count * n]
        for algo in ("auto", "ring"):
            lib.b200mpi_set_algo(L.COLL_ALLGATHER, ALGOS[algo])
            mpi.Allgather(send, g)
            check_equal(g.to_host(), O.allgather(ins), "unaligned allgather %s %s" % (dn, algo))
            done += 1
        lib.b200mpi_set_algo(L.COLL_ALLGATHER, 0)
        for algo in ("oneshot", "twoshot"):
            lib.b200mpi_set_algo(L.COLL_BCAST, ALGOS[algo])
            b = big[so:so + count].copy_from_host(ins[1 % n] if rank == 1 % n else np.zeros(count, dtype=dt))
            mpi.Bcast(b, 1 % n)
            check_equal(b.to_host(), ins[1 % n], "unaligned bcast %s %s" % (dn, algo))
            done += 1
        lib.b200mpi_set_algo(L.COLL_BCAST, 0)
        # mixed access widths: the size is a multiple of 16 but the offsets are 8/16/24 bytes
        # depending on the rank, and the message spans many CTAs
        if dt != np.float32:
            big_n = 65536
            wide = mpi.Alloc(big_n * (n + 1) + 16, dt)
            wsrc = mpi.Alloc(big_n + 16, dt)
            wins = inputs_for(dt, n, big_n, salt=9)
            ws = wsrc[so:so + big_n].copy_from_host(wins[rank])
            wr = wide[2:2 + big_n * n]  # 16-byte aligned everywhere: the send offset alone decides each rank's width
            for algo in ("auto", "ring"):
                lib.b200mpi_set_algo(L.COLL_ALLGATHER, ALGOS[algo])
                mpi.Allgather(ws, wr)
                check_equal(wr.to_host(), O.allgather(wins), "mixed-width allgather %s %s" % (dn, algo))
                done += 1
            lib.b200mpi_set_algo(L.COLL_ALLGATHER, 0)
            for algo in ("oneshot", "twoshot"):
                lib.b200mpi_set_algo(L.COLL_BCAST, ALGOS[algo])
                root = (n - 1) % n
                wb = wsrc[so:so + big_n].copy_from_host(wins[root] if rank == root else np.zeros(big_n, dtype=dt))
                mpi.Bcast(wb, root)
                check_equal(wb.to_host(), wins[root], "mixed-width bcast %s %s" % (dn, algo))
                done += 1
            lib.b200mpi_set_algo(L.COLL_BCAST, 0)
            wide.free()
            wsrc.free()
        # bytes: odd length, odd offset
        raw = np.frombuffer(O.fill(np.int64, SEED + rank, 200).tobytes(), dtype=np.uint8)[:1501]
        rb = np.zeros(1501 * n, dtype=np.uint8)
        mpi.Allgather(np.array(raw), rb)
        want = np.concatenate([np.frombuffer(O.fill(np.int64, SEED + r, 200).tobytes(), dtype=np.uint8)[:1501] for r in range(n)])
        check_equal(rb, want, "byte allgather")
        big.free()
        out.free()
        gath.free()
        done += 1
    return {"checked": done}


def scenario_p2p(a):
    """bounce (examples/bounce/bounce.go:85-138): even/odd ping-pong over the size ladder, []byte then
    []float64, equality checked on the even rank; plus device-resident buffers."""
    rank, n = mpi.Rank(), mpi.Size()
    if n % 2:
        raise AssertionError("Must have an even number of nodes for this example")
    even = rank % 2 == 0
    lengths = [int(s) for s in a.sizes.split(",")]
    maxlen = max(lengths + [8])
    message = np.frombuffer(O.fill(np.int64, SEED + rank, maxlen // 8 + 1).tobytes(), dtype=np.uint8)[:maxlen].copy()
    message_f = O.fill(np.float64, SEED + 100 + rank, maxlen // 8 + 1)
    done = 0
    for l in lengths:
        for rep in range(2):
            msg = message[:l]
            rcv = np.zeros(l, dtype=np.uint8)
            if even:
                mpi.Send(msg, rank + 1, 0)
                rcv = mpi.Receive(rcv, rank + 1, 0)
                check_equal(rcv, msg, "bounce bytes len %d" % l)
            else:
                rcv = mpi.Receive(rcv, rank - 1, 0)
                mpi.Send(rcv, rank - 1, 0)
            msg_f = message_f[: l // 8]
            rcv_f = np.zeros(l // 8, dtype=np.float64)
            if even:
                mpi.Send(msg_f, rank + 1, 0)
                rcv_f = mpi.Receive(rcv_f, rank + 1, 0)
                check_equal(rcv_f, msg_f, "bounce float64 len %d" % (l // 8))
            else:
                rcv_f = mpi.Receive(rcv_f, rank - 1, 0)
                mpi.Send(rcv_f, rank - 1, 0)
            done += 2
        # device-resident: heap -> heap
        cnt = l // 8
        d_msg = mpi.Alloc(cnt, np.float64).copy_from_host(message_f[:cnt])
        d_rcv = mpi.Alloc(cnt, np.float64)
        if even:
            mpi.Send(d_msg, rank + 1, 7)
            got = mpi.Receive(d_rcv, rank + 1, 7)
            if len(got) != cnt:
                raise AssertionError("device recv count %d != %d" % (len(got), cnt))
            check_equal(got.to_host(), message_f[:cnt], "bounce device float64 %d" % cnt)
        else:
            got = mpi.Receive(d_rcv, rank - 1, 7)
            mpi.Send(got, rank - 1, 7)
        d_msg.free()
        d_rcv.free()
        done += 1
    # receive into a too-small buffer: the value still arrives whole (gob resize analogue)
    if even:
        mpi.Send(message_f[:1000], rank + 1, 11)
    else:
        got = mpi.Receive(np.zeros(10, dtype=np.float64), rank - 1, 11)
        src = O.fill(np.float64, SEED + 100 + rank - 1, maxlen // 8 + 1)[:1000]
        check_equal(got, src, "resize-on-receive")
    # int64 and float32 typed slices
    for dt in (np.int64, np.float32):
        x = O.fill(dt, SEED + 5 + rank, 4097)
        if even:
            mpi.Send(x, rank + 1, 3)
        else:
            got = mpi.Receive(np.zeros(4097, dtype=dt), rank - 1, 3)
            check_equal(got, O.fill(dt, SEED + 5 + rank - 1, 4097), "typed p2p %s" % np.dtype(dt).name)
        done += 1
    mpi.Barrier()
    return {"checked": done}


def scenario_helloworld(a):
    """examples/helloworld/helloworld.go:54-81: every rank concurrently sends a string to every rank
    (itself included) and receives from every rank, tag 0."""
    rank, n = mpi.Rank(), mpi.Size()
    errs, got = [], {}

    def send(i):
        try:
            s = '"Hello node %d, I\'m node %d"' % (i, rank)
            if i == rank:
                s = '"I\'m just node %d talking to myself"' % rank
            mpi.Send(s, i, 0)
        except Exception as e:  # noqa: BLE001
            errs.append("send %d: %s" % (i, e))

    def recv(i):
        try:
            got[i] = mpi.Receive(str, i, 0)
        except Exception as e:  # noqa: BLE001
            errs.append("recv %d: %s" % (i, e))

    ths = [threading.Thread(target=send, args=(i,)) for i in range(n)] + [threading.Thread(target=recv, args=(i,)) for i in range(n)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    if errs:
        raise AssertionError("; ".join(errs))
    for i in range(n):
        want = '"Hello node %d, I\'m node %d"' % (rank, i) if i != rank else '"I\'m just node %d talking to myself"' % rank
        if got.get(i) != want:
            raise AssertionError("from %d got %r want %r" % (i, got.get(i), want))
    return {"checked": n}


def scenario_tags(a):
    """Concurrent sends with distinct tags to one peer; duplicate in-flight tag -> TagExists."""
    rank, n = mpi.Rank(), mpi.Size()
    peer = rank ^ 1
    ntags = 6
    payloads = {t: O.fill(np.int64, SEED + 31 * t + rank, 100 + 37 * t) for t in range(ntags)}
    errs, got = [], {}

    def send(t):
        try:
            mpi.Send(payloads[t], peer, t)
        except Exception as e:  # noqa: BLE001
            errs.append("send tag %d: %r" % (t, e))

    def recv(t):
        try:
            got[t] = mpi.Receive(np.zeros(1000, dtype=np.int64), peer, t)
        except Exception as e:  # noqa: BLE001
            errs.append("recv tag %d: %r" % (t, e))

    # receivers start in reverse tag order so matching is really by tag
    ths = [threading.Thread(target=send, args=(t,)) for t in range(ntags)] + [threading.Thread(target=recv, args=(t,)) for t in reversed(range(ntags))]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    if errs:
        raise AssertionError("; ".join(errs))
    for t in range(ntags):
        check_equal(got[t], O.fill(np.int64, SEED + 31 * t + peer, 100 + 37 * t), "tag %d" % t)
    mpi.Barrier()
    # duplicate tag: second Send on the same {dest, tag} while the first is still unmatched
    dup = {}
    if rank == 0:
        first = threading.Thread(target=lambda: mpi.Send(np.arange(4, dtype=np.int64), 1, 99))
        first.start()
        import time
        time.sleep(0.3)
        try:
            mpi.Send(np.arange(4, dtype=np.int64), 1, 99)
            dup["raised"] = False
        except mpi.TagExists as e:
            dup["raised"] = True
            dup["tag"] = e.Tag
        mpi.Send(np.arange(1, dtype=np.int64), 1, 100)  # tell rank 1 to go on
        first.join()
        if not dup.get("raised") or dup.get("tag") != 99:
            raise AssertionError("duplicate tag did not raise TagExists: %s" % dup)
    elif rank == 1:
        mpi.Receive(np.zeros(1, dtype=np.int64), 0, 100)
        got99 = mpi.Receive(np.zeros(4, dtype=np.int64), 0, 99)
        check_equal(got99, np.arange(4, dtype=np.int64), "message behind duplicate tag")
    mpi.Barrier()
    return {"checked": ntags + 1}


def scenario_fullsize(a):
    """Full-size points checked through size-independent properties plus the oracle on the same
    seeded inputs (the oracle finishes these sizes in a second or two)."""
    lib = L.load()
    rank, n = mpi.Rank(), mpi.Size()
    done = 0
    if a.what == "allgather":
        count = 1 << 20  # "1M indices per rank" (BASELINE.json configs[4]); also the decimal million
        for cnt in (count, 1000000):
            mine = O.fill(np.int64, SEED + rank, cnt)
            send = mpi.Alloc(cnt, np.int64).copy_from_host(mine)
            recv = mpi.Alloc(cnt * n, np.int64)
            for algo in ("auto", "ring"):
                lib.b200mpi_set_algo(L.COLL_ALLGATHER, ALGOS[algo])
                mpi.Allgather(send, recv)
                got = recv.to_host()
                for r in range(n):
                    check_equal(got[r * cnt:(r + 1) * cnt], O.fill(np.int64, SEED + r, cnt), "allgather i64 %d block %d algo %s" % (cnt, r, algo))
                done += 1
            lib.b200mpi_set_algo(L.COLL_ALLGATHER, 0)
            send.free()
            recv.free()
    else:
        count = 1 << 24
        ins = [O.fill(np.float32, SEED + r, count) for r in range(n)]
        send = mpi.Alloc(count, np.float32).copy_from_host(ins[rank])
        recv = mpi.Alloc(count, np.float32)
        for algo in ("twoshot", "ring", "oneshot", "nvls", "smem"):
            lib.b200mpi_set_algo(L.COLL_ALLREDUCE, ALGOS[algo])
            used = lib.b200mpi_get_algo(L.COLL_ALLREDUCE, count, L.F32)
            mpi.Allreduce(send, recv)
            want, order = expect_allreduce(ins, O.SUM, used, n, count, np.float32)
            check_equal(recv.to_host(), want, "allreduce f32 16Mi algo=%s" % algo, exact=order != O.ORDER_F64, ins=ins)
            # linearity: allreduce(2x) == 2 * allreduce(x) exactly (scaling by 2 is exact in binary fp)
            twice = mpi.Alloc(count, np.float32).copy_from_host(ins[rank] * np.float32(2))
            mpi.Allreduce(twice, twice)
            check_equal(twice.to_host(), want * np.float32(2), "linearity algo=%s" % algo, exact=order != O.ORDER_F64, ins=[x * 2 for x in ins])
            twice.free()
            done += 2
        lib.b200mpi_set_algo(L.COLL_ALLREDUCE, 0)
        # bcast 64 MiB from rank n-1, both P2P algorithms
        for algo in ("oneshot", "twoshot", "nvls"):
            lib.b200mpi_set_algo(L.COLL_BCAST, ALGOS[algo])
            buf = mpi.Alloc(count, np.float32).copy_from_host(ins[n - 1] if rank == n - 1 else np.zeros(count, dtype=np.float32))
            mpi.Bcast(buf, n - 1)
            check_equal(buf.to_host(), ins[n - 1], "bcast 64MiB algo=%s" % algo)
            buf.free()
            done += 1
        lib.b200mpi_set_algo(L.COLL_BCAST, 0)
        send.free()
        recv.free()
    return {"checked": done}


def scenario_stream(a):
    """Caller-provided stream (b200mpi_set_stream) + enqueue-only calls + the event stopwatch."""
    import ctypes
    import torch
    lib = L.load()
    rank, n = mpi.Rank(), mpi.Size()
    dev = lib.b200mpi_device()
    torch.cuda.set_device(dev)
    st = torch.cuda.Stream(device=dev)
    own = ctypes.c_void_p()
    assert lib.b200mpi_get_stream(ctypes.byref(own)) == 0 and own.value
    assert lib.b200mpi_set_stream(ctypes.c_void_p(st.cuda_stream)) == 0
    cur = ctypes.c_void_p()
    lib.b200mpi_get_stream(ctypes.byref(cur))
    assert cur.value == st.cuda_stream
    count = 1 << 18
    ins = [O.fill(np.float32, SEED + r, count) for r in range(n)]
    send = mpi.Alloc(count, np.float32).copy_from_host(ins[rank])
    recv = mpi.Alloc(count, np.float32)
    gath = mpi.Alloc(count * n, np.float32)
    l0 = lib.b200mpi_launch_count()
    assert lib.b200mpi_timer_start() == 0
    assert lib.b200mpi_allreduce_async(send.ptr, recv.ptr, count, L.F32, L.SUM) == 0, L.last_error()
    assert lib.b200mpi_allgather_async(send.ptr, gath.ptr, count, L.F32) == 0, L.last_error()
    assert lib.b200mpi_bcast_async(send.ptr, count, L.F32, 0) == 0, L.last_error()
    ms = ctypes.c_float()
    assert lib.b200mpi_timer_stop(ctypes.byref(ms)) == 0 and ms.value > 0
    st.synchronize()
    assert lib.b200mpi_stream_sync() == 0
    assert lib.b200mpi_launch_count() - l0 == (3 if n > 1 else 2)  # world of 1: bcast is a no-op
    used = lib.b200mpi_get_algo(L.COLL_ALLREDUCE, count, L.F32) if n > 1 else L.ALGO_TWOSHOT
    want, order = expect_allreduce(ins, O.SUM, used, n, count, np.float32)
    check_equal(recv.to_host(), want, "allreduce on caller stream", exact=order != O.ORDER_F64, ins=ins)
    check_equal(gath.to_host(), O.allgather(ins), "allgather on caller stream")
    check_equal(send.to_host(), ins[0], "bcast on caller stream")
    assert lib.b200mpi_set_stream(None) == 0
    lib.b200mpi_get_stream(ctypes.byref(cur))
    assert cur.value == own.value
    mpi.Barrier()
    return {"checked": 3}


def scenario_mismatch(a):
    """Ranks that disagree on count / dtype / collective get B200MPI_ERR_PEER, not a hang and not
    an out-of-bounds access; the library keeps working afterwards."""
    rank, n = mpi.Rank(), mpi.Size()
    lib = L.load()
    done = 0
    # different counts
    cnt = 1000 if rank == 0 else 999
    x = mpi.Alloc(1000, np.float32).copy_from_host(np.ones(1000, dtype=np.float32))
    y = mpi.Alloc(1000, np.float32).copy_from_host(np.full(1000, -5, dtype=np.float32))
    rc = lib.b200mpi_allreduce(x.ptr, y.ptr, cnt, L.F32, L.SUM, L.DEVICE)
    assert rc == L.ERR_PEER, (rc, L.last_error())
    check_equal(y.to_host(), np.full(1000, -5, dtype=np.float32), "recv untouched after a mismatched call")
    done += 1
    # different dtypes (same byte size)
    rc = lib.b200mpi_allreduce(x.ptr, y.ptr, 500, L.F64 if rank == 0 else L.I64, L.SUM, L.DEVICE)
    assert rc == L.ERR_PEER, (rc, L.last_error())
    done += 1
    # different collectives
    if rank == 0:
        rc = lib.b200mpi_bcast(x.ptr, 1000, L.F32, 0, L.DEVICE)
    else:
        rc = lib.b200mpi_allgather(x.ptr, y.ptr, 1000 // n, L.F32, L.DEVICE)
    assert rc == L.ERR_PEER, (rc, L.last_error())
    done += 1
    # and the world still works
    mpi.Allreduce(x, y)
    check_equal(y.to_host(), np.full(1000, n, dtype=np.float32), "allreduce after mismatches")
    mpi.Barrier()
    return {"checked": done + 1}


def scenario_smoke(a):
    rank, n = mpi.Rank(), mpi.Size()
    x = O.fill(np.float32, SEED + rank, 1 << 12)
    out = np.zeros_like(x)
    mpi.Allreduce(x, out)
    want = O.allreduce([O.fill(np.float32, SEED + r, 1 << 12) for r in range(n)], order=O.ORDER_TREE if n in (2, 4, 8) else O.ORDER_RANK)
    check_equal(out, want, "smoke allreduce")
    return {"checked": 1, "device": L.load().b200mpi_device(), "launches": int(L.load().b200mpi_launch_count())}


def scenario_control_only(a):
    """CPU plumbing: bootstrap over TCP loopback, rank/size, barrier; data calls must refuse."""
    rank, n = mpi.Rank(), mpi.Size()
    lib = L.load()
    rc = lib.b200mpi_barrier()
    if rc:
        raise AssertionError("control-plane barrier failed: %s" % L.last_error())
    x = np.zeros(4, dtype=np.float32)
    try:
        mpi.Allreduce(x, x)
        raise AssertionError("data call succeeded without a device")
    except mpi.MpiError as e:
        if e.code != L.ERR_NO_DEVICE:
            raise
    return {"checked": 1, "rank": rank, "size": n}


# ------------------------------------------------------------------------------------------------
# Reducing collectives at ragged ownership shapes, every op, checked twice: against tests/_exact.py
# (order-independent: exact sum + error bound, wrap-around sum, numpy max/min) and bit for bit
# against the oracle in the order of the kernel that ran.  Every case reports what ran, both
# verdicts and a SHA-256 of the rank's result; the pytest side compares the digests across ranks.
# Every rank makes the same calls with the same settings (the grid is part of the call signature).
SHAPE_ALGOS = (("oneshot", 1, None), ("twoshot_u0", 2, 0), ("twoshot_u1", 2, 1), ("smem", 5, None), ("ring", 3, None))
OPNAMES = ("sum", "max", "min")


def _ok(rc):
    if rc:
        raise RuntimeError(L.last_error())


def _multicast():
    info = (L.ctypes.c_size_t(), L.ctypes.c_size_t(), L.ctypes.c_int())
    L.load().b200mpi_heap_info(L.ctypes.byref(info[0]), L.ctypes.byref(info[1]), L.ctypes.byref(info[2]))
    return bool(info[2].value)


_INPUTS = {}


def _inputs(gen, dt, n, count, seed):
    key = (gen, np.dtype(dt).name, n, count, seed)
    if key not in _INPUTS:
        _INPUTS.clear()
        _INPUTS[key] = X.generate(gen, dt, n, count, seed)
    return _INPUTS[key]


def _row(label, algo, opn, dn, got, xs, want, digest=True):
    """One reported case: the algorithm that ran, the order-independent verdict, the oracle verdict
    (None when the order is switch-defined), the result digest."""
    trace(label)
    return {"case": label, "algo": L.ALGO_NAMES.get(algo, str(algo)), "op": opn, "dtype": dn,
            "exact": X.check(got, xs, X.OPS[opn]) if xs is not None else None,
            "oracle": X.bit_diff(got, want) if want is not None else None,
            "digest": X.digest(got) if digest else None}


def _gen_for(dn, opn, k):
    if dn == "i64":
        return "i64"
    if opn == "sum":
        return ("signed", "cancel", "uniform01")[k % 3]
    return ("signed", "cancel")[k % 2]  # max/min over non-negative data would prove little


def _allreduce_case(lib, label, dn, opn, gen, count, inplace, kind, seed):
    rank, n = mpi.Rank(), mpi.Size()
    dt = DTYPES[dn]
    op = X.OPS[opn]
    xs = _inputs(gen, dt, n, count, seed)
    used = lib.b200mpi_get_algo(L.COLL_ALLREDUCE, count, O.NP2DT[np.dtype(dt)])
    send = make_buffer(kind, xs[rank])
    recv = send if inplace else make_buffer(kind, np.zeros(count, dtype=dt))
    mpi.Allreduce(send, recv, op)
    got = np.array(read_buffer(recv), copy=True)
    want, _ = expect_allreduce(xs, op, used, n, count, dt)
    if not inplace:
        check_equal(read_buffer(send), xs[rank], label + ": send buffer untouched")
        free_buffer(recv)
    free_buffer(send)
    return _row("%s %s %s %s n=%d count=%d %s%s" % (label, dn, opn, gen, n, count, kind, " inplace" if inplace else ""),
                used, opn, dn, got, xs, want)


def scenario_shapes(a):
    """Allreduce with every forced P2P algorithm, op and dtype at ragged shapes (own_block_bytes =
    4 KiB, grids of 1, 3 and all CTAs), at the shuffle / plain one-shot switch, and once at the
    default 1 MiB block with every rank's share above 1 MiB."""
    lib = L.load()
    n = mpi.Size()
    rows = []
    _ok(lib.b200mpi_set_param(b"own_block_bytes", X.SMALL_BLOCK))
    for ai, (aname, aid, unroll) in enumerate(SHAPE_ALGOS):
        _ok(lib.b200mpi_set_algo(L.COLL_ALLREDUCE, aid))
        if unroll is not None:
            _ok(lib.b200mpi_set_param(b"twoshot_unroll", unroll))
        if aname == "smem" and n not in (2, 4, 8):  # the TMA kernel needs 2, 4 or 8 ranks
            used = lib.b200mpi_get_algo(L.COLL_ALLREDUCE, X.ragged_counts(n, np.float32)[0], L.F32)
            if used != L.ALGO_TWOSHOT:
                raise AssertionError("forced smem at n=%d reports %s, not two-shot" % (n, L.ALGO_NAMES.get(used)))
            continue
        for di, dn in enumerate(("f32", "f64", "i64")):
            counts = X.ragged_counts(n, DTYPES[dn])
            for oi, opn in enumerate(OPNAMES):
                gen = _gen_for(dn, opn, ai + di + oi)
                for inplace in (False, True):
                    combo = (di * 3 + oi + 3 * inplace) % 6  # every (count, grid) pair 3 times per algorithm
                    mb = (0, 1, 3)[combo % 3]
                    _ok(lib.b200mpi_set_max_blocks(mb))
                    rows.append(_allreduce_case(lib, "shapes %s blocks=%d" % (aname, mb), dn, opn, gen, counts[combo // 3], inplace, "heap",
                                                SEED + 17 * ai + di))
        _ok(lib.b200mpi_set_max_blocks(0))
    # host slices: one case per dtype
    _ok(lib.b200mpi_set_algo(L.COLL_ALLREDUCE, ALGOS["twoshot"]))
    for dn in ("f32", "f64", "i64"):
        rows.append(_allreduce_case(lib, "shapes host twoshot", dn, "sum", _gen_for(dn, "sum", 0), X.ragged_counts(n, DTYPES[dn])[1], False, "host", SEED + 5))
    _ok(lib.b200mpi_set_param(b"twoshot_unroll", 1))
    # 4095 / 4096 / 4097 vectors: shuffle one-shot up to 4096, plain one-shot above
    if n in (4, 8):
        _ok(lib.b200mpi_set_algo(L.COLL_ALLREDUCE, ALGOS["oneshot"]))
        for di, dn in enumerate(("f32", "f64", "i64")):
            for oi, opn in enumerate(OPNAMES):
                for ci, count in enumerate(X.switch_counts(DTYPES[dn])):
                    rows.append(_allreduce_case(lib, "switch oneshot", dn, opn, _gen_for(dn, opn, ci + oi), count, (ci + oi) % 2 == 1, "heap", SEED + 9))
    # the default 1 MiB block: every rank's share above 1 MiB, odd count
    _ok(lib.b200mpi_set_param(b"own_block_bytes", 1 << 20))
    for dn, opn in (("f32", "sum"), ("i64", "max")):
        for ai, (aname, aid, unroll) in enumerate(SHAPE_ALGOS):
            if aname == "smem" and n not in (2, 4, 8):
                continue
            _ok(lib.b200mpi_set_algo(L.COLL_ALLREDUCE, aid))
            if unroll is not None:
                _ok(lib.b200mpi_set_param(b"twoshot_unroll", unroll))
            rows.append(_allreduce_case(lib, "big %s" % aname, dn, opn, _gen_for(dn, opn, 0), X.big_count(n, DTYPES[dn]), ai % 2 == 1, "heap", SEED + 3))
    _ok(lib.b200mpi_set_param(b"twoshot_unroll", 1))
    _ok(lib.b200mpi_set_algo(L.COLL_ALLREDUCE, 0))
    mpi.Barrier()
    return {"rows": rows}


def scenario_reduce_ops(a):
    """Reduce (every op, roots 0, 1, n-1; in place on the root; NULL recv on non-roots through the
    C ABI), ReduceScatter (every op, ragged blocks, grids of 1 and all CTAs) and, up to 4 ranks,
    Allgather in place (send = the caller's block of recv), push and ring, heap and host."""
    lib = L.load()
    rank, n = mpi.Rank(), mpi.Size()
    switch = _multicast()  # Reduce / ReduceScatter sums then go through the switch: no fixed order
    rows = []
    _ok(lib.b200mpi_set_param(b"own_block_bytes", X.SMALL_BLOCK))
    for di, dn in enumerate(("f32", "f64", "i64")):
        dt = DTYPES[dn]
        code = O.NP2DT[np.dtype(dt)]
        count = X.ragged_counts(n, dt)[0]
        for oi, opn in enumerate(OPNAMES):
            op = X.OPS[opn]
            gen = _gen_for(dn, opn, di + oi)
            xs = _inputs(gen, dt, n, count, SEED + 40 + di)
            for ri, root in enumerate(sorted({0, 1, n - 1})):
                mode = ("out", "null", "inplace")[(di + oi + ri) % 3]
                mb = (0, 1, 3)[(di + 2 * oi + ri) % 3]
                _ok(lib.b200mpi_set_max_blocks(mb))
                send = mpi.Alloc(count, dt).copy_from_host(xs[rank])
                sentinel = np.full(count, -7, dtype=dt)
                if rank == root:
                    recv = send if mode == "inplace" else mpi.Alloc(count, dt).copy_from_host(sentinel)
                else:
                    recv = None if mode == "null" else mpi.Alloc(count, dt).copy_from_host(sentinel)
                _ok(lib.b200mpi_reduce(send.ptr, recv.ptr if recv is not None else None, count, code, op, root, L.DEVICE))
                label = "reduce %s %s %s root=%d %s blocks=%d n=%d count=%d" % (dn, opn, gen, root, mode, mb, n, count)
                if rank == root:
                    got = recv.to_host()
                    exact_order = not (switch and op == X.SUM and dn != "i64" and n >= 4)
                    want = O.allreduce(xs, op=op, order=O.ORDER_RANK) if exact_order else None
                    rows.append(_row(label, L.ALGO_TWOSHOT, opn, dn, got, xs, want, digest=False))
                else:  # the same case on every rank; here the check is that nothing was written
                    check_equal(send.to_host(), xs[rank], label + ": non-root send untouched")
                    if recv is not None:
                        check_equal(recv.to_host(), sentinel, label + ": non-root recv untouched")
                    rows.append({"case": label, "algo": L.ALGO_NAMES[L.ALGO_TWOSHOT], "op": opn, "dtype": dn, "exact": None, "oracle": None, "digest": None})
                if recv is not None and recv is not send:
                    recv.free()
                send.free()
        # ReduceScatter: rank j receives block j (of `count`, ragged) reduced over the ranks
        for ci, count in enumerate(X.ragged_counts(n, dt)):
            for oi, opn in enumerate(OPNAMES):
                op = X.OPS[opn]
                gen = _gen_for(dn, opn, ci + oi)
                xs = _inputs(gen, dt, n, count * n, SEED + 50 + di)
                mb = (0, 1)[(ci + oi) % 2]
                inplace = (di + ci + oi) % 2 == 1
                _ok(lib.b200mpi_set_max_blocks(mb))
                send = mpi.Alloc(count * n, dt).copy_from_host(xs[rank])
                recv = send[rank * count:(rank + 1) * count] if inplace else mpi.Alloc(count, dt)
                mpi.ReduceScatter(send, recv, op)
                got = recv.to_host()
                blocks = [x[rank * count:(rank + 1) * count] for x in xs]
                exact_order = not (switch and op == X.SUM and dn != "i64")
                want = O.reduce_scatter(xs, rank, op=op, order=O.ORDER_RANK) if exact_order else None
                label = "reduce_scatter %s %s %s blocks=%d%s n=%d count=%d" % (dn, opn, gen, mb, " inplace" if inplace else "", n, count)
                rows.append(_row(label, L.ALGO_TWOSHOT, opn, dn, got, blocks, want, digest=False))
                if not inplace:
                    check_equal(send.to_host(), xs[rank], label + ": send untouched")
                    recv.free()
                send.free()
    _ok(lib.b200mpi_set_max_blocks(0))
    # Allgather in place: the caller's block of recv is the send buffer
    if n <= 4:
        for dn in ("f32", "i64"):
            dt = DTYPES[dn]
            count = X.ragged_counts(n, dt)[0]
            xs = _inputs(_gen_for(dn, "sum", 0), dt, n, count, SEED + 60)
            full = np.concatenate(xs)
            for ai, algo in enumerate(("oneshot", "ring")):
                _ok(lib.b200mpi_set_algo(L.COLL_ALLGATHER, ALGOS[algo]))
                for ki, kind in enumerate(("heap", "host")):
                    mb = (0, 1)[(ai + ki) % 2]
                    _ok(lib.b200mpi_set_max_blocks(mb))
                    init = np.full(count * n, -1, dtype=dt)
                    init[rank * count:(rank + 1) * count] = xs[rank]
                    recv = make_buffer(kind, init)
                    mpi.Allgather(recv[rank * count:(rank + 1) * count], recv)
                    got = np.array(read_buffer(recv), copy=True)
                    label = "allgather inplace %s %s %s blocks=%d n=%d count=%d" % (algo, kind, dn, mb, n, count)
                    row = _row(label, ALGOS[algo], "sum", dn, got, None, full)
                    row["op"] = "copy"
                    rows.append(row)
                    free_buffer(recv)
        _ok(lib.b200mpi_set_max_blocks(0))
        _ok(lib.b200mpi_set_algo(L.COLL_ALLGATHER, 0))
    _ok(lib.b200mpi_set_param(b"own_block_bytes", 1 << 20))
    mpi.Barrier()
    return {"rows": rows, "multicast": switch}


EDGE_F32 = np.array([np.nan, 0.0, -0.0, np.inf, -np.inf, np.finfo(np.float32).max, -np.finfo(np.float32).max,
                     2.0 ** -149, -2.0 ** -149, 2.0 ** -130, 1.0, -1.0], dtype=np.float32)
EDGE_F64 = np.array([np.nan, 0.0, -0.0, np.inf, -np.inf, np.finfo(np.float64).max, -np.finfo(np.float64).max,
                     2.0 ** -1074, -2.0 ** -1074, 2.0 ** -1050, 1.0, -1.0], dtype=np.float64)
EDGE_I64 = np.array([-2 ** 63, 2 ** 63 - 1, -2 ** 63 + 1, 2 ** 63 - 2, -1, 0, 1, 42], dtype=np.int64)


def edge_inputs(dt, n, count, seed):
    """Per element, each rank picks a value of the edge set; for floats, the first two elements of
    ring chunk 1 are set so that the order shows: {x0 = 1, x1 = NaN, rest 1} and {x0 = +0, x1 = -0,
    rest +0}.  max/min keep the left operand on NaN and ties, so rank order yields 1 and +0 there
    while the ring, which starts chunk 1 at rank 1, yields NaN and -0."""
    edge = {np.dtype(np.float32): EDGE_F32, np.dtype(np.float64): EDGE_F64, np.dtype(np.int64): EDGE_I64}[np.dtype(dt)]
    xs = [edge[(X.splitmix64(seed + r, count) % np.uint64(edge.size)).astype(np.int64)] for r in range(n)]
    planted = []
    if np.dtype(dt).kind == "f":
        e = X.epv(dt)
        per = -(-(count // e) // n)
        lo = per * e  # first element of ring chunk 1
        for k, (first, second, rest) in enumerate(((1.0, np.nan, 1.0), (0.0, -0.0, 0.0))):
            for r in range(n):
                xs[r][lo + k] = first if r == 0 else second if r == 1 else rest
            planted.append(lo + k)
    return xs, planted


def scenario_edge_ops(a):
    """MAX and MIN over NaN, +-0, +-inf, +-max, subnormals and the int64 extremes, every forced P2P
    algorithm, bit for bit against the oracle in that algorithm's order."""
    lib = L.load()
    rank, n = mpi.Rank(), mpi.Size()
    rows, pinned = [], 0
    for ai, (aname, aid, unroll) in enumerate(SHAPE_ALGOS):
        if aname == "smem" and n not in (2, 4, 8):
            continue
        _ok(lib.b200mpi_set_algo(L.COLL_ALLREDUCE, aid))
        if unroll is not None:
            _ok(lib.b200mpi_set_param(b"twoshot_unroll", unroll))
        for dn in ("f32", "f64", "i64"):
            dt = DTYPES[dn]
            count = 64 * n * X.epv(dt) + X.epv(dt) - 1  # ring chunks of 64 vectors, a scalar tail
            xs, planted = edge_inputs(dt, n, count, SEED + 70 + ai)
            for opn in ("max", "min"):
                op = X.OPS[opn]
                used = lib.b200mpi_get_algo(L.COLL_ALLREDUCE, count, O.NP2DT[np.dtype(dt)])
                send = mpi.Alloc(count, dt).copy_from_host(xs[rank])
                recv = mpi.Alloc(count, dt)
                mpi.Allreduce(send, recv, op)
                got = recv.to_host()
                send.free()
                recv.free()
                want, order = expect_allreduce(xs, op, used, n, count, dt)
                rows.append(_row("edge %s %s %s n=%d count=%d" % (aname, dn, opn, n, count), used, opn, dn, got, None, want))
                if used == L.ALGO_RING and planted:
                    rank_order = O.allreduce(xs, op=op, order=O.ORDER_RANK)
                    if not X.bit_diff(got[planted], rank_order[planted]):
                        raise AssertionError("ring %s %s: the planted NaN / -0 elements do not show the ring order" % (dn, opn))
                    pinned += 1
    _ok(lib.b200mpi_set_param(b"twoshot_unroll", 1))
    _ok(lib.b200mpi_set_algo(L.COLL_ALLREDUCE, 0))
    mpi.Barrier()
    return {"rows": rows, "ring_order_pinned": pinned}


def scenario_oneshot_budget(a):
    """One CTA per rank: the largest count whose one-shot plan fits in the mid-barrier budget runs
    one-shot, one vector more runs two-shot; both out of place, then the limit once in place."""
    import time
    lib = L.load()
    rank, n = mpi.Rank(), mpi.Size()
    _ok(lib.b200mpi_set_max_blocks(1))
    _ok(lib.b200mpi_set_algo(L.COLL_ALLREDUCE, ALGOS["oneshot"]))
    lim = X.oneshot_limit(np.float32, n, 1)
    rows, times = [], {}
    for count, inplace, expect in ((lim, False, L.ALGO_ONESHOT), (lim + 4, False, L.ALGO_TWOSHOT), (lim, True, L.ALGO_ONESHOT)):
        used = lib.b200mpi_get_algo(L.COLL_ALLREDUCE, count, L.F32)
        if used != expect:
            raise AssertionError("count %d: get_algo reports %s, want %s" % (count, L.ALGO_NAMES.get(used), L.ALGO_NAMES[expect]))
        mpi.Barrier()
        t0 = time.time()
        rows.append(_allreduce_case(lib, "budget", "f32", "sum", "signed", count, inplace, "heap", SEED + 80))
        times["%d%s" % (count, " inplace" if inplace else "")] = time.time() - t0
    _ok(lib.b200mpi_set_max_blocks(0))
    _ok(lib.b200mpi_set_algo(L.COLL_ALLREDUCE, 0))
    mpi.Barrier()
    return {"rows": rows, "limit": lim, "seconds": times}


def scenario_switch_bound(a):
    """NVLS and hybrid Allreduce and NVLS ReduceScatter (f32, f64 sums) held to the any-order error
    bound of tests/_exact.py.  Needs a multicast mapping (one GPU per rank)."""
    lib = L.load()
    rank, n = mpi.Rank(), mpi.Size()
    if not _multicast():
        raise AssertionError("no multicast mapping: the switch paths cannot run in this world")
    _ok(lib.b200mpi_set_param(b"hybrid_p2p_permille", 250))
    _ok(lib.b200mpi_set_param(b"hybrid_min_bytes", 0))
    rows = []
    for dn in ("f32", "f64"):
        dt = DTYPES[dn]
        for ci, count in enumerate((X.ragged_counts(n, dt)[0], X.big_count(n, dt))):
            for algo in ("nvls", "hybrid"):
                _ok(lib.b200mpi_set_algo(L.COLL_ALLREDUCE, ALGOS[algo]))
                for gi, gen in enumerate(("signed", "cancel", "uniform01")):
                    xs = _inputs(gen, dt, n, count, SEED + 90 + ci)
                    used = lib.b200mpi_get_algo(L.COLL_ALLREDUCE, count, O.NP2DT[np.dtype(dt)])
                    send = mpi.Alloc(count, dt).copy_from_host(xs[rank])
                    recv = send if gi == 1 else mpi.Alloc(count, dt)  # the cancelling data in place
                    mpi.Allreduce(send, recv, mpi.SUM)
                    got = recv.to_host()
                    if recv is not send:
                        recv.free()
                    send.free()
                    rows.append(_row("switch allreduce %s %s %s n=%d count=%d" % (algo, dn, gen, n, count), used, "sum", dn, got, xs, None))
            _ok(lib.b200mpi_set_algo(L.COLL_REDUCE_SCATTER, ALGOS["nvls"]))
            rc = count - count % X.epv(dt)  # whole vectors per block: the switch form
            for gen in ("signed", "cancel"):
                xs = _inputs(gen, dt, n, rc * n, SEED + 95 + ci)
                send = mpi.Alloc(rc * n, dt).copy_from_host(xs[rank])
                recv = mpi.Alloc(rc, dt)
                mpi.ReduceScatter(send, recv, mpi.SUM)
                got = recv.to_host()
                send.free()
                recv.free()
                rows.append(_row("switch reduce_scatter nvls %s %s n=%d count=%d" % (dn, gen, n, rc), L.ALGO_NVLS, "sum", dn, got,
                                 [x[rank * rc:(rank + 1) * rc] for x in xs], None, digest=False))
    _ok(lib.b200mpi_set_algo(L.COLL_ALLREDUCE, 0))
    _ok(lib.b200mpi_set_algo(L.COLL_REDUCE_SCATTER, 0))
    mpi.Barrier()
    return {"rows": rows}


SCENARIOS = {k[len("scenario_"):]: v for k, v in list(globals().items()) if k.startswith("scenario_")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("scenario")
    ap.add_argument("--out", required=True)
    ap.add_argument("--sizes", default="0,1,3,4,5,255,256,257,4096,65537")
    ap.add_argument("--dtypes", default="f32,f64,i64")
    ap.add_argument("--algos", default="default", help="default: every P2P algorithm, plus the switch forms where a multicast mapping exists")
    ap.add_argument("--kinds", default="heap,host")
    ap.add_argument("--gpu", type=int, default=None)
    ap.add_argument("--what", default="allgather")
    ap.add_argument("--control-only", action="store_true")
    args, rest = ap.parse_known_args()
    sys.argv = [sys.argv[0]] + rest  # leave the -mpi-* flags for the library's flag parser
    result = {"ok": False}
    try:
        gpu = -2 if args.control_only else args.gpu
        mpi.api._reset_for_tests(mpi.Cuda(Gpu=gpu))
        mpi.Init()
        result.update(SCENARIOS[args.scenario](args))
        result["rank_reported"] = mpi.Rank()
        result["size_reported"] = mpi.Size()
        mpi.Finalize()
        result["ok"] = True
    except Exception as e:  # noqa: BLE001
        result["error"] = "%s: %s" % (type(e).__name__, e)
        traceback.print_exc()
    with open(args.out, "w") as f:
        json.dump(result, f)
    sys.exit(0 if result["ok"] else 1)


if __name__ == "__main__":
    main()
