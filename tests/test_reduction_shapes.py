"""The reducing collectives at ragged multi-block shapes, every op, against an order-independent
reference (tests/_exact.py) and the oracle's per-kernel order.

CPU part: the reference's error bound accepts every order the kernels use and rejects arithmetic
mutants; the shape selector's counts really reach the ragged ownership cases.  GPU part: worlds of
3, 4 and 8 ranks (sharing GPU 0 on a 1-GPU box) run the scenarios of tests/_worker.py; every case
must pass both checks, every rank must hold the same bits, and the (algorithm, op, dtype) matrix
that actually ran must be complete."""
import numpy as np
import pytest

import _exact as X
from oracle import oracle as O

ORDERS = {"rank": O.ORDER_RANK, "tree": O.ORDER_TREE, "ring": O.ORDER_RING, "f64": O.ORDER_F64}
FLOAT_GENS = ("uniform01", "signed", "cancel")


# ---- CPU: the reference ------------------------------------------------------------------------
@pytest.mark.parametrize("dn", ["f32", "f64"])
@pytest.mark.parametrize("n", range(2, 9))
def test_bound_accepts_every_kernel_order(n, dn):
    dt = X.DTYPES[dn]
    count = 4 * 97 + 3  # several ring chunks and a scalar tail
    for gen in FLOAT_GENS:
        xs = X.generate(gen, dt, n, count, 0xB2000000 + n)
        for oname, order in ORDERS.items():
            got = O.allreduce(xs, op=O.SUM, order=order)
            assert X.check(got, xs, X.SUM) is None, (gen, oname, X.check(got, xs, X.SUM))


@pytest.mark.parametrize("n", [2, 3, 8])
def test_exact_sum_matches_fsum(n):
    import math
    for dn in ("f32", "f64"):
        for gen in FLOAT_GENS:
            xs = X.generate(gen, X.DTYPES[dn], n, 300, 7)
            s, c = X.exact_sum(xs)
            want = np.array([math.fsum(float(x[i]) for x in xs) for i in range(300)])
            assert np.array_equal(s + c, want), (dn, gen)


def test_integer_and_minmax_references():
    xs = X.generate("i64", np.int64, 5, 999, 3)
    want = np.array([sum(int(x[i]) for x in xs) for i in range(999)], dtype=object)
    want = np.array([((v + 2 ** 63) % 2 ** 64) - 2 ** 63 for v in want], dtype=np.int64)
    assert np.array_equal(X.reference(xs, X.SUM), want)
    wraps = sum(1 for i in range(999) if not -2 ** 63 <= sum(int(x[i]) for x in xs) < 2 ** 63)
    assert wraps > 100  # the generator really makes sums wrap
    for op, oop in ((X.MAX, O.MAX), (X.MIN, O.MIN)):
        for gen, dt in (("signed", np.float32), ("cancel", np.float64), ("i64", np.int64)):
            xs = X.generate(gen, dt, 6, 501, 11)
            assert X.check(O.allreduce(xs, op=oop), xs, op) is None


def _worst(xs, bound_of):
    """(rank, element) whose term is largest relative to the bound there."""
    ratio = np.stack([np.abs(np.asarray(x, dtype=np.float64)) for x in xs]) / bound_of
    r, e = np.unravel_index(int(np.argmax(ratio)), ratio.shape)
    return int(r), int(e), float(ratio[r, e])


@pytest.mark.parametrize("n", [2, 3, 4, 8])
def test_bound_rejects_mutants(n):
    count = 4 * 64 + 3
    for dn in ("f32", "f64"):
        dt = X.DTYPES[dn]
        for gen in FLOAT_GENS:
            xs = X.generate(gen, dt, n, count, 99 + n)
            good = O.allreduce(xs, op=O.SUM)
            s, c = X.exact_sum(xs)
            bound = X.sum_bound(xs, s, c)
            # one rank's term dropped at one element
            r, e, ratio = _worst(xs, bound)
            assert ratio > 4
            bad = good.copy()
            bad[e] = O.allreduce([x[e:e + 1] for k, x in enumerate(xs) if k != r], op=O.SUM)[0]
            assert X.check(bad, xs, X.SUM) is not None, ("dropped term", dn, gen)
            # the last (tail) element read from index e-1 (cancelling data leaves the bound too wide
            # for this one: there rank order itself loses the small terms)
            if gen == "cancel":
                continue
            bad = good.copy()
            bad[-1] = good[-2]
            assert X.check(bad, xs, X.SUM) is not None, ("tail from e-1", dn, gen)
        # f64 summed through f32
        xs = X.generate("signed", np.float64, n, count, 5)
        bad = O.allreduce([x.astype(np.float32) for x in xs], op=O.SUM).astype(np.float64)
        assert X.check(bad, xs, X.SUM) is not None
    # i64 saturating instead of wrapping
    xs = X.generate("i64", np.int64, n, count, 8)
    sat = np.array([max(-2 ** 63, min(2 ** 63 - 1, sum(int(x[i]) for x in xs))) for i in range(count)], dtype=np.int64)
    assert X.check(sat, xs, X.SUM) is not None
    # MAX computed as MIN
    for gen, dt in (("signed", np.float32), ("i64", np.int64)):
        xs = X.generate(gen, dt, n, count, 12)
        assert X.check(O.allreduce(xs, op=O.MIN), xs, X.MAX) is not None
        assert X.check(O.allreduce(xs, op=O.MAX), xs, X.MAX) is None


# ---- CPU: the shapes really are ragged -----------------------------------------------------------
@pytest.mark.parametrize("n", [3, 4, 8])
@pytest.mark.parametrize("dn", ["f32", "f64", "i64"])
def test_ragged_counts_have_the_promised_properties(n, dn):
    dt = X.DTYPES[dn]
    owners = set()
    for count in X.ragged_counts(n, dt):
        for min_shift in (0, 8):  # LDG / ring / NVLS, and the TMA kernel (a block is whole 4 KiB tiles)
            o = X.ownership(count, dt, n, X.SMALL_BLOCK, min_shift)
            assert o["shift"] == 8, o  # 4 KiB blocks
            assert o["nblk"] > 2 * n, o  # ownership wraps around the ranks more than twice
            assert o["last_partial"] and o["last_owner"] != 0, o
            assert 0 < o["tail"] < X.epv(dt), o  # the last rank reduces a scalar tail
            assert min(o["owned"]) > 2 * X.SMEM_STAGES, o  # one CTA turns the stage ring over twice
            assert sum(o["owned"]) == o["nblk"]
        owners.add(X.ownership(count, dt, n, X.SMALL_BLOCK)["last_owner"])
    assert owners == {1, n - 1}
    big = X.big_count(n, dt)
    o = X.ownership(big, dt, n, 1 << 20)
    assert o["shift"] == 16 and big % 2 == 1 and o["tail"] > 0
    assert big * np.dtype(dt).itemsize / n > (1 << 20)  # every rank's share is more than 1 MiB
    assert o["nblk"] > 2 * n and o["last_partial"] and o["last_owner"] != 0, o
    sw = X.switch_counts(dt)
    assert [-(-c // X.epv(dt)) for c in sw] == [4095, 4096, 4097]


def test_oneshot_limit_is_the_boundary():
    for n, dt in ((2, np.float32), (2, np.float64), (4, np.int64)):
        lim = X.oneshot_limit(dt, n, 1)
        assert X.oneshot_rounds(lim, dt, n, 1) <= X.MAX_MIDS < X.oneshot_rounds(lim + X.epv(dt), dt, n, 1)


# ---- GPU ---------------------------------------------------------------------------------------
ENV = {"B200MPI_WATCHDOG_S": "90"}


def _world(n, scenario, env=None, timeout=900):
    from _launch import assert_world_ok, run_world
    e = dict(ENV)
    e.update(env or {})
    res = run_world(n, scenario, timeout=timeout, env=e)
    assert_world_ok(res)
    return res


def _assert_rows(res):
    """Every case passed both checks on every rank, and every rank holds the same bits."""
    n = len(res)
    rows = [r["rows"] for r in res]
    assert all(len(x) == len(rows[0]) for x in rows)
    bad = []
    for i, case in enumerate(rows[0]):
        for r in range(n):
            row = rows[r][i]
            assert row["case"] == case["case"]
            if row["exact"] or row["oracle"]:
                bad.append("rank %d %s [%s]: exact: %s; oracle: %s" % (r, row["case"], row["algo"], row["exact"], row["oracle"]))
        if case["digest"] is not None:
            digests = {rows[r][i]["digest"] for r in range(n)}
            if len(digests) != 1:
                bad.append("%s: ranks hold different results" % case["case"])
    assert not bad, "\n".join(bad[:40])
    return rows[0]


def _coverage(rows):
    return {(r["algo"], r["op"], r["dtype"]) for r in rows}


def _intended(n):
    algos = ["oneshot", "twoshot", "ring"] + (["twoshot_smem"] if n in (2, 4, 8) else [])
    return {(a, op, dn) for a in algos for op in ("sum", "max", "min") for dn in ("f32", "f64", "i64")}


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 4, 8])
def test_shapes(n):
    res = _world(n, "shapes", env={"B200MPI_HEAP_BYTES": str(512 << 20)})
    rows = _assert_rows(res)
    missing = _intended(n) - _coverage(rows)
    assert not missing, "never ran: %s" % sorted(missing)
    print("\nworld of %d: %d cases, coverage %s" % (n, len(rows), sorted(_coverage(rows))))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 3, 4, 8])
def test_reduce_ops(n):
    rows = _assert_rows(_world(n, "reduce_ops"))
    ops = {r["op"] for r in rows if r["case"].startswith("reduce ")}
    assert ops == {"sum", "max", "min"}
    assert {r["op"] for r in rows if r["case"].startswith("reduce_scatter")} == {"sum", "max", "min"}
    if n <= 4:
        assert {r["algo"] for r in rows if r["case"].startswith("allgather")} == {"oneshot", "ring"}


@pytest.mark.gpu
@pytest.mark.parametrize("n", [3, 4, 8])
def test_edge_ops(n):
    res = _world(n, "edge_ops")
    rows = _assert_rows(res)
    assert _coverage(rows) >= {(a, op, dn) for a, _, dn in _intended(n) for op in ("max", "min")}
    assert res[0]["ring_order_pinned"] == 4  # f32 and f64, max and min


@pytest.mark.gpu
def test_oneshot_budget():
    res = _world(2, "oneshot_budget")
    rows = _assert_rows(res)
    assert [r["algo"] for r in rows] == ["oneshot", "twoshot", "oneshot"]
    print("\none-shot limit %d elements (f32, 1 CTA): seconds %s" % (res[0]["limit"], res[0]["seconds"]))


@pytest.mark.gpu
def test_switch_paths_meet_the_exact_bound():
    """NVLS / hybrid Allreduce and NVLS ReduceScatter held to the any-order error bound."""
    from test_gpu_worlds import need_gpus
    have = need_gpus(2, "the switch (NVLS) reductions")
    n = 8 if have >= 8 else 4 if have >= 4 else 2
    rows = _assert_rows(_world(n, "switch_bound", env={"B200MPI_HEAP_BYTES": str(1 << 30)}))
    assert {r["algo"] for r in rows if "allreduce nvls" in r["case"]} == {"nvls"}
    assert {r["algo"] for r in rows if "allreduce hybrid" in r["case"]} == {"hybrid"}
