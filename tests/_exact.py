"""Order-independent references for the reducing collectives, with no call into oracle/.

The oracle restates each kernel's order of operations, so a misreading shared by the oracle and a
kernel passes a bit-exact comparison.  This module checks the same results against what any order
must satisfy:

  * float SUM: the exact sum S, and the forward error bound of recursive summation, valid for any
    order and any reduction tree (Higham, Accuracy and Stability of Numerical Algorithms, 4.2):
        |got - S| <= gamma_{n-1} * sum|x| + 2^-53 * |S| + (n-1) * eta,
    gamma_k = k*u / (1 - k*u), u = 2^-24 (f32) or 2^-53 (f64), eta = 2^-150 (f32) or 2^-1074 (f64,
    the nearest double above 2^-1075) the subnormal term, 2^-53 * |S| the rounding of the reference itself to f64;
  * i64 SUM: the sum mod 2^64, compared exactly;
  * MAX / MIN: numpy's maximum / minimum, compared bit for bit (valid on data without NaN and
    without a +0 / -0 tie, which the generators here never produce).

It also holds the seeded input generators and the shape selector of tests/test_reduction_shapes.py,
with the kernels' ownership arithmetic (own_shift in b200mpi.cu, Owner in kernels.cuh) restated.
"""
import hashlib

import numpy as np

SUM, MAX, MIN = 0, 1, 2
OPS = {"sum": SUM, "max": MAX, "min": MIN}
DTYPES = {"f32": np.float32, "f64": np.float64, "i64": np.int64}
UNIT = {np.dtype(np.float32): 2.0 ** -24, np.dtype(np.float64): 2.0 ** -53}
ETA = {np.dtype(np.float32): 2.0 ** -150, np.dtype(np.float64): 2.0 ** -1074}  # f64: 2^-1075 is not representable; its upper neighbour


def epv(dtype):
    """Elements per 16-byte vector."""
    return 16 // np.dtype(dtype).itemsize


# ---- seeded generators (the same arrays on every rank) -------------------------------------------
def splitmix64(seed, count, start=0):
    """splitmix64(seed, i) for i in [start, start+count): the stream oracle_fill_* also uses."""
    i = np.arange(start, start + count, dtype=np.uint64)
    z = np.uint64(seed & 0xFFFFFFFFFFFFFFFF) + (i + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def _mantissa(bits, dtype):
    """A value in [1, 2) with every mantissa bit of `dtype` random."""
    if np.dtype(dtype) == np.float32:
        return 1.0 + (bits >> np.uint64(41)).astype(np.float64) * 2.0 ** -23
    return 1.0 + (bits >> np.uint64(12)).astype(np.float64) * 2.0 ** -52


def uniform01(dtype, n, count, seed):
    """The suite's usual fill: uniform [0, 1) with 24 (f32) or 53 (f64) random bits; raw bits for i64."""
    out = []
    for r in range(n):
        z = splitmix64(seed + r, count)
        if np.dtype(dtype) == np.int64:
            out.append(z.view(np.int64))
        elif np.dtype(dtype) == np.float32:
            out.append(((z >> np.uint64(40)).astype(np.float64) * 2.0 ** -24).astype(np.float32))
        else:
            out.append((z >> np.uint64(11)).astype(np.float64) * 2.0 ** -53)
    return out


def signed(dtype, n, count, seed):
    """Random sign, full mantissa, exponent within +-20 of a per-element base that itself spans
    +-20: sums cancel at every magnitude.  |x| < 2^41, so no f32 sum of 8 terms overflows."""
    base = (splitmix64(seed ^ 0x5151, count) % np.uint64(41)).astype(np.int64) - 20
    out = []
    for r in range(n):
        z = splitmix64(seed + 101 * (r + 1), count)
        e = base + (z % np.uint64(41)).astype(np.int64) - 20
        sgn = np.where((z >> np.uint64(7)) & np.uint64(1), -1.0, 1.0)
        out.append(np.ldexp(sgn * _mantissa(z, dtype), e).astype(dtype))
    return out


def cancel(dtype, n, count, seed):
    """x_0 = +B, x_{n-1} = -B with B ~ 2^10..2^30, the ranks between small (|x| < 1): the exact
    sum is the small part, which rank order mostly loses.  n = 2: S == 0."""
    zb = splitmix64(seed ^ 0xCA7CE1, count)
    big = np.ldexp(_mantissa(zb, dtype), (zb % np.uint64(21)).astype(np.int64) + 10).astype(dtype)
    out = []
    for r in range(n):
        if r == 0:
            out.append(big.copy())
        elif r == n - 1:
            out.append(-big)
        else:
            z = splitmix64(seed + 7 * r, count)
            sgn = np.where((z >> np.uint64(5)) & np.uint64(1), -1.0, 1.0)
            e = -(z % np.uint64(21)).astype(np.int64) - 1
            out.append(np.ldexp(sgn * _mantissa(z, dtype), e).astype(dtype))
    return out


def i64(dtype, n, count, seed):
    """Full-range int64, every third element within 2^20 of +-2^63: sums wrap around."""
    assert np.dtype(dtype) == np.int64
    out = []
    for r in range(n):
        z = splitmix64(seed + 31 * (r + 1), count)
        x = z.view(np.int64).copy()
        near = (z & np.uint64(0xFFFFF)).astype(np.int64)
        hi = np.int64(2 ** 63 - 1) - near
        lo = np.int64(-2 ** 63) + near
        sel = np.arange(count) % 3 == 0
        x[sel] = np.where((z[sel] >> np.uint64(63)) == 1, hi[sel], lo[sel])
        out.append(x)
    return out


GENERATORS = {"uniform01": uniform01, "signed": signed, "cancel": cancel, "i64": i64}


def generate(name, dtype, n, count, seed):
    return GENERATORS[name](np.dtype(dtype), n, count, seed)


# ---- exact references --------------------------------------------------------------------------
def _two_sum(a, b):
    s = a + b
    bp = s - a
    return s, (a - (s - bp)) + (b - bp)


def exact_sum(xs):
    """Ogita-Rump-Oishi Sum2 over the ranks, vectorised over elements, in f64: returns (s, c) with
    S ~= s + c.  TwoSum is error free, so S - (s + c) is only the rounding of the c accumulation,
    |S - (s + c)| <= gamma_{n-1}^2 * sum|x| with u = 2^-53; sum_bound adds that term.  f32 inputs
    convert to f64 exactly."""
    s = np.asarray(xs[0], dtype=np.float64).copy()
    c = np.zeros_like(s)
    for x in xs[1:]:
        s, e = _two_sum(s, np.asarray(x, dtype=np.float64))
        c += e
    return s, c


def gamma(k, u):
    return k * u / (1.0 - k * u)


def sum_bound(xs, s, c):
    """Per-element bound on |got - S| for any summation order of xs in their own precision."""
    dt = np.asarray(xs[0]).dtype
    n = len(xs)
    absum = np.zeros(np.asarray(xs[0]).shape, dtype=np.float64)
    for x in xs:
        absum += np.abs(np.asarray(x, dtype=np.float64))
    u = UNIT[dt]
    b = gamma(n - 1, u) * absum + 2.0 ** -53 * np.abs(s + c) + (n - 1) * ETA[dt]
    b += 2.0 * gamma(n - 1, 2.0 ** -53) ** 2 * absum  # the reference's own Sum2 error, twice over
    return b * (1.0 + 2.0 ** -30)  # the bound and |got - S| are themselves computed in f64


def wrap_sum(xs):
    acc = np.zeros(np.asarray(xs[0]).shape, dtype=np.uint64)
    for x in xs:
        acc += np.asarray(x, dtype=np.int64).view(np.uint64)  # mod 2^64, as Go's int64
    return acc.view(np.int64)


def reference(xs, op):
    """The order-independent expected value: for float SUM a pair (s, c), else an array."""
    dt = np.asarray(xs[0]).dtype
    if op == SUM:
        return wrap_sum(xs) if dt == np.int64 else exact_sum(xs)
    stack = np.stack([np.asarray(x) for x in xs])
    return (np.maximum if op == MAX else np.minimum).reduce(stack, axis=0)


def check(got, xs, op):
    """None when `got` is right whatever the order, else a one-line description of the first miss."""
    got = np.asarray(got)
    dt = got.dtype
    ref = reference(xs, op)
    if op == SUM and dt != np.int64:
        s, c = ref
        err = np.abs((got.astype(np.float64) - s) - c)
        bound = sum_bound(xs, s, c)
        bad = ~(err <= bound)
        if bad.any():
            i = int(np.flatnonzero(bad)[0])
            return "element %d of %d: got %r, exact %r, |err| %.3g > bound %.3g (%d bad)" % (
                i, got.size, float(got[i]), float(s[i] + c[i]), err[i], bound[i], int(bad.sum()))
        return None
    return bit_diff(got, ref)


def bit_diff(got, want):
    """None when the two arrays hold the same bits, else where they first differ."""
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    if got.shape != want.shape or got.dtype != want.dtype:
        return "shape/dtype %s %s != %s %s" % (got.shape, got.dtype, want.shape, want.dtype)
    ui = np.dtype("u%d" % got.dtype.itemsize)
    bad = np.flatnonzero(got.view(ui) != want.view(ui))
    if bad.size:
        i = int(bad[0])
        return "element %d of %d: got %r want %r (bit-exact, %d differ)" % (i, got.size, got[i], want[i], bad.size)
    return None


def digest(arr):
    return hashlib.sha256(np.ascontiguousarray(arr).tobytes()).hexdigest()


# ---- ownership arithmetic, restated from b200mpi.cu (own_shift) and kernels.cuh (Owner) -----------
def own_shift(nvec, n, own_block_bytes, min_shift=0):
    """log2 of the ownership block in vectors; nvec is ceil(count / EPV), as the host passes it."""
    per = max((nvec + n - 1) // n, 1)
    sh = per.bit_length() - 1
    cap = (own_block_bytes // 16).bit_length() - 1
    return max(min(sh, cap), min_shift)


def ownership(count, dtype, n, own_block_bytes, min_shift=0):
    """What the owner-reduces kernels see: whole vectors (floor), block shift, number of blocks,
    owner of the last block, whether it is partial, blocks owned per rank, scalar tail length."""
    e = epv(dtype)
    nvec_whole = count // e
    sh = own_shift(-(-count // e), n, own_block_bytes, min_shift)
    blk = 1 << sh
    nblk = -(-nvec_whole // blk)
    owned = [(nblk - r + n - 1) // n if nblk > r else 0 for r in range(n)]
    return {"nvec": nvec_whole, "shift": sh, "nblk": nblk, "last_owner": (nblk - 1) % n if nblk else None,
            "last_partial": nvec_whole % blk != 0, "owned": owned, "tail": count % e}


SMALL_BLOCK = 4096  # own_block_bytes for the ragged shapes: 256 vectors per block
SMEM_STAGES = 4     # kSmemStages: the TMA kernel's ring of shared-memory stages


def ragged_counts(n, dtype, block_bytes=SMALL_BLOCK):
    """Counts at which, with own_block_bytes = block_bytes: ownership wraps around the ranks more
    than twice; the last block is partial and held by rank 1 or rank n-1 (never 0); count % EPV != 0,
    so the last rank reduces the scalar tail; every rank owns more than 2 * SMEM_STAGES blocks, so
    one CTA of the TMA two-shot turns its stage ring over at least twice."""
    e = epv(dtype)
    bv = block_bytes // 16
    out = []
    for last_blk in (9 * n + 1, 10 * n - 1):  # owners 1 and n-1
        nvec = last_blk * bv + 37
        out.append(nvec * e + (e - 1))
    return out


def switch_counts(dtype):
    """Counts of 4095, 4096 and 4097 whole vectors: the shuffle one-shot runs up to 4096 vectors,
    the plain one-shot above (oneshot_plan in b200mpi.cu)."""
    return [v * epv(dtype) for v in (4095, 4096, 4097)]


def big_count(n, dtype, block_bytes=1 << 20):
    """An odd count at the default 1 MiB block: every rank's share is more than 1 MiB, ownership wraps
    twice, the last block is partial and belongs to rank 1."""
    e = epv(dtype)
    bv = block_bytes // 16
    nvec = (2 * n + 1) * bv + 1023
    return nvec * e + 1


# ---- one-shot plan, restated from oneshot_plan in b200mpi.cu ------------------------------------
THREADS = 512   # kThreads
MAX_MIDS = 4094  # kMaxMids = kEpochStride - 2


def oneshot_rounds(count, dtype, n, blocks_cap):
    """Mid-barrier budget the one-shot plan reserves for `count` elements with a grid cap of
    `blocks_cap` CTAs (the SM count or set_max_blocks)."""
    es = np.dtype(dtype).itemsize
    e = 16 // es
    nvec = -(-count // e)
    shfl = n in (2, 4, 8) and nvec <= 4096
    units = nvec * n if shfl else nvec
    blocks = max(1, min(-(-units // THREADS), blocks_cap))
    per_round = blocks * THREADS
    return -(-count // per_round) + (-(-(nvec * n) // per_round) if shfl else 0) + 2


def oneshot_limit(dtype, n, blocks_cap):
    """Largest count whose one-shot plan fits in MAX_MIDS (searched over whole vectors)."""
    e = epv(dtype)
    lo, hi = 1, 1
    while oneshot_rounds(hi * e, dtype, n, blocks_cap) <= MAX_MIDS:
        hi *= 2
    while hi - lo > 1:  # rounds is monotone in the vector count
        mid = (lo + hi) // 2
        if oneshot_rounds(mid * e, dtype, n, blocks_cap) <= MAX_MIDS:
            lo = mid
        else:
            hi = mid
    return lo * e
