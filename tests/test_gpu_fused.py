"""The fused iterated product against an exact reference of its contract.

Seven entry points (include/spmv_b200.h) on four kernel families: spmv_b200_csr_spmv_fused / _fused_mail
(csr_row_fused_kernel<B>, or the fused csr_stream_kernel at batch 0), _fused_flat (csr_row_flat_kernel<B>), _fused_async
(csr_row_async_kernel<B>), and spmv_b200_hll_spmv_fused / _fused_mail (hll_row_fused_kernel<B>) and _fused_flat
(hll_row_flat_kernel<B>).  One launch computes y = (A x) * s, mirrors rows [lo, hi) of every peer into peers.dst[p] and
leaves per-CTA partial sums of y^2.  The reference, all in fp64 ("serial" = spmv_csr_serial: one lane, index order, every
multiply and add rounded):

  s         fused: fl(1 / fl(sqrt(*prev_sumsq))); mail, launch k > 0: the same of the mailbox total; flat: *inv_norm;
            async: fl(1 / fl(sqrt(S[k-2]))) for k >= 2, else 1; without scaling no multiply happens.  The mailbox totals
            and S are read bit for bit from the mailbox slots, never recomputed.
  y         EXACT    y_i = fl(serial_i * s) bit for bit: every row of the row / flat / async / HLL kernels, rows of <= 12
                     nonzeros in the fused stream kernel.  (Dividing by the norm differs by up to 1 ulp: the exact
                     assertion tells the two apart.)
            BOUNDED  the fused stream kernel's longer rows: |y_i - serial_i s| <= (len_i + 3) 2^-53 S_i s, S_i = sum_j |a_ij x_j|.
            HLL y equals CSR y bit for bit (a padding slot adds +0.0).
  partials  flat: CTA b owns rows [256 b, 256 b + 256).  Grid-stride (g CTAs): CTA b owns the 256-row chunks of walk steps
            q = b (mod g); the walk is the natural chunk order, or with boundary-first (SPMV_B200_FUSED_BOUNDARY_FIRST, and
            always in the async form) the chunks holding peer rows first, then the others in order.  Each partial lies
            within (n_b + 1) 2^-53 of the exact sum of y_r^2 over its n_b rows; entries past the grid are 0.0; with the
            CSR row kernel the HLL partials equal the CSR partials bit for bit.  Stream form: only the total is bounded.
  peers     dst[p][lo:hi] = y[lo:hi] bit for bit, every other element of dst[p] untouched.
  protocol  (world = 1) after every launch: status and the CTA counter (async: and the boundary counter) at 0, tag k + 1
            in slot [k&1][0] (mail) or [k&3][0] (async), the halo tag k + 1 when a peer sends to rank 0, and the published
            sum within g 2^-53 of the sum of the partials.

test_the_assertions_catch_broken_kernels shows, without a GPU, that these assertions fail on numpy models of kernels that
break the contract in the ways a fused kernel can.
"""
import math
import zlib

import numpy as np
import pytest

U53 = 2.0 ** -53
CHUNK = 256
MAX_PEERS = 7


# ---------------------------------------------------------------------------------------------------
# the reference and the assertions
# ---------------------------------------------------------------------------------------------------
def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def inv_sqrt(total):
    """fl(1 / fl(sqrt(total))): the scale factor of the fused kernels."""
    return 1.0 / math.sqrt(total)


def random_csr(rng, M, N, lengths):
    """Sorted, duplicate-free rows of the given lengths, each inside a random window of columns; normal values."""
    lengths = np.asarray(lengths, np.int64)
    w = min(N, max(16, int(lengths.max(initial=0)) + 8))
    taken = np.arange(w)[None, :] < lengths[:, None]
    offs = np.sort(np.where(taken, np.argsort(rng.random((M, w)), axis=1), w), axis=1)
    base = rng.integers(0, N - w + 1, M)
    ci = (base[:, None] + offs)[taken].astype(np.int32)
    rp = np.zeros(M + 1, np.int64)
    np.cumsum(lengths, out=rp[1:])
    return rp.astype(np.int32), ci, rng.standard_normal(int(rp[-1]))


class Ref:
    """serial = A x in the serial order, S = |A| |x| (the bound's scale), the row lengths."""

    def __init__(self, checker, rp, ci, va, x):
        self.serial = checker.spmv_csr_serial(rp, ci, va, x)
        self.S = checker.spmv_csr_serial(rp, ci, np.abs(va), np.abs(x))
        self.lens = np.diff(np.asarray(rp, np.int64))

    def y(self, s):
        return self.serial.copy() if s is None else self.serial * s


def y_violations(y, ref, s, exact):
    """Rows of y that break the contract: `exact` marks the rows that must be fl(serial * s) bit for bit, the others must
    lie within (len + 3) 2^-53 S s of serial * s."""
    want = ref.y(s)
    scale = 1.0 if s is None else s
    bound = (ref.lens + 3.0) * U53 * ref.S * scale
    ok = np.where(exact, bits(y) == bits(want), np.abs(y - want) <= bound)
    return np.nonzero(~ok)[0]


def assert_y(y, ref, s, what, exact=True):
    exact = np.broadcast_to(np.asarray(exact, bool), y.shape)
    bad = y_violations(y, ref, s, exact)
    want = ref.y(s)
    assert bad.size == 0, (f"{what}: y: {bad.size} of {y.size} rows off ({int(exact[bad].sum())} of them exact rows), "
                           f"first rows {bad[:5]}: got {y[bad[:5]]}, want {want[bad[:5]]}")


def exact_squares(y):
    """(p, e) with p + e = y^2 exactly (Veltkamp split; |y| well inside the exponent range)."""
    p = y * y
    c = 134217729.0 * y
    hi = c - (c - y)
    lo = y - hi
    return p, ((hi * hi - p) + 2.0 * hi * lo) + lo * lo


def partial_violations(partials, y, owner, g):
    """CTAs b < g whose partial is not within (n_b + 1) 2^-53 of the exact sum of y_r^2 over the rows r with owner[r] = b
    (rows with owner < 0 are not checked), and the entries past g that are not exactly 0.0."""
    p, e = exact_squares(np.asarray(y, np.float64))
    owner = np.asarray(owner, np.int64)
    keep = owner >= 0
    rows = np.nonzero(keep)[0]
    rows = rows[np.argsort(owner[rows], kind="stable")]
    counts = np.bincount(owner[keep], minlength=g)[:g]
    starts = np.concatenate([[0], np.cumsum(counts)])
    bad = []
    for b in range(g):
        mine = rows[starts[b]:starts[b + 1]]
        exact = math.fsum(np.concatenate([p[mine], e[mine]]))
        if not abs(partials[b] - exact) <= (counts[b] + 1) * U53 * exact:
            bad.append(int(b))
    tail = np.nonzero(np.asarray(partials[g:]) != 0.0)[0] + g
    return np.array(bad + tail.tolist(), np.int64)


def assert_partials(partials, y, owner, g, what):
    bad = partial_violations(partials, y, owner, g)
    assert bad.size == 0, f"{what}: partials of CTAs {bad[:8]} ({bad.size} in all, grid {g}) outside (n_b + 1) 2^-53 or not 0.0"


def assert_total(partials, y, what):
    """The sum of all partials (the stream form groups rows its own way) within (M + 2) 2^-53 of the exact sum of y^2."""
    p, e = exact_squares(np.asarray(y, np.float64))
    exact = math.fsum(np.concatenate([p, e]))
    got = math.fsum(partials)
    assert abs(got - exact) <= (y.size + 2) * U53 * exact, f"{what}: sum of the partials {got!r}, exact sum of y^2 {exact!r}"


def peer_violations(dst, y, lo, hi):
    """Elements of a NaN-filled peer buffer that are not y on [lo, hi) bit for bit, or not NaN elsewhere."""
    inside = np.zeros(dst.size, bool)
    inside[lo:hi] = True
    want = np.full(dst.size, np.nan)
    want[:y.size] = y
    return np.nonzero(np.where(inside, bits(dst) == bits(want), np.isnan(dst)) == 0)[0]


def assert_peers(dsts, y, ranges, what):
    for p, (dst, (lo, hi)) in enumerate(zip(dsts, ranges)):
        bad = peer_violations(dst, y, lo, hi)
        assert bad.size == 0, f"{what}: peer {p} [{lo},{hi}): {bad.size} elements wrong, first {bad[:5]}: {dst[bad[:5]]}"


def flat_owner(M):
    return np.arange(M) // CHUNK


def boundary_order(ranges):
    """Twin of boundary_first_order: the union of the peers' row ranges in chunks, ascending and disjoint."""
    merged = []
    for a, b in sorted((lo // CHUNK, (hi + CHUNK - 1) // CHUNK) for lo, hi in ranges if hi > lo):
        if merged and a <= merged[-1][1]:
            merged[-1][1] = max(merged[-1][1], b)
        else:
            merged.append([a, b])
    return merged


def stride_owner(M, g, order=()):
    """CTA of every row under the grid-stride walk of g CTAs: walk step q visits the q-th chunk of the walk order (twin of
    ordered_chunk: the chunks of `order` first, then the others ascending) and belongs to CTA q mod g."""
    chunks = (M + CHUNK - 1) // CHUNK
    first = [c for lo, hi in order for c in range(lo, hi)]
    boundary = np.zeros(chunks, bool)
    boundary[first] = True
    walk = np.array(first + np.nonzero(~boundary)[0].tolist(), np.int64)
    cta = np.empty(chunks, np.int64)
    cta[walk] = np.arange(chunks) % g
    return cta[np.arange(M) // CHUNK]


def peer_ranges(M, count=3):
    """`count` peer row ranges of an M-row matrix: a head, a tail and overlapping ranges around chunk edges (clamped to M,
    possibly empty)."""
    cand = [(0, 37), (M - 40, M), (M // 4, M // 4 + 300), (M // 4 + 150, M // 2 + 7), (255, 257), (M // 2, M // 2), (M // 3, M // 3 + 513)]
    out = []
    for lo, hi in cand[:count]:
        lo, hi = min(max(lo, 0), M), min(max(hi, 0), M)
        out.append((lo, max(lo, hi)))
    return out


# ---------------------------------------------------------------------------------------------------
# CPU: numpy models of broken kernels fail the assertions meant to catch them
# ---------------------------------------------------------------------------------------------------
def model_launch(ref, s, M, owner, g, ranges, flaw=None, total=None):
    """y, partials[g] and peer buffers of one launch of a model kernel (s = 1/sqrt(total) when total is given)."""
    if flaw == "divides by the norm":
        y = ref.serial / math.sqrt(total)
    else:
        y = ref.y(s)
    sq = y * y
    if flaw == "partials one row off":
        sq = np.append(sq[1:], 0.0)
    if flaw == "last ragged chunk left out of the partials" and M % CHUNK:
        sq[M - M % CHUNK:] = 0.0
    partials = np.bincount(owner, weights=sq, minlength=g)
    dsts = []
    for lo, hi in ranges:
        d = np.full(M + 32, np.nan)
        d[lo:hi] = (ref.serial if flaw == "boundary rows mirrored before scaling" else y)[lo:hi]
        dsts.append(d)
    return y, partials, dsts


def model_async(checker, rp, ci, va, x, launches, late=False):
    """Outputs y_k and published sums S[k] of `launches` async launches on a ring (x_{k+1} = y_k), scale from S[k-2]
    (late: from S[k-3])."""
    ys, S = [], []
    lag = 3 if late else 2
    for k in range(launches):
        s = inv_sqrt(S[k - lag]) if k >= lag else None
        y = Ref(checker, rp, ci, va, x).y(s)
        ys.append(y)
        S.append(math.fsum(y * y))
        x = y
    return ys, S


def test_the_assertions_catch_broken_kernels(checker):
    """No GPU: the correct model passes every assertion; each broken model fails the one meant to catch it on a
    meaningful share of rows or CTAs."""
    rng = np.random.default_rng(7)
    M, N = 3000, 3500                                      # 12 chunks, the last one ragged (184 rows)
    lengths = rng.integers(0, 13, M)
    rp, ci, va = random_csr(rng, M, N, lengths)
    x = rng.standard_normal(N)
    ref = Ref(checker, rp, ci, va, x)
    total = 12345.678
    s = inv_sqrt(total)
    ranges = peer_ranges(M, 3)
    for name, owner, g in (("flat", flat_owner(M), (M + 255) // 256), ("grid-stride, 5 CTAs", stride_owner(M, 5), 5),
                           ("boundary-first, 5 CTAs", stride_owner(M, 5, boundary_order(ranges)), 5)):
        y, partials, dsts = model_launch(ref, s, M, owner, g, ranges)
        assert_y(y, ref, s, f"correct model, {name}")
        assert_partials(partials, y, owner, g, f"correct model, {name}")
        assert_total(partials, y, f"correct model, {name}")
        assert_peers(dsts, y, ranges, f"correct model, {name}")
        live = np.count_nonzero(ref.serial)
        y_div, _, _ = model_launch(ref, s, M, owner, g, ranges, "divides by the norm", total)
        off = y_violations(y_div, ref, s, np.ones(M, bool)).size
        assert off > 0.1 * live, f"dividing by the norm: only {off} of {live} rows caught"
        for flaw, share in (("partials one row off", 0.9), ("last ragged chunk left out of the partials", None)):
            y2, p2, _ = model_launch(ref, s, M, owner, g, ranges, flaw)
            bad = partial_violations(p2, y2, owner, g)
            if share is None:                              # exactly the CTA that owns the ragged chunk
                assert bad.tolist() == [int(owner[-1])], f"{name}: {flaw}: CTAs {bad}"
            else:
                assert bad.size >= share * g, f"{name}: {flaw}: only {bad.size} of {g} CTAs caught"
        y3, _, d3 = model_launch(ref, s, M, owner, g, ranges, "boundary rows mirrored before scaling")
        for p, (lo, hi) in enumerate(ranges):
            caught = peer_violations(d3[p], y3, lo, hi).size
            assert caught >= 0.9 * np.count_nonzero(ref.serial[lo:hi]), f"mirrored before scaling: peer {p}: {caught} caught"
    # the async scale one launch late: launch 2 multiplies by 1 instead of 1/sqrt(S[0])
    x0 = rng.standard_normal(M)
    rp_sq, ci_sq, va_sq = random_csr(rng, M, M, lengths)
    for late in (False, True):
        ys, S = model_async(checker, rp_sq, ci_sq, va_sq, x0, 4, late)
        xk = x0
        caught = 0
        for k in range(4):
            rk = Ref(checker, rp_sq, ci_sq, va_sq, xk)
            sk = inv_sqrt(S[k - 2]) if k >= 2 else None
            caught += y_violations(ys[k], rk, sk, np.ones(M, bool)).size
            xk = ys[k]
        if late:
            assert caught >= 0.9 * np.count_nonzero(ys[2]), f"async scale one launch late: only {caught} rows caught"
        else:
            assert caught == 0


# ---------------------------------------------------------------------------------------------------
# GPU fixtures and launch helpers
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    import torch
    from sparsematrixvectormultiplication_b200 import device
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    return device


def _t(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, np.float64)).cuda()


def _nan(n):
    import torch
    return torch.full((max(n, 1),), float("nan"), dtype=torch.float64, device="cuda")


def _peers(N, ranges, M):
    """A Peers struct whose dst[p] are NaN-filled device buffers of M + 32 doubles (the tail catches stores past M)."""
    ps = N.Peers()
    ps.count = len(ranges)
    bufs = []
    for p, (lo, hi) in enumerate(ranges):
        b = _nan(M + 32)
        bufs.append(b)
        ps.dst[p] = b.data_ptr()
        ps.lo[p], ps.hi[p] = lo, hi
    return ps, bufs


def fused_grid(dev, M):
    """Grid of the fused row kernels at the current SPMV_B200_FUSED_CTAS_PER_SM."""
    import os
    ctas = max(1, min(int(os.environ.get("SPMV_B200_FUSED_CTAS_PER_SM", "8") or 8), 256))
    return max(1, min(ctas * dev.device_info()["sm_count"], (M + CHUNK - 1) // CHUNK))


class Mailbox:
    """World-1 mailbox (mail form: 2 x 1 slots; async form: 4 x 1 slots + halo tags) and its counters, zeroed with
    iteration 0, so that every wait of launch k is answered by launch k - 1 on the same stream."""

    def __init__(self, N, async_form=False):
        import torch
        self.async_form = async_form
        self.box = torch.zeros((N.ASYNC_MAILBOX_BYTES if async_form else N.MAILBOX_BYTES) // 8, dtype=torch.int64, device="cuda")
        self.sync = torch.zeros(4, dtype=torch.int32, device="cuda")   # counter, boundary counter (async), status
        self.d = (N.Async if async_form else N.Mail)()
        self.d.world, self.d.rank, self.d.iteration = 1, 0, 0
        self.d.box[0] = self.box.data_ptr()
        self.d.counter = self.sync.data_ptr()
        if async_form:
            self.d.bcounter = self.sync.data_ptr() + 4
            self.d.status = self.sync.data_ptr() + 8
        else:
            self.d.status = self.sync.data_ptr() + 8

    def slot(self, k):
        """(sum, tag) that launch k published."""
        at = 2 * (k & (3 if self.async_form else 1))
        raw = self.box.cpu().numpy()
        return float(raw[at:at + 1].view(np.float64)[0]), int(raw[at + 1])

    def check(self, k, partials, g, what, halo=False):
        """Protocol state after launch k; returns the published sum."""
        sync = self.sync.cpu().numpy()
        assert sync[2] == 0, f"{what}: launch {k}: status {sync[2]} (a wait gave up)"
        assert sync[0] == 0, f"{what}: launch {k}: CTA counter left at {sync[0]}"
        if self.async_form:
            assert sync[1] == 0, f"{what}: launch {k}: boundary counter left at {sync[1]}"
        total, tag = self.slot(k)
        assert tag == k + 1, f"{what}: launch {k}: tag {tag} in slot [{k & (3 if self.async_form else 1)}][0]"
        if halo:
            got = int(self.box.cpu().numpy()[8])
            assert got == k + 1, f"{what}: launch {k}: halo tag {got}"
        ref = math.fsum(partials[:g])
        assert abs(total - ref) <= g * U53 * ref, f"{what}: launch {k}: published {total!r}, partials add to {ref!r}"
        return total


# ---------------------------------------------------------------------------------------------------
# the matrices
# ---------------------------------------------------------------------------------------------------
CASES = {   # name: (M, N, lengths(rng, M))
    "M1": (1, 16, lambda r, M: np.array([7])),
    "M31": (31, 64, lambda r, M: r.integers(0, 13, M)),
    "M255": (255, 400, lambda r, M: r.integers(0, 13, M)),
    "M256": (256, 300, lambda r, M: r.integers(0, 13, M)),
    "M257": (257, 257, lambda r, M: r.integers(0, 13, M)),
    "prime7919": (7919, 7919, lambda r, M: r.integers(0, 13, M)),
    "rank_slice": (1000, 5000, lambda r, M: r.integers(0, 13, M)),        # M rows reading an x of N != M elements
    "rows13to40": (3001, 4000, lambda r, M: np.where(r.random(M) < 0.5, r.integers(13, 41, M), r.integers(0, 13, M))),
    "plan_timed": (600_011, 600_011, lambda r, M: r.integers(6, 13, M)),   # >= 2^22 nonzeros: the plan times the batches
}


def case_lengths(name, rng):
    M, _, make = {**CASES, **WALK}[name]
    lengths = np.asarray(make(rng, M), np.int64)
    for r in (255, 256, 511, 512, M - 1):                  # empty rows at chunk edges and at the end
        if 0 < r < M and M > 1:
            lengths[r] = 0
    return lengths


WALK = {"walk": (200_003, 200_003, lambda r, M: r.integers(0, 13, M))}   # 782 chunks
_built = {}


def case(dev, checker, name):
    """Host arrays, reference and device handles of a case (built once per module)."""
    if name not in _built:
        M, N, _ = {**CASES, **WALK}[name]
        rng = np.random.default_rng(zlib.crc32(name.encode()))
        rp, ci, va = random_csr(rng, M, N, case_lengths(name, rng))
        x = rng.standard_normal(N)
        A = dev.DeviceCSR.upload(M, N, rp, ci, va)
        _built[name] = dict(M=M, N=N, rp=rp, ci=ci, va=va, x=x, xd=_t(x), ref=Ref(checker, rp, ci, va, x), A=A, H=A.to_hll(),
                            total=float(rng.uniform(0.5, 1e6)), short=np.diff(rp) <= 12)
    return _built[name]


# ---------------------------------------------------------------------------------------------------
# one launch of each entry point, checked in full: y, partials, peers (and the protocol state)
# ---------------------------------------------------------------------------------------------------
def run_fused(dev, c, fmt, what, scaled=True, ranges=(), order=None, hll_partials_of=None):
    """spmv_b200_{csr,hll}_spmv_fused; returns (y, partials, g) with g the row kernel's grid (None: stream kernel)."""
    import torch
    from sparsematrixvectormultiplication_b200 import _native as N
    M, ref = c["M"], c["ref"]
    X = c["A"] if fmt == "csr" else c["H"]
    info = X.info()
    g = None if fmt == "csr" and batch_of(info.fused_batch, "SPMV_B200_FUSED_BATCH") == 0 else fused_grid(dev, M)
    count = X.partials_count()
    partials = torch.full((count,), float("nan"), dtype=torch.float64, device="cuda")
    prev = _t([c["total"]]) if scaled else None
    s = inv_sqrt(c["total"]) if scaled else None
    ps, bufs = _peers(N, ranges, M) if ranges else (None, [])
    y = _nan(M)
    X.spmv_fused(c["xd"], y, prev_sumsq=prev, partials=partials, peers=ps)
    yh, ph = y.cpu().numpy()[:M], partials.cpu().numpy()
    assert_y(yh, ref, s, what, exact=True if g is not None else c["short"])
    if g is None:
        assert_total(ph, yh, what)
    else:
        owner = stride_owner(M, g, boundary_order(ranges) if ranges and order else ())
        assert_partials(ph, yh, owner, g, what)
    assert_peers([b.cpu().numpy() for b in bufs], yh, ranges, what)
    return yh, ph, g


def run_mail(dev, c, fmt, what, launches=2, ranges=(), order=False):
    """spmv_b200_{csr,hll}_spmv_fused_mail at world 1: launch 0 unscaled, launch k > 0 scaled by the mailbox total."""
    import torch
    from sparsematrixvectormultiplication_b200 import _native as N
    M, ref = c["M"], c["ref"]
    X = c["A"] if fmt == "csr" else c["H"]
    stream_form = fmt == "csr" and batch_of(X.info().fused_batch, "SPMV_B200_FUSED_BATCH") == 0
    g = fused_grid(dev, M)
    mb = Mailbox(N)
    partials = torch.full((X.partials_count(),), float("nan"), dtype=torch.float64, device="cuda")
    total = None
    for k in range(launches):
        mb.d.iteration = k
        ps, bufs = _peers(N, ranges, M) if ranges else (None, [])
        y = _nan(M)
        X.spmv_fused_mail(c["xd"], y, partials, mb.d, peers=ps)
        s = inv_sqrt(total) if k > 0 else None
        yh, ph = y.cpu().numpy()[:M], partials.cpu().numpy()
        tag = f"{what}, launch {k}"
        assert_y(yh, ref, s, tag, exact=c["short"] if stream_form else True)
        if stream_form:                                    # its grid is its own: the whole buffer is summed
            assert_total(ph, yh, tag)
            total = mb.check(k, ph, ph.size, tag)
        else:
            assert_partials(ph, yh, stride_owner(M, g, boundary_order(ranges) if ranges and order else ()), g, tag)
            total = mb.check(k, ph, g, tag)
        assert_peers([b.cpu().numpy() for b in bufs], yh, ranges, tag)


def run_flat(dev, c, fmt, what, scaled=True, ranges=()):
    import torch
    from sparsematrixvectormultiplication_b200 import _native as N
    M, ref = c["M"], c["ref"]
    X = c["A"] if fmt == "csr" else c["H"]
    g = X.flat_partials_count()
    assert g == (M + CHUNK - 1) // CHUNK
    partials = torch.full((g,), float("nan"), dtype=torch.float64, device="cuda")
    s = inv_sqrt(c["total"]) if scaled else None
    inv = _t([s]) if scaled else None
    ps, bufs = _peers(N, ranges, M) if ranges else (None, [])
    y = _nan(M)
    X.spmv_fused_flat(c["xd"], y, inv_norm=inv, partials=partials, peers=ps)
    yh, ph = y.cpu().numpy()[:M], partials.cpu().numpy()
    assert_y(yh, ref, s, what)
    assert_partials(ph, yh, flat_owner(M), g, what)
    assert_peers([b.cpu().numpy() for b in bufs], yh, ranges, what)
    return yh, ph


def run_async(dev, c, what, launches=4, ranges=()):
    """spmv_b200_csr_spmv_fused_async at world 1 on a fixed x: launch k scaled by 1/sqrt(S[k-2]) read from the mailbox; a
    peer sends to rank 0, which also receives from itself (the halo tag of launch k-1 answers launch k)."""
    import torch
    from sparsematrixvectormultiplication_b200 import _native as N
    M, ref, A = c["M"], c["ref"], c["A"]
    g = fused_grid(dev, M)
    mb = Mailbox(N, async_form=True)
    if ranges:
        mb.d.num_recv, mb.d.recv_from[0] = 1, 0
        for p in range(len(ranges)):
            mb.d.send_to[p] = 0
    partials = torch.full((A.partials_count(),), float("nan"), dtype=torch.float64, device="cuda")
    owner = stride_owner(M, g, boundary_order(ranges))
    S = []
    for k in range(launches):
        mb.d.iteration = k
        ps, bufs = _peers(N, ranges, M) if ranges else (None, [])
        y = _nan(M)
        A.spmv_fused_async(c["xd"], y, partials, mb.d, peers=ps)
        s = inv_sqrt(S[k - 2]) if k >= 2 else None
        yh, ph = y.cpu().numpy()[:M], partials.cpu().numpy()
        tag = f"{what}, launch {k}"
        assert_y(yh, ref, None if s is None else s, tag)
        assert_partials(ph[:g], yh, owner, g, tag)
        S.append(mb.check(k, ph, g, tag, halo=bool(ranges)))
        assert_peers([b.cpu().numpy() for b in bufs], yh, ranges, tag)


def batch_of(planned, env):
    import os
    v = os.environ.get(env, "")
    return int(v) if v else planned


def form_name(kernel, planned, env):
    import os
    forced = os.environ.get(env, "")
    b = int(forced) if forced else planned
    if kernel == "csr_row_fused_kernel" and b == 0:
        return f"fused csr_stream_kernel ({'forced' if forced else 'plan'})"
    return f"{kernel}<{b}> ({'forced' if forced else 'plan'})"


FUSED_BATCHES = [None, 0, 2, 3, 4, 5, 6, 7]   # None: the form the plan chose
ROW_BATCHES = [None, 2, 3, 4, 5, 6, 7]


# ---------------------------------------------------------------------------------------------------
# step-level exactness: every forced form, every entry point, every shape
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_csr_fused_and_mail_every_batch(dev, checker, monkeypatch, name):
    c = case(dev, checker, name)
    info = c["A"].info()
    if name == "plan_timed":
        assert info.nnz >= 1 << 22
    for batch in FUSED_BATCHES:
        if batch is None:
            monkeypatch.delenv("SPMV_B200_FUSED_BATCH", raising=False)
        else:
            monkeypatch.setenv("SPMV_B200_FUSED_BATCH", str(batch))
        form = form_name("csr_row_fused_kernel", info.fused_batch, "SPMV_B200_FUSED_BATCH")
        what = f"{name}: spmv_b200_csr_spmv_fused, {form}"
        run_fused(dev, c, "csr", what, ranges=peer_ranges(c["M"], 3))
        if batch is None:
            run_fused(dev, c, "csr", what + ", unscaled", scaled=False)
        run_mail(dev, c, "csr", f"{name}: spmv_b200_csr_spmv_fused_mail, {form}", ranges=peer_ranges(c["M"], 2))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_hll_fused_and_mail_every_batch(dev, checker, monkeypatch, name):
    """The HLL twins, also on hacks wider than 12 and on the padding of M % 32 != 0; y and the partials are those of the
    CSR row kernel bit for bit."""
    c = case(dev, checker, name)
    info = c["H"].info()
    monkeypatch.setenv("SPMV_B200_FUSED_BATCH", "4")
    _, csr_partials, _ = run_fused(dev, c, "csr", f"{name}: spmv_b200_csr_spmv_fused, csr_row_fused_kernel<4>")
    planned = info.fused_batch if info.fused_batch > 0 else info.row_batch
    for batch in ROW_BATCHES:
        if batch is None:
            monkeypatch.delenv("SPMV_B200_HLL_FUSED_BATCH", raising=False)
        else:
            monkeypatch.setenv("SPMV_B200_HLL_FUSED_BATCH", str(batch))
        form = form_name("hll_row_fused_kernel", planned, "SPMV_B200_HLL_FUSED_BATCH")
        what = f"{name}: spmv_b200_hll_spmv_fused, {form}"
        _, ph, g = run_fused(dev, c, "hll", what, ranges=peer_ranges(c["M"], 3))
        bad = np.nonzero(bits(ph) != bits(csr_partials[:ph.size]))[0]
        assert bad.size == 0, f"{what}: partials of CTAs {bad[:8]} differ from the CSR row kernel's"
        if batch is None:
            run_fused(dev, c, "hll", what + ", unscaled", scaled=False)
        run_mail(dev, c, "hll", f"{name}: spmv_b200_hll_spmv_fused_mail, {form}", ranges=peer_ranges(c["M"], 2))


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_flat_every_batch(dev, checker, monkeypatch, name):
    """The FLAT forms, CSR (rows of <= 12 only) and HLL (any width); the HLL partials equal the CSR partials bit for bit."""
    c = case(dev, checker, name)
    ci, hi = c["A"].info(), c["H"].info()
    csr_ok = ci.max_row_nnz <= 12
    for batch in ROW_BATCHES:
        for env in ("SPMV_B200_FLAT_BATCH", "SPMV_B200_HLL_FLAT_BATCH"):
            if batch is None:
                monkeypatch.delenv(env, raising=False)
            else:
                monkeypatch.setenv(env, str(batch))
        hform = form_name("hll_row_flat_kernel", hi.flat_batch, "SPMV_B200_HLL_FLAT_BATCH")
        yh, ph = run_flat(dev, c, "hll", f"{name}: spmv_b200_hll_spmv_fused_flat, {hform}", ranges=peer_ranges(c["M"], 3))
        if batch is None:
            run_flat(dev, c, "hll", f"{name}: spmv_b200_hll_spmv_fused_flat, {hform}, unscaled", scaled=False)
        if csr_ok:
            cform = form_name("csr_row_flat_kernel", ci.flat_batch, "SPMV_B200_FLAT_BATCH")
            what = f"{name}: spmv_b200_csr_spmv_fused_flat, {cform}"
            yc, pc = run_flat(dev, c, "csr", what, ranges=peer_ranges(c["M"], 3))
            if batch is None:
                run_flat(dev, c, "csr", what + ", unscaled", scaled=False)
            assert np.array_equal(bits(yh), bits(yc)), f"{what}: HLL y differs from CSR y"
            bad = np.nonzero(bits(ph) != bits(pc))[0]
            assert bad.size == 0, f"{what}: HLL partials of CTAs {bad[:8]} differ from the CSR partials"


@pytest.mark.gpu
@pytest.mark.parametrize("name", [n for n in CASES if n != "rows13to40"])
def test_async_launches(dev, checker, name):
    """Four launches of the asynchronous form: lagged scale, tags, counters, partials, a peer sending to rank 0 and
    overlapping peer ranges."""
    c = case(dev, checker, name)
    info = c["A"].info()
    form = f"csr_row_async_kernel<{info.fused_batch if info.fused_batch > 0 else info.row_batch}>"
    run_async(dev, c, f"{name}: spmv_b200_csr_spmv_fused_async, {form}, no peers")
    run_async(dev, c, f"{name}: spmv_b200_csr_spmv_fused_async, {form}, 3 peers", ranges=peer_ranges(c["M"], 3))


@pytest.mark.gpu
@pytest.mark.parametrize("ctas", [1, 3])
@pytest.mark.parametrize("boundary_first", [0, 1])
def test_grid_stride_walk(dev, checker, monkeypatch, ctas, boundary_first):
    """SPMV_B200_FUSED_CTAS_PER_SM = 1 / 3: every CTA walks several chunks, the chunk count (782) is not a multiple of the
    grid; with boundary-first and up to 7 peers the chunks holding peer rows come first."""
    monkeypatch.setenv("SPMV_B200_FUSED_CTAS_PER_SM", str(ctas))   # before partials_count(): the grid follows it
    monkeypatch.setenv("SPMV_B200_FUSED_BOUNDARY_FIRST", str(boundary_first))
    monkeypatch.setenv("SPMV_B200_FUSED_BATCH", "4")
    c = case(dev, checker, "walk")
    g = fused_grid(dev, c["M"])
    chunks = (c["M"] + CHUNK - 1) // CHUNK
    assert chunks > g and chunks % g, (chunks, g)
    for npeers in (2, MAX_PEERS):
        ranges = peer_ranges(c["M"], npeers)
        tag = f"walk, {ctas} CTAs/SM, boundary-first {boundary_first}, {npeers} peers"
        for fmt in ("csr", "hll"):
            run_fused(dev, c, fmt, f"spmv_b200_{fmt}_spmv_fused, {fmt}_row_fused_kernel<4>, {tag}", ranges=ranges,
                      order=bool(boundary_first))
            run_mail(dev, c, fmt, f"spmv_b200_{fmt}_spmv_fused_mail, {fmt}_row_fused_kernel<4>, {tag}", launches=3,
                     ranges=ranges, order=bool(boundary_first))
        run_async(dev, c, f"spmv_b200_csr_spmv_fused_async, {tag}", launches=3, ranges=ranges)
    # results repeat bit for bit
    tag = f"walk, {ctas} CTAs/SM, boundary-first {boundary_first}, second launch"
    y1, p1, _ = run_fused(dev, c, "csr", tag, ranges=peer_ranges(c["M"], 2), order=bool(boundary_first))
    y2, p2, _ = run_fused(dev, c, "csr", tag, ranges=peer_ranges(c["M"], 2), order=bool(boundary_first))
    assert np.array_equal(bits(y1), bits(y2)) and np.array_equal(bits(p1), bits(p2)), f"{tag}: a second launch differs"


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [1, 2, 3])
def test_private_image_is_ignored(dev, checker, monkeypatch, mode):
    """A handle that holds a private image (set_image 1 / 2 / 3) gives the same bits in every fused form: those kernels
    read the CSR arrays."""
    import torch
    from sparsematrixvectormultiplication_b200 import synth
    n = 96                                                 # lap2d: 9 distinct rows, 3 distinct values
    rp, ci, va = synth.lap2d_csr(n)
    M = n * n
    rng = np.random.default_rng(mode)
    x = rng.standard_normal(M)
    c = dict(M=M, N=M, rp=rp, ci=ci, va=va, x=x, xd=_t(x), ref=Ref(checker, rp, ci, va, x), total=7.25,
             short=np.ones(M, bool))
    c["A"] = dev.DeviceCSR.upload(M, M, rp, ci, va)
    c["A"].set_image(0)
    c["H"] = c["A"].to_hll()
    monkeypatch.setenv("SPMV_B200_FUSED_BATCH", "4")
    ranges = peer_ranges(M, 3)
    plain = [run_fused(dev, c, "csr", "no image: csr fused", ranges=ranges)[:2],
             run_flat(dev, c, "csr", "no image: csr flat", ranges=ranges)]
    c["A"].set_image(mode)
    assert c["A"].image_form() != "none"
    what = f"image {c['A'].image_form()}"
    imaged = [run_fused(dev, c, "csr", f"{what}: csr fused", ranges=ranges)[:2],
              run_flat(dev, c, "csr", f"{what}: csr flat", ranges=ranges)]
    for (ya, pa), (yb, pb) in zip(plain, imaged):
        assert np.array_equal(bits(ya), bits(yb)) and np.array_equal(bits(pa), bits(pb)), what
    run_mail(dev, c, "csr", f"{what}: csr mail", ranges=ranges)
    run_async(dev, c, f"{what}: csr async", ranges=ranges)


# ---------------------------------------------------------------------------------------------------
# iterations: the async class against the oracle, and general matrices through the entry points directly
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_async_power_iteration_matches_the_oracle(dev, port):
    from sparsematrixvectormultiplication_b200 import synth
    from sparsematrixvectormultiplication_b200.distributed import AsyncPowerIteration
    n, K = 14, 24
    rp, ci, va = synth.lap3d_csr(n)
    x_ref, _, lam_ref = port.power_iteration(rp, ci, va, np.ones(n ** 3), K)
    P = AsyncPowerIteration(synth.SYNTH_LAP3D, n, single=True)
    for k in range(1, K + 1):
        P.step()
        if k >= 3:
            lam = P.eigenvalue_estimate()
            assert abs(lam - lam_ref[k - 1]) <= 1e-12 * lam_ref[k - 1], f"launch {k}: lambda {lam!r}, oracle {lam_ref[k - 1]!r}"
    v = P.normalized_x().cpu().numpy()
    assert np.max(np.abs(v - x_ref)) <= 1e-12 * np.max(np.abs(x_ref))
    P.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["csr", "hll"])
@pytest.mark.parametrize("form", ["mailbox", "split"])
def test_general_matrix_iteration(dev, port, fmt, form):
    """The iterated product on a general (unsymmetric, irregular, positive) matrix through the entry points: one mailbox
    launch, or a FLAT launch plus the exchange kernel, per iteration; lambda and x against the oracle's power iteration."""
    import torch
    from sparsematrixvectormultiplication_b200 import _native as N
    rng = np.random.default_rng(11)
    M, iters = 5003, 14
    rp, ci, va = random_csr(rng, M, M, rng.integers(1, 13, M))
    va = np.abs(va) + 0.1
    x_ref, _, lam_ref = port.power_iteration(rp, ci, va, np.ones(M), iters)
    A = dev.DeviceCSR.upload(M, M, rp, ci, va)
    A.set_image(0)
    X = A if fmt == "csr" else A.to_hll()
    xs = [torch.ones(M, dtype=torch.float64, device="cuda"), torch.zeros(M, dtype=torch.float64, device="cuda")]
    mb = Mailbox(N)
    partials = torch.zeros(X.flat_partials_count() if form == "split" else X.partials_count(), dtype=torch.float64, device="cuda")
    scale = torch.ones(2, dtype=torch.float64, device="cuda")
    for k in range(iters):
        x, y = xs[k & 1], xs[(k & 1) ^ 1]
        mb.d.iteration = k
        if form == "split":
            X.spmv_fused_flat(x, y, inv_norm=scale.data_ptr() + 8 if k else None, partials=partials)
            dev.mail_exchange(partials, partials.numel(), mb.d, scale)
            lam = float(scale[0]) ** 0.5                   # at world 1 the exchange kernel has no one to publish to
        else:
            X.spmv_fused_mail(x, y, partials, mb.d)
            assert mb.slot(k)[1] == k + 1
            lam = mb.slot(k)[0] ** 0.5
        assert int(mb.sync[2]) == 0 and int(mb.sync[0]) == 0
        assert abs(lam - lam_ref[k]) <= 1e-12 * lam_ref[k], f"{fmt} {form}, iteration {k}: lambda {lam!r}, oracle {lam_ref[k]!r}"
    v = (xs[iters & 1] / lam).cpu().numpy()
    assert np.max(np.abs(v - x_ref)) <= 1e-12 * np.max(np.abs(x_ref)), f"{fmt} {form}: x"


# ---------------------------------------------------------------------------------------------------
# full size: lap3d 512^3, row windows where the nnz offset crosses 2^28 and 2^29, and the last 2^20 rows
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_full_size_lap3d_512(dev, checker, monkeypatch):
    """One launch of the tuned fused form, the fused form at batch 5 and the flat form (CSR), and of the fused and flat
    forms (HLL), bit for bit on the numpy twin's windows (as test_gpu_fp32.py::test_offsets_past_2_31_bytes_lap3d_512);
    the flat partials of the CTAs inside the windows bounded, the total of every form bounded against sum y^2 on the
    device."""
    import torch
    from sparsematrixvectormultiplication_b200 import synth
    n = 512
    M = n ** 3
    n2 = n * n
    seed = 0x3D512
    half = 1 << 20
    rows = []
    for target in (1 << 28, 1 << 29):
        lo, hi = 0, M
        while hi - lo > 1:
            mid = (lo + hi) // 2
            if synth.row_offset(synth.SYNTH_LAP3D, n, 0, 0, mid) <= target:
                lo = mid
            else:
                hi = mid
        rows.append(lo)
    windows = [(max(0, r - half) // CHUNK * CHUNK, min(M, r + half) // CHUNK * CHUNK) for r in rows] + [(M - half, M)]
    total = 3.0e7
    s = inv_sqrt(total)
    refs = []
    for lo, hi in windows:
        rp, ci, va = synth.lap3d_csr(n, lo, hi)
        base, top = max(0, lo - n2), min(M, hi + n2)
        xw = synth.hash_vector(top - base, seed, begin=base)
        refs.append(Ref(checker, rp, ci - np.int32(base), va, xw))
        del rp, ci, va, xw

    def check(y, partials, what, flat):
        for (lo, hi), ref in zip(windows, refs):
            got = y[lo:hi].cpu().numpy()
            assert_y(got, ref, s, f"{what}, rows [{lo},{hi})")
            if flat:
                p = partials[lo // CHUNK: hi // CHUNK].cpu().numpy()
                assert_partials(p, got, np.arange(hi - lo) // CHUNK, p.size, f"{what}, CTAs of rows [{lo},{hi})")
        sq = float((y * y).sum())
        got = math.fsum(partials.cpu().numpy())
        assert abs(got - sq) <= 2 * (M + 2) * U53 * sq, f"{what}: partials add to {got!r}, sum of y^2 {sq!r}"

    A = dev.DeviceCSR.synth(synth.SYNTH_LAP3D, n)
    A.set_image(0)
    info = A.info()
    x = torch.empty(M, dtype=torch.float64, device="cuda")
    dev.synth_vector(x, seed)
    y = torch.empty(M, dtype=torch.float64, device="cuda")
    prev = _t([total])
    inv = _t([s])
    for batch in (None, 5):
        if batch is None:
            monkeypatch.delenv("SPMV_B200_FUSED_BATCH", raising=False)
        else:
            monkeypatch.setenv("SPMV_B200_FUSED_BATCH", str(batch))
        partials = torch.full((A.partials_count(),), float("nan"), dtype=torch.float64, device="cuda")
        y.fill_(float("nan"))
        A.spmv_fused(x, y, prev_sumsq=prev, partials=partials)
        check(y, partials, "lap3d 512: spmv_b200_csr_spmv_fused, " + form_name("csr_row_fused_kernel", info.fused_batch,
                                                                                  "SPMV_B200_FUSED_BATCH"), False)
    monkeypatch.delenv("SPMV_B200_FUSED_BATCH", raising=False)
    partials = torch.full((A.flat_partials_count(),), float("nan"), dtype=torch.float64, device="cuda")
    y.fill_(float("nan"))
    A.spmv_fused_flat(x, y, inv_norm=inv, partials=partials)
    check(y, partials, f"lap3d 512: spmv_b200_csr_spmv_fused_flat, csr_row_flat_kernel<{info.flat_batch}> (plan)", True)
    H = A.to_hll()
    A.close()
    del A
    hi = H.info()
    partials = torch.full((H.partials_count(),), float("nan"), dtype=torch.float64, device="cuda")
    y.fill_(float("nan"))
    H.spmv_fused(x, y, prev_sumsq=prev, partials=partials)
    check(y, partials, f"lap3d 512: spmv_b200_hll_spmv_fused, hll_row_fused_kernel<{hi.fused_batch or hi.row_batch}> (plan)", False)
    partials = torch.full((H.flat_partials_count(),), float("nan"), dtype=torch.float64, device="cuda")
    y.fill_(float("nan"))
    H.spmv_fused_flat(x, y, inv_norm=inv, partials=partials)
    check(y, partials, f"lap3d 512: spmv_b200_hll_spmv_fused_flat, hll_row_flat_kernel<{hi.flat_batch}> (plan)", True)
    H.close()


# ---------------------------------------------------------------------------------------------------
# validation: bad arguments are rejected before anything is written
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_entry_points_reject_bad_arguments(dev, checker):
    import torch
    from sparsematrixvectormultiplication_b200 import _native as N
    c = case(dev, checker, "M257")
    M = c["M"]
    rng = np.random.default_rng(5)
    wrp, wci, wva = random_csr(rng, 300, 300, rng.integers(13, 20, 300))   # rows above 12
    wide = dev.DeviceCSR.upload(300, 300, wrp, wci, wva)
    rp, ci, va = random_csr(rng, 300, 3000, np.r_[rng.integers(0, 13, 299), 2000])   # one row past the long-row threshold
    longrow = dev.DeviceCSR.upload(300, 3000, rp, ci, va)
    empty = dev.DeviceCSR.upload(0, 8, np.zeros(1, np.int32), np.zeros(0, np.int32), np.zeros(0))
    empty_h = empty.to_hll()

    y = _nan(M)
    partials = torch.full((4096,), float("nan"), dtype=torch.float64, device="cuda")
    buf = _nan(M + 32)
    before = [t.clone() for t in (y, partials, buf)]

    def peers(count=1, lo=0, hi=10):
        ps = N.Peers()
        ps.count = count
        for p in range(MAX_PEERS):
            ps.dst[p], ps.lo[p], ps.hi[p] = buf.data_ptr(), lo, hi
        return ps

    def calls(X, fmt, ps=None, mb=None, ab=None, partials_ptr=partials, yv=y, xv=None):
        xv = c["xd"] if xv is None else xv
        out = {f"spmv_b200_{fmt}_spmv_fused": lambda: X.spmv_fused(xv, yv, partials=partials_ptr, peers=ps),
               f"spmv_b200_{fmt}_spmv_fused_flat": lambda: X.spmv_fused_flat(xv, yv, partials=partials_ptr, peers=ps),
               f"spmv_b200_{fmt}_spmv_fused_mail": lambda: X.spmv_fused_mail(xv, yv, partials_ptr, (mb or Mailbox(N)).d, peers=ps)}
        if fmt == "csr":
            out["spmv_b200_csr_spmv_fused_async"] = lambda: X.spmv_fused_async(xv, yv, partials_ptr,
                                                                              (ab or Mailbox(N, True)).d, peers=ps)
        return out

    def rejected(fn, what):
        with pytest.raises(N.SpmvError):
            fn()
        torch.cuda.synchronize()
        for t, b in zip((y, partials, buf), before):
            assert bool(torch.equal(t.isnan(), b.isnan())) and bool(torch.equal(t.nan_to_num(), b.nan_to_num())), \
                f"{what}: rejected, but a vector was written"

    for X, fmt in ((c["A"], "csr"), (c["H"], "hll")):
        for bad in (peers(-1), peers(MAX_PEERS + 1), peers(1, 0, M + 1), peers(2, 20, 10), peers(1, -1, 5),
                    peers(MAX_PEERS, 0, M + 5)):
            for name, fn in calls(X, fmt, ps=bad).items():
                rejected(fn, f"{name}: peers count {bad.count}, range [{bad.lo[0]},{bad.hi[0]})")
        for name, fn in calls(X, fmt, partials_ptr=0).items():
            if "mail" in name or "async" in name:
                rejected(fn, f"{name}: NULL partials")
        for field in ("counter", "status") + (("bcounter",) if fmt == "csr" else ()):
            for async_form in ((False, True) if fmt == "csr" else (False,)):
                if field == "bcounter" and not async_form:
                    continue
                m = Mailbox(N, async_form)
                setattr(m.d, field, None)
                name = "spmv_b200_csr_spmv_fused_async" if async_form else f"spmv_b200_{fmt}_spmv_fused_mail"
                rejected(calls(X, fmt, mb=m, ab=m)[name], f"{name}: NULL {field}")
        for world, rank in ((0, 0), (9, 0), (1, 1), (1, -1), (2, 0)):   # world 2: box[1] is NULL
            for async_form in ((False, True) if fmt == "csr" else (False,)):
                m = Mailbox(N, async_form)
                m.d.world, m.d.rank = world, rank
                name = "spmv_b200_csr_spmv_fused_async" if async_form else f"spmv_b200_{fmt}_spmv_fused_mail"
                rejected(calls(X, fmt, mb=m, ab=m)[name], f"{name}: world {world}, rank {rank}")
    m = Mailbox(N, True)
    m.d.num_recv, m.d.recv_from[0] = 1, 3
    rejected(lambda: c["A"].spmv_fused_async(c["xd"], y, partials, m.d), "async: receives from rank 3 of 1")
    m = Mailbox(N, True)
    m.d.send_to[0] = 1
    rejected(lambda: c["A"].spmv_fused_async(c["xd"], y, partials, m.d, peers=peers(1)), "async: sends to rank 1 of 1")
    xw = _t(np.ones(3000))
    for name, fn in calls(wide, "csr", xv=xw).items():
        if "flat" in name or "async" in name:
            rejected(fn, f"{name}: rows above 12")
    for name, fn in calls(longrow, "csr", xv=xw).items():
        if name.endswith("fused") or "mail" in name:
            rejected(fn, f"{name}: a row past the long-row threshold")
    for name, fn in list(calls(empty, "csr", xv=xw).items()) + list(calls(empty_h, "hll", xv=xw).items()):
        if "mail" in name or "async" in name:
            rejected(fn, f"{name}: M = 0")
    # HLL flat has no width limit (one lane sums a row), and accepts every range inside the matrix, empty ones too
    Hw = wide.to_hll()
    yw = _nan(300)
    Hw.spmv_fused_flat(xw, yw)
    assert_y(yw.cpu().numpy(), Ref(checker, wrp, wci, wva, np.ones(300)), None, "spmv_b200_hll_spmv_fused_flat, rows above 12")
    ps = peers(2, M, M)
    c["A"].spmv_fused(c["xd"], _nan(M), peers=ps)
    c["H"].spmv_fused_flat(c["xd"], _nan(M), peers=ps)
    torch.cuda.synchronize()
    assert bool(torch.isnan(buf).all()), "an empty peer range was written"
    for X in (wide, longrow, empty, empty_h, Hw):
        X.close()
