"""Multi-vector products Y = A X (spmv_b200_csr_spmm / spmv_b200_hll_spmm, DeviceCSR.spmm / DeviceHLL.spmm).

Contract (include/spmv_b200.h, SpMM section): X is N x k, Y is M x k, row-major with leading dimensions >= k.
  * CSR rows up to the long-row threshold, and every HLL row: column c of Y is bit for bit the serial loop on column c
    of X (csr_matrix_vector_mult / spmv_hll_serial), with accumulate starting from Y's value (CSR only).
  * CSR long rows: within (len + 2) 2^-53 sum_j |a_ij x_jc| (+ |y0| with accumulate) of the exact sum, identical bits
    from call to call, and the bits of a column independent of k, ldx, ldy and the column's position in X.
  * Only rows < M and columns < k of Y are written.

References: the oracle's serial loops per column, the library's own single-vector products per column and, for sampled
rows of huge matrices, `serial_rows` below (numpy, one product column at a time in index order: acc = acc + v * x with
the multiply and the add rounded separately, which is what the serial loop does).
"""
import ctypes as C

import numpy as np
import pytest

from conftest import GOLDEN, golden_names, load_golden

U53 = 2.0 ** -53
KS = (1, 2, 3, 5, 8, 16, 31, 32, 33, 64, 100)
XCOLS = 105                      # columns of the source block; a slice at column 2 leaves room for k = 100
SENTINEL = np.array([0x7FF8DEADBEEF0001], np.uint64).view(np.float64)[0]  # a NaN with a payload of its own


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def sentinel_bits():
    """The bits of SENTINEL as torch.full stores them on the device."""
    import torch
    return bits(torch.full((1,), SENTINEL, dtype=torch.float64, device="cuda").cpu().numpy())[0]


# ---------------------------------------------------------------------------------------------------
# the sequential per-row reference (numpy)
# ---------------------------------------------------------------------------------------------------
def serial_rows(rp, ci, va, X, rows, Y0=None):
    """Rows `rows` of A X, every column summed sequentially in index order: acc = acc + v * X[col] (numpy rounds the
    multiply and the add separately).  Y0 (len(rows) x k): starting values, as the serial loop with accumulate."""
    X = np.asarray(X, np.float64)
    out = np.zeros((len(rows), X.shape[1]), np.float64) if Y0 is None else np.array(Y0, np.float64, copy=True)
    for i, r in enumerate(rows):
        acc = out[i].copy()
        for j in range(int(rp[r]), int(rp[r + 1])):
            acc = acc + va[j] * X[ci[j]]
        out[i] = acc
    return out


def golden_csr(name):
    g = load_golden(name)
    return int(g["M"]), int(g["N"]), g["row_ptr"].astype(np.int32), g["col_idx"].astype(np.int32), g["values"]


@pytest.mark.parametrize("name", golden_names())
def test_serial_rows_is_the_serial_loop(port, name):
    """The numpy helper equals the oracle's spmv_csr_serial bit for bit, column by column, with and without a start."""
    M, N, rp, ci, va = golden_csr(name)
    rng = np.random.default_rng(7)
    X = np.column_stack([np.ones(N), 1.0 + (np.arange(N) % 7) / 8.0, rng.standard_normal(N), rng.standard_normal(N) * 1e3])
    Y0 = rng.standard_normal((M, X.shape[1]))
    got = serial_rows(rp, ci, va, X, range(M))
    got_acc = serial_rows(rp, ci, va, X, range(M), Y0)
    for c in range(X.shape[1]):
        assert np.array_equal(bits(got[:, c]), bits(port.spmv_csr_serial(rp, ci, va, X[:, c]))), f"{name} column {c}"
        want = port.spmv_csr_serial(rp, ci, va, X[:, c], y=Y0[:, c].copy())
        assert np.array_equal(bits(got_acc[:, c]), bits(want)), f"{name} column {c} with a start"


def test_bad_arguments_without_a_device():
    """Both entry points refuse a NULL handle, a negative k and a leading dimension below k before touching anything
    (the dummy handle / array addresses below are never dereferenced)."""
    from sparsematrixvectormultiplication_b200 import _native as N
    lib = N.lib()
    h, p = C.c_void_p(64), C.c_void_p(4096)
    assert lib.spmv_b200_csr_spmm(None, 4, p, 4, p, 4, 0, None) != 0
    assert lib.spmv_b200_hll_spmm(None, 4, p, 4, p, 4, None) != 0
    assert lib.spmv_b200_csr_spmm(h, -1, p, 4, p, 4, 0, None) != 0
    assert lib.spmv_b200_hll_spmm(h, -1, p, 4, p, 4, None) != 0
    assert lib.spmv_b200_csr_spmm(h, 4, p, 3, p, 4, 0, None) != 0
    assert lib.spmv_b200_hll_spmm(h, 4, p, 3, p, 4, None) != 0
    assert lib.spmv_b200_csr_spmm(h, 4, p, 4, p, 3, 1, None) != 0
    assert lib.spmv_b200_hll_spmm(h, 4, p, 4, p, 3, None) != 0
    assert lib.spmv_b200_csr_spmm(h, 2, None, 4, p, 4, 0, None) != 0
    assert lib.spmv_b200_hll_spmm(h, 2, p, 4, None, 4, None) != 0
    assert lib.spmv_b200_version() >= 101


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    import torch
    from sparsematrixvectormultiplication_b200 import device
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    return device


def random_csr(rng, M, N, lengths):
    """Rows of the given lengths, distinct sorted columns, column 0 and N-1 used when N allows; normal values."""
    lengths = np.minimum(np.asarray(lengths, np.int64), N)
    rp = np.zeros(M + 1, np.int64)
    np.cumsum(lengths, out=rp[1:])
    cols = []
    for i, n in enumerate(lengths):
        c = np.sort(rng.choice(N, size=int(n), replace=False)) if n else np.zeros(0, np.int64)
        cols.append(c)
    ci = np.concatenate(cols).astype(np.int32) if cols else np.zeros(0, np.int32)
    if len(ci) and N > 1:
        first = int(np.argmax(lengths > 0))
        ci[rp[first]] = 0                                    # column 0 ...
        last = M - 1 - int(np.argmax(lengths[::-1] > 0))
        if lengths[last] and ci[rp[last + 1] - 1] != 0:
            ci[rp[last + 1] - 1] = N - 1                     # ... and column N-1 (rows stay sorted and distinct)
    return rp.astype(np.int32), ci, rng.standard_normal(len(ci))


def hll_of(checker, M, N, rp, ci, va):
    from oracle import oracle as O
    rows = np.repeat(np.arange(M, dtype=np.int32), np.diff(rp))
    return checker.coo_to_hll(O.Coo(M, N, len(ci), rows, ci.astype(np.int32), va))


def host_hll(M, N, rp, ci, va):
    from sparsematrixvectormultiplication_b200 import host
    rows = np.repeat(np.arange(M, dtype=np.int32), np.diff(rp))
    return host.convert_to_hll(host.PreMatrix(M, N, rows, ci.astype(np.int32), np.asarray(va, np.float64)))


class Operands:
    """X and Y for one product: 'tight' (ld = k, fresh tensors) or 'slice' (column slices of wider buffers, ld > k).
    Y's block is prefilled with NaN (or Y0), everything else of its buffer with SENTINEL."""

    def __init__(self, Xsrc_d, M, k, layout, Y0=None):
        import torch
        self.k, self.layout = k, layout
        self.xcol = 0 if layout == "tight" else 2
        if layout == "tight":
            self.X = Xsrc_d[:, :k].contiguous()
            self.buf = torch.full((M, k), float("nan"), dtype=torch.float64, device="cuda")
            self.Y = self.buf
        else:
            self.X = Xsrc_d[:, 2:2 + k]
            self.buf = torch.full((M, k + 4), SENTINEL, dtype=torch.float64, device="cuda")
            self.Y = self.buf[:, 1:1 + k]
            self.Y.fill_(float("nan"))
        if Y0 is not None:
            self.Y.copy_(Y0[:, :k])

    def cols(self):
        return slice(self.xcol, self.xcol + self.k)

    def result(self, what):
        """Y's block on the host; asserts that no element outside it changed."""
        buf = self.buf.cpu().numpy()
        if self.layout == "slice":
            outside = np.concatenate([buf[:, :1], buf[:, 1 + self.k:]], axis=1)
            assert np.all(bits(outside) == sentinel_bits()), f"{what}: wrote outside the M x k block"
            return buf[:, 1:1 + self.k]
        return buf


def assert_bitwise(got, want, what):
    bad = np.argwhere(bits(got) != bits(want))
    assert bad.size == 0, f"{what}: {len(bad)} elements differ, first (row, column) {bad[:4].tolist()}: got {got[tuple(bad[0])]}, want {want[tuple(bad[0])]}"


def reference_columns(fn, ncols):
    return np.column_stack([fn(c) for c in range(ncols)])


def check_all_k(dev, A, Hs, M, N, ref, ref_acc, hll_ref, Xsrc, Y0src, what):
    """Every k of KS, both layouts, CSR plain and accumulating, every HLL image: bitwise per column."""
    import torch
    Xd = torch.from_numpy(Xsrc).cuda()
    Y0d = torch.from_numpy(Y0src).cuda()
    for k in KS:
        for layout in ("tight", "slice"):
            tag = f"{what} k={k} {layout}"
            op = Operands(Xd, M, k, layout)
            A.spmm(op.X, op.Y)
            assert_bitwise(op.result(tag), ref[:, op.cols()], tag + " csr")
            op = Operands(Xd, M, k, layout, Y0d[:, op.cols()])
            A.spmm(op.X, op.Y, accumulate=True)
            assert_bitwise(op.result(tag), ref_acc[:, op.cols()], tag + " csr accumulate")
            for hname, H in Hs:
                op = Operands(Xd, M, k, layout)
                H.spmm(op.X, op.Y)
                assert_bitwise(op.result(tag), hll_ref[:, op.cols()], f"{tag} hll {hname}")


def single_vector_columns(fn, Xsrc, M, cols):
    """The library's single-vector product on columns `cols` of Xsrc."""
    import torch
    out = []
    for c in cols:
        x = torch.from_numpy(np.ascontiguousarray(Xsrc[:, c])).cuda()
        y = torch.full((max(M, 1),), float("nan"), dtype=torch.float64, device="cuda")
        fn(x, y)
        out.append(y.cpu().numpy()[:M])
    return np.column_stack(out)


SHAPES = {"M1": (1, 50, [7]), "M31": (31, 300, None), "M33": (33, 300, None), "M257": (257, 1000, None),
          "prime7919": (7919, 3001, None), "N1": (300, 1, None), "nnz0": (100, 80, [0] * 100)}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(SHAPES))
def test_shapes_bitwise(dev, checker, case):
    """Row counts of 1, 31, 33, 257 and 7919, N = 1, no nonzero at all, empty rows, columns 0 and N-1; every k of KS,
    ld = k and ld > k, CSR plain and accumulating, HLL uploaded from the host layout and converted on the device."""
    rng = np.random.default_rng(sum(map(ord, case)))
    M, N, lengths = SHAPES[case]
    if lengths is None:
        lengths = rng.integers(0, 30, M)
        lengths[rng.random(M) < 0.1] = 0                     # empty rows
    rp, ci, va = random_csr(rng, M, N, lengths)
    Xsrc = rng.standard_normal((N, XCOLS))
    Y0src = rng.standard_normal((M, XCOLS))
    ref = reference_columns(lambda c: checker.spmv_csr_serial(rp, ci, va, Xsrc[:, c]), XCOLS)
    ref_acc = reference_columns(lambda c: checker.spmv_csr_serial(rp, ci, va, Xsrc[:, c], y=Y0src[:, c].copy()), XCOLS)
    h = hll_of(checker, M, N, rp, ci, va)
    hll_ref = reference_columns(lambda c: checker.spmv_hll_serial(h, Xsrc[:, c], M), XCOLS)
    if int(rp[-1]) == 0:
        assert not bits(ref).any(), "a matrix without nonzeros gives +0.0"
    A = dev.DeviceCSR.upload(M, N, rp, ci, va)
    Hs = [("from_host", dev.DeviceHLL.from_host(host_hll(M, N, rp, ci, va), M, N)), ("to_hll", A.to_hll())]
    check_all_k(dev, A, Hs, M, N, ref, ref_acc, hll_ref, Xsrc, Y0src, case)
    cols = [0, 2, XCOLS - 1]
    assert_bitwise(single_vector_columns(lambda x, y: A.spmv(x, y, algo=dev.ALGO_ROW), Xsrc, M, cols), ref[:, cols], "spmv ROW")
    assert_bitwise(single_vector_columns(lambda x, y: Hs[1][1].spmv(x, y, slice_kernel="rows"), Xsrc, M, cols),
                   hll_ref[:, cols], "hll spmv rows")


@pytest.mark.gpu
@pytest.mark.parametrize("name", golden_names())
def test_golden_fixtures_bitwise(dev, checker, name):
    """Every golden fixture: CSR against the serial loop per column; the HLL image uploaded from convert_to_hll against
    the library's own lane-per-row product (the bits of spmv_hll_serial, test_gpu_parity.py) per column."""
    from sparsematrixvectormultiplication_b200 import host
    M, N, rp, ci, va = golden_csr(name)
    rng = np.random.default_rng(11)
    Xsrc = rng.standard_normal((N, XCOLS))
    Y0src = rng.standard_normal((M, XCOLS))
    ref = reference_columns(lambda c: checker.spmv_csr_serial(rp, ci, va, Xsrc[:, c]), XCOLS)
    ref_acc = reference_columns(lambda c: checker.spmv_csr_serial(rp, ci, va, Xsrc[:, c], y=Y0src[:, c].copy()), XCOLS)
    pre = host.read_matrix_market(GOLDEN / "mtx" / f"{name}.mtx")
    A = dev.DeviceCSR.upload(M, N, rp, ci, va)
    H = dev.DeviceHLL.from_host(host.convert_to_hll(pre))
    hll_ref = single_vector_columns(lambda x, y: H.spmv(x, y, slice_kernel="rows"), Xsrc, M, range(XCOLS))
    check_all_k(dev, A, [("from_host", H)], M, N, ref, ref_acc, hll_ref, Xsrc, Y0src, name)


# ---------------------------------------------------------------------------------------------------
# long rows
# ---------------------------------------------------------------------------------------------------
def exact_bound(rp, ci, va, X, Y0=None):
    """(near-exact sums in long double, the allowed error) per element: (len + 2) 2^-53 (|y0| + sum_j |a_ij x_jc|)."""
    M, k = len(rp) - 1, X.shape[1]
    exact = np.zeros((M, k), np.longdouble)
    S = np.zeros((M, k), np.float64)
    Xl = X.astype(np.longdouble)
    for r in range(M):
        lo, hi = int(rp[r]), int(rp[r + 1])
        prods = va[lo:hi, None].astype(np.longdouble) * Xl[ci[lo:hi]]
        exact[r] = prods.sum(axis=0)
        S[r] = np.abs(va[lo:hi, None] * X[ci[lo:hi]]).sum(axis=0)
    if Y0 is not None:
        exact += Y0.astype(np.longdouble)
        S += np.abs(Y0)
    lens = np.diff(rp.astype(np.int64)).astype(np.float64)[:, None]
    return exact, (lens + 2.0) * U53 * S


def check_long(dev, A, rp, ci, va, Xsrc, Y0src, threshold, what):
    import torch
    M = len(rp) - 1
    lens = np.diff(rp.astype(np.int64))
    short, long_ = lens <= threshold, lens > threshold
    assert long_.any() and A.info().num_long_rows == int(long_.sum())
    Xd, Y0d = torch.from_numpy(Xsrc).cuda(), torch.from_numpy(Y0src).cuda()
    k = 33
    for acc in (False, True):
        Y0 = Y0src[:, 2:2 + k] if acc else None
        exact, bound = exact_bound(rp, ci, va, Xsrc[:, 2:2 + k], Y0)
        ref = serial_rows(rp, ci, va, Xsrc[:, 2:2 + k], np.nonzero(short)[0], None if Y0 is None else Y0[short])
        runs = []
        for rep in range(2):
            op = Operands(Xd, M, k, "slice", Y0d[:, 2:2 + k] if acc else None)
            A.spmm(op.X, op.Y, accumulate=acc)
            runs.append(op.result(what).copy())
        tag = f"{what}{' accumulate' if acc else ''}"
        assert_bitwise(runs[1], runs[0], tag + ": two calls")
        y = runs[0]
        assert_bitwise(y[short], ref, tag + ": rows up to the threshold")
        err = np.abs(y[long_].astype(np.longdouble) - exact[long_]).astype(np.float64)
        assert np.all(err <= bound[long_]), f"{tag}: split rows outside the bound, worst ratio {np.max(err / np.maximum(bound[long_], 1e-300))}"
        # the same columns from calls of other widths, at other positions in X and other leading dimensions
        for kk, start in ((1, 2), (1, 20), (8, 2), (8, 27), (33, 2)):
            for layout in ("tight", "slice"):
                if layout == "slice":
                    Xv = Xd[:, start:start + kk]
                    buf = torch.full((M, kk + 9), SENTINEL, dtype=torch.float64, device="cuda")
                    Yv = buf[:, 5:5 + kk]
                    if acc:
                        Yv.copy_(Y0d[:, start:start + kk])
                    A.spmm(Xv, Yv, accumulate=acc)
                    got = Yv.cpu().numpy()
                else:
                    Xv = Xd[:, start:start + kk].contiguous()
                    Yv = Y0d[:, start:start + kk].clone() if acc else torch.full((M, kk), float("nan"), dtype=torch.float64, device="cuda")
                    A.spmm(Xv, Yv, accumulate=acc)
                    got = Yv.cpu().numpy()
                want = y[:, start - 2:start - 2 + kk]
                assert_bitwise(got, want, f"{tag}: columns {start}..{start + kk - 1} with k={kk} ({layout})")


@pytest.mark.gpu
def test_long_rows(dev):
    """Rows of 513, 8192, 8193 and 20 000 nonzeros among short ones (default threshold 512): split rows within the bound,
    every other row bitwise, two calls bitwise equal, and a column's bits the same whatever k, position and ld."""
    rng = np.random.default_rng(513)
    M, N = 64, 24000
    lengths = rng.integers(0, 60, M)
    lengths[[3, 10, 11, 40]] = [513, 8192, 8193, 20000]
    lengths[50] = 512
    rp, ci, va = random_csr(rng, M, N, lengths)
    Xsrc = rng.standard_normal((N, 40))
    Y0src = rng.standard_normal((M, 40))
    A = dev.DeviceCSR.upload(M, N, rp, ci, va)
    assert A.info().long_threshold == 512
    check_long(dev, A, rp, ci, va, Xsrc, Y0src, 512, "long rows")


@pytest.mark.gpu
def test_long_rows_after_replan(dev):
    """replan(long_threshold=16) on a random irregular matrix: every row above 16 nonzeros takes the fragment path."""
    rng = np.random.default_rng(16)
    M, N = 3000, 5000
    lengths = rng.choice([0, 1, 5, 16, 17, 40, 100, 700], size=M)
    rp, ci, va = random_csr(rng, M, N, lengths)
    Xsrc = rng.standard_normal((N, 40))
    Y0src = rng.standard_normal((M, 40))
    A = dev.DeviceCSR.upload(M, N, rp, ci, va)
    A.replan(long_threshold=16)
    check_long(dev, A, rp, ci, va, Xsrc, Y0src, 16, "replan(long_threshold=16)")
    A.replan(long_threshold=512)                             # the partials buffer follows the plan
    check_long(dev, A, rp, ci, va, Xsrc, Y0src, 512, "replan(long_threshold=512)")


# ---------------------------------------------------------------------------------------------------
# HLL images
# ---------------------------------------------------------------------------------------------------
def hack_runs(rng, widths, hacks_per_run, tail_rows):
    """Row lengths whose hacks come in runs of equal width (the regular-image case), last hack short."""
    lengths = []
    for w in widths:
        for _ in range(hacks_per_run):
            row = rng.integers(0, w + 1, 32)
            row[rng.integers(0, 32)] = w
            lengths.extend(row.tolist())
    return np.array(lengths[: len(lengths) - 32 + tail_rows], np.int64)


@pytest.mark.gpu
@pytest.mark.parametrize("image", ["lap2d", "runs7", "runs9", "wide", "tail"])
def test_hll_images(dev, checker, image):
    """lap2d, images with seven and nine runs of equal hack width, wide hacks (MAXNZ 33 and above: the slice-kernel case
    of the single-vector product) and M off a multiple of 32: every column bit for bit spmv_hll_serial."""
    from sparsematrixvectormultiplication_b200 import synth
    rng = np.random.default_rng(sum(map(ord, image)))
    if image == "lap2d":
        rp, ci, va = synth.lap2d_csr(48)
        M = N = 48 * 48
    else:
        if image == "runs7":
            lengths = hack_runs(rng, [3, 5, 2, 7, 4, 6, 1], 3, 32)
        elif image == "runs9":
            lengths = hack_runs(rng, [5, 6, 2, 9, 4, 12, 3, 8, 6], 2, 32)
        elif image == "wide":
            lengths = hack_runs(rng, [33, 40, 100, 7, 64], 2, 19)
        else:
            lengths = rng.integers(0, 20, 32 * 9 + 13)
        M, N = len(lengths), 700
        rp, ci, va = random_csr(rng, M, N, lengths)
    rp, ci = np.asarray(rp, np.int32), np.asarray(ci, np.int32)
    Xsrc = rng.standard_normal((N, XCOLS))
    h = hll_of(checker, M, N, rp, ci, va)
    hll_ref = reference_columns(lambda c: checker.spmv_hll_serial(h, Xsrc[:, c], M), XCOLS)
    A = dev.DeviceCSR.upload(M, N, rp, ci, va)
    H = A.to_hll()
    if image == "wide":
        assert H.info().max_maxnz >= 33
    H2 = dev.DeviceHLL.from_host(host_hll(M, N, rp, ci, va), M, N)
    import torch
    Xd = torch.from_numpy(Xsrc).cuda()
    for k in (1, 2, 3, 8, 16, 32, 33, 100):
        for layout in ("tight", "slice"):
            for hname, img in (("to_hll", H), ("from_host", H2)):
                op = Operands(Xd, M, k, layout)
                img.spmm(op.X, op.Y)
                assert_bitwise(op.result(image), hll_ref[:, op.cols()], f"{image} {hname} k={k} {layout}")
    assert_bitwise(single_vector_columns(lambda x, y: H.spmv(x, y, slice_kernel="rows"), Xsrc, M, [0, 50]),
                   hll_ref[:, [0, 50]], f"{image}: spmv rows")


# ---------------------------------------------------------------------------------------------------
# past 2^31 elements
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_offsets_past_2_31_elements(dev):
    """lap2d 4096^2 with k = 4 and ldx = ldy = 136: row * ld passes 2^31 for the last 1.0 M rows (about 37 GB).  Sampled
    rows on both sides of the crossing, and at both ends, bitwise against serial_rows; the ldy gap of those rows untouched."""
    import torch
    from sparsematrixvectormultiplication_b200 import synth
    n, k, ld = 4096, 4, 136
    M = n * n
    cross = (1 << 31) // ld
    assert M - cross > 980_000
    rng = np.random.default_rng(2 ** 31)
    X4 = rng.standard_normal((M, k))
    Xbuf = torch.full((M, ld), SENTINEL, dtype=torch.float64, device="cuda")
    Xbuf[:, :k].copy_(torch.from_numpy(X4))
    windows = [(0, 600), (cross - 3000, cross + 3000), (M - 3000, M)]
    A = dev.DeviceCSR.synth(dev.SYNTH_LAP2D, n)
    formats = [("csr", A), ("hll", A.to_hll())]
    for fname, Mat in formats:
        Ybuf = torch.full((M, ld), SENTINEL, dtype=torch.float64, device="cuda")
        Mat.spmm(Xbuf[:, :k], Ybuf[:, :k])
        torch.cuda.synchronize()
        for lo, hi in windows:
            rp, ci, va = synth.lap2d_csr(n, lo, hi)
            want = serial_rows(rp, ci, va, X4, range(hi - lo))
            got = Ybuf[lo:hi].cpu().numpy()
            assert_bitwise(got[:, :k], want, f"{fname} rows {lo}..{hi}")
            assert np.all(bits(got[:, k:]) == sentinel_bits()), f"{fname}: gap written"
        del Ybuf
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------
# validation
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_wrapper_validation(dev):
    """Every bad operand raises ValueError before a launch, and Y is left as it was."""
    import torch
    from sparsematrixvectormultiplication_b200 import _native as N
    rng = np.random.default_rng(3)
    M = N_ = 200
    rp, ci, va = random_csr(rng, M, N_, rng.integers(0, 9, M))
    A = dev.DeviceCSR.upload(M, N_, rp, ci, va)
    H = A.to_hll()
    k = 4
    cuda = dict(dtype=torch.float64, device="cuda")
    X = torch.randn(N_, k, **cuda)
    Ybuf = torch.full((M, 2 * k), SENTINEL, **cuda)
    before = bits(Ybuf.cpu().numpy()).copy()
    Y = Ybuf[:, :k]
    Xstrided = torch.empty(3 * N_ + k, **cuda).as_strided((N_, k), (3, 1))  # row stride 3 < k
    bad = {
        "float32 X": (X.float(), Y), "float32 Y": (X, Ybuf[:, :k].float()),
        "CPU X": (X.cpu(), Y), "CPU Y": (X, torch.zeros(M, k, dtype=torch.float64)),
        "1-D X": (X[:, 0], Y[:, :1]), "3-D Y": (X, Ybuf.view(M, 2, k)[:, :1, :]),
        "X rows": (torch.randn(N_ + 1, k, **cuda), Y), "Y rows": (X, torch.full((M - 1, 2 * k), 0.0, **cuda)[:, :k]),
        "column counts": (X[:, :3], Y),
        "X column stride": (torch.randn(k, N_, **cuda).t(), Y), "Y column stride": (X, Ybuf[:, ::2]),
        "X row stride": (Xstrided, Y),
        "Y = X": (Ybuf[:, :k], Ybuf[:, :k]), "Y overlaps X": (Ybuf[:, 2:2 + k], Ybuf[:, :k]),
    }
    for what, (Xb, Yb) in bad.items():
        for name, call in (("csr", lambda: A.spmm(Xb, Yb)), ("csr accumulate", lambda: A.spmm(Xb, Yb, accumulate=True)),
                           ("hll", lambda: H.spmm(Xb, Yb))):
            with pytest.raises(ValueError):
                call()
            torch.cuda.synchronize()
            assert np.array_equal(bits(Ybuf.cpu().numpy()), before), f"{what} ({name}): Y was written"
    # interleaved column slices of one buffer do not overlap: accepted
    Z = torch.full((N_, 2 * k), 0.0, **cuda)
    Z[:, :k] = X
    A.spmm(Z[:, :k], Z[:, k:])
    H.spmm(Z[:, :k], Z[:, k:])
    # k = 0 and an empty Y are no-ops; a size-1 dimension's stride does not matter
    A.spmm(torch.empty(N_, 0, **cuda), torch.empty(M, 0, **cuda))
    H.spmm(torch.empty(N_, 0, **cuda), torch.empty(M, 0, **cuda))
    col = torch.randn(N_, 1, **cuda)
    yc = torch.full((M, 1), float("nan"), **cuda)
    A.spmm(col.as_strided((N_, 1), (1, 7)), yc.as_strided((M, 1), (1, 3)))
    y1 = torch.full((M,), float("nan"), **cuda)
    A.spmv(col[:, 0].contiguous(), y1, algo=dev.ALGO_ROW)
    assert np.array_equal(bits(yc[:, 0].cpu().numpy()), bits(y1.cpu().numpy()))
    # the C layer on a real handle: negative k, ld < k, NULL arrays return SPMV_B200_ERR_INVALID and write nothing
    lib, s = N.lib(), C.c_void_p(torch.cuda.current_stream().cuda_stream)
    px, py = C.c_void_p(X.data_ptr()), C.c_void_p(Ybuf.data_ptr())
    for rc in (lib.spmv_b200_csr_spmm(A._h, -1, px, k, py, 2 * k, 0, s), lib.spmv_b200_csr_spmm(A._h, k, px, k - 1, py, 2 * k, 0, s),
               lib.spmv_b200_csr_spmm(A._h, k, px, k, py, k - 1, 0, s), lib.spmv_b200_csr_spmm(A._h, k, None, k, py, 2 * k, 0, s),
               lib.spmv_b200_hll_spmm(H._h, -1, px, k, py, 2 * k, s), lib.spmv_b200_hll_spmm(H._h, k, px, k - 1, py, 2 * k, s),
               lib.spmv_b200_hll_spmm(H._h, k, px, k, py, k - 1, s), lib.spmv_b200_hll_spmm(H._h, k, px, k, None, 2 * k, s)):
        assert rc == -1
    torch.cuda.synchronize()
    assert np.array_equal(bits(Ybuf.cpu().numpy()), before), "the C layer wrote Y on an invalid call"
