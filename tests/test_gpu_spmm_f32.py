"""Multi-vector products on the fp32 copy (spmv_b200_csr_spmm_f32 / spmv_b200_hll_spmm_f32, DeviceCSR.spmm_f32 /
DeviceHLL.spmm_f32) against the exact reference of the fp32 contract.

Contract (include/spmv_b200.h, fp32 section): X, Y and the values are float; products and sums in double, one rounding
to float per element.  Per column c, with vw = float64(float32(values)) and xw = float64(X[:, c]):
  * CSR rows up to the long-row threshold and every HLL row (hacks of any width): float32 of the serial fp64 loop, the
    EXACT assertion of test_gpu_fp32.py; CSR with accumulate starts from float64(Y[:, c]).  CSR columns are also bit for
    bit spmv_f32(ALGO_ROW) on that column.
  * CSR long rows: the BOUNDED assertion of test_gpu_fp32.py, identical bits from call to call and whatever k, ldx, ldy
    or the column's position in X.

`ref32_columns` below is the numpy form of that reference for all columns at once (serial_rows of test_gpu_spmm.py on the
widened operands, rounded to float); test_ref32_columns_is_the_exact_reference ties it to Ref of test_gpu_fp32.py.
"""
import ctypes as C

import numpy as np
import pytest

from conftest import GOLDEN, golden_names
from test_gpu_fp32 import Ref, adversarial_matrix, assert_bounded, assert_exact, hll_reference, u32, widen
from test_gpu_spmm import KS, SHAPES, XCOLS, golden_csr, hack_runs, host_hll, random_csr, serial_rows

SENTINEL32 = 0x7FDEAD01            # bits of a float NaN with a payload of its own, written into the ldy gap


# ---------------------------------------------------------------------------------------------------
# the reference
# ---------------------------------------------------------------------------------------------------
def ref32_columns(rp, ci, va, X32, Y0=None, rows=None):
    """float32 of the serial fp64 loop over the widened values and columns of X32 (and widened Y0 as the start)."""
    rows = range(len(rp) - 1) if rows is None else rows
    Y0w = None if Y0 is None else np.asarray(Y0, np.float32).astype(np.float64)
    return serial_rows(rp, ci, widen(va), np.asarray(X32, np.float32).astype(np.float64), rows, Y0w).astype(np.float32)


def hll_columns(checker, rp, ci, va, X32, M, N):
    """spmv_hll_serial per column on the oracle's HLL image with AS widened, rounded to float (hll_reference of
    test_gpu_fp32.py, which also asserts that it equals the CSR reference on column 0)."""
    h = hll_reference(checker, rp, ci, va, X32[:, 0], M, N, Ref(checker, rp, ci, va, X32[:, 0]))
    return np.column_stack([checker.spmv_hll_serial(h, X32[:, c].astype(np.float64), M).astype(np.float32)
                            for c in range(X32.shape[1])])


def image_columns(checker, H, X32, M):
    """spmv_hll_serial per column on the device image itself (downloaded in the reference layout, AS widened)."""
    from oracle import oracle as O
    rows, maxnz, offset, JA, AS = H.download().flat()
    h = O.Hll(len(rows), rows, maxnz, offset, JA, widen(AS))
    return np.column_stack([checker.spmv_hll_serial(h, X32[:, c].astype(np.float64), M).astype(np.float32)
                            for c in range(X32.shape[1])])


def assert_bitwise32(got, want, what):
    bad = np.argwhere(u32(got) != u32(want))
    assert bad.size == 0, (f"{what}: {len(bad)} elements differ, first (row, column) {bad[:4].tolist()}: "
                           f"got {got[tuple(bad[0])]}, want {want[tuple(bad[0])]}")


def random_x32(rng, rows, cols):
    X = rng.standard_normal((rows, cols)).astype(np.float32)
    X[:, 1] = 1.0 + (np.arange(rows) % 7) / 8.0            # the ramp of the golden fixtures
    return X


@pytest.mark.parametrize("name", golden_names())
def test_ref32_columns_is_the_exact_reference(checker, name):
    """No GPU: the numpy per-column reference equals Ref(...).ref32 of test_gpu_fp32.py on every golden fixture, with and
    without a start, bit for bit."""
    M, N, rp, ci, va = golden_csr(name)
    rng = np.random.default_rng(32)
    X32 = random_x32(rng, N, 4)
    X32[:, 3] *= 1e3
    Y0 = rng.standard_normal((M, 4)).astype(np.float32)
    got, got_acc = ref32_columns(rp, ci, va, X32), ref32_columns(rp, ci, va, X32, Y0)
    for c in range(4):
        assert np.array_equal(u32(got[:, c]), u32(Ref(checker, rp, ci, va, X32[:, c]).ref32)), f"{name} column {c}"
        assert np.array_equal(u32(got_acc[:, c]), u32(Ref(checker, rp, ci, va, X32[:, c], Y0[:, c]).ref32)), \
            f"{name} column {c} with a start"


def test_bad_arguments_without_a_device():
    """Both fp32 entry points refuse a NULL handle, a negative k, a leading dimension below k and NULL arrays before
    touching anything (the dummy handle / array addresses are never dereferenced)."""
    from sparsematrixvectormultiplication_b200 import _native as N
    lib = N.lib()
    h, p = C.c_void_p(64), C.c_void_p(4096)
    for csr, hll in (((None, 4, p, 4, p, 4, 0, None), (None, 4, p, 4, p, 4, None)),
                     ((h, -1, p, 4, p, 4, 0, None), (h, -1, p, 4, p, 4, None)),
                     ((h, 4, p, 3, p, 4, 0, None), (h, 4, p, 3, p, 4, None)),
                     ((h, 4, p, 4, p, 3, 1, None), (h, 4, p, 4, p, 3, None)),
                     ((h, 2, None, 4, p, 4, 0, None), (h, 2, None, 4, p, 4, None)),
                     ((h, 2, p, 4, None, 4, 0, None), (h, 2, p, 4, None, 4, None))):
        assert lib.spmv_b200_csr_spmm_f32(*csr) == -1
        assert lib.spmv_b200_hll_spmm_f32(*hll) == -1
    assert lib.spmv_b200_version() >= 105


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


def sentinel_block(rows, cols):
    import torch
    buf = torch.zeros((rows, cols), dtype=torch.float32, device="cuda")
    buf.view(torch.int32).fill_(SENTINEL32)
    return buf


class Operands32:
    """The layouts of test_gpu_spmm.Operands in float32: 'tight' (ld = k) or 'slice' (column slices of wider buffers,
    ld > k); Y's block prefilled with NaN (or Y0), the rest of its buffer with the SENTINEL32 bits."""

    def __init__(self, Xsrc_d, M, k, layout, Y0=None):
        import torch
        self.k, self.layout = k, layout
        self.xcol = 0 if layout == "tight" else 2
        if layout == "tight":
            self.X = Xsrc_d[:, :k].contiguous()
            self.buf = torch.full((M, k), float("nan"), dtype=torch.float32, device="cuda")
            self.Y = self.buf
        else:
            self.X = Xsrc_d[:, 2:2 + k]
            self.buf = sentinel_block(M, k + 4)
            self.Y = self.buf[:, 1:1 + k]
            self.Y.fill_(float("nan"))
        if Y0 is not None:
            self.Y.copy_(Y0[:, :k])

    def cols(self):
        return slice(self.xcol, self.xcol + self.k)

    def result(self, what):
        buf = self.buf.cpu().numpy()
        if self.layout == "slice":
            outside = np.concatenate([buf[:, :1], buf[:, 1 + self.k:]], axis=1)
            assert np.all(u32(outside) == SENTINEL32), f"{what}: wrote outside the M x k block"
            return buf[:, 1:1 + self.k]
        return buf


def check_all_k(A, Hs, M, ref, ref_acc, hll_ref, X32, Y0, what):
    """Every k, both layouts, CSR plain and accumulating, every HLL image: bitwise per column."""
    import torch
    Xd, Y0d = torch.from_numpy(X32).cuda(), torch.from_numpy(Y0).cuda()
    for k in KS:
        for layout in ("tight", "slice"):
            tag = f"{what} k={k} {layout}"
            op = Operands32(Xd, M, k, layout)
            A.spmm_f32(op.X, op.Y)
            assert_bitwise32(op.result(tag), ref[:, op.cols()], tag + " csr")
            op = Operands32(Xd, M, k, layout, Y0d[:, op.cols()])
            A.spmm_f32(op.X, op.Y, accumulate=True)
            assert_bitwise32(op.result(tag), ref_acc[:, op.cols()], tag + " csr accumulate")
            for hname, H in Hs:
                op = Operands32(Xd, M, k, layout)
                H.spmm_f32(op.X, op.Y)
                assert_bitwise32(op.result(tag), hll_ref[:, op.cols()], f"{tag} hll {hname}")


def spmv_f32_columns(A, algo, X32, M, cols):
    import torch
    out = []
    for c in cols:
        x = torch.from_numpy(np.ascontiguousarray(X32[:, c])).cuda()
        y = torch.full((max(M, 1),), float("nan"), dtype=torch.float32, device="cuda")
        A.spmv_f32(x, y, algo=algo)
        out.append(y.cpu().numpy()[:M])
    return np.column_stack(out)


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(SHAPES))
def test_shapes_exact(dev, checker, case):
    """The shapes of test_gpu_spmm.py (M = 1, 31, 33, 257, 7919, N = 1, no nonzero, empty rows, columns 0 and N-1): every
    k, ld = k and ld > k, CSR plain and accumulating, HLL uploaded and converted; CSR columns also spmv_f32(ALGO_ROW)."""
    rng = np.random.default_rng(sum(map(ord, case)) + 32)
    M, N, lengths = SHAPES[case]
    if lengths is None:
        lengths = rng.integers(0, 30, M)
        lengths[rng.random(M) < 0.1] = 0
    rp, ci, va = random_csr(rng, M, N, lengths)
    X32 = random_x32(rng, N, XCOLS)
    Y0 = rng.standard_normal((M, XCOLS)).astype(np.float32)
    ref, ref_acc = ref32_columns(rp, ci, va, X32), ref32_columns(rp, ci, va, X32, Y0)
    hll_ref = hll_columns(checker, rp, ci, va, X32, M, N)
    assert np.array_equal(u32(hll_ref), u32(ref)), "the HLL and CSR references differ"
    if int(rp[-1]) == 0:
        assert not u32(ref).any(), "a matrix without nonzeros gives +0.0"
    A = dev.DeviceCSR.upload(M, N, rp, ci, va).enable_f32()
    Hs = [("from_host", dev.DeviceHLL.from_host(host_hll(M, N, rp, ci, va), M, N).enable_f32()),
          ("to_hll", A.to_hll().enable_f32())]
    check_all_k(A, Hs, M, ref, ref_acc, hll_ref, X32, Y0, case)
    cols = [0, 2, XCOLS - 1]
    assert_bitwise32(spmv_f32_columns(A, dev.ALGO_ROW, X32, M, cols), ref[:, cols], "spmv_f32 ROW")


@pytest.mark.gpu
@pytest.mark.parametrize("name", golden_names())
def test_golden_fixtures_exact(dev, checker, name):
    """Every golden fixture: CSR (plain, accumulating, spmv_f32 ROW per column) and the HLL image of convert_to_hll,
    against spmv_hll_serial on that image (duplicates may sit in other slots than in the CSR arrays)."""
    from sparsematrixvectormultiplication_b200 import host
    M, N, rp, ci, va = golden_csr(name)
    rng = np.random.default_rng(33)
    X32 = random_x32(rng, N, XCOLS)
    Y0 = rng.standard_normal((M, XCOLS)).astype(np.float32)
    ref, ref_acc = ref32_columns(rp, ci, va, X32), ref32_columns(rp, ci, va, X32, Y0)
    A = dev.DeviceCSR.upload(M, N, rp, ci, va).enable_f32()
    H = dev.DeviceHLL.from_host(host.convert_to_hll(host.read_matrix_market(GOLDEN / "mtx" / f"{name}.mtx"))).enable_f32()
    check_all_k(A, [("from_host", H)], M, ref, ref_acc, image_columns(checker, H, X32, M), X32, Y0, name)
    assert_bitwise32(spmv_f32_columns(A, dev.ALGO_ROW, X32, M, [0, 50]), ref[:, [0, 50]], f"{name}: spmv_f32 ROW")


# ---------------------------------------------------------------------------------------------------
# adversarial rows: arithmetic in float, products rounded to float or flushed subnormals cannot pass
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_adversarial_rows_exact(dev, checker):
    """The rows of adversarial_matrix (cancellation, float overflow, float subnormals, random cancellation; the matrix of
    test_gpu_fp32.py::test_the_reference_catches_float_arithmetic, which shows on the CPU that float arithmetic fails
    there) in several columns of X -- x, -x, 2x (the special values keep their effect) and x with its random part
    permuted -- at positions in the first and the second column tile: CSR (plain, accumulating) and HLL, EXACT."""
    import torch
    rng = np.random.default_rng(31)
    M, N = 4000, 3000
    rp, ci, va, x32, kinds = adversarial_matrix(rng, M, N, rng.integers(0, 41, M))
    perm = x32.copy()
    perm[24:] = rng.permutation(perm[24:])
    variants = [x32, -x32, x32 * np.float32(2), perm]
    A = dev.DeviceCSR.upload(M, N, rp, ci, va).enable_f32()
    H = A.to_hll().enable_f32()
    assert H.info().max_maxnz > 12                           # wide hacks: spmv_f32 would take the slice kernel here
    for k in (4, 37):
        X32 = np.column_stack([variants[c % 4] for c in range(k)])
        Y0 = rng.standard_normal((M, k)).astype(np.float32)
        Xd = torch.from_numpy(X32).cuda()
        for fmt, call, acc in (("csr", lambda X, Y: A.spmm_f32(X, Y), False),
                               ("csr accumulate", lambda X, Y: A.spmm_f32(X, Y, accumulate=True), True),
                               ("hll", lambda X, Y: H.spmm_f32(X, Y), False)):
            Y = torch.from_numpy(Y0).cuda() if acc else torch.full((M, k), float("nan"), dtype=torch.float32, device="cuda")
            call(Xd, Y)
            y = Y.cpu().numpy()
            for c in range(k):
                assert_exact(y[:, c], Ref(checker, rp, ci, va, X32[:, c], Y0[:, c] if acc else None), f"{fmt} k={k} column {c}")
    hll_reference(checker, rp, ci, va, x32, M, N, Ref(checker, rp, ci, va, x32))


# ---------------------------------------------------------------------------------------------------
# long rows
# ---------------------------------------------------------------------------------------------------
def check_long(dev, A, rp, ci, va, checker, X32, Y0, threshold, what):
    import torch
    M = len(rp) - 1
    lens = np.diff(rp.astype(np.int64))
    short, long_ = lens <= threshold, lens > threshold
    assert long_.any() and A.info().num_long_rows == int(long_.sum())
    Xd, Y0d = torch.from_numpy(X32).cuda(), torch.from_numpy(Y0).cuda()
    k = 33
    for acc in (False, True):
        runs = []
        for rep in range(2):
            op = Operands32(Xd, M, k, "slice", Y0d[:, 2:2 + k] if acc else None)
            A.spmm_f32(op.X, op.Y, accumulate=acc)
            runs.append(op.result(what).copy())
        tag = f"{what}{' accumulate' if acc else ''}"
        assert_bitwise32(runs[1], runs[0], tag + ": two calls")
        y = runs[0]
        for c in range(k):
            r = Ref(checker, rp, ci, va, X32[:, 2 + c], Y0[:, 2 + c] if acc else None)
            assert_exact(y[:, c], r, f"{tag} column {c}: rows up to the threshold", rows=short)
            assert_bounded(y[long_, c], _rows(r, long_), f"{tag} column {c}: split rows")
        # the same columns from calls of other widths, at other positions in X and other leading dimensions
        for kk, start in ((1, 2), (1, 20), (8, 2), (8, 27), (33, 2)):
            for layout in ("tight", "slice"):
                if layout == "slice":
                    Xv = Xd[:, start:start + kk]
                    buf = sentinel_block(M, kk + 9)
                    Yv = buf[:, 5:5 + kk]
                    if acc:
                        Yv.copy_(Y0d[:, start:start + kk])
                else:
                    Xv = Xd[:, start:start + kk].contiguous()
                    Yv = Y0d[:, start:start + kk].clone() if acc else torch.full((M, kk), float("nan"), dtype=torch.float32, device="cuda")
                A.spmm_f32(Xv, Yv, accumulate=acc)
                assert_bitwise32(Yv.cpu().numpy(), y[:, start - 2:start - 2 + kk],
                                 f"{tag}: columns {start}..{start + kk - 1} with k={kk} ({layout})")


def _rows(r, mask):
    """Ref restricted to the rows of a boolean mask."""
    out = object.__new__(Ref)
    out.y64, out.ref32, out.S, out.lens = r.y64[mask], r.ref32[mask], r.S[mask], r.lens[mask]
    return out


@pytest.mark.gpu
def test_long_rows(dev, checker):
    """Rows of 513, 8192, 8193 and 20 000 nonzeros among short ones (default threshold 512): split rows BOUNDED, every
    other row EXACT, two calls bitwise equal, a column's bits the same whatever k, position and ld."""
    rng = np.random.default_rng(514)
    M, N = 64, 24000
    lengths = rng.integers(0, 60, M)
    lengths[[3, 10, 11, 40]] = [513, 8192, 8193, 20000]
    lengths[50] = 512
    rp, ci, va = random_csr(rng, M, N, lengths)
    X32 = random_x32(rng, N, 40)
    Y0 = rng.standard_normal((M, 40)).astype(np.float32)
    A = dev.DeviceCSR.upload(M, N, rp, ci, va).enable_f32()
    assert A.info().long_threshold == 512
    check_long(dev, A, rp, ci, va, checker, X32, Y0, 512, "long rows")


@pytest.mark.gpu
def test_long_rows_after_replan(dev, checker):
    """replan(long_threshold=16) on a random irregular matrix, then back to 512: the fp32 product follows the plan."""
    rng = np.random.default_rng(17)
    M, N = 3000, 5000
    lengths = rng.choice([0, 1, 5, 16, 17, 40, 100, 700], size=M)
    rp, ci, va = random_csr(rng, M, N, lengths)
    X32 = random_x32(rng, N, 40)
    Y0 = rng.standard_normal((M, 40)).astype(np.float32)
    A = dev.DeviceCSR.upload(M, N, rp, ci, va).enable_f32()
    A.replan(long_threshold=16)
    check_long(dev, A, rp, ci, va, checker, X32, Y0, 16, "replan(long_threshold=16)")
    A.replan(long_threshold=512)
    check_long(dev, A, rp, ci, va, checker, X32, Y0, 512, "replan(long_threshold=512)")


# ---------------------------------------------------------------------------------------------------
# HLL images
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("image", ["lap2d", "runs7", "runs9", "wide13", "wide", "tail"])
def test_hll_images(dev, checker, image):
    """lap2d (a regular image), seven and nine runs of equal hack width, hacks wider than 12 (and than 32) and M off a
    multiple of 32: every column EXACT, for the image converted on the device and the one uploaded from the host."""
    import torch
    from sparsematrixvectormultiplication_b200 import synth
    rng = np.random.default_rng(sum(map(ord, image)) + 32)
    if image == "lap2d":
        rp, ci, va = synth.lap2d_csr(48)
        va = va * rng.uniform(0.5, 1.5, va.size)             # values off the float grid: the storage rounding matters
        M = N = 48 * 48
    else:
        lengths = {"runs7": lambda: hack_runs(rng, [3, 5, 2, 7, 4, 6, 1], 3, 32),
                   "runs9": lambda: hack_runs(rng, [5, 6, 2, 9, 4, 12, 3, 8, 6], 2, 32),
                   "wide13": lambda: hack_runs(rng, [13, 20, 5, 16], 2, 32),
                   "wide": lambda: hack_runs(rng, [33, 40, 100, 7, 64], 2, 19),
                   "tail": lambda: rng.integers(0, 20, 32 * 9 + 13)}[image]()
        M, N = len(lengths), 700
        rp, ci, va = random_csr(rng, M, N, lengths)
    rp, ci = np.asarray(rp, np.int32), np.asarray(ci, np.int32)
    X32 = random_x32(rng, N, XCOLS)
    hll_ref = hll_columns(checker, rp, ci, va, X32, M, N)
    A = dev.DeviceCSR.upload(M, N, rp, ci, va)
    H = A.to_hll().enable_f32()
    if image.startswith("wide"):
        assert H.info().max_maxnz > 12
    H2 = dev.DeviceHLL.from_host(host_hll(M, N, rp, ci, va), M, N).enable_f32()
    Xd = torch.from_numpy(X32).cuda()
    for k in (1, 2, 3, 8, 16, 32, 33, 100):
        for layout in ("tight", "slice"):
            for hname, img in (("to_hll", H), ("from_host", H2)):
                op = Operands32(Xd, M, k, layout)
                img.spmm_f32(op.X, op.Y)
                assert_bitwise32(op.result(image), hll_ref[:, op.cols()], f"{image} {hname} k={k} {layout}")


# ---------------------------------------------------------------------------------------------------
# past 2^31 elements
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_offsets_past_2_31_elements(dev):
    """lap2d 4096^2 with k = 4 and ldx = ldy = 136 float32: row * ld passes 2^31 for the last 1.0 M rows (about 18 GB).
    Sampled rows on both sides of the crossing and at both ends EXACT, CSR and HLL; the ldy gap of those rows untouched."""
    import torch
    from sparsematrixvectormultiplication_b200 import synth
    n, k, ld = 4096, 4, 136
    M = n * n
    cross = (1 << 31) // ld
    assert M - cross > 980_000
    rng = np.random.default_rng(2 ** 31 + 32)
    X4 = rng.standard_normal((M, k)).astype(np.float32)
    Xbuf = sentinel_block(M, ld)
    Xbuf[:, :k].copy_(torch.from_numpy(X4))
    windows = [(0, 600), (cross - 3000, cross + 3000), (M - 3000, M)]
    A = dev.DeviceCSR.synth(dev.SYNTH_LAP2D, n).enable_f32()
    for fname, Mat in (("csr", A), ("hll", A.to_hll().enable_f32())):
        Ybuf = sentinel_block(M, ld)
        Mat.spmm_f32(Xbuf[:, :k], Ybuf[:, :k])
        torch.cuda.synchronize()
        for lo, hi in windows:
            rp, ci, va = synth.lap2d_csr(n, lo, hi)
            got = Ybuf[lo:hi].cpu().numpy()
            assert_bitwise32(got[:, :k], ref32_columns(rp, ci, va, X4), f"{fname} rows {lo}..{hi}")
            assert np.all(u32(got[:, k:]) == SENTINEL32), f"{fname}: gap written"
        del Ybuf
        if fname == "hll":
            Mat.close()
        torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------
# validation
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_validation(dev):
    """Without enable_f32: SpmvError and Y untouched.  float64 operands for spmm_f32 (and float32 ones for spmm), CPU
    tensors, bad strides, wrong shapes and overlap: ValueError before any launch, Y untouched.  The C layer on real
    handles: a negative k, ld < k and NULL arrays return SPMV_B200_ERR_INVALID and write nothing."""
    import torch
    from sparsematrixvectormultiplication_b200 import _native as N
    rng = np.random.default_rng(4)
    M = N_ = 200
    rp, ci, va = random_csr(rng, M, N_, rng.integers(0, 9, M))
    k = 4
    f32 = dict(dtype=torch.float32, device="cuda")
    X = torch.randn(N_, k, **f32)
    Ybuf = sentinel_block(M, 2 * k)
    Y = Ybuf[:, :k]

    def unchanged(what):
        torch.cuda.synchronize()
        assert np.all(u32(Ybuf.cpu().numpy()) == SENTINEL32), f"{what}: Y was written"

    # no float copy yet
    A = dev.DeviceCSR.upload(M, N_, rp, ci, va)
    H = A.to_hll()
    for what, call in (("csr", lambda: A.spmm_f32(X, Y)), ("csr accumulate", lambda: A.spmm_f32(X, Y, accumulate=True)),
                       ("hll", lambda: H.spmm_f32(X, Y))):
        with pytest.raises(N.SpmvError):
            call()
        unchanged(f"{what} without enable_f32")
    A.enable_f32()
    H.enable_f32()
    X64, Y64 = X.double(), torch.zeros(M, k, dtype=torch.float64, device="cuda")
    Xstrided = torch.empty(3 * N_ + k, **f32).as_strided((N_, k), (3, 1))
    bad = {
        "float64 X": (X64, Y), "float64 Y": (X, Y64), "float64 X and Y": (X64, Y64),
        "float16 X": (X.half(), Y), "CPU X": (X.cpu(), Y), "CPU Y": (X, torch.zeros(M, k)),
        "1-D X": (X[:, 0], Y[:, :1]), "X rows": (torch.randn(N_ + 1, k, **f32), Y), "column counts": (X[:, :3], Y),
        "X column stride": (torch.randn(k, N_, **f32).t(), Y), "Y column stride": (X, Ybuf[:, ::2]),
        "X row stride": (Xstrided, Y),
        "Y = X": (Ybuf[:, :k], Ybuf[:, :k]), "Y overlaps X": (Ybuf[:, 2:2 + k], Ybuf[:, :k]),
    }
    for what, (Xb, Yb) in bad.items():
        for name, call in (("csr", lambda: A.spmm_f32(Xb, Yb)), ("csr accumulate", lambda: A.spmm_f32(Xb, Yb, accumulate=True)),
                           ("hll", lambda: H.spmm_f32(Xb, Yb))):
            with pytest.raises(ValueError):
                call()
            unchanged(f"{what} ({name})")
    # float32 operands for the fp64 products
    Y64buf = torch.full((M, k), 7.0, dtype=torch.float64, device="cuda")
    for what, call in (("csr X", lambda: A.spmm(X, Y64buf)), ("csr Y", lambda: A.spmm(X64, Y)), ("hll X", lambda: H.spmm(X, Y64buf)),
                       ("hll Y", lambda: H.spmm(X64, Y))):
        with pytest.raises(ValueError):
            call()
        unchanged(f"spmm {what}")
    assert bool((Y64buf == 7.0).all())
    # interleaved column slices of one float buffer do not overlap; k = 0 is a no-op
    Z = torch.zeros(N_, 2 * k, **f32)
    Z[:, :k] = X
    A.spmm_f32(Z[:, :k], Z[:, k:])
    H.spmm_f32(Z[:, :k], Z[:, k:])
    A.spmm_f32(torch.empty(N_, 0, **f32), torch.empty(M, 0, **f32))
    H.spmm_f32(torch.empty(N_, 0, **f32), torch.empty(M, 0, **f32))
    lib, s = N.lib(), C.c_void_p(torch.cuda.current_stream().cuda_stream)
    px, py = C.c_void_p(X.data_ptr()), C.c_void_p(Ybuf.data_ptr())
    for rc in (lib.spmv_b200_csr_spmm_f32(A._h, -1, px, k, py, 2 * k, 0, s), lib.spmv_b200_csr_spmm_f32(A._h, k, px, k - 1, py, 2 * k, 0, s),
               lib.spmv_b200_csr_spmm_f32(A._h, k, px, k, py, k - 1, 0, s), lib.spmv_b200_csr_spmm_f32(A._h, k, None, k, py, 2 * k, 0, s),
               lib.spmv_b200_hll_spmm_f32(H._h, -1, px, k, py, 2 * k, s), lib.spmv_b200_hll_spmm_f32(H._h, k, px, k - 1, py, 2 * k, s),
               lib.spmv_b200_hll_spmm_f32(H._h, k, px, k, py, k - 1, s), lib.spmv_b200_hll_spmm_f32(H._h, k, px, k, None, 2 * k, s)):
        assert rc == -1
    unchanged("the C layer on an invalid call")
    H.close()
    A.close()
