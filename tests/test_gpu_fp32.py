"""The fp32-storage path against an exact reference of its contract.

Contract (include/spmv_b200.h, fp32 section): values, x and y are stored as float; every product is formed and summed in
double; the result is rounded once, on the store.  The reference of exactly that:

    vw    = float64(float32(values))   what enable_f32 stores (round to nearest even), exact when widened
    xw    = float64(x32), y0w = float64(y0)
    y64   = spmv_csr_serial(row_ptr, col_idx, vw, xw[, y = y0w])   the serial loop, every multiply and add rounded in double
    ref32 = float32(y64)

Two assertions:
  * EXACT -- a kernel that sums a row in one lane in index order (csr_row_kernel, csr_rowm_kernel, hll_row_kernel,
    hll_rowm_kernel, hll_rowu_kernel, the one-lane class of the binned kernel, the vector path at width 1) gives ref32
    bit for bit, with or without accumulate.  The HLL kernels also add the padding slots of their hack, as
    spmv_hll_serial does; a padding slot adds 0.0 * x = +-0.0, which changes no finite sum (a sum of non-zero terms that
    cancels is +0.0 in round-to-nearest, and +0.0 + -0.0 = +0.0), so the HLL reference equals the CSR one bit for bit --
    asserted where both are computed.
  * BOUNDED -- every other kernel: |y - y64| <= ulp32(ref32) + (len_i + 2) * 2^-53 * S_i with S_i = |y0w_i| + sum_j
    |vw_ij xw_j|: the float rounding of SOME fp64 sum of the same terms, in any order (vector and vec4 kernels at every
    width, binned multi-lane classes, long-row fragments and their combine, the HLL slice kernel).

The old 1e-5 * S check (test_gpu_parity.py::test_fp32_path_within_1e_5) cannot see arithmetic done in float;
test_the_reference_catches_float_arithmetic shows, without a GPU, that these assertions do on the rows used here.
"""
import numpy as np
import pytest

U53 = 2.0 ** -53
SPECIAL = 24                           # columns 0..23 of an adversarial x hold the special values below
PLAIN, CANCEL, OVERFLOW, SUBNORMAL, RANDOM_CANCEL = range(5)
KIND_NAMES = ("plain", "cancellation", "overflow", "subnormal", "random cancellation")


# ---------------------------------------------------------------------------------------------------
# the reference and the two assertions
# ---------------------------------------------------------------------------------------------------
def widen(a):
    """float32 storage of fp64 values, widened back (exact)."""
    return np.asarray(a, np.float64).astype(np.float32).astype(np.float64)


def u32(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


class Ref:
    """y64 / ref32 / S / row lengths of the fp32 contract on host CSR arrays (fp64 values, float32 x and y0)."""

    def __init__(self, checker, rp, ci, va, x32, y0=None):
        vw, xw = widen(va), np.asarray(x32, np.float32).astype(np.float64)
        y0w = None if y0 is None else np.asarray(y0, np.float32).astype(np.float64)
        self.y64 = checker.spmv_csr_serial(rp, ci, vw, xw, y=None if y0w is None else y0w.copy())
        self.ref32 = self.y64.astype(np.float32)
        self.S = checker.spmv_csr_serial(rp, ci, np.abs(vw), np.abs(xw)) + (0.0 if y0w is None else np.abs(y0w))
        self.lens = np.diff(np.asarray(rp, np.int64)).astype(np.float64)

    def window(self, lo, hi):
        out = object.__new__(Ref)
        out.y64, out.ref32, out.S, out.lens = self.y64[lo:hi], self.ref32[lo:hi], self.S[lo:hi], self.lens[lo:hi]
        return out

    def bound(self):
        return np.spacing(np.abs(self.ref32)).astype(np.float64) + (self.lens + 2.0) * U53 * self.S

    def violations(self, y):
        """Rows outside the bounded assertion (NaN counts as outside)."""
        err = np.abs(np.asarray(y, np.float32).astype(np.float64) - self.y64)
        return np.nonzero(~(err <= self.bound()))[0]


def assert_exact(y, r, what, rows=None):
    y = np.asarray(y, np.float32)
    want = r.ref32
    if rows is not None:
        y, want = y[rows], want[rows]
    bad = np.nonzero(u32(y) != u32(want))[0]
    assert bad.size == 0, (f"{what}: {bad.size} of {y.size} rows are not the exact reference, first {bad[:5]}: "
                           f"got {y[bad[:5]]}, want {want[bad[:5]]}")


def assert_bounded(y, r, what):
    bad = r.violations(y)
    y = np.asarray(y, np.float32)
    assert bad.size == 0, (f"{what}: {bad.size} of {y.size} rows outside ulp32 + (len+2) 2^-53 S, first {bad[:5]}: "
                           f"got {y[bad[:5]]}, want {r.y64[bad[:5]]}, S {r.S[bad[:5]]}")


# ---------------------------------------------------------------------------------------------------
# adversarial rows: arithmetic done in float (or a storage conversion other than round-to-nearest) cannot pass them
# ---------------------------------------------------------------------------------------------------
def adversarial_matrix(rng, M, N, lengths):
    """Sorted, duplicate-free CSR rows of the given lengths and a float32 x.  With N >= 64, x[0:8] = 1, x[8:16] = 1e20,
    x[16:24] = 1e30 and the rows of length >= 3 take turns among
      CANCEL         1, 2^27, -2^27 against x = 1 (then random terms): float addition loses the 1;
      OVERFLOW       1e20, -1e20, 3 against x = 1e20: the products overflow float (inf - inf), not double;
      SUBNORMAL      values of 1e-44..1e-38 (float subnormals) against x = 1e30 (rows of <= 8): a flush to zero gives 0;
      RANDOM_CANCEL  random terms and a first term that cancels their sum up to the float storage of its value: the
                     rounding of any product or stored value to float is thousands of ulps of what remains;
    other rows are random normal values (the storage rounding matters everywhere), every seventh ending in column N-1.
    Returns row_ptr, col_idx, values (fp64), x32, kind per row."""
    lengths = np.asarray(lengths, np.int64)
    x = rng.standard_normal(N)
    special = N >= 64
    if special:
        x[0:8], x[8:16], x[16:24] = 1.0, 1e20, 1e30
    x32 = x.astype(np.float32)
    xw = x32.astype(np.float64)
    first = SPECIAL if special else 0
    kinds = np.zeros(M, np.int8)
    cols, vals = [], []
    for i, L in enumerate(lengths.tolist()):
        kind = PLAIN if not special or L < 3 else 1 + i % 4
        if kind == SUBNORMAL and L > 8:
            kind = RANDOM_CANCEL
        kinds[i] = kind
        if kind == SUBNORMAL:
            c = 16 + np.sort(rng.choice(8, L, replace=False))
            v = rng.choice([-1.0, 1.0], L) * 10.0 ** rng.uniform(-44.5, -38.0, L)
        else:
            head = {PLAIN: [], CANCEL: [0, 1, 2], OVERFLOW: [8, 9, 10], RANDOM_CANCEL: [3]}[kind]
            rest = np.sort(rng.choice(N - first, L - len(head), replace=False)) + first
            if kind == PLAIN and L and i % 7 == 0 and rest[-1] != N - 1:
                rest[-1] = N - 1
            c = np.concatenate([np.array(head, np.int64), rest])
            v = rng.standard_normal(L)
            if kind == CANCEL:
                v[:3] = [1.0, 2.0 ** 27, -(2.0 ** 27)]
            elif kind == OVERFLOW:
                v[:3] = [1e20, -1e20, 3.0]
            elif kind == RANDOM_CANCEL:
                v[0] = -np.dot(widen(v[1:]), xw[c[1:]])
        cols.append(c)
        vals.append(v)
    rp = np.zeros(M + 1, np.int64)
    np.cumsum(lengths, out=rp[1:])
    ci = np.concatenate(cols).astype(np.int32) if rp[-1] else np.zeros(0, np.int32)
    va = np.concatenate(vals).astype(np.float64) if rp[-1] else np.zeros(0, np.float64)
    return rp.astype(np.int32), ci, va, x32, kinds


# numpy models of kernels that break the contract (and of two that keep it), rows padded to a dense block
def _dense(rp, ci, vals, xs):
    lens = np.diff(rp)
    pos = np.arange(int(lens.max()))
    mask = pos[None, :] < lens[:, None]
    idx = np.where(mask, rp[:-1, None] + pos[None, :], 0)
    return np.where(mask, vals[idx], 0), np.where(mask, xs[ci[idx]], 0)


def _serial(V, X, acc, rounded_product=lambda p: p):
    with np.errstate(all="ignore"):
        for j in range(V.shape[1]):
            acc = acc + rounded_product(V[:, j] * X[:, j])
    return acc


def model_products(name, rp, ci, va, x32):
    """float32 y of the model kernel `name` (no accumulate)."""
    M = len(rp) - 1
    xw = x32.astype(np.float64)
    with np.errstate(all="ignore"):
        if name == "float arithmetic":                      # multiply and add in float32
            V, X = _dense(rp, ci, va.astype(np.float32), x32)
            return _serial(V, X, np.zeros(M, np.float32))
        if name == "products rounded to float":           # (double)(float)(v * x)
            V, X = _dense(rp, ci, widen(va), xw)
            return _serial(V, X, np.zeros(M), lambda p: p.astype(np.float32).astype(np.float64)).astype(np.float32)
        if name == "storage truncated toward zero":       # a conversion that is not round-to-nearest
            f = va.astype(np.float32)
            up = np.abs(f.astype(np.float64)) > np.abs(va)
            f[up] = np.nextafter(f[up], np.float32(0))
            V, X = _dense(rp, ci, f.astype(np.float64), xw)
            return _serial(V, X, np.zeros(M)).astype(np.float32)
        if name == "float subnormals flushed":             # FTZ on the load of the stored values
            vw = widen(va)
            vw[np.abs(vw) < 2.0 ** -126] = 0.0
            V, X = _dense(rp, ci, vw, xw)
            return _serial(V, X, np.zeros(M)).astype(np.float32)
        V, X = _dense(rp, ci, widen(va), xw)
        if name == "widened fp64, serial":                 # the contract in the serial order
            return _serial(V, X, np.zeros(M)).astype(np.float32)
        if name == "widened fp64, four lanes":            # the contract in a vector kernel's order
            lanes = [_serial(V[:, k::4], X[:, k::4], np.zeros(M)) for k in range(4)]
            return ((lanes[0] + lanes[1]) + (lanes[2] + lanes[3])).astype(np.float32)
        if name == "widened fp64, reversed":
            return _serial(V[:, ::-1], X[:, ::-1], np.zeros(M)).astype(np.float32)
    raise KeyError(name)


def test_the_reference_catches_float_arithmetic(checker):
    """No GPU: on the adversarial rows every contract-breaking model violates the BOUNDED assertion on the kind of row
    meant to catch it, while fp64 arithmetic on the widened values passes it in any order (and the serial order is the
    EXACT reference).  What the GPU tests below assert can therefore fail."""
    rng = np.random.default_rng(31)
    M, N = 4000, 3000
    rp, ci, va, x32, kinds = adversarial_matrix(rng, M, N, rng.integers(0, 41, M))
    r = Ref(checker, rp, ci, va, x32)
    assert np.isfinite(r.y64).all() and np.isfinite(r.ref32).all()
    for kind in range(5):
        assert (kinds == kind).sum() >= 100, KIND_NAMES[kind]
    assert_exact(model_products("widened fp64, serial", rp, ci, va, x32), r, "widened fp64, serial")
    for name in ("widened fp64, four lanes", "widened fp64, reversed"):
        assert_bounded(model_products(name, rp, ci, va, x32), r, name)
    catches = {"float arithmetic": (CANCEL, OVERFLOW, RANDOM_CANCEL),
               "products rounded to float": (OVERFLOW, RANDOM_CANCEL),
               "storage truncated toward zero": (RANDOM_CANCEL,),
               "float subnormals flushed": (SUBNORMAL,)}
    for name, by in catches.items():
        bad = np.zeros(M, bool)
        bad[r.violations(model_products(name, rp, ci, va, x32))] = True
        for kind in by:
            rows = kinds == kind
            assert bad[rows].mean() > 0.5, f"{name}: only {bad[rows].sum()} of {rows.sum()} {KIND_NAMES[kind]} rows caught"
    # the old componentwise 1e-5 tolerance lets the float-arithmetic kernel through on plain random rows
    y = model_products("float arithmetic", rp, ci, va, x32).astype(np.float64)
    plain = kinds == PLAIN
    assert np.all(np.abs(y - r.y64)[plain] <= 1e-5 * r.S[plain])


# ---------------------------------------------------------------------------------------------------
# GPU: every fp32 entry point
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    import torch
    from sparsematrixvectormultiplication_b200 import device
    assert torch.cuda.is_available()
    torch.cuda.set_device(0)
    return device


def _nan32(M):
    import torch
    return torch.full((max(M, 1),), float("nan"), dtype=torch.float32, device="cuda")


def _product(fn, M, y0=None):
    """y from fn(y) on a NaN-filled (or y0-filled) float32 vector: a row the kernel skips stays NaN."""
    import torch
    y = _nan32(M) if y0 is None else torch.from_numpy(np.ascontiguousarray(y0, np.float32)).cuda()
    fn(y)
    return y.cpu().numpy()[:M]


def hll_reference(checker, rp, ci, va, x32, M, N, r):
    """spmv_hll_serial on the oracle's HLL of the same rows (AS widened), rounded to float; asserted equal to the CSR
    reference (the padding slots add +-0.0)."""
    from oracle import oracle as O
    rows = np.repeat(np.arange(M, dtype=np.int32), np.diff(rp))
    h = checker.coo_to_hll(O.Coo(M, N, len(ci), rows, ci.astype(np.int32), va))
    h.AS = widen(h.AS)
    y64 = checker.spmv_hll_serial(h, x32.astype(np.float64), M)
    assert np.array_equal(y64.view(np.uint64), r.y64.view(np.uint64)), "spmv_hll_serial and the serial CSR loop differ"
    return h


def check_csr_f32(dev, A, M, rp, r, r_acc, y0, x32d, what, exact_auto):
    """Every CSR fp32 algorithm, plain and accumulating, plus the host round trip."""
    lens = np.diff(rp)
    for name, algo in (("auto", dev.ALGO_AUTO), ("row", dev.ALGO_ROW), ("vector", dev.ALGO_VECTOR), ("binned", dev.ALGO_BINNED)):
        for acc, ref in ((False, r), (True, r_acc)):
            y = _product(lambda y: A.spmv_f32(x32d, y, accumulate=acc, algo=algo), M, y0 if acc else None)
            tag = f"{what} csr {name}{' accumulate' if acc else ''}"
            if name == "row" or (name == "auto" and exact_auto):
                assert_exact(y, ref, tag)
            else:
                assert_bounded(y, ref, tag)
                if name == "binned":                      # rows of <= 8: the one-lane class, serial order
                    assert_exact(y, ref, tag + " (rows of <= 8)", rows=lens <= 8)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["M1", "M31", "M33", "M257", "M4900", "prime7919", "N1", "nnz0", "bin_edges", "long_rows",
                                  "skewed"])
def test_every_f32_entry_point(dev, checker, case):
    """CSR spmv_f32 (AUTO / ROW / VECTOR / BINNED, plain and accumulating onto random float32 y0) on an uploaded and on a
    wrapped matrix, HLL spmv_f32 and both host round trips, against the exact reference.  Row counts that are no
    multiple of 32 or 256, N = 1, no nonzero at all, empty rows, columns 0 and N-1, rows that start off a multiple of four
    and nnz that is no multiple of four (the masking of the aligned-group loads and of their safe_nnz limit), every
    row-length bin edge and long rows at the fragment edges (8192, 8193, 16385), also after replan(long_threshold)."""
    import torch
    rng = np.random.default_rng(sum(map(ord, case)))
    shapes = {"M1": (1, 50, [7]), "M31": (31, 300, rng.integers(0, 13, 31)), "M33": (33, 300, rng.integers(0, 21, 33)),
              "M257": (257, 1000, rng.integers(0, 41, 257)), "M4900": (4900, 4900, rng.integers(0, 31, 4900)),
              "prime7919": (7919, 3001, rng.integers(0, 17, 7919)), "N1": (300, 1, rng.integers(0, 2, 300)),
              "nnz0": (100, 80, np.zeros(100, np.int64)),
              "bin_edges": (64, 5000, np.tile([0, 1, 8, 9, 12, 13, 24, 25, 48, 49, 96, 97, 2048, 2049, 3, 5], 4)),
              "long_rows": (40, 40000, np.concatenate([[8192, 8193, 16385, 0, 7, 8191], rng.integers(0, 40, 34)])),
              "skewed": (6000, 5000, np.concatenate([[4900, 3000, 600], rng.integers(0, 30, 5997)]))}
    M, N, lengths = shapes[case]
    lengths = np.array(lengths, np.int64)
    if lengths.sum() % 4 == 0 and lengths.sum() > 0:    # nnz off a multiple of four
        lengths[np.argmax((lengths > 0) & (lengths < N) & (lengths != 8) & (lengths != 2048))] += 1
    rp, ci, va, x32, kinds = adversarial_matrix(rng, M, N, lengths)
    nnz = int(rp[-1])
    assert nnz % 4 != 0 or nnz == 0
    if M > 4 and nnz:
        assert (rp[:-1] % 4 != 0).any()
    y0 = rng.standard_normal(M).astype(np.float32)
    r, r_acc = Ref(checker, rp, ci, va, x32), Ref(checker, rp, ci, va, x32, y0)
    if nnz == 0:
        assert not u32(r.ref32).any(), "every row of a matrix without nonzeros is +0.0"
    x32d = torch.from_numpy(x32).cuda()
    short = int(np.diff(rp).max(initial=0)) <= 12
    t = [torch.from_numpy(a).cuda() for a in (rp, ci, va)]
    for how in ("upload", "wrap"):
        A = dev.DeviceCSR.upload(M, N, rp, ci, va) if how == "upload" else dev.DeviceCSR.wrap(M, N, *t)
        A.enable_f32()
        check_csr_f32(dev, A, M, rp, r, r_acc, y0, x32d, f"{case}/{how}", exact_auto=short)
        yh = A.spmv_host_f32(x32, np.full(M, np.nan, np.float32))
        (assert_exact if short else assert_bounded)(yh, r, f"{case}/{how} csr spmv_host_f32")
        if case in ("long_rows", "skewed"):
            for L in (512, 4096):                          # other long-row plans: the automatic choice changes with them
                A.replan(long_threshold=L)
                check_csr_f32(dev, A, M, rp, r, r_acc, y0, x32d, f"{case}/{how}/long_threshold={L}", exact_auto=short)
        if how == "upload":
            hll_reference(checker, rp, ci, va, x32, M, N, r)
            H = A.to_hll().enable_f32()
            exact = H.info().max_maxnz <= 12               # lane-per-row kernels; wider hacks take the slice kernel
            y = _product(lambda y: H.spmv_f32(x32d, y), M)
            (assert_exact if exact else assert_bounded)(y, r, f"{case} hll spmv_f32 (max width {H.info().max_maxnz})")
            yh = H.spmv_host_f32(x32, np.full(M, np.nan, np.float32))
            (assert_exact if exact else assert_bounded)(yh, r, f"{case} hll spmv_host_f32")
            H.close()
        A.close()


def _mixed_matrix(rng, M=3001, N=4000):
    lengths = rng.choice([0, 1, 3, 5, 8, 9, 13, 17, 25, 33, 49, 70, 97, 130], size=M)
    lengths[:3] = [3, 97, 2]
    return lengths


@pytest.mark.gpu
def test_vector_widths_vec4_and_binned_split(dev, checker, monkeypatch):
    """SPMV_B200_VECTOR_WIDTH in {1,2,4,8,16,32} x SPMV_B200_VEC4 in {0,1,2} (read at every launch; the binned kernel
    reads VEC4 too) and SPMV_B200_BINNED_SPLIT in {0,1} (long-row fragments in the binned launch or in one of their
    own), on an uploaded (arrays padded to a multiple of four) and a wrapped matrix (aligned loads stop at nnz & ~3):
    width 1 and the binned one-lane class exact, everything else bounded."""
    import torch
    rng = np.random.default_rng(404)
    M, N = 3001, 10000
    lengths = np.concatenate([_mixed_matrix(rng, M - 3, N), [8193, 2049, 6]])
    rp, ci, va, x32, _ = adversarial_matrix(rng, M, N, lengths)
    assert int(rp[-1]) % 4 != 0
    y0 = rng.standard_normal(M).astype(np.float32)
    r, r_acc = Ref(checker, rp, ci, va, x32), Ref(checker, rp, ci, va, x32, y0)
    x32d = torch.from_numpy(x32).cuda()
    t = [torch.from_numpy(a).cuda() for a in (rp, ci, va)]
    lens = np.diff(rp)
    for how in ("upload", "wrap"):
        A = dev.DeviceCSR.upload(M, N, rp, ci, va) if how == "upload" else dev.DeviceCSR.wrap(M, N, *t)
        A.enable_f32()
        for vec4 in (0, 1, 2):
            monkeypatch.setenv("SPMV_B200_VEC4", str(vec4))
            for width in (1, 2, 4, 8, 16, 32):
                monkeypatch.setenv("SPMV_B200_VECTOR_WIDTH", str(width))
                for acc, ref in ((False, r), (True, r_acc)):
                    y = _product(lambda y: A.spmv_f32(x32d, y, accumulate=acc, algo=dev.ALGO_VECTOR), M, y0 if acc else None)
                    tag = f"{how} vector width {width} vec4 {vec4}{' accumulate' if acc else ''}"
                    (assert_exact if width == 1 else assert_bounded)(y, ref, tag)
            monkeypatch.delenv("SPMV_B200_VECTOR_WIDTH")
            for split in (0, 1):
                monkeypatch.setenv("SPMV_B200_BINNED_SPLIT", str(split))
                for acc, ref in ((False, r), (True, r_acc)):
                    y = _product(lambda y: A.spmv_f32(x32d, y, accumulate=acc, algo=dev.ALGO_BINNED), M, y0 if acc else None)
                    tag = f"{how} binned split {split} vec4 {vec4}{' accumulate' if acc else ''}"
                    assert_bounded(y, ref, tag)
                    assert_exact(y, ref, tag + " (rows of <= 8)", rows=lens <= 8)
            monkeypatch.delenv("SPMV_B200_BINNED_SPLIT")
        A.close()


@pytest.mark.gpu
@pytest.mark.parametrize("batch", range(1, 9))
def test_row_batches(dev, checker, monkeypatch, batch):
    """SPMV_B200_ROW_BATCH / SPMV_B200_HLL_ROW_BATCH = 1..8 (read when the plan is made, so set before the upload): the
    one-row kernels at every batch, CSR (plain and accumulating) and HLL, exact; M = 4903, rows of 0..12 whose lengths
    are no multiple of any batch."""
    import torch
    monkeypatch.setenv("SPMV_B200_ROW_BATCH", str(batch))
    monkeypatch.setenv("SPMV_B200_HLL_ROW_BATCH", str(batch))
    rng = np.random.default_rng(100 + batch)
    M, N = 4903, 3500
    rp, ci, va, x32, _ = adversarial_matrix(rng, M, N, rng.integers(0, 13, M))
    y0 = rng.standard_normal(M).astype(np.float32)
    r, r_acc = Ref(checker, rp, ci, va, x32), Ref(checker, rp, ci, va, x32, y0)
    hll_reference(checker, rp, ci, va, x32, M, N, r)
    x32d = torch.from_numpy(x32).cuda()
    A = dev.DeviceCSR.upload(M, N, rp, ci, va).enable_f32()
    assert A.info().row_batch == batch and A.row_form_f32() == f"csr_row_kernel<{batch},float>"
    for algo in (dev.ALGO_AUTO, dev.ALGO_ROW):
        assert_exact(_product(lambda y: A.spmv_f32(x32d, y, algo=algo), M), r, f"csr batch {batch} algo {algo}")
        assert_exact(_product(lambda y: A.spmv_f32(x32d, y, accumulate=True, algo=algo), M, y0), r_acc,
                     f"csr batch {batch} algo {algo} accumulate")
    H = A.to_hll().enable_f32()
    assert H.row_form_f32() == f"hll_row_kernel<{batch},float>"
    assert_exact(_product(lambda y: H.spmv_f32(x32d, y), M), r, f"hll batch {batch}")
    H.close()
    A.close()


# ---------------------------------------------------------------------------------------------------
# HLL images: regular ones (hll_rowu_kernel), one that is not, wide hacks (slice kernel)
# ---------------------------------------------------------------------------------------------------
def image_lengths(rng, runs, M):
    """Row lengths whose HLL image has the given runs [(width, hacks), ...]: every hack of a run has one row of the full
    width and others shorter; a width-0 run is a run of empty hacks.  M may end inside the last hack."""
    out = []
    for width, hacks in runs:
        for _ in range(hacks):
            rows = rng.integers(0, width + 1, 32)
            rows[rng.integers(0, 32)] = width
            out.append(rows)
    lengths = np.concatenate(out)[:M]
    full = (M // 32) * 32
    if M > full:
        lengths[full] = runs[-1][0]          # the short last hack keeps its run's width
    return lengths


def run_count(widths):
    widths = np.asarray(widths)
    return int(1 + np.count_nonzero(widths[1:] != widths[:-1])) if widths.size else 0


@pytest.mark.gpu
@pytest.mark.parametrize("image", ["lap2d", "one_run", "seven_runs", "eight_runs", "nine_runs", "wide13", "wide33"])
def test_hll_images(dev, checker, monkeypatch, image):
    """Regular images (at most 8 runs of hacks of equal width: lap2d 70^2 with M % 32 != 0, and images of exactly 1, 7 and
    8 runs with empty hacks and with runs whose width is and is not the batch -- the straight-line and the loop branch of
    hll_rowu_kernel) under every SPMV_B200_HLL_UNIFORM in 3..7, exact; a 9-run image (not regular: the forced form must
    change nothing); images with hacks wider than 12 and wider than 32 (the slice kernel), bounded."""
    import torch
    from sparsematrixvectormultiplication_b200 import synth
    rng = np.random.default_rng(sum(map(ord, image)))
    if image == "lap2d":
        rp, ci, va = synth.lap2d_csr(70)
        M = N = 4900
        va = va * rng.uniform(0.5, 1.5, va.size)       # values off the float grid: the storage rounding matters
        x32 = rng.standard_normal(N).astype(np.float32)
        runs = 3
    else:
        spec = {"one_run": [(5, 40)], "seven_runs": [(3, 3), (0, 2), (7, 4), (4, 1), (6, 5), (5, 2), (2, 3)],
                "eight_runs": [(5, 2), (4, 3), (0, 2), (7, 2), (6, 4), (3, 1), (12, 3), (1, 2)],
                "nine_runs": [(1, 2), (2, 2), (3, 2), (4, 2), (5, 2), (6, 2), (7, 2), (8, 2), (9, 2)],
                "wide13": [(13, 4), (5, 2), (20, 3), (0, 1), (16, 2)], "wide33": [(33, 3), (40, 2), (7, 2), (64, 2)]}[image]
        runs = len(spec)
        M = 32 * sum(h for _, h in spec) - 13
        N = 3000
        rp, ci, va, x32, _ = adversarial_matrix(rng, M, N, image_lengths(rng, spec, M))
    r = Ref(checker, rp, ci, va, x32)
    hll_reference(checker, rp, ci, va, x32, M, N, r)
    x32d = torch.from_numpy(x32).cuda()
    A = dev.DeviceCSR.upload(M, N, rp, ci, va)
    H = A.to_hll().enable_f32()
    A.close()
    _, widths, _, _, _ = H.download().flat()
    assert run_count(widths) == runs and M % 32 != 0, f"{image}: the image has {run_count(widths)} runs"
    wide = H.info().max_maxnz > 12
    plain = _product(lambda y: H.spmv_f32(x32d, y), M)
    if wide:
        assert_bounded(plain, r, f"{image}: slice kernel (max width {H.info().max_maxnz})")
    else:
        assert_exact(plain, r, f"{image}: {H.row_form_f32()}")
    for b in (3, 4, 5, 6, 7):
        monkeypatch.setenv("SPMV_B200_HLL_UNIFORM", str(b))
        y = _product(lambda y: H.spmv_f32(x32d, y), M)
        assert np.array_equal(u32(y), u32(plain)), f"{image}: SPMV_B200_HLL_UNIFORM={b} changed the result"
        if not wide:
            assert_exact(y, r, f"{image}: SPMV_B200_HLL_UNIFORM={b}")
        yh = H.spmv_host_f32(x32, np.full(M, np.nan, np.float32))
        assert np.array_equal(u32(yh), u32(plain)), f"{image}: host round trip, SPMV_B200_HLL_UNIFORM={b}"
    H.close()


# ---------------------------------------------------------------------------------------------------
# the forms enable_f32 chooses on matrices large enough to be tuned
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["lap2d_4096", "irregular_short_rows"])
def test_forms_chosen_at_plan_time(dev, checker, monkeypatch, kind):
    """lap2d 4096^2 (the fp32 headline shape; its HLL image is regular, so hll_rowu_kernel competes) and an irregular matrix
    of 6.3 M nonzeros (rows of 0..12 at random columns): the form the plan-time timing chose gives the exact reference on
    every row, CSR and HLL; so does every form forced through SPMV_B200_ROW_MULTI and SPMV_B200_HLL_UNIFORM."""
    import torch
    from sparsematrixvectormultiplication_b200 import synth
    for key in ("SPMV_B200_ROW_MULTI", "SPMV_B200_HLL_UNIFORM", "SPMV_B200_ROW_BATCH", "SPMV_B200_HLL_ROW_BATCH"):
        monkeypatch.delenv(key, raising=False)
    if kind == "lap2d_4096":
        n = 4096
        A = dev.DeviceCSR.synth(synth.SYNTH_LAP2D, n)
        rp, ci, va = A.download()
        M = N = n * n
    else:
        rng = np.random.default_rng(2026)
        M = N = 1 << 20
        lengths = rng.integers(0, 13, M)
        rp = np.zeros(M + 1, np.int64)
        np.cumsum(lengths, out=rp[1:])
        rp = rp.astype(np.int32)
        ci = rng.integers(0, N, int(rp[-1])).astype(np.int32)
        va = rng.standard_normal(int(rp[-1]))
        assert rp[-1] >= 6_000_000
        A = dev.DeviceCSR.upload(M, N, rp, ci, va)
    x32 = synth.hash_vector(N, 0xF32).astype(np.float32)
    r = Ref(checker, rp, ci, va, x32)
    del rp, ci, va
    x32d = torch.from_numpy(x32).cuda()
    A.enable_f32()
    form = A.row_form_f32()
    y = _product(lambda y: A.spmv_f32(x32d, y), M)
    assert_exact(y, r, f"{kind} CSR, tuned form {form}")
    for k in range(1, len(dev.row_forms(dev.FORMAT_CSR)) + 1):
        monkeypatch.setenv("SPMV_B200_ROW_MULTI", str(k))
        assert_exact(_product(lambda y: A.spmv_f32(x32d, y), M), r,
                     f"{kind} CSR, SPMV_B200_ROW_MULTI={k} ({dev.row_form_name(dev.FORMAT_CSR, 15 + k)}; tuned {form})")
    monkeypatch.delenv("SPMV_B200_ROW_MULTI")
    H = A.to_hll().enable_f32()
    form = H.row_form_f32()
    assert_exact(_product(lambda y: H.spmv_f32(x32d, y), M), r, f"{kind} HLL, tuned form {form}")
    for b in (3, 4, 5, 6, 7):
        monkeypatch.setenv("SPMV_B200_HLL_UNIFORM", str(b))
        assert_exact(_product(lambda y: H.spmv_f32(x32d, y), M), r, f"{kind} HLL, SPMV_B200_HLL_UNIFORM={b} (tuned {form})")
    monkeypatch.delenv("SPMV_B200_HLL_UNIFORM")
    H.close()
    # a tuned hll_rowu_kernel form takes precedence over SPMV_B200_ROW_MULTI: an image whose batch is fixed at plan time
    # (no timing) runs every multi-hack form when it is forced
    monkeypatch.setenv("SPMV_B200_HLL_ROW_BATCH", "5")
    H = A.to_hll().enable_f32()
    monkeypatch.delenv("SPMV_B200_HLL_ROW_BATCH")
    assert H.row_form_f32() == "hll_row_kernel<5,float>"
    for k in range(1, len(dev.row_forms(dev.FORMAT_HLL)) + 1):
        monkeypatch.setenv("SPMV_B200_ROW_MULTI", str(k))
        assert_exact(_product(lambda y: H.spmv_f32(x32d, y), M), r,
                     f"{kind} HLL, SPMV_B200_ROW_MULTI={k} ({dev.row_form_name(dev.FORMAT_HLL, 15 + k)})")
    monkeypatch.delenv("SPMV_B200_ROW_MULTI")
    H.close()
    A.close()


# ---------------------------------------------------------------------------------------------------
# element offsets past 2^31 bytes: lap3d 512^3 (938 M nonzeros)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_offsets_past_2_31_bytes_lap3d_512(dev, checker):
    """Row windows of +-2^20 rows around the rows where the CSR nnz offset and the HLL slot offset cross 2^28 (fp64 values
    past 2^31 bytes) and 2^29 (column indices, fp32 values, JA past 2^31 bytes), and the last 2^20 rows, with x a hash
    vector (not ones: every interior row sums to 0 against ones), against the numpy twin of the generator through the
    serial oracle.  fp64: CSR AUTO / ROW / STREAM / VECTOR / BINNED and HLL automatic / rows / stream sum rows of 7 in the
    serial order (bitwise), the HLL slice kernel within 1e-12 componentwise; fp32: CSR and HLL exact.  The HLL slot
    offsets are computed independently on the device from the closed-form row lengths.  About 40 GB of device memory."""
    import torch
    from sparsematrixvectormultiplication_b200 import synth
    n = 512
    M = n ** 3
    n2 = n * n
    seed = 0x3D512
    half = 1 << 20
    # rows where the CSR nnz offset crosses 2^28 / 2^29 (closed form)
    csr_rows = []
    for target in (1 << 28, 1 << 29):
        lo, hi = 0, M                                   # last row whose offset is <= target
        while hi - lo > 1:
            mid = (lo + hi) // 2
            if synth.row_offset(synth.SYNTH_LAP3D, n, 0, 0, mid) <= target:
                lo = mid
            else:
                hi = mid
        assert synth.row_offset(synth.SYNTH_LAP3D, n, 0, 0, lo) <= target < synth.row_offset(synth.SYNTH_LAP3D, n, 0, 0, lo + 1)
        csr_rows.append(lo)
    # HLL slot offsets: hack width = the longest of its 32 rows, row length = 7 minus the missing neighbours
    r_all = torch.arange(M, device="cuda", dtype=torch.int64)
    length = torch.full((M,), 7, dtype=torch.int8, device="cuda")
    for c in (r_all // n2, (r_all // n) % n, r_all % n):
        length -= (c == 0).to(torch.int8) + (c == n - 1).to(torch.int8)
    del r_all
    width = length.view(-1, 32).amax(dim=1).to(torch.int64)
    del length
    hack_end = torch.cumsum(width * 32, 0)             # slots of hacks [0, h]
    slots_total = int(hack_end[-1])
    hll_rows = [32 * int(torch.searchsorted(hack_end, torch.tensor([target], device="cuda"), right=True)[0])
                for target in (1 << 28, 1 << 29)]     # first row of the hack holding slot `target`
    del width, hack_end
    windows = [(max(0, r - half), min(M, r + half)) for r in csr_rows + hll_rows] + [(M - half, M)]
    # references from the numpy twin: only the columns [lo - n^2, hi + n^2) of x are needed
    refs = []
    for lo, hi in windows:
        rp, ci, va = synth.lap3d_csr(n, lo, hi)
        base, top = max(0, lo - n2), min(M, hi + n2)
        xw = synth.hash_vector(top - base, seed, begin=base)
        ci = ci - np.int32(base)
        y64 = checker.spmv_csr_serial(rp, ci, va, xw)
        S = checker.spmv_csr_serial(rp, ci, np.abs(va), np.abs(xw))
        refs.append((y64, S, Ref(checker, rp, ci, va, xw.astype(np.float32))))
        del rp, ci, va, xw

    def check64(y, what, exact=True):
        for (lo, hi), (y64, S, _) in zip(windows, refs):
            got = y[lo:hi].cpu().numpy()
            if exact:
                bad = np.nonzero(got.view(np.uint64) != y64.view(np.uint64))[0]
            else:
                bad = np.nonzero(~(np.abs(got - y64) <= 1e-12 * S))[0]
            assert bad.size == 0, f"{what}, rows [{lo},{hi}): {bad.size} rows off, first {lo + bad[:5]}: {got[bad[:5]]} vs {y64[bad[:5]]}"

    def check32(y, what):
        for (lo, hi), (_, _, r) in zip(windows, refs):
            assert_exact(y[lo:hi].cpu().numpy(), r, f"{what}, rows [{lo},{hi})")

    A = dev.DeviceCSR.synth(synth.SYNTH_LAP3D, n)
    assert A.info().nnz == 937_951_232 and A.info().max_row_nnz == 7
    x = torch.empty(M, dtype=torch.float64, device="cuda")
    dev.synth_vector(x, seed)
    x32 = x.float()
    y = torch.empty(M, dtype=torch.float64, device="cuda")
    for name, algo in (("auto", dev.ALGO_AUTO), ("row", dev.ALGO_ROW), ("stream", dev.ALGO_STREAM), ("vector", dev.ALGO_VECTOR),
                       ("binned", dev.ALGO_BINNED)):
        y.fill_(float("nan"))
        A.spmv(x, y, algo=algo)
        check64(y, f"fp64 CSR {name}")
    A.enable_f32()
    y32 = torch.empty(M, dtype=torch.float32, device="cuda")
    for name, algo in (("auto", dev.ALGO_AUTO), ("row", dev.ALGO_ROW), ("vector", dev.ALGO_VECTOR), ("binned", dev.ALGO_BINNED)):
        y32.fill_(float("nan"))
        A.spmv_f32(x32, y32, algo=algo)
        check32(y32, f"fp32 CSR {name} (tuned form {A.row_form_f32()})")
    H = A.to_hll()
    A.close()
    del A
    assert H.info().slots == slots_total and H.info().max_maxnz == 7
    for name, flag in (("automatic", None), ("rows", "rows"), ("stream", False), ("slice", True)):
        y.fill_(float("nan"))
        H.spmv(x, y, slice_kernel=flag)
        check64(y, f"fp64 HLL {name}", exact=name != "slice")
    H.enable_f32()
    y32.fill_(float("nan"))
    H.spmv_f32(x32, y32)
    check32(y32, f"fp32 HLL (tuned form {H.row_form_f32()})")
    H.close()


# ---------------------------------------------------------------------------------------------------
# the Python wrappers check their vectors before anything is launched
# ---------------------------------------------------------------------------------------------------
def _small_pair(dev):
    from sparsematrixvectormultiplication_b200 import synth
    A = dev.DeviceCSR.synth(synth.SYNTH_LAP2D, 9).enable_f32()       # 81 x 81
    H = A.to_hll().enable_f32()
    return A, H, 81


@pytest.mark.gpu
def test_f32_products_reject_a_wider_dtype(dev):
    """float64 tensors where spmv_f32 expects float32 (as many elements, twice the bytes): ValueError, and the vectors are
    left as they were -- nothing was launched."""
    import torch
    A, H, M = _small_pair(dev)
    x32 = torch.ones(M, dtype=torch.float32, device="cuda")
    y32 = torch.full((M,), 7.0, dtype=torch.float32, device="cuda")
    x64 = torch.ones(M, dtype=torch.float64, device="cuda")
    y64 = torch.full((M,), 7.0, dtype=torch.float64, device="cuda")
    for what, call in (("csr x", lambda: A.spmv_f32(x64, y32)), ("csr y", lambda: A.spmv_f32(x32, y64)),
                       ("hll x", lambda: H.spmv_f32(x64, y32)), ("hll y", lambda: H.spmv_f32(x32, y64))):
        with pytest.raises(ValueError):
            call()
        torch.cuda.synchronize()
        assert bool((y32 == 7.0).all()) and bool((y64 == 7.0).all()), f"{what}: a vector was written"
    for what, obj in (("csr", A), ("hll", H)):
        yh = np.full(M, 7.0)
        with pytest.raises(ValueError):
            obj.spmv_host_f32(np.ones(M, np.float32), yh)            # float64 y for a float32 product
        assert (yh == 7.0).all(), f"{what} spmv_host_f32 wrote into a float64 y"
    H.close()
    A.close()


@pytest.mark.gpu
def test_wrappers_reject_bad_vectors(dev):
    """CPU, short, narrower-dtype and non-contiguous tensors for spmv_f32 / spmv_rows / spmv_hacks; host round trips with
    a y or x of the wrong length or dtype: ValueError, and nothing is written."""
    import torch
    A, H, M = _small_pair(dev)
    good32 = torch.ones(M, dtype=torch.float32, device="cuda")
    good64 = torch.ones(M, dtype=torch.float64, device="cuda")
    bad32 = {"cpu": torch.ones(M, dtype=torch.float32), "short": torch.ones(M - 1, dtype=torch.float32, device="cuda"),
             "float16": torch.ones(M, dtype=torch.float16, device="cuda"),
             "strided": torch.ones(2 * M, dtype=torch.float32, device="cuda")[::2]}
    bad64 = {"cpu": torch.ones(M, dtype=torch.float64), "short": torch.ones(M - 1, dtype=torch.float64, device="cuda"),
             "float32": torch.ones(M, dtype=torch.float32, device="cuda"),
             "strided": torch.ones(2 * M, dtype=torch.float64, device="cuda")[::2]}
    for tag, bad in bad32.items():
        for what, call in (("csr x", lambda: A.spmv_f32(bad, good32)), ("csr y", lambda: A.spmv_f32(good32, bad)),
                           ("hll x", lambda: H.spmv_f32(bad, good32)), ("hll y", lambda: H.spmv_f32(good32, bad))):
            with pytest.raises(ValueError):
                call()
    for tag, bad in bad64.items():
        for what, call in (("csr rows x", lambda: A.spmv_rows(0, M, bad, good64)), ("csr rows y", lambda: A.spmv_rows(0, M, good64, bad)),
                           ("hll hacks x", lambda: H.spmv_hacks(0, 3, bad, good64)), ("hll hacks y", lambda: H.spmv_hacks(0, 3, good64, bad))):
            with pytest.raises(ValueError):
                call()
    torch.cuda.synchronize()
    assert bool((good32 == 1.0).all()) and bool((good64 == 1.0).all())
    for obj in (A, H):
        for fn, dt, wrong in ((obj.spmv_host_f32, np.float32, np.float16), (obj.spmv_host, np.float64, np.float32)):
            for y in (np.zeros(M - 1, dt), np.zeros(M, wrong), np.zeros(2 * M, dt)[::2], np.zeros(M + 1, dt)):
                with pytest.raises(ValueError):
                    fn(np.ones(M, dt), y)
            with pytest.raises(ValueError):
                fn(np.ones(M - 1, dt))                                    # x shorter than N
            assert fn(np.ones(M, dt)).dtype == dt
    H.close()
    A.close()
