"""The pattern form of a CSR handle's private image: one byte per row when the rows hold at most 256 distinct patterns.

Contract (include/spmv_b200.h, "Private image"): a row's pattern is its length, then col - row of each nonzero, then the
64-bit pattern of each value (+0.0 and -0.0 count apart).  When there are at most 256 of them and the dictionary (12
bytes per pattern and slot of the longest row, W) takes at most 24 KB, set_image(3) stores one byte per row naming its
pattern (image_patterns P, image_form 256 + W, image_device_bytes M + P * (12 W + 4)); it fails otherwise and leaves the
handle as it was.  The kernel gathers all W slots of a row -- a slot past the row's length gathers x[min(row, N - 1)]
-- and adds v * x for the slots below the length in order, mul and add rounded separately: bit for bit
SPMV_B200_ALGO_ROW for every x and with accumulate from any y, except which payload a NaN carries where two NaNs meet in
one sum (as for the coded image, test_gpu_csr_image_values.py).
"""
import numpy as np
import pytest

from test_gpu_csr_image import (adversarial_csr, adversarial_x, bits, dev, minus_zero_start, products_equal_row, serial,
                                special_x, tbits)
from test_gpu_csr_image_values import same_bits_up_to_nan_payload

MAX_PATTERNS = 256
DICT_BYTES = 24 * 1024


# ---------------------------------------------------------------------------------------------------
# numpy model of the dictionary and the product (no GPU)
# ---------------------------------------------------------------------------------------------------
def row_patterns(rp, ci, va):
    """(W, sorted distinct pattern keys, id per row), or None when the matrix does not qualify.  A key is (len, deltas
    as uint32, value bits), zero past len -- the order the library sorts its dictionary in."""
    rp, ci = np.asarray(rp, np.int64), np.asarray(ci, np.int64)
    vb = np.ascontiguousarray(va, np.float64).view(np.uint64)
    M = len(rp) - 1
    W = int(np.diff(rp).max()) if M else 0
    if W < 1 or W > 12:
        return None
    keys = []
    for r in range(M):
        lo, hi = rp[r], rp[r + 1]
        pad = [0] * (W - (hi - lo))
        keys.append(tuple([int(hi - lo)] + [int(c - r) & 0xffffffff for c in ci[lo:hi]] + pad + [int(v) for v in vb[lo:hi]] + pad))
    table = sorted(set(keys))
    if len(table) > MAX_PATTERNS or 12 * W * len(table) > DICT_BYTES:
        return None
    index = {k: i for i, k in enumerate(table)}
    return W, table, np.array([index[k] for k in keys], np.int64)


def pattern_product(pats, M, N, x, y0=None):
    """The kernel's loop on the model: every slot gathers, slots below the length add, in order."""
    W, table, ids = pats
    y = np.zeros(M) if y0 is None else np.array(y0, np.float64, copy=True)
    for r in range(M):
        key = table[ids[r]]
        n = key[0]
        deltas = [int(np.int32(np.uint32(d))) for d in key[1:1 + W]]
        vals = np.array(key[1 + W:], np.uint64).view(np.float64)
        xv = [x[min(r + deltas[s], N - 1)] for s in range(W)]
        acc = y[r]
        for s in range(n):
            acc = acc + vals[s] * xv[s]
        y[r] = acc
    return y


def banded_pool(M, N, pool, seed):
    """Rows drawn from a pool of (deltas, values) patterns; a row takes one whose columns all lie in [0, N), else it stays
    empty; when N < 8, every fourth row holds column 0 only (a pattern of its own per row)."""
    rng = np.random.default_rng(seed)
    rp, ci, va = [0], [], []
    for r in range(M):
        fits = [p for p in pool if all(0 <= r + d < N for d in p[0])]
        if N < 8 and r % 4 == 1:
            cols, vals = [0], [1.5]
        elif fits and r % 9 != 4:
            deltas, vals = fits[int(rng.integers(len(fits)))]
            cols = [r + d for d in deltas]
        else:
            cols, vals = [], []
        ci.extend(cols)
        va.extend(vals)
        rp.append(len(ci))
    return np.array(rp, np.int32), np.array(ci, np.int32), np.array(va, np.float64)


def make_pool(count, seed, span=40, lengths=(1, 12)):
    """count patterns of lengths[0]-lengths[1] sorted distinct deltas in [-span, span] and values from a small set with
    stored zeros."""
    rng = np.random.default_rng(seed)
    choices = np.array([1.0, -1.0, 4.0, 0.0, -0.0, 0.25, 3.0e-300, -7.5])
    pool = []
    for _ in range(count):
        n = int(rng.integers(lengths[0], lengths[1] + 1))
        deltas = sorted(rng.choice(np.arange(-span, span + 1), size=n, replace=False).tolist())
        pool.append((deltas, rng.choice(choices, size=n).tolist()))
    return pool


def test_pattern_model_keeps_the_serial_bits():
    """lap2d has 9 patterns and lap3d 27; on them and on adversarial rows (empty rows, stored +-0.0, Inf and NaN in x,
    accumulate from -0.0) the model's product equals the serial loop up to NaN payloads, bit for bit on finite x."""
    from sparsematrixvectormultiplication_b200 import synth
    cases = [synth.lap2d_csr(64) + (64 * 64, 64 * 64, 9), synth.lap2d_csr(128) + (128 * 128, 128 * 128, 9),
             synth.lap3d_csr(24) + (24 ** 3, 24 ** 3, 27)]
    rp, ci, va, M, N = adversarial_csr()
    cases.append((rp, ci, va, M, N, None))
    rpb, cib, vab = banded_pool(300, 250, make_pool(30, 3), 4)
    cases.append((rpb, cib, vab, 300, 250, None))
    for rp, ci, va, M, N, expect in cases:
        pats = row_patterns(rp, ci, va)
        assert pats is not None
        if expect is not None:
            assert len(pats[1]) == expect
        y0 = np.full(M, -0.0)
        y0[::4] = np.random.default_rng(9).standard_normal(len(y0[::4]))
        x = adversarial_x(rp, ci, N)
        xf = np.nan_to_num(x, nan=0.5, posinf=3.0, neginf=-3.0)
        with np.errstate(invalid="ignore"):
            for start in (None, y0):
                ref, got = serial(rp, ci, va, x, start), pattern_product(pats, M, N, x, start)
                assert np.array_equal(np.isnan(ref), np.isnan(got))
                assert np.array_equal(bits(ref)[~np.isnan(ref)], bits(got)[~np.isnan(ref)])
                assert np.array_equal(bits(serial(rp, ci, va, xf, start)), bits(pattern_product(pats, M, N, xf, start)))


def count_matrix(count, M=2000):
    """The diagonal with `count` distinct values: exactly `count` patterns."""
    rp = np.arange(M + 1, dtype=np.int32)
    ci = np.arange(M, dtype=np.int32)
    va = 1.0 + np.arange(M) % count
    return rp, ci, va


def wide_count_matrix(count, W, M=2000):
    """Rows of W nonzeros at col - row = 0 .. W - 1 with `count` distinct first values: exactly `count` patterns of
    width W, every column in [0, M + W - 1)."""
    rp = np.arange(M + 1, dtype=np.int32) * W
    ci = (np.arange(M, dtype=np.int32)[:, None] + np.arange(W, dtype=np.int32)[None, :]).ravel()
    va = np.tile(np.linspace(-1.0, 0.5, W), (M, 1))
    va[:, 0] = 1.0 + np.arange(M) % count
    return rp, ci, va.ravel()


def test_pattern_model_limits():
    """256 patterns qualify, 257 do not; equal deltas with different values (+0.0 against -0.0 included) are different
    patterns, and so are equal values at different deltas; a row of 13 nonzeros or no nonzero at all never qualifies."""
    assert len(row_patterns(*count_matrix(256))[1]) == 256
    assert row_patterns(*count_matrix(257)) is None
    rp, ci, va = mixed_rows()
    assert len(row_patterns(rp, ci, va)[1]) == 6
    assert row_patterns(np.array([0, 13]), np.arange(13), np.ones(13)) is None
    assert row_patterns(np.array([0, 0, 0]), np.zeros(0, np.int64), np.zeros(0)) is None


def mixed_rows(M=200):
    """Six patterns: deltas (0, 1) with values (1, 2), (1, 3), (1, +0.0), (1, -0.0); deltas (0, 2) and (-1, 0) with
    values (1, 2); the last row takes (-1, 0) so that no column leaves [0, M)."""
    kinds = [((0, 1), (1.0, 2.0)), ((0, 1), (1.0, 3.0)), ((0, 1), (1.0, 0.0)), ((0, 1), (1.0, -0.0)),
             ((0, 2), (1.0, 2.0)), ((-1, 0), (1.0, 2.0))]
    rp, ci, va = [0], [], []
    for r in range(M):
        k = 5 if r >= M - 2 else (r % 5 if r > 0 else 0)
        if r % 7 == 3 and r > 0:
            k = 5
        deltas, vals = kinds[k]
        ci.extend(r + d for d in deltas)
        va.extend(vals)
        rp.append(len(ci))
    return np.array(rp, np.int32), np.array(ci, np.int32), np.array(va)


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
def patterns_equal_row(A, x, y0=None, algos=None):
    """AUTO and ROW_IMAGE against ALGO_ROW with and without accumulate, NaN payloads aside."""
    import torch
    d = dev()
    M = A.info().M
    for start in ([None] if y0 is None else [None, y0]):
        ref = torch.zeros(M, dtype=torch.float64, device="cuda") if start is None else start.clone()
        A.spmv(x, ref, accumulate=start is not None, algo=d.ALGO_ROW)
        for algo in algos or (d.ALGO_AUTO, d.ALGO_ROW_IMAGE):
            y = torch.zeros(M, dtype=torch.float64, device="cuda") if start is None else start.clone()
            A.spmv(x, y, accumulate=start is not None, algo=algo)
            torch.cuda.synchronize()
            assert same_bits_up_to_nan_payload(y, ref), f"algo {algo}, accumulate={start is not None}"


def check_pattern_form(A, M, N, W, P, x):
    """The info fields of the form, then the products: NaN payloads aside for x, bit for bit for x free of NaN and Inf,
    a row-range product that starts and ends inside a hack, and the host-buffer call."""
    import torch
    d = dev()
    i = A.info()
    assert (i.image_patterns, i.image_form, i.image_index_bytes, i.image_value_bytes) == (P, 256 + W, 0, 0)
    assert i.image_device_bytes == i.image_bytes == M + P * (12 * W + 4)
    assert A.image_form() == f"csr_pattern_kernel<{W}>"
    assert i.auto_algo == d.ALGO_ROW_IMAGE
    patterns_equal_row(A, x, minus_zero_start(M))
    products_equal_row(A, torch.nan_to_num(x, nan=0.5, posinf=3.0, neginf=-3.0), minus_zero_start(M))
    ref = torch.zeros(M, dtype=torch.float64, device="cuda")
    A.spmv(x, ref, algo=d.ALGO_ROW)
    lo, hi = min(45, M // 3), max(M - 13, M // 3 + 1)
    y = torch.full((M,), 7.0, dtype=torch.float64, device="cuda")
    A.spmv_rows(lo, hi, x, y)
    torch.cuda.synchronize()
    assert same_bits_up_to_nan_payload(y[lo:hi], ref[lo:hi])
    assert bool((y[:lo] == 7.0).all()) and bool((y[hi:] == 7.0).all())
    refh = ref.cpu().numpy().view(np.int64)
    for algo in (d.ALGO_AUTO, d.ALGO_ROW_IMAGE):
        assert np.array_equal(A.spmv_host(x.cpu().numpy(), algo=algo).view(np.int64), refh)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n", [("lap2d", 64), ("lap2d", 4096), ("lap3d", 24), ("lap3d", 256)])
def test_patterns_on_stencils(kind, n):
    d = dev()
    A = d.DeviceCSR.synth(d.SYNTH_LAP2D if kind == "lap2d" else d.SYNTH_LAP3D, n)
    A.set_image(3)
    i = A.info()
    if n <= 64:
        rp, ci, va = A.download()
        assert len(row_patterns(rp, ci, va)[1]) == (9 if kind == "lap2d" else 27)
    rp_last = A.download()[1][::9973]
    check_pattern_form(A, i.M, i.N, 5 if kind == "lap2d" else 7, 9 if kind == "lap2d" else 27, special_x(i.N, rp_last))
    A.close()


@pytest.mark.gpu
@pytest.mark.parametrize("M,N,W", [(1000, 777, None), (33, 5, None), (31, 1, None), (4900, 4900, None), (700, 1400, None)]
                         + [(1500 + 37 * w, 1300, w) for w in range(1, 13)],
                         ids=["1000-777", "33-5", "31-1", "4900-4900", "700-1400"] + [f"W{w}" for w in range(1, 13)])
def test_patterns_on_irregular_rows(M, N, W):
    """M > N and M < N, empty rows, rows of 1-12 nonzeros from a pool, stored +-0.0; x with +-Inf and NaN.  W: every
    width of csr_pattern_kernel, on M > N with rows of 1 to W nonzeros."""
    d = dev()
    pool = make_pool(60, M)
    if W is not None:  # rows of 1 to W nonzeros, one pattern of exactly W
        pool = make_pool(40, M, span=20, lengths=(1, W)) + [(list(range(-(W // 2), W - W // 2)), [2.0] * W)]
    rp, ci, va = banded_pool(M, N, pool, M + N)
    pats = row_patterns(rp, ci, va)
    assert pats is not None and pats[0] == (W or pats[0])
    A = d.DeviceCSR.upload(M, N, rp, ci, va)
    A.set_image(3)
    last = [ci[rp[r + 1] - 1] for r in range(M) if rp[r + 1] > rp[r]]
    check_pattern_form(A, M, N, pats[0], len(pats[1]), special_x(N, last, seed=M))
    A.close()


@pytest.mark.gpu
def test_equal_deltas_or_equal_values():
    d = dev()
    rp, ci, va = mixed_rows()
    A = d.DeviceCSR.upload(200, 200, rp, ci, va)
    A.set_image(3)
    check_pattern_form(A, 200, 200, 2, 6, special_x(200, ci[1::2], seed=5))
    A.close()


@pytest.mark.gpu
@pytest.mark.parametrize("count,W", [(256, 1), (257, 1), (170, 12), (171, 12), (186, 11), (187, 11)],
                         ids=["256", "257", "W12-170", "W12-171", "W11-186", "W11-187"])
def test_pattern_count_boundary(count, W):
    """256 patterns build; 257 fail with SpmvError and leave the held image (here the fp64 column-major one) as it was.
    The dictionary's bytes bound it too: 12 W P <= 24576, so W = 12 holds 170 patterns (24480 bytes, the largest
    dictionary) and not 171, W = 11 holds 186 and not 187."""
    import torch
    from sparsematrixvectormultiplication_b200 import _native as NN
    d = dev()
    rp, ci, va = count_matrix(count) if W == 1 else wide_count_matrix(count, W)
    M, N = len(rp) - 1, int(ci.max()) + 1
    builds = count <= MAX_PATTERNS and 12 * W * count <= DICT_BYTES
    assert (row_patterns(rp, ci, va) is not None) == builds
    A = d.DeviceCSR.upload(M, N, rp, ci, va)
    x = special_x(N, ci[::37], seed=count)
    if builds:
        A.set_image(3)
        check_pattern_form(A, M, N, W, count, x)
    else:
        A.set_image(1)
        before = A.info()
        with pytest.raises(NN.SpmvError):
            A.set_image(3)
        after = A.info()
        assert (after.image_patterns, after.image_form, after.image_device_bytes, after.image_value_bytes) == \
            (0, before.image_form, before.image_device_bytes, 8)
        products_equal_row(A, torch.nan_to_num(x, nan=0.5, posinf=3.0, neginf=-3.0), minus_zero_start(M))
    A.close()


@pytest.mark.gpu
def test_pattern_lifecycle():
    """3 -> 1 -> 3 -> 0; replan decides again (no image at this size); remap_columns drops the form and a new one
    multiplies the remapped matrix; wrapped arrays, a row of 13 nonzeros and an empty matrix never get one."""
    import torch
    from sparsematrixvectormultiplication_b200 import _native as NN
    d = dev()
    A = d.DeviceCSR.synth(d.SYNTH_LAP2D, 64)
    i = A.info()
    x = torch.randn(i.N, dtype=torch.float64, device="cuda")
    assert i.image_patterns == 0 and A.image_form() == "none"
    for mode in (3, 1, 3, 3, 0):
        A.set_image(mode)
        j = A.info()
        assert j.image_patterns == (9 if mode == 3 else 0)
        assert j.image_value_bytes == (8 if mode == 1 else 0)
        products_equal_row(A, x, minus_zero_start(i.M), algos=None if mode else (d.ALGO_AUTO,))
    A.set_image(3)
    A.replan()
    assert A.info().image_patterns == 0 and A.info().image_bytes == 0
    products_equal_row(A, x, algos=(d.ALGO_AUTO,))
    A.set_image(3)
    N0 = i.N
    half = N0 // 2
    stride = half + 3
    A.remap_columns([0, half, N0], stride)
    assert A.info().image_patterns == 0 and A.info().image_bytes == 0
    xr = torch.zeros(2 * stride, dtype=torch.float64, device="cuda")
    xr[:half] = x[:half]
    xr[stride:stride + N0 - half] = x[half:]
    products_equal_row(A, xr, algos=(d.ALGO_AUTO,))
    A.set_image(3)
    assert A.info().image_patterns > 9  # the remapped columns move col - row on the rows past the split
    products_equal_row(A, xr, minus_zero_start(i.M))
    A.close()

    rp = torch.as_tensor(np.arange(0, 2 * 64 + 1, 2, dtype=np.int32), device="cuda")
    ci = torch.as_tensor(np.tile(np.array([0, 5], np.int32), 64), device="cuda")
    va = torch.ones(128, dtype=torch.float64, device="cuda")
    W = d.DeviceCSR.wrap(64, 8, rp, ci, va)
    with pytest.raises(NN.SpmvError):
        W.set_image(3)
    assert W.info().image_patterns == 0
    W.close()
    for rp_, ci_, N_ in ((np.array([0, 13, 14], np.int32), np.array(list(range(13)) + [0], np.int32), 13),
                         (np.zeros(5, np.int32), np.zeros(0, np.int32), 3)):
        B = d.DeviceCSR.upload(len(rp_) - 1, N_, rp_, ci_, np.ones(len(ci_)))
        with pytest.raises(NN.SpmvError):
            B.set_image(3)
        assert B.info().image_patterns == 0 and B.info().auto_algo != d.ALGO_ROW_IMAGE
        B.close()
