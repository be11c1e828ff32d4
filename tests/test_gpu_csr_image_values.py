"""The coded private image of a CSR handle: 1-byte value codes when the matrix holds at most 256 distinct value patterns.

Contract (include/spmv_b200.h, "Private image"): the distinct 64-bit patterns of the values (+0.0 and -0.0, and NaNs of
different payloads, count apart) form a table sorted as uint64; every slot of the image stores the index of its value's
pattern, a padding slot code 0.  The kernels multiply by table[code], the stored double itself, and keep the masked
padding rule, so products stay bit for bit SPMV_B200_ALGO_ROW for every x and with accumulate from any y.
set_image(2) builds the coded image (image_value_bytes 1, image_device_bytes (index + 1) per slot plus 8 per table
entry) and fails on a matrix of more than 256 patterns, leaving the handle as it was; set_image(1) keeps meaning the
fp64 image and replaces a coded one.

Bits are compared as integers.  Where two different NaNs meet in one row's sum (a NaN value or x entry and an invalid
product such as 0 * Inf), which payload the sum carries depends on the order in which ptxas puts the operands of an add,
and that order differs between the coded kernels and csr_row_kernel; there only NaN-ness is compared.
"""
import numpy as np
import pytest

from test_gpu_csr_image import (HACK, adversarial_csr, adversarial_x, bits, dev, image, image_slots, minus_zero_start,
                                products_equal_row, serial, special_x, tbits)
from test_gpu_csr_image_narrow import narrow_fits

MAX_VALUES = 256
MARK = 0x80000000


# ---------------------------------------------------------------------------------------------------
# numpy model of the value table and the coded kernels (no GPU)
# ---------------------------------------------------------------------------------------------------
def value_table(va):
    """The distinct 64-bit patterns of the values, ascending as uint64; None when there are more than 256."""
    pats = np.unique(np.ascontiguousarray(va, np.float64).view(np.uint64))
    return None if len(pats) > MAX_VALUES else pats


def coded_image(hacks, table):
    """The wide image (test_gpu_csr_image.image) with AS replaced by codes: a real slot's pattern index, padding 0."""
    out = []
    for JA, AS in hacks:
        AC = np.searchsorted(table, AS.view(np.uint64)).astype(np.uint8)
        AC[(JA & MARK) != 0] = 0
        real = (JA & MARK) == 0
        assert np.array_equal(table[AC[real]], AS.view(np.uint64)[real])
        out.append((JA, AC))
    return out


def coded_product(hacks, table, M, x, y0=None):
    """The masked kernels on the coded image: every slot gathers, a marked slot skips the add, a value is table[code]."""
    tab = table.view(np.float64)
    y = np.zeros(M) if y0 is None else np.array(y0, np.float64, copy=True)
    for h, (JA, AC) in enumerate(hacks):
        for lr in range(HACK):
            r = h * HACK + lr
            if r >= M:
                continue
            acc = y[r]
            for j in range(JA.shape[0]):
                c = int(JA[j, lr])
                xv = x[c & ~MARK]
                if not c & MARK:
                    acc = acc + tab[AC[j, lr]] * xv
            y[r] = acc
    return y


def special_values():
    """+-0.0, +-Inf, NaNs of two payloads, the all-ones pattern (a NaN, and the empty mark of the library's distinct-value
    set), subnormals and a few normal numbers."""
    pats = np.array([0x0000000000000000, 0x8000000000000000, 0x7FF0000000000000, 0xFFF0000000000000,
                     0x7FF8000000000000, 0x7FF8000000000123, 0xFFFFFFFFFFFFFFFF, 0x0000000000000001, 0x800FFFFFFFFFFFFF],
                    np.uint64).view(np.float64)
    return np.concatenate([pats, [1.0, -2.5, 4.0, -1.0]])


def test_value_table_model():
    """Sorted uint64 patterns; 256 patterns fit, 257 do not; +-0.0 and NaN payloads are separate patterns."""
    rng = np.random.default_rng(3)
    va = rng.choice(rng.standard_normal(200), 5000)
    t = value_table(va)
    assert t is not None and len(t) == len(np.unique(va.view(np.uint64)))
    assert np.all(t[1:] > t[:-1])
    assert value_table(np.arange(256.0)) is not None and len(value_table(np.arange(256.0))) == 256
    assert value_table(np.arange(257.0)) is None
    t = value_table(special_values())
    assert len(t) == len(special_values())   # +0.0 / -0.0 and the two NaNs are four patterns
    assert list(t) == sorted(int(p) for p in special_values().view(np.uint64))


def test_coded_product_model_keeps_the_serial_bits():
    """Codes of a 17-pattern value set (stored zeros of both signs included): the coded masked product equals the serial
    loop bit for bit, with +-Inf/NaN in x and accumulate from -0.0."""
    rp, ci, va, M, N = adversarial_csr()
    rng = np.random.default_rng(4)
    pool = np.concatenate([rng.standard_normal(15), [0.0, -0.0]])
    va = rng.choice(pool, len(va))
    va[1::7] = -0.0
    table = value_table(va)
    assert table is not None and len(table) <= 17
    hacks = coded_image(image(rp, ci, va), table)
    x = adversarial_x(rp, ci, N)
    y0 = np.full(M, -0.0)
    y0[::4] = np.random.default_rng(9).standard_normal(len(y0[::4]))
    with np.errstate(invalid="ignore"):
        for start in (None, y0):
            assert np.array_equal(bits(coded_product(hacks, table, M, x, start)), bits(serial(rp, ci, va, x, start)))


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
def check_coded(A, rp, ci, va, N):
    """image_value_bytes, image_device_bytes and the form's name as the model predicts them."""
    i = A.info()
    index = 2 if narrow_fits(rp, ci, N) else 4
    K = len(value_table(va))
    slots = image_slots(rp)
    assert i.image_value_bytes == 1 and i.image_index_bytes == index
    assert i.image_device_bytes == (index + 1) * slots + 8 * K
    assert i.image_bytes == 12 * slots
    assert A.image_form().endswith((",uint16_t,uint8_t>" if index == 2 else ",int,uint8_t>")), A.image_form()
    assert i.auto_algo == dev().ALGO_ROW_IMAGE


def same_bits_up_to_nan_payload(y, ref):
    """Every non-NaN entry bit for bit (+-0.0 and +-Inf included), NaN exactly where ref has NaN."""
    import torch
    nan = torch.isnan(ref)
    return bool(torch.equal(nan, torch.isnan(y))) and bool(torch.equal(tbits(y)[~nan], tbits(ref)[~nan]))


def coded_equal_row(A, x, y0=None):
    """AUTO and ROW_IMAGE against ALGO_ROW, with and without accumulate (products_equal_row, NaN payloads aside)."""
    import torch
    d = dev()
    M = A.info().M
    for start in ([None] if y0 is None else [None, y0]):
        ref = torch.zeros(M, dtype=torch.float64, device="cuda") if start is None else start.clone()
        A.spmv(x, ref, accumulate=start is not None, algo=d.ALGO_ROW)
        for algo in (d.ALGO_AUTO, d.ALGO_ROW_IMAGE):
            y = torch.zeros(M, dtype=torch.float64, device="cuda") if start is None else start.clone()
            A.spmv(x, y, accumulate=start is not None, algo=algo)
            torch.cuda.synchronize()
            assert same_bits_up_to_nan_payload(y, ref), f"algo {algo}, accumulate={start is not None}"


def check_products(A, x, M, finite_values=True):
    """AUTO and ROW_IMAGE give ALGO_ROW's bits with and without accumulate from -0.0: NaN payloads aside for this x, bit
    for bit for the same x free of NaN and Inf (on finite values).  A row-range product that starts and ends inside a
    hack and the host-buffer call (both on the row kernel) give ALGO_ROW's bits."""
    import torch
    d = dev()
    coded_equal_row(A, x, minus_zero_start(M))
    if finite_values:
        products_equal_row(A, torch.nan_to_num(x, nan=0.5, posinf=3.0, neginf=-3.0), minus_zero_start(M))
    ref = torch.zeros(M, dtype=torch.float64, device="cuda")
    A.spmv(x, ref, algo=d.ALGO_ROW)
    lo, hi = min(45, M // 3), max(M - 13, M // 3 + 1)
    y = torch.full((M,), 7.0, dtype=torch.float64, device="cuda")
    A.spmv_rows(lo, hi, x, y)
    torch.cuda.synchronize()
    assert torch.equal(tbits(y[lo:hi]), tbits(ref[lo:hi]))
    assert bool((y[:lo] == 7.0).all()) and bool((y[hi:] == 7.0).all())
    xh = x.cpu().numpy()
    refh = ref.cpu().numpy().view(np.int64)
    for algo in (d.ALGO_AUTO, d.ALGO_ROW_IMAGE):
        assert np.array_equal(A.spmv_host(xh, algo=algo).view(np.int64), refh)


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n", [("lap2d", 64), ("lap2d", 4096), ("lap3d", 64), ("lap3d", 128)])
def test_coded_image_on_stencils(kind, n):
    """Two distinct values each: lap2d and lap3d 64 with the 2-byte column field, lap3d 128 with the 4-byte one."""
    d = dev()
    A = d.DeviceCSR.synth(d.SYNTH_LAP2D if kind == "lap2d" else d.SYNTH_LAP3D, n)
    A.set_image(2)
    i = A.info()
    rp, ci, va = A.download()
    assert len(value_table(va)) == 2
    check_coded(A, rp, ci, va, i.N)
    last = ci[rp[1:][np.diff(rp) > 0] - 1][::97]
    check_products(A, special_x(i.N, last), i.M)
    A.close()


def irregular(M, N, pool, seed):
    """Random rows of 0-12 nonzeros (every 9th row empty), columns 0 and N-1, values drawn from `pool`."""
    rng = np.random.default_rng(seed)
    rp, ci, va = [0], [], []
    for r in range(M):
        n = 0 if r % 9 == 4 else int(rng.integers(0, min(N, 12) + 1))
        cols = np.sort(rng.choice(N, size=n, replace=False)) if n else np.zeros(0, np.int64)
        if n and r % 4 == 0:
            cols[0] = 0
        if n and r % 6 == 1:
            cols[-1] = N - 1
        cols = np.unique(cols)
        ci.extend(cols.tolist())
        va.extend(rng.choice(pool, len(cols)).tolist())
        rp.append(len(ci))
    va = np.array(va)
    va[:len(pool)] = pool[:min(len(pool), len(va))]   # every pattern present
    return np.array(rp, np.int32), np.array(ci, np.int32), va


@pytest.mark.gpu
@pytest.mark.parametrize("M,N", [(9001, 3000), (3001, 40000)])
def test_coded_image_on_irregular_rows(M, N):
    """M > N with a padded last hack (2-byte column field) and M < N with columns past 2^14 (4-byte), empty rows, values
    from a 17-element set with stored zeros of both signs."""
    d = dev()
    rng = np.random.default_rng(M + N)
    pool = np.concatenate([rng.standard_normal(15), [0.0, -0.0]])
    rp, ci, va = irregular(M, N, pool, M)
    A = d.DeviceCSR.upload(M, N, rp, ci, va)
    A.set_image(2)
    assert len(value_table(va)) == 17
    check_coded(A, rp, ci, va, N)
    last = [ci[rp[r + 1] - 1] for r in range(M) if rp[r + 1] > rp[r]]
    check_products(A, special_x(N, last, seed=M), M)
    A.close()


@pytest.mark.gpu
@pytest.mark.parametrize("count,all_ones", [(256, False), (257, False), (256, True), (257, True)],
                         ids=["256", "257", "256-all-ones", "257-all-ones"])
def test_value_count_boundary(count, all_ones):
    """Exactly 256 patterns gets the coded image; 257 raises and leaves the handle as it was (no image, then the fp64
    image).  With the all-ones pattern among them -- counted on the host, not in the device's set -- 256 patterns build
    with it as code 255, and 257 fail where the device counts 256."""
    import torch
    d = dev()
    from sparsematrixvectormultiplication_b200 import _native as NN
    pool = np.random.default_rng(count).standard_normal(count)
    if all_ones:
        pool[-1] = np.array([0xFFFFFFFFFFFFFFFF], np.uint64).view(np.float64)[0]
    M = N = 2000
    rp, ci, va = irregular(M, N, pool, count)
    assert len(np.unique(va.view(np.uint64))) == count
    A = d.DeviceCSR.upload(M, N, rp, ci, va)
    x = special_x(N, [], seed=count)
    if all_ones:  # no NaN of another payload in x to meet the all-ones one in a sum
        x = torch.nan_to_num(x, nan=float("-inf"), posinf=float("inf"), neginf=float("-inf"))
    if count <= MAX_VALUES:
        A.set_image(2)
        check_coded(A, rp, ci, va, N)
        assert value_table(va)[-1] == 0xFFFFFFFFFFFFFFFF or not all_ones
        check_products(A, x, M)
    else:
        before = A.info()
        with pytest.raises(NN.SpmvError):
            A.set_image(2)
        after = A.info()
        assert (after.image_bytes, after.image_form, after.image_value_bytes) == (before.image_bytes, before.image_form, 0)
        A.set_image(1)
        held = A.info()
        assert held.image_value_bytes == 8
        with pytest.raises(NN.SpmvError):
            A.set_image(2)
        i = A.info()
        assert (i.image_value_bytes, i.image_device_bytes, i.image_form) == (8, held.image_device_bytes, held.image_form)
        products_equal_row(A, x, minus_zero_start(M))   # the fp64 image: bit for bit
    A.close()
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_special_values():
    """A value set of +0.0, -0.0, +-Inf, NaNs of two payloads and subnormals: each its own code, products bit for bit
    ALGO_ROW."""
    d = dev()
    pool = special_values()
    M, N = 4000, 3000
    rp, ci, va = irregular(M, N, pool, 5)
    assert len(value_table(va)) == len(pool)
    A = d.DeviceCSR.upload(M, N, rp, ci, va)
    A.set_image(2)
    check_coded(A, rp, ci, va, N)
    last = [ci[rp[r + 1] - 1] for r in range(M) if rp[r + 1] > rp[r]]
    check_products(A, special_x(N, last, seed=6), M, finite_values=False)
    A.close()


@pytest.mark.gpu
def test_coded_lifecycle():
    """2 -> 1 -> 2 -> 0, then replan (decides again: no image at this size) and remap_columns (drops the image; a new
    coded one multiplies the remapped matrix)."""
    import torch
    d = dev()
    A = d.DeviceCSR.synth(d.SYNTH_LAP2D, 64)
    i = A.info()
    rp, ci, va = A.download()
    x = torch.randn(i.N, dtype=torch.float64, device="cuda")
    slots = image_slots(rp)
    for mode, value_bytes in ((2, 1), (1, 8), (2, 1), (0, 0)):
        A.set_image(mode)
        j = A.info()
        assert j.image_value_bytes == value_bytes, mode
        assert j.image_device_bytes == (0 if mode == 0 else (2 + value_bytes) * slots + (16 if value_bytes == 1 else 0))
        products_equal_row(A, x, minus_zero_start(i.M), algos=None if mode else (d.ALGO_AUTO,))
    A.set_image(2)
    A.replan()
    assert A.info().image_bytes == 0 and A.info().image_value_bytes == 0
    products_equal_row(A, x, algos=(d.ALGO_AUTO,))
    A.set_image(2)
    N0 = i.N
    half = N0 // 2
    stride = half + 3
    A.remap_columns([0, half, N0], stride)
    assert A.info().image_bytes == 0 and A.info().image_value_bytes == 0
    xr = torch.zeros(2 * stride, dtype=torch.float64, device="cuda")
    xr[:half] = x[:half]
    xr[stride:stride + N0 - half] = x[half:]
    products_equal_row(A, xr, algos=(d.ALGO_AUTO,))
    A.set_image(2)
    assert A.info().image_value_bytes == 1
    products_equal_row(A, xr, minus_zero_start(i.M))
    A.close()
