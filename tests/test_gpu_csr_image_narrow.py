"""The narrow private image of a CSR handle: a 2-byte column field when every slot's column lies within 2^14 of its row.

Contract (include/spmv_b200.h, "Private image"): when col - row lies in [-16384, 16383] for every slot of the image,
padding included, the column field holds col - row in bits 0-14 (two's complement) and the padding mark in bit 15, so the
image takes 10 bytes per slot instead of 12 (image_index_bytes 2, image_device_bytes 10 per slot; image_bytes keeps its
definition of 12 per slot).  A padding slot of a row without real columns (empty, or past M in the last hack) gathers
column min(row, N - 1); a matrix where that is out of reach keeps the wide image.  Products stay bit for bit
SPMV_B200_ALGO_ROW for every x and with accumulate from any y, as with the wide image (tests/test_gpu_csr_image.py).

Bits are compared as integers, so NaN payloads count.
"""
import numpy as np
import pytest

from test_gpu_csr_image import (HACK, adversarial_csr, adversarial_x, bits, dev, image_slots, minus_zero_start,
                                products_equal_row, serial, special_x, tbits)

DMIN, DMAX, MARK16 = -16384, 16383, 0x8000


# ---------------------------------------------------------------------------------------------------
# numpy model of the narrow field (no GPU)
# ---------------------------------------------------------------------------------------------------
def encode16(col, row, pad):
    d = col - row
    assert DMIN <= d <= DMAX
    return (d & 0x7FFF) | (MARK16 if pad else 0)


def decode16(field, row):
    d = field & 0x7FFF
    return row + (d - 0x8000 if d & 0x4000 else d), bool(field & MARK16)


def narrow_fits(rp, ci, N):
    """hll_narrow_check_kernel: every real slot's col - row in range, and every row without real columns that still has
    slots (empty, or past M in a hack with any nonzero) reaches column min(row, N - 1)."""
    rp = np.asarray(rp, np.int64)
    lens = np.diff(rp)
    M = len(lens)
    rows = np.repeat(np.arange(M), lens)
    d = np.asarray(ci, np.int64) - rows
    if len(d) and (d.min() < DMIN or d.max() > DMAX):
        return False
    padded = np.concatenate([lens, np.zeros((-M) % HACK, np.int64)])
    width = padded.reshape(-1, HACK).max(axis=1) if len(padded) else np.zeros(0, np.int64)
    r = np.arange(len(padded))
    empty_with_slots = (padded == 0) & (np.repeat(width, HACK) > 0)
    return bool(np.all(r[empty_with_slots] - (N - 1) <= -DMIN))


def image16(rp, ci, va, N):
    """The narrow image: per hack (JA16, AS) of shape (width, 32), padded rows past M included."""
    M = len(rp) - 1
    hacks = []
    for h in range((M + HACK - 1) // HACK):
        rows = range(h * HACK, (h + 1) * HACK)
        w = max([rp[r + 1] - rp[r] for r in rows if r < M] + [0])
        JA = np.zeros((w, HACK), np.uint16)
        AS = np.zeros((w, HACK))
        for lr, r in enumerate(rows):
            last = min(r, N - 1)
            n = rp[r + 1] - rp[r] if r < M else 0
            for j in range(w):
                if j < n:
                    last = ci[rp[r] + j]
                    JA[j, lr], AS[j, lr] = encode16(last, r, False), va[rp[r] + j]
                else:
                    JA[j, lr] = encode16(last, r, True)
        hacks.append((JA, AS))
    return hacks


def image16_product(hacks, M, N, x, y0=None):
    """The narrow masked kernels: every slot gathers x[row + d] (asserted in bounds), a marked slot skips the add."""
    y = np.zeros(M) if y0 is None else np.array(y0, np.float64, copy=True)
    for h, (JA, AS) in enumerate(hacks):
        for lr in range(HACK):
            r = h * HACK + lr
            acc = y[r] if r < M else 0.0
            for j in range(JA.shape[0]):
                c, pad = decode16(int(JA[j, lr]), r)
                assert 0 <= c < N, (r, j, c)
                xv = x[c]
                if not pad:
                    acc = acc + AS[j, lr] * xv
            if r < M:
                y[r] = acc
    return y


def test_narrow_field_model():
    """The extreme deltas round-trip and +16384 / -16385 do not fit; on the narrow image every gather, padding included,
    stays in bounds and the masked rule keeps the serial bits with +-Inf/NaN in x and -0.0 accumulate."""
    for d in (DMIN, -1, 0, 1, DMAX):
        for pad in (False, True):
            assert decode16(encode16(40000 + d, 40000, pad), 40000) == (40000 + d, pad)
    for d in (DMAX + 1, DMIN - 1):
        with pytest.raises(AssertionError):
            encode16(40000 + d, 40000, False)
        M = 40000
        rp = np.arange(M + 1, dtype=np.int64)
        ci = np.arange(M, dtype=np.int64)
        ci[20000] += d
        assert not narrow_fits(rp, ci, M + DMAX + 1)
        ci[20000] -= d + (1 if d > 0 else -1)
        assert narrow_fits(rp, ci, M + DMAX + 1)
    # a row without columns past the reach of column N - 1 (rows past M included) disqualifies the matrix
    assert narrow_fits(np.arange(16481), np.minimum(np.arange(16480), 99), 100)
    assert not narrow_fits(np.arange(16485), np.minimum(np.arange(16484), 99), 100)
    rp, ci, va, M, N = adversarial_csr()
    assert narrow_fits(rp, ci, N)
    x = adversarial_x(rp, ci, N)
    hacks = image16(rp, ci, va, N)
    y0 = np.full(M, -0.0)
    y0[::4] = np.random.default_rng(9).standard_normal(len(y0[::4]))
    with np.errstate(invalid="ignore"):
        for start in (None, y0):
            assert np.array_equal(bits(image16_product(hacks, M, N, x, start)), bits(serial(rp, ci, va, x, start)))


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
def check_image_size(A, rp, ci, N):
    """image_index_bytes and image_device_bytes as the numpy model of the eligibility test predicts them."""
    i = A.info()
    index = 2 if narrow_fits(rp, ci, N) else 4
    slots = image_slots(rp)
    assert i.image_index_bytes == index
    assert i.image_device_bytes == (8 + index) * slots
    assert i.image_bytes == 12 * slots
    assert A.image_form().endswith(",uint16_t>" if index == 2 else ",int>"), A.image_form()
    return index


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n", [("lap2d", 33), ("lap2d", 1000), ("lap2d", 4096), ("lap3d", 64), ("lap3d", 127),
                                    ("lap3d", 128), ("lap3d", 200)])
def test_image_width_on_stencils(kind, n):
    """lap2d, and lap3d up to n = 127 (plane offset n^2 <= 16383), get the narrow image; lap3d from n = 128 on the wide."""
    d = dev()
    A = d.DeviceCSR.synth(d.SYNTH_LAP2D if kind == "lap2d" else d.SYNTH_LAP3D, n)
    A.set_image(1)
    i = A.info()
    assert i.auto_algo == d.ALGO_ROW_IMAGE
    rp, ci, _ = A.download()
    assert check_image_size(A, rp, ci, i.N) == (2 if kind == "lap2d" or n * n <= DMAX else 4)
    last = ci[rp[1:][np.diff(rp) > 0] - 1][::97]
    products_equal_row(A, special_x(i.N, last), minus_zero_start(i.M))
    A.close()


@pytest.mark.gpu
@pytest.mark.parametrize("M,N", [(1000, 777), (9001, 3000), (3001, 9000), (40001, 100), (20000, 20000)])
def test_image_width_on_irregular_rows(M, N):
    """Random rows of 0-12 nonzeros, empty rows, columns 0 and N-1, stored zeros, M > N with a padded last hack and
    M < N; narrow up to 9001 x 3000 / 3001 x 9000, wide where columns reach past 2^14."""
    d = dev()
    rng = np.random.default_rng(M)
    rp, ci, va = [0], [], []
    for r in range(M):
        n = 0 if r % 9 == 4 else int(rng.integers(0, min(N, 12) + 1))
        cols = np.sort(rng.choice(N, size=n, replace=False)) if n else np.zeros(0, np.int64)
        if n and r % 4 == 0:
            cols[0] = 0
        if n and r % 6 == 1:
            cols[-1] = N - 1
        cols = np.unique(cols)
        vals = rng.standard_normal(len(cols))
        vals[::5] = 0.0
        ci.extend(cols.tolist())
        va.extend(vals.tolist())
        rp.append(len(ci))
    rp, ci, va = np.array(rp, np.int32), np.array(ci, np.int32), np.array(va)
    A = d.DeviceCSR.upload(M, N, rp, ci, va)
    A.set_image(1)
    assert check_image_size(A, rp, ci, N) == (2 if max(M, N) <= 9001 else 4)
    last = [ci[rp[r + 1] - 1] for r in range(M) if rp[r + 1] > rp[r]]
    products_equal_row(A, special_x(N, last, seed=M), minus_zero_start(M))
    A.close()


def banded(M, N, delta, empty_from=None):
    """Row r: the diagonal column min(r, N - 1), plus r + delta where that is a column; every 7th row empty, and rows from
    empty_from on empty too."""
    rp, ci = [0], []
    for r in range(M):
        if r % 7 != 3 and (empty_from is None or r < empty_from):
            cols = {min(r, N - 1)}
            if delta is not None and 0 <= r + delta < N:
                cols.add(r + delta)
            ci.extend(sorted(cols))
        rp.append(len(ci))
    return np.array(rp, np.int32), np.array(ci, np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("case,index", [("+16383", 2), ("-16384", 2), ("+16384", 4), ("-16385", 4),
                                        ("reach_M16480", 2), ("reach_M16484", 4), ("reach_empty_rows", 4)])
def test_narrow_image_boundaries(case, index):
    """The narrow image exactly where every slot fits, the wide one one step past; rows without columns (empty, or past
    M in the last hack) must reach column N - 1.  Bit for bit ALGO_ROW with +-Inf/NaN in x and accumulate from -0.0, and
    a row-range product that starts and ends inside a hack."""
    import torch
    d = dev()
    if case.startswith("reach"):
        M = {"reach_M16480": 16480, "reach_M16484": 16484, "reach_empty_rows": 16512}[case]
        rp, ci = banded(M, 100, None, empty_from=16484 if case == "reach_empty_rows" else None)
        N = 100
    else:
        M = N = 40000
        rp, ci = banded(M, N, int(case))
    va = np.random.default_rng(len(ci)).standard_normal(len(ci))
    va[::11] = 0.0
    va[5::11] = -0.0
    assert narrow_fits(rp, ci, N) == (index == 2)
    A = d.DeviceCSR.upload(M, N, rp, ci, va)
    A.set_image(1)
    assert check_image_size(A, rp, ci, N) == index
    last = [ci[rp[r + 1] - 1] for r in range(M) if rp[r + 1] > rp[r]]
    x = special_x(N, last[::5], seed=index)
    products_equal_row(A, x, minus_zero_start(M))
    ref = torch.zeros(M, dtype=torch.float64, device="cuda")
    A.spmv(x, ref, algo=d.ALGO_ROW)
    y = torch.full((M,), 7.0, dtype=torch.float64, device="cuda")
    A.spmv_rows(45, M - 13, x, y)
    torch.cuda.synchronize()
    assert torch.equal(tbits(y[45:M - 13]), tbits(ref[45:M - 13]))
    assert bool((y[:45] == 7.0).all()) and bool((y[M - 13:] == 7.0).all())
    A.close()
