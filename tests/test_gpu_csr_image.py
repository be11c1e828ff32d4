"""The private column-major image of a CSR handle (spmv_b200_csr_set_image, SPMV_B200_ALGO_ROW_IMAGE).

Contract (include/spmv_b200.h, "Private image"): a handle that owns its arrays and has no row above 12 nonzeros may hold
an HLL-layout copy of its matrix whose padding slots carry bit 31 of the column.  The masked kernels gather
x[c & 0x7fffffff] for such a slot and skip its add, so every product on the image is bit for bit SPMV_B200_ALGO_ROW (the
serial loop), for every x -- infinities and NaNs included -- and with accumulate from any y, -0.0 included.  The HLL
format's own semantics (add 0 * x[c] for a padding slot) would not be: the CPU test below shows both on a numpy model.

Bits are compared as integers, so NaN payloads count.
"""
import numpy as np
import pytest

HACK = 32
MARK = 0x80000000


# ---------------------------------------------------------------------------------------------------
# numpy model of the two padding schemes (no GPU)
# ---------------------------------------------------------------------------------------------------
def serial(rp, ci, va, x, y0=None):
    """The serial loop: acc = acc + v * x[c] in index order, the multiply and the add rounded separately."""
    M = len(rp) - 1
    y = np.zeros(M) if y0 is None else np.array(y0, np.float64, copy=True)
    for r in range(M):
        acc = y[r]
        for j in range(rp[r], rp[r + 1]):
            acc = acc + va[j] * x[ci[j]]
        y[r] = acc
    return y


def image(rp, ci, va):
    """Column-major, hack-aligned image: per hack (JA, AS) of shape (width, 32); a padding slot repeats the row's last
    real column (0 for an empty row) with bit 31 set and holds 0.0."""
    M = len(rp) - 1
    hacks = []
    for h in range((M + HACK - 1) // HACK):
        rows = range(h * HACK, min(M, (h + 1) * HACK))
        w = max([rp[r + 1] - rp[r] for r in rows] + [0])
        JA = np.full((w, HACK), MARK, np.uint32)
        AS = np.zeros((w, HACK))
        for lr, r in enumerate(rows):
            last = 0
            for j in range(w):
                if rp[r] + j < rp[r + 1]:
                    last = ci[rp[r] + j]
                    JA[j, lr], AS[j, lr] = last, va[rp[r] + j]
                else:
                    JA[j, lr] = last | MARK
        hacks.append((JA, AS))
    return hacks


def image_product(hacks, M, x, masked, y0=None):
    """One lane per row over the image.  masked: a marked slot is skipped (the masked kernels); otherwise it adds
    0 * x[c] like any slot (the HLL format's semantics)."""
    y = np.zeros(M) if y0 is None else np.array(y0, np.float64, copy=True)
    for h, (JA, AS) in enumerate(hacks):
        for lr in range(HACK):
            r = h * HACK + lr
            if r >= M:
                continue
            acc = y[r]
            for j in range(JA.shape[0]):
                c = int(JA[j, lr])
                if masked and c & MARK:
                    continue
                acc = acc + AS[j, lr] * x[c & ~MARK]
            y[r] = acc
    return y


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.int64)


def adversarial_csr(seed=7, M=77, N=41):
    """Rows of 0-12 nonzeros (several empty), columns 0 and N-1, explicitly stored zeros (+0.0 and -0.0)."""
    rng = np.random.default_rng(seed)
    rp, ci, va = [0], [], []
    for r in range(M):
        n = 0 if r % 11 == 3 else int(rng.integers(0, 13))
        cols = np.sort(rng.choice(N, size=n, replace=False))
        if r % 7 == 0 and n:
            cols[0] = 0
        if r % 5 == 0 and n:
            cols[-1] = N - 1
        cols = np.unique(cols)
        vals = rng.standard_normal(len(cols))
        if len(vals) > 2:
            vals[1] = 0.0
            vals[2] = -0.0
        ci.extend(cols.tolist())
        va.extend(vals.tolist())
        rp.append(len(ci))
    return np.array(rp, np.int64), np.array(ci, np.int64), np.array(va), M, N


def adversarial_x(rp, ci, N, seed=8):
    """x with +-Inf and NaN at column 0 and at the last column of rows that have padding slots."""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal(N)
    x[0] = np.inf
    specials = [-np.inf, np.nan, np.inf]
    for r in range(len(rp) - 1):
        if rp[r + 1] > rp[r] and r % 3 == 0:
            x[ci[rp[r + 1] - 1]] = specials[r % len(specials)]
    return x


def test_padding_model_masked_keeps_the_serial_bits():
    """The masked scheme equals the serial loop bit for bit; adding 0 * x[c] for padding does not (NaN from 0 * Inf, and
    +0 flips an untouched -0.0)."""
    rp, ci, va, M, N = adversarial_csr()
    x = adversarial_x(rp, ci, N)
    hacks = image(rp, ci, va)
    y0 = np.full(M, -0.0)
    y0[::4] = np.random.default_rng(9).standard_normal(len(y0[::4]))
    with np.errstate(invalid="ignore"):
        for start in (None, y0):
            ref = serial(rp, ci, va, x, start)
            assert np.array_equal(bits(image_product(hacks, M, x, True, start)), bits(ref))
            assert not np.array_equal(bits(image_product(hacks, M, x, False, start)), bits(ref))
        # each failure mode on its own: an infinite x at a padded row's last column, and a -0.0 start of an empty row
        empty = next(r for r in range(M) if rp[r + 1] == rp[r] and any(rp[q + 1] > rp[q] for q in range(r // HACK * HACK, min(M, r // HACK * HACK + HACK))))
        ref = serial(rp, ci, va, x, y0)
        unmasked = image_product(hacks, M, x, False, y0)
        assert bits(ref)[empty] != bits(unmasked)[empty] or np.isnan(unmasked[empty])
        assert np.isnan(image_product(hacks, M, x, False)).sum() > np.isnan(serial(rp, ci, va, x)).sum()


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
def dev():
    from sparsematrixvectormultiplication_b200 import device
    return device


def tbits(t):
    import torch
    return t.view(torch.int64)


def image_slots(rp):
    lens = np.diff(np.asarray(rp, np.int64))
    pad = (-len(lens)) % HACK
    lens = np.concatenate([lens, np.zeros(pad, np.int64)])
    return int(HACK * lens.reshape(-1, HACK).max(axis=1).sum()) if len(lens) else 0


def products_equal_row(A, x, y0=None, algos=None):
    """AUTO and ROW_IMAGE (and any `algos`) give ALGO_ROW's bits, with and without accumulate."""
    import torch
    d = dev()
    M = A.info().M
    starts = [None] if y0 is None else [None, y0]
    for start in starts:
        ref = torch.zeros(M, dtype=torch.float64, device="cuda") if start is None else start.clone()
        A.spmv(x, ref, accumulate=start is not None, algo=d.ALGO_ROW)
        for algo in algos or (d.ALGO_AUTO, d.ALGO_ROW_IMAGE):
            y = torch.zeros(M, dtype=torch.float64, device="cuda") if start is None else start.clone()
            A.spmv(x, y, accumulate=start is not None, algo=algo)
            torch.cuda.synchronize()
            assert torch.equal(tbits(y), tbits(ref)), f"algo {algo}, accumulate={start is not None}"


def special_x(N, ci_last, seed=1):
    import torch
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(N, dtype=torch.float64, device="cuda", generator=g)
    x[0] = float("inf")
    x[N - 1] = float("nan")
    if len(ci_last):
        idx = torch.as_tensor(np.asarray(ci_last, np.int64), device="cuda")
        x[idx[0::3]] = float("-inf")
        x[idx[1::3]] = float("nan")
    return x


def minus_zero_start(M, seed=2):
    import torch
    y0 = torch.full((M,), -0.0, dtype=torch.float64, device="cuda")
    y0[::3] = torch.randn(len(y0[::3]), dtype=torch.float64, device="cuda")
    return y0


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n", [("lap2d", 64), ("lap2d", 257), ("lap2d", 4096), ("lap3d", 64), ("lap3d", 256)])
def test_image_equals_row_kernel_on_stencils(kind, n):
    d = dev()
    A = d.DeviceCSR.synth(d.SYNTH_LAP2D if kind == "lap2d" else d.SYNTH_LAP3D, n)
    A.set_image(1)
    i = A.info()
    assert i.auto_algo == d.ALGO_ROW_IMAGE
    rp, ci, _ = A.download()
    assert i.image_bytes == 12 * image_slots(rp)
    if kind == "lap2d":
        assert i.image_form >= 64, A.image_form()   # three width runs: the offset-free form
    elif n == 256:
        assert 0 < i.image_form < 64, A.image_form()  # many runs: hll_row_kernel
    last = ci[rp[1:][np.diff(rp) > 0] - 1][::97]
    x = special_x(i.N, last)
    products_equal_row(A, x, minus_zero_start(i.M))
    A.close()


@pytest.mark.gpu
@pytest.mark.parametrize("M,N", [(1000, 777), (33, 5), (31, 1), (4900, 4900)])
def test_image_equals_row_kernel_on_irregular_rows(M, N):
    """M not a multiple of 32, empty rows, random rows of 0-12 nonzeros, columns 0 and N-1, stored zeros; x with +-Inf and
    NaN at column 0 and at padded rows' last columns; accumulate from -0.0."""
    import torch
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
    assert A.info().image_bytes == 12 * image_slots(rp)
    last = [ci[rp[r + 1] - 1] for r in range(M) if rp[r + 1] > rp[r]]
    x = special_x(N, last, seed=M)
    products_equal_row(A, x, minus_zero_start(M))
    # the host-buffer call: the same bits
    xh = x.cpu().numpy()
    ref = torch.zeros(M, dtype=torch.float64, device="cuda")
    A.spmv(x, ref, algo=d.ALGO_ROW)
    for algo in (d.ALGO_AUTO, d.ALGO_ROW_IMAGE):
        yh = A.spmv_host(xh, algo=algo)
        assert np.array_equal(yh.view(np.int64), ref.cpu().numpy().view(np.int64))
    A.close()


def small_lap(n=64):
    d = dev()
    return d.DeviceCSR.synth(d.SYNTH_LAP2D, n)


@pytest.mark.gpu
def test_eligibility_and_lifecycle():
    import torch
    d = dev()
    from sparsematrixvectormultiplication_b200 import _native as NN
    A = small_lap()
    i = A.info()
    x = torch.randn(i.N, dtype=torch.float64, device="cuda")
    # too small for plan-time timing: no image until asked for
    assert i.image_bytes == 0 and i.image_form == 0 and A.image_form() == "none"
    with pytest.raises(NN.SpmvError):
        A.spmv(x, torch.zeros(i.M, dtype=torch.float64, device="cuda"), algo=d.ALGO_ROW_IMAGE)
    A.set_image(1)
    assert A.info().image_bytes > 0 and A.image_form().startswith("hll_rowu_kernel<")
    products_equal_row(A, x)
    # set_image(0) frees the image; AUTO goes back to csr_row_kernel with the same bits
    A.set_image(0)
    assert A.info().image_bytes == 0 and A.info().auto_algo == d.ALGO_ROW
    products_equal_row(A, x, algos=(d.ALGO_AUTO,))
    # replan decides again (no image at this size); the products still equal ALGO_ROW
    A.set_image(1)
    A.replan()
    assert A.info().image_bytes == 0
    products_equal_row(A, x, algos=(d.ALGO_AUTO,))
    # remap_columns rewrites col_idx: the image goes, and a new one multiplies the remapped matrix
    A.set_image(1)
    N0 = i.N
    half = N0 // 2
    stride = half + 3
    A.remap_columns([0, half, N0], stride)
    assert A.info().image_bytes == 0
    xr = torch.zeros(2 * stride, dtype=torch.float64, device="cuda")
    xr[:half] = x[:half]
    xr[stride:stride + N0 - half] = x[half:]
    products_equal_row(A, xr, algos=(d.ALGO_AUTO,))
    A.set_image(1)
    products_equal_row(A, xr)
    A.close()

    # wrapped arrays are the caller's: never an image
    rp = torch.as_tensor(np.arange(0, 2 * 64 + 1, 2, dtype=np.int32), device="cuda")
    ci = torch.as_tensor(np.tile(np.array([0, 5], np.int32), 64), device="cuda")
    va = torch.ones(128, dtype=torch.float64, device="cuda")
    W = d.DeviceCSR.wrap(64, 8, rp, ci, va)
    assert W.info().image_bytes == 0
    with pytest.raises(NN.SpmvError):
        W.set_image(1)
    assert W.info().image_bytes == 0
    W.close()

    # a row of 13 nonzeros: no image
    rp13 = np.array([0, 13, 14], np.int32)
    ci13 = np.array(list(range(13)) + [0], np.int32)
    B = d.DeviceCSR.upload(2, 13, rp13, ci13, np.ones(14))
    with pytest.raises(NN.SpmvError):
        B.set_image(1)
    assert B.info().image_bytes == 0 and B.info().auto_algo != d.ALGO_ROW_IMAGE
    B.close()
