"""The dictionaries of the CSR handle's private image under crafted keys.

distinct_kernel (image.cu) collects the distinct value patterns of the coded form and the distinct rows of the pattern
form in an open-addressing set of 1024 slots: a key's probe starts at slot hash & 1023, walks at most 257 slots and wraps
at 1024.  A value's hash is mix64 of its 64-bit pattern; the all-ones pattern (the set's empty mark) never enters the set
and is added to the table on the host.  A row's hash chains mix64 over its length, then col - row and the value bits of
each nonzero; the set stores the top 33 bits of that hash (the tag) and a representative row, and a probe that meets its
own tag compares the two rows in full.  The warp merge ahead of the probe trusts the 64-bit hash alone, so two different
rows of equal hash in one warp cannot both be placed, and pattern_fill_kernel then fails the build.

Random and stencil data never reach these branches.  mix64 is a bijection, so they can be reached on purpose: the CPU
part below models mix64, its inverse and both hashes, and crafts the last value of a row (or a value) so that its hash
equals a target, or matches it in chosen bits.  The model is trusted through its controls on the GPU: every crafted case
comes with a twin that must come out the other way (one builds, one fails).
"""
import struct

import numpy as np
import pytest

from test_gpu_csr_image import dev, minus_zero_start, products_equal_row, special_x
from test_gpu_csr_image_patterns import check_pattern_form, row_patterns
from test_gpu_csr_image_values import check_coded, check_products, irregular, value_table

MASK = (1 << 64) - 1
SET_SLOTS = 1024
MAX_DISTINCT = 256
ALL_ONES = 0xFFFFFFFFFFFFFFFF
ROW_SEED = 0x9E3779B97F4A7C15
FREE_BITS = ((1 << 31) - 1) & ~(SET_SLOTS - 1)  # bits 10-30: neither in the tag nor in the start slot


# ---------------------------------------------------------------------------------------------------
# the model (no GPU)
# ---------------------------------------------------------------------------------------------------
def mix64(z):
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & MASK
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & MASK
    return z ^ (z >> 31)


def _unshift(z, s):
    """The inverse of z ^ (z >> s)."""
    r = z
    for _ in range(64 // s + 1):
        r = z ^ (r >> s)
    return r & MASK


def unmix64(z):
    z = _unshift(z, 31)
    z = (z * pow(0x94D049BB133111EB, -1, 1 << 64)) & MASK
    z = _unshift(z, 27)
    z = (z * pow(0xBF58476D1CE4E5B9, -1, 1 << 64)) & MASK
    return _unshift(z, 30)


def f2u(v):
    return struct.unpack("<Q", struct.pack("<d", v))[0]


def u2f(b):
    return struct.unpack("<d", struct.pack("<Q", b))[0]


def value_key(v):
    """ValueKeys::key: mix64 of the value's 64-bit pattern."""
    return mix64(f2u(v))


def _row_state(deltas, vals, length):
    h = mix64((ROW_SEED + length) & MASK)
    for d, v in zip(deltas, vals):
        h = mix64(h ^ (d & 0xFFFFFFFF))
        h = mix64(h ^ f2u(v))
    return h


def row_key(deltas, vals):
    """RowKeys::key of a row with nonzeros at col - row = deltas holding vals."""
    assert len(deltas) == len(vals)
    return _row_state(deltas, vals, len(deltas))


def tag(h):
    return h >> 31


def start_slot(h):
    return h & (SET_SLOTS - 1)


def last_value_for(deltas, vals, target):
    """The value v that gives the row (deltas, vals + [v]) the hash target."""
    h = _row_state(deltas[:-1], vals, len(deltas))
    h = mix64(h ^ (deltas[-1] & 0xFFFFFFFF))
    return u2f(unmix64(target) ^ h)


def moderate(v):
    return v == v and 2.0 ** -20 <= abs(v) <= 2.0 ** 20


def craft_one(target, deltas):
    """A row of one nonzero whose hash is target, its delta from `deltas` chosen so that the value is moderate."""
    for d in deltas:
        v = last_value_for([d], [], target)
        if moderate(v):
            return d, v
    raise AssertionError("no moderate value")


def craft_matching(target, keep, delta, rng):
    """A row of one nonzero at `delta` whose hash agrees with target in the bits of `keep` and differs from it; the
    free bits are drawn until the value is moderate."""
    while True:
        h = (target & keep) | (int(rng.integers(0, 1 << 63)) * 2 + int(rng.integers(0, 2))) & ~keep & MASK
        if h == target:
            continue
        v = last_value_for([delta], [], h)
        if moderate(v):
            return v


def craft_values_at_slot(count, slot, rng):
    """count distinct moderate values whose hashes all start their probe at `slot`."""
    out = set()
    while len(out) < count:
        h = (int(rng.integers(0, 1 << 53)) << 10) | slot
        v = u2f(unmix64(h & MASK))
        if moderate(v):
            out.add(v)
    return sorted(out)


def craft_rows_at_slot(count, slot, rng):
    """count distinct one-nonzero rows (delta 0) whose hashes all start their probe at `slot`."""
    out = set()
    while len(out) < count:
        h = (int(rng.integers(0, 1 << 53)) << 10) | slot
        v = last_value_for([0], [], h & MASK)
        if moderate(v):
            out.add(v)
    return sorted(out)


ROW_A = ((0, 1), (4.0, -1.0))  # the row every crafted collision is aimed at


def full_collision():
    """(delta, value) of a one-nonzero row whose 64-bit hash equals ROW_A's."""
    return craft_one(row_key(*ROW_A), range(2, 60))


def tag_collision(seed=11):
    """(delta, value) of a one-nonzero row whose hash shares ROW_A's tag (top 33 bits) and start slot (low 10 bits) but
    not bits 10-30."""
    d = 3
    return d, craft_matching(row_key(*ROW_A), MASK & ~FREE_BITS, d, np.random.default_rng(seed))


def test_mix64_round_trip():
    rng = np.random.default_rng(1)
    for z in [0, 1, MASK, ALL_ONES - 1, ROW_SEED] + [int(v) for v in rng.integers(0, 1 << 63, 2000, dtype=np.int64)]:
        assert unmix64(mix64(z)) == z and mix64(unmix64(z)) == z
    # the model of RowKeys::key sees what the patterns are made of: length, deltas as uint32, value bits
    assert row_key([0, 1], [4.0, -1.0]) != row_key([0, 2], [4.0, -1.0])
    assert row_key([0], [0.0]) != row_key([0], [-0.0])
    assert row_key([0], [1.0]) != row_key([0, 0], [1.0, 1.0])
    assert row_key([-1], [1.0]) == row_key([0xFFFFFFFF], [1.0])  # col - row is hashed as a 32-bit word


def test_crafted_keys_under_the_model():
    """Each crafted case has the property its GPU test relies on, and the deltas stay small."""
    hA = row_key(*ROW_A)
    d, v = full_collision()
    assert moderate(v) and 2 <= d < 60 and row_key([d], [v]) == hA and ([d], [v]) != list(map(list, ROW_A))
    d, v = tag_collision()
    h = row_key([d], [v])
    assert moderate(v) and h != hA and tag(h) == tag(hA) and start_slot(h) == start_slot(hA)
    assert (h & FREE_BITS) != (hA & FREE_BITS)
    rng = np.random.default_rng(2)
    vals = craft_values_at_slot(MAX_DISTINCT + 1, SET_SLOTS - 1, rng)
    assert len(set(f2u(x) for x in vals)) == MAX_DISTINCT + 1
    assert all(start_slot(value_key(x)) == SET_SLOTS - 1 and moderate(x) for x in vals)
    rows = craft_rows_at_slot(MAX_DISTINCT + 1, SET_SLOTS - 1, rng)
    assert len(set(rows)) == MAX_DISTINCT + 1
    assert all(start_slot(row_key([0], [x])) == SET_SLOTS - 1 and moderate(x) for x in rows)
    # the empty mark is a value like any other in the model of the table
    assert u2f(ALL_ONES) != u2f(ALL_ONES) and value_table(np.array([1.0, u2f(ALL_ONES)]))[-1] == ALL_ONES


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
def rows_matrix(M, placed, fill=((0,), (2.0,))):
    """M x M: row r holds placed[r] = (deltas, values) where given, else the one-nonzero row `fill`."""
    rp, ci, va = [0], [], []
    for r in range(M):
        deltas, vals = placed.get(r, fill)
        assert all(0 <= r + d < M for d in deltas)
        ci.extend(r + d for d in deltas)
        va.extend(vals)
        rp.append(len(ci))
    return np.array(rp, np.int32), np.array(ci, np.int32), np.array(va, np.float64)


def exact_products(A, rp, ci, va, checker, seed=3):
    """AUTO and ROW_IMAGE on a finite x, plain and accumulating from -0.0, against the serial oracle bit for bit."""
    import torch
    d = dev()
    M = len(rp) - 1
    x = torch.randn(A.info().N, dtype=torch.float64, device="cuda", generator=torch.Generator(device="cuda").manual_seed(seed))
    y0 = minus_zero_start(M)
    xh = x.cpu().numpy()
    for start in (None, y0):
        ref = checker.spmv_csr_serial(rp, ci, va, xh, y=None if start is None else start.cpu().numpy().copy())
        for algo in (d.ALGO_AUTO, d.ALGO_ROW_IMAGE):
            y = torch.zeros(M, dtype=torch.float64, device="cuda") if start is None else start.clone()
            A.spmv(x, y, accumulate=start is not None, algo=algo)
            assert np.array_equal(y.cpu().numpy().view(np.int64), ref.view(np.int64)), (algo, start is not None)


def held_state(A):
    i = A.info()
    return (i.image_form, i.image_bytes, i.image_device_bytes, i.image_index_bytes, i.image_value_bytes, i.image_patterns,
            i.auto_algo, A.image_form())


def assert_build_fails_unchanged(A, mode, M, x):
    """set_image(mode) raises SpmvError and leaves the held image, its info and its products as they were."""
    from sparsematrixvectormultiplication_b200 import _native as NN
    before = held_state(A)
    with pytest.raises(NN.SpmvError):
        A.set_image(mode)
    assert held_state(A) == before
    products_equal_row(A, x, minus_zero_start(M), algos=None if before[0] else (dev().ALGO_AUTO,))


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["same_warp", "other_warp", "repeated"])
def test_full_hash_collision(where, checker):
    """Two different rows of equal 64-bit hash.  In one warp, and nowhere else, the warp merge keeps one of them and the
    build must fail cleanly; with the second row in another warp, or repeated in one, both patterns are counted."""
    import torch
    d = dev()
    M = 2000
    dB, vB = full_collision()
    B = ((dB,), (vB,))
    placed = {0: ROW_A, 1: B} if where != "other_warp" else {0: ROW_A, 40: B}
    if where == "repeated":
        placed[100] = B
    rp, ci, va = rows_matrix(M, placed)
    assert len(row_patterns(rp, ci, va)[1]) == 3
    A = d.DeviceCSR.upload(M, M, rp, ci, va)
    x = torch.randn(M, dtype=torch.float64, device="cuda")
    if where == "same_warp":
        A.set_image(1)
        assert_build_fails_unchanged(A, 3, M, x)
        A.set_image(0)
        assert_build_fails_unchanged(A, 3, M, x)
    else:
        A.set_image(3)
        check_pattern_form(A, M, M, 2, 3, special_x(M, ci[::7], seed=4))
        exact_products(A, rp, ci, va, checker)
    A.close()


@pytest.mark.gpu
def test_tag_collision(checker):
    """Two rows of one warp with the same tag and start slot but different bits 10-30: the probe's full-row compare keeps
    both, every row gets its own id (the crafted row's value is not ROW_A's, so a shared id changes the product)."""
    d = dev()
    M = 2000
    dB, vB = tag_collision()
    placed = {0: ROW_A, 1: ((dB,), (vB,)), 2: ROW_A, 33: ((dB,), (vB,)), 70: ROW_A}
    rp, ci, va = rows_matrix(M, placed)
    assert len(row_patterns(rp, ci, va)[1]) == 3
    A = d.DeviceCSR.upload(M, M, rp, ci, va)
    A.set_image(3)
    check_pattern_form(A, M, M, 2, 3, special_x(M, ci[::7], seed=5))
    exact_products(A, rp, ci, va, checker)
    A.close()


@pytest.mark.gpu
@pytest.mark.parametrize("count", [256, 257])
def test_one_probe_chain_of_rows(count, checker):
    """count distinct rows whose hashes all start at slot 1023: the chain wraps to slot 0 and holds 256 of them; a 257th
    fails the build and leaves the handle as it was."""
    import torch
    d = dev()
    vals = craft_rows_at_slot(count, SET_SLOTS - 1, np.random.default_rng(count))
    M = 2000
    placed = {r: ((0,), (vals[r % count],)) for r in range(M)}
    rp, ci, va = rows_matrix(M, placed)
    A = d.DeviceCSR.upload(M, M, rp, ci, va)
    if count <= MAX_DISTINCT:
        A.set_image(3)
        check_pattern_form(A, M, M, 1, count, special_x(M, ci[::37], seed=count))
        exact_products(A, rp, ci, va, checker)
    else:
        A.set_image(1)
        assert_build_fails_unchanged(A, 3, M, torch.randn(M, dtype=torch.float64, device="cuda"))
    A.close()


@pytest.mark.gpu
@pytest.mark.parametrize("count", [256, 257])
def test_one_probe_chain_of_values(count):
    """The same for the coded form: count distinct values whose mix64 all start at slot 1023."""
    import torch
    d = dev()
    pool = np.array(craft_values_at_slot(count, SET_SLOTS - 1, np.random.default_rng(count + 7)))
    M = N = 2000
    rp, ci, va = irregular(M, N, pool, count)
    assert len(np.unique(va.view(np.uint64))) == count
    A = d.DeviceCSR.upload(M, N, rp, ci, va)
    if count <= MAX_DISTINCT:
        A.set_image(2)
        check_coded(A, rp, ci, va, N)
        check_products(A, special_x(N, [], seed=count), M)
    else:
        A.set_image(1)
        assert_build_fails_unchanged(A, 2, M, torch.randn(N, dtype=torch.float64, device="cuda"))
    A.close()


@pytest.mark.gpu
def test_all_ones_value_in_patterns(checker):
    """Rows whose values include the all-ones pattern (a NaN): the pattern form stores it in its dictionary like any
    other value; a row entry of the set never equals the empty mark."""
    import torch
    d = dev()
    M = 3000
    ones = u2f(ALL_ONES)
    kinds = [((0, 1), (ones, 2.0)), ((0, 1), (1.0, ones)), ((-1, 0), (ones, ones)), ((0,), (3.0,))]
    placed = {r: kinds[(r * 7) % 4] for r in range(1, M - 1)}
    placed[0] = kinds[0]
    placed[M - 1] = kinds[2]
    rp, ci, va = rows_matrix(M, placed)
    assert len(row_patterns(rp, ci, va)[1]) == 4
    A = d.DeviceCSR.upload(M, M, rp, ci, va)
    A.set_image(3)
    x = special_x(M, ci[::11], seed=9)  # +-Inf, and no NaN of another payload to meet the all-ones one in a sum
    check_pattern_form(A, M, M, 2, 4, torch.nan_to_num(x, nan=float("-inf"), posinf=float("inf"), neginf=float("-inf")))
    A.close()
