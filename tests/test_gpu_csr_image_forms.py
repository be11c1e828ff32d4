"""Every form the plan can pick for the private image of a CSR handle.

On a matrix of at least 2^22 nonzeros that owns its arrays and has no row above 12 nonzeros, the plan builds every image
form the matrix qualifies for (image_candidates in image.cu), times them on a zero x against the plain row kernels and
keeps the fastest.  The candidates, in the plan's order:
  * column-major, when the image takes at most nnz + nnz / 4 slots: hll_rowu_kernel<4..7> on a regular layout (at most
    8 runs of hacks of equal width), else hll_row_kernel<2..7>; first on the fp64 values, then on 1-byte codes when the
    values hold at most 256 distinct 64-bit patterns; with the 2-byte column field when every slot's col - row fits
    (test_gpu_csr_image_narrow.narrow_fits), else the 4-byte one;
  * then csr_pattern_kernel<W>, when M * W <= nnz + nnz / 4 and the rows hold at most 256 patterns in a dictionary of
    at most 24 KB (test_gpu_csr_image_patterns.row_patterns).
Which form wins depends on the machine and the run, so SPMV_B200_IMAGE_CANDIDATE=i makes the plan keep candidate i
instead (no image past the last one).  The tests walk i = 0, 1, ... until the handle holds no image, check the names
against the model above, and check each kept form's products: bit for bit the serial loop on a finite x, with and without
accumulate from -0.0, and ALGO_ROW's bits up to NaN payloads with +-Inf and NaN in x.
"""
import numpy as np
import pytest

from test_gpu_csr_image import HACK, dev, minus_zero_start, special_x, tbits
from test_gpu_csr_image_narrow import narrow_fits
from test_gpu_csr_image_patterns import make_pool
from test_gpu_csr_image_values import same_bits_up_to_nan_payload, special_values, value_table

ENV = "SPMV_B200_IMAGE_CANDIDATE"
MAX_SEGMENTS = 8
MAX_DISTINCT = 256
DICT_BYTES = 24 * 1024
MIN_NNZ = 1 << 22


# ---------------------------------------------------------------------------------------------------
# the model of image_candidates (no GPU)
# ---------------------------------------------------------------------------------------------------
def hack_widths(lens):
    """The width of every hack of 32 rows (rows past M count as empty)."""
    lens = np.asarray(lens, np.int64)
    lens = np.concatenate([lens, np.zeros((-len(lens)) % HACK, np.int64)])
    return lens.reshape(-1, HACK).max(axis=1) if len(lens) else np.zeros(0, np.int64)


def regular(widths):
    """hll_find_segments: at most 8 runs of hacks of equal width."""
    return len(widths) > 0 and 1 + int(np.count_nonzero(widths[1:] != widths[:-1])) <= MAX_SEGMENTS


def pattern_count(rp, ci, va):
    """The number of distinct row patterns (length, col - row as uint32, value bits; zero past the length)."""
    rp = np.asarray(rp, np.int64)
    lens = np.diff(rp)
    M, W = len(lens), int(lens.max())
    rows = np.repeat(np.arange(M), lens)
    slot = np.arange(len(ci)) - np.repeat(rp[:-1], lens)
    key = np.zeros((M, 1 + 2 * W), np.uint64)
    key[:, 0] = lens
    key[rows, 1 + slot] = (np.asarray(ci, np.int64) - rows).astype(np.uint32)
    key[rows, 1 + W + slot] = np.ascontiguousarray(va, np.float64).view(np.uint64)
    return len(np.unique(key, axis=0))


def candidate_names(regular_layout, index, coded, pattern_width):
    """The names image_form() gives the candidates, in the plan's order.  index: 'uint16_t', 'int' or None (no
    column-major form); pattern_width: W of the pattern form, or None."""
    names = []
    if index:
        kernel, batches = ("hll_rowu_kernel", range(4, 8)) if regular_layout else ("hll_row_kernel", range(2, 8))
        for stream in [""] + ([",uint8_t"] if coded else []):
            names += [f"{kernel}<{b},double,true,{index}{stream}>" for b in batches]
    if pattern_width:
        names.append(f"csr_pattern_kernel<{pattern_width}>")
    return names


def image_candidates(rp, ci, va, N):
    rp = np.asarray(rp, np.int64)
    lens = np.diff(rp)
    M, nnz = len(lens), len(ci)
    W = int(lens.max()) if M else 0
    limit = nnz + nnz // 4
    widths = hack_widths(lens)
    index = None
    if HACK * int(widths.sum()) <= limit:
        index = "uint16_t" if narrow_fits(rp, ci, N) else "int"
    pattern = None
    if 1 <= W <= 12 and M * W <= limit:
        P = pattern_count(rp, ci, va)
        pattern = W if P <= MAX_DISTINCT and 12 * W * P <= DICT_BYTES else None
    return candidate_names(regular(widths), index, value_table(va) is not None, pattern)


# ---------------------------------------------------------------------------------------------------
# the matrices
# ---------------------------------------------------------------------------------------------------
def hack_lengths(M, widths, rng):
    """Row lengths for hacks of the given widths: each hack's first row and 15 in 16 of the others at the width, the
    rest shorter (0 up to the width), so the image wastes few slots and the padding is real."""
    w = np.repeat(np.asarray(widths, np.int64), HACK)[:M]
    lens = np.where(rng.random(M) < 15 / 16, w, rng.integers(0, w + 1))
    lens[::HACK] = w[::HACK]
    return lens


def csr_from_lengths(lens, N, rng, narrow, values):
    """Columns for the given row lengths: near the row (col - row in [-6, 5], clamped into [0, N), narrow) or one per
    twelfth of [0, N) (wide, with column 0 and N - 1 in some rows); values drawn from `values` (an array: every entry
    present) or standard normal (None)."""
    lens = np.asarray(lens, np.int64)
    M = len(lens)
    rp = np.concatenate([[0], np.cumsum(lens)])
    nnz = int(rp[-1])
    rows = np.repeat(np.arange(M), lens)
    k = np.arange(nnz) - np.repeat(rp[:-1], lens)
    if narrow:
        ci = np.clip(rows - 6, 0, N - 12) + k
    else:
        band = N // 12
        ci = k * band + rng.integers(0, band, nnz)
        nz = np.nonzero(lens > 0)[0]
        ci[rp[nz[nz % 4 == 0]]] = 0
        ci[rp[nz[nz % 6 == 1] + 1] - 1] = N - 1
    if values is None:
        va = rng.standard_normal(nnz)
    else:
        va = rng.choice(values, nnz)
        va[:len(values)] = values
    return rp.astype(np.int32), ci.astype(np.int32), va


def pool_rows(M, N, pool, rng):
    """banded_pool's rows, drawn without its per-row search: a row takes a random pattern of the pool and stays empty
    when that pattern leaves [0, N) or r % 12 == 5."""
    lens = np.array([len(p[0]) for p in pool])
    W = int(lens.max())
    deltas = np.array([p[0] + [0] * (W - len(p[0])) for p in pool])
    vals = np.array([p[1] + [0.0] * (W - len(p[1])) for p in pool])
    pick = rng.integers(0, len(pool), M)
    r = np.arange(M)
    cols = r[:, None] + deltas[pick]
    inside = np.arange(W)[None, :] < lens[pick][:, None]
    ok = np.all(~inside | ((cols >= 0) & (cols < N)), axis=1) & (r % 12 != 5)
    keep = inside & ok[:, None]
    rp = np.concatenate([[0], np.cumsum(keep.sum(axis=1))]).astype(np.int32)
    return rp, cols[keep].astype(np.int32), vals[pick][keep]


RUNS8 = [0, 1, 3, 4, 5, 7, 12, 6]


def matrix(name):
    """(rp, ci, va, M, N, values_special) of the named case; the stencils are generated on the device instead."""
    rng = np.random.default_rng(sum(map(ord, name)))
    if name in ("random_special", "random_distinct"):
        M = N = 1 << 20
        lens = hack_lengths(M, rng.integers(0, 13, M // HACK), rng)
        pool = np.concatenate([special_values(), rng.standard_normal(20)]) if name == "random_special" else None
        return csr_from_lengths(lens, N, rng, False, pool) + (M, N, name == "random_special")
    if name in ("runs8", "runs9"):
        widths = RUNS8 + ([2] if name == "runs9" else [])
        M = 1_000_003 if name == "runs8" else 1_100_011
        N = (1 << 20) if name == "runs8" else M - 1000
        nh = (M + HACK - 1) // HACK
        per_hack = np.array(widths)[np.arange(nh) * len(widths) // nh]
        lens = hack_lengths(M, per_hack, rng)
        pool = np.array([1.0, -2.0, 0.5, -0.0, 3.75])
        return csr_from_lengths(lens, N, rng, name == "runs9", pool) + (M, N, False)
    if name == "pattern_pool":
        M = N = 460_000
        pool = make_pool(100, 12, span=40, lengths=(10, 12))
        return pool_rows(M, N, pool, rng) + (M, N, False)
    raise KeyError(name)


GENERATED = {
    "random_special": candidate_names(False, "int", True, None),
    "random_distinct": candidate_names(False, "int", False, None),
    "runs8": candidate_names(True, "int", True, None),
    "runs9": candidate_names(False, "uint16_t", True, None),
    "pattern_pool": candidate_names(True, "uint16_t", True, 12),
}
STENCILS = {
    ("lap2d", 1024): candidate_names(True, "uint16_t", True, 5),
    ("lap3d", 96): candidate_names(False, "uint16_t", True, 7),
}


def test_candidate_model_on_small_layouts():
    """The runs rule at 8 and 9 runs, the slot limit, the narrow field and the pattern limits, on small matrices."""
    assert regular(np.array(RUNS8).repeat(3)) and not regular(np.array(RUNS8 + [2]).repeat(3))
    assert regular(np.array([5])) and not regular(np.zeros(0, np.int64))
    assert not regular(np.array([4, 5, 4, 5, 4, 5, 4, 5, 4]))
    # the diagonal with 3 values: 1 run, narrow, 3 patterns of width 1
    M = 64
    rp, ci, va = np.arange(M + 1), np.arange(M), 1.0 + np.arange(M) % 3
    assert image_candidates(rp, ci, va, M) == candidate_names(True, "uint16_t", True, 1)
    assert len(image_candidates(rp, ci, va, M)) == 9
    # one row of 12 among rows of 1: the hack of width 12 takes 12 * 32 slots, past nnz + nnz / 4
    lens = np.ones(M, np.int64)
    lens[5] = 12
    rp = np.concatenate([[0], np.cumsum(lens)])
    ci = np.concatenate([[r] if n == 1 else np.arange(12) for r, n in enumerate(lens)])
    assert image_candidates(rp, ci, np.ones(len(ci)), 100) == []
    # 257 distinct values: no codes, and 257 patterns: no pattern form; a column 2^14 + 1 away: the wide field
    M = 512
    rp, ci, va = np.arange(M + 1), np.arange(M), np.arange(M, dtype=np.float64) % 257
    assert image_candidates(rp, ci, va, M) == candidate_names(True, "uint16_t", False, None)
    ci = ci.copy()
    ci[7] = 7 + 16384
    assert image_candidates(rp, ci, np.ones(M), M + 16384) == candidate_names(True, "int", True, 1)


@pytest.mark.parametrize("name", sorted(GENERATED))
def test_generated_matrices_offer_the_intended_forms(name):
    """Each generated matrix is large enough for the plan to time its candidates and offers the forms it is meant to
    reach (every batch, both column fields, both value streams, the pattern form at W = 12)."""
    rp, ci, va, M, N, _ = matrix(name)
    assert len(ci) >= MIN_NNZ
    if name.startswith("runs"):
        assert M % HACK != 0 and (N < M) == (name == "runs9")
    assert image_candidates(rp, ci, va, N) == GENERATED[name]


def test_stencils_offer_the_intended_forms():
    from sparsematrixvectormultiplication_b200 import synth
    for (kind, n), expect in STENCILS.items():
        rp, ci, va = (synth.lap2d_csr if kind == "lap2d" else synth.lap3d_csr)(n)
        assert len(ci) >= MIN_NNZ
        assert image_candidates(rp, ci, va, len(rp) - 1) == expect, (kind, n)


def test_coverage_of_the_walk():
    """Together the matrices offer every batch of both kernels with both column fields and both value streams."""
    names = set()
    for expect in list(GENERATED.values()) + list(STENCILS.values()):
        names.update(expect)
    for index in ("int", "uint16_t"):
        for stream in ("", ",uint8_t"):
            for b in range(2, 8):
                assert f"hll_row_kernel<{b},double,true,{index}{stream}>" in names
            for b in range(4, 8):
                assert f"hll_rowu_kernel<{b},double,true,{index}{stream}>" in names


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
def walk(A, monkeypatch):
    """Yields the name of every image candidate the plan keeps under SPMV_B200_IMAGE_CANDIDATE = 0, 1, ...; the walk
    ends at the first index that leaves the handle without an image, and there are at most 13 candidates."""
    d = dev()
    for i in range(14):
        monkeypatch.setenv(ENV, str(i))
        A.replan()
        name = A.image_form()
        if name == "none":
            assert A.info().auto_algo != d.ALGO_ROW_IMAGE
            return
        assert A.info().auto_algo == d.ALGO_ROW_IMAGE
        yield name
    raise AssertionError(f"{ENV}=13 still leaves an image: the plan ignores the switch")


class Oracle:
    """The serial loop's y for one finite x, plain and accumulating from a start that holds -0.0."""

    def __init__(self, rp, ci, va, M, N, checker, seed=5):
        import torch
        g = torch.Generator(device="cuda").manual_seed(seed)
        self.x = torch.randn(N, dtype=torch.float64, device="cuda", generator=g)
        self.y0 = minus_zero_start(M)
        xh = self.x.cpu().numpy()
        self.ref = {False: checker.spmv_csr_serial(rp, ci, va, xh),
                    True: checker.spmv_csr_serial(rp, ci, va, xh, y=self.y0.cpu().numpy().copy())}


def equal(y, ref, nan_payloads_free):
    import torch
    ref = torch.as_tensor(ref, device=y.device)
    return same_bits_up_to_nan_payload(y, ref) if nan_payloads_free else torch.equal(tbits(y), tbits(ref))


def check_kept_form(A, name, orc, xs, M, nan_values):
    """The products of the form the handle holds: AUTO and ROW_IMAGE against the serial oracle on a finite x (NaN
    payloads aside only when the values hold NaN), and against ALGO_ROW up to NaN payloads on x with +-Inf and NaN;
    plain and accumulating.  Under the pattern form, spmv_rows over rows that start and end inside a hack too."""
    import torch
    d = dev()
    for acc in (False, True):
        for algo in (d.ALGO_AUTO, d.ALGO_ROW_IMAGE):
            y = orc.y0.clone() if acc else torch.zeros(M, dtype=torch.float64, device="cuda")
            A.spmv(orc.x, y, accumulate=acc, algo=algo)
            assert equal(y, orc.ref[acc], nan_values), f"{name}: algo {algo}, accumulate={acc}, finite x"
            ref = orc.y0.clone() if acc else torch.zeros(M, dtype=torch.float64, device="cuda")
            A.spmv(xs, ref, accumulate=acc, algo=d.ALGO_ROW)
            y = orc.y0.clone() if acc else torch.zeros(M, dtype=torch.float64, device="cuda")
            A.spmv(xs, y, accumulate=acc, algo=algo)
            assert same_bits_up_to_nan_payload(y, ref), f"{name}: algo {algo}, accumulate={acc}, x with +-Inf and NaN"
    if name.startswith("csr_pattern_kernel"):
        lo, hi = 45, M - 13
        y = torch.full((M,), 7.0, dtype=torch.float64, device="cuda")
        A.spmv_rows(lo, hi, orc.x, y)
        assert equal(y[lo:hi], orc.ref[False][lo:hi], nan_values), f"{name}: spmv_rows"
        assert bool((y[:lo] == 7.0).all()) and bool((y[hi:] == 7.0).all())


def walk_and_check(A, rp, ci, va, M, N, expect, nan_values, checker, monkeypatch):
    import torch
    orc = Oracle(rp, ci, va, M, N, checker)
    lens = np.diff(np.asarray(rp, np.int64))
    widths = np.repeat(hack_widths(lens), HACK)[:M]
    padded = np.nonzero((lens > 0) & (lens < widths))[0]
    xs = special_x(N, np.asarray(ci)[np.asarray(rp)[padded[::97] + 1] - 1], seed=M)
    walked = []
    for name in walk(A, monkeypatch):
        walked.append(name)
        check_kept_form(A, name, orc, xs, M, nan_values)
        torch.cuda.synchronize()
    assert walked == expect
    print(f"walked {len(walked)}: {', '.join(walked)}")
    # without the switch the plan keeps whichever form is fastest here, or none
    monkeypatch.delenv(ENV)
    A.replan()
    assert A.image_form() in walked + ["none"]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n", sorted(STENCILS))
def test_walk_stencils(kind, n, checker, monkeypatch):
    d = dev()
    A = d.DeviceCSR.synth(d.SYNTH_LAP2D if kind == "lap2d" else d.SYNTH_LAP3D, n)
    rp, ci, va = A.download()
    i = A.info()
    walk_and_check(A, rp, ci, va, i.M, i.N, STENCILS[(kind, n)], False, checker, monkeypatch)
    A.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(GENERATED))
def test_walk_generated(name, checker, monkeypatch):
    d = dev()
    rp, ci, va, M, N, nan_values = matrix(name)
    A = d.DeviceCSR.upload(M, N, rp, ci, va)
    walk_and_check(A, rp, ci, va, M, N, GENERATED[name], nan_values, checker, monkeypatch)
    A.close()


# ---------------------------------------------------------------------------------------------------
# lap3d 512: images past 2^31 bytes
# ---------------------------------------------------------------------------------------------------
def lap3d_hack_offsets(n):
    """The image's first slot of every hack (and the total), from the row lengths of the 7-point stencil."""
    import torch
    r = torch.arange(n ** 3, device="cuda")
    lens = torch.full((n ** 3,), 7, dtype=torch.int8, device="cuda")
    for c in (r // (n * n), (r // n) % n, r % n):
        lens -= (c == 0).to(torch.int8) + (c == n - 1).to(torch.int8)
    del r
    widths = torch.nn.functional.pad(lens, (0, (-n ** 3) % HACK)).view(-1, HACK).amax(dim=1).long()
    return torch.cat([torch.zeros(1, dtype=torch.long, device="cuda"), torch.cumsum(widths * HACK, 0)]).cpu().numpy()


class MemoryPeak:
    """The most device memory in use, sampled every 5 ms (cudaMemGetInfo, so other processes' memory counts too)."""

    def __enter__(self):
        import threading
        import torch
        self.peak, self._stop = 0, threading.Event()

        def sample():
            while not self._stop.is_set():
                free, total = torch.cuda.mem_get_info()
                self.peak = max(self.peak, total - free)
                self._stop.wait(0.005)
        self._thread = threading.Thread(target=sample, daemon=True)
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join()


@pytest.mark.gpu
def test_walk_lap3d_512(checker, monkeypatch):
    """lap3d 512 (938 M nonzeros): the column-major images hold about 938 M slots, so fp64 values pass 2^31 bytes at
    slot 2^28 and the 4-byte column field at slot 2^29.  Every candidate: the whole y torch.equal to ALGO_ROW for a hash
    x, and 2^21-row windows around those slots and at the end bit for bit the serial loop on the numpy twin."""
    import time
    import torch
    from sparsematrixvectormultiplication_b200 import synth
    d = dev()
    n = 512
    M = n ** 3
    off = lap3d_hack_offsets(n)
    assert off[-1] > 1 << 29
    rows = [int(np.searchsorted(off, s, side="right") - 1) * HACK for s in (1 << 28, 1 << 29)]
    half = 1 << 20
    windows = [(r - half, r + half) for r in rows] + [(M - 2 * half, M)]
    A = d.DeviceCSR.synth(d.SYNTH_LAP3D, n)
    x = torch.empty(M, dtype=torch.float64, device="cuda")
    d.synth_vector(x, 4242)
    xh = x.cpu().numpy()
    want = []
    for lo, hi in windows:
        rp, ci, va = synth.lap3d_csr(n, lo, hi)
        want.append(checker.spmv_csr_serial(rp, ci, va, xh))
    del xh
    ref = torch.empty(M, dtype=torch.float64, device="cuda")
    A.spmv(x, ref, algo=d.ALGO_ROW)
    y = torch.empty_like(ref)
    base = torch.cuda.mem_get_info()
    expect = candidate_names(False, "int", True, 7)
    walked = []
    t0 = time.perf_counter()
    with MemoryPeak() as peak:
        for name in walk(A, monkeypatch):
            walked.append(name)
            for algo in (d.ALGO_AUTO, d.ALGO_ROW_IMAGE):
                y.fill_(float("nan"))
                A.spmv(x, y, algo=algo)
                assert torch.equal(y, ref), f"{name}: algo {algo}"
                for (lo, hi), w in zip(windows, want):
                    assert np.array_equal(y[lo:hi].cpu().numpy().view(np.int64), w.view(np.int64)), (name, algo, lo)
    seconds = time.perf_counter() - t0
    assert walked == expect
    print(f"lap3d 512 walk: {len(walked)} candidates in {seconds:.1f} s; device memory in use at most "
          f"{peak.peak / 2 ** 30:.1f} GiB ({(base[1] - base[0]) / 2 ** 30:.1f} GiB before the walk); windows {windows}")
    A.close()
