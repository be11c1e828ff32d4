"""The tiled kernel of the pattern form: a CTA multiplies 1024 rows from windows of x staged in shared memory.

Contract (include/spmv_b200.h, image_windows): at build time the distinct col - row of the real slots of all patterns are
sorted and clustered, neighbours less than 32 apart sharing a cluster.  A tile stages one window of x per cluster when
there are at most min(W, 3) clusters, none spans more than 256, and the slot records (16 bytes per pattern and slot)
plus the windows (1024 + span + 1 words, rounded up to whole 16-byte vectors) take at most 26 KB; image_windows is then
the cluster count, else 0 and the form gathers x from global memory.  Either way the image's bytes, its form number and
the product's bits are those of test_gpu_csr_image_patterns.py: ALGO_ROW's up to NaN payloads, the serial loop's on
finite x.
"""
import numpy as np
import pytest

from test_gpu_csr_image import bits, dev, minus_zero_start, serial, special_x, tbits
from test_gpu_csr_image_patterns import banded_pool, check_pattern_form, make_pool, row_patterns
from test_gpu_csr_image_values import same_bits_up_to_nan_payload

TILE_ROWS = 1024
MAX_WINDOWS = 3
GAP = 32
MAX_SPAN = 256
SMEM_MAX = 26 * 1024


# ---------------------------------------------------------------------------------------------------
# numpy model of the window plan (no GPU)
# ---------------------------------------------------------------------------------------------------
def window_plan(pats):
    """The windows a tile stages for the dictionary `pats` (row_patterns' result): 0 when the plan does not qualify."""
    W, table, _ = pats
    deltas = sorted({int(np.int32(np.uint32(d))) for key in table for d in key[1:1 + key[0]]})
    clusters = []
    for d in deltas:
        if clusters and d - clusters[-1][1] < GAP:
            clusters[-1][1] = d
        else:
            clusters.append([d, d])
    if not clusters or len(clusters) > min(W, MAX_WINDOWS) or any(hi - lo > MAX_SPAN for lo, hi in clusters):
        return 0
    words = 2 * W * len(table) + sum((TILE_ROWS + hi - lo + 3) & ~1 for lo, hi in clusters)
    return len(clusters) if 8 * words <= SMEM_MAX else 0


def rows_of(kinds, M, N=None, values=None):
    """Row r takes the deltas kinds[r % len(kinds)] (each row gets the ones whose columns lie in [0, N)), every value
    1.0, or values[r % len(values)] on the first slot: len(values) times as many patterns."""
    N = M if N is None else N
    rp, ci, va = [0], [], []
    for r in range(M):
        cols = [r + d for d in sorted(kinds[r % len(kinds)]) if 0 <= r + d < N]
        ci.extend(cols)
        va.extend([1.0] * len(cols))
        if values is not None and cols:
            va[-len(cols)] = values[r % len(values)]
        rp.append(len(ci))
    return np.array(rp, np.int32), np.array(ci, np.int32), np.array(va, np.float64)


def count_limit(windows, width=None):
    """`windows` clusters 100 apart in rows of `width` nonzeros (default: the cluster count): wider rows add deltas to
    the first cluster, narrower ones cycle through the clusters."""
    W = width or windows
    deltas = [100 * c for c in range(windows)]
    if W >= windows:  # the first cluster holds deltas 0 .. W - windows
        kinds = [deltas + list(range(1, W - windows + 1))]
    else:
        kinds = [[deltas[(k + s) % windows] for s in range(W)] for k in range(windows)]
    return rows_of(kinds, 3000, 3000 + 100 * windows)


def span_limit(span):
    """One cluster from delta 0 to `span` in steps of at most 16, spread over rows of up to 12 nonzeros."""
    deltas = sorted(set(list(range(0, span, 16)) + [span]))
    kinds = [deltas[i:i + 12] for i in range(0, len(deltas), 12)]
    return rows_of(kinds, 3000, 3000 + span + 1)


def smem_limit(patterns):
    """Rows of 4 nonzeros at deltas 0, 1, 1000, 1001 with `patterns` distinct first values: two windows of span 1
    (2 x 1028 words) and 16 * 4 * patterns bytes of slot records, exactly 26 KB at 159 patterns."""
    return rows_of([[0, 1, 1000, 1001]], 2000, 2000 + 1002, values=[1.0 + k for k in range(patterns)])


def scattered(M=30000):
    """Rows of 2 nonzeros: the diagonal and one of 40 deltas 500 apart -- 41 clusters for W = 2."""
    return rows_of([[0, 500 * k - 10010] for k in range(40)], M)


def test_window_plan_model():
    from sparsematrixvectormultiplication_b200 import synth
    assert window_plan(row_patterns(*synth.lap2d_csr(64))) == 3     # {-64}, {-1, 0, 1}, {+64}
    assert window_plan(row_patterns(*synth.lap3d_csr(34))) == 0     # {-n^2}, {-n}, {-1, 0, 1}, {+n}, {+n^2}: 5 > 3
    assert window_plan(row_patterns(*synth.lap3d_csr(24))) == 0     # 3 clusters, but 27 x 7 slot records: 27.4 KB
    assert window_plan(row_patterns(*banded_pool(3000, 2500, make_pool(30, 3), 4))) == 1
    assert window_plan(row_patterns(*scattered())) == 0
    # the cluster count: at most W, and at most 3
    assert window_plan(row_patterns(*count_limit(3))) == 3
    assert window_plan(row_patterns(*count_limit(3, width=2))) == 0
    assert window_plan(row_patterns(*count_limit(2, width=5))) == 2
    assert window_plan(row_patterns(*count_limit(4, width=6))) == 0
    # the span of one window, and the shared memory of records and windows
    assert window_plan(row_patterns(*span_limit(MAX_SPAN))) == 1
    assert window_plan(row_patterns(*span_limit(MAX_SPAN + 1))) == 0
    assert window_plan(row_patterns(*smem_limit(159))) == 2
    assert window_plan(row_patterns(*smem_limit(160))) == 0


def test_shapes_of_the_limit_matrices():
    """The limit matrices hold what their names say: W, the pattern count and the clusters' extent."""
    assert row_patterns(*count_limit(2, width=5))[0] == 5
    assert row_patterns(*count_limit(4, width=6))[0] == 6
    assert row_patterns(*count_limit(3, width=2))[0] == 2
    assert row_patterns(*span_limit(MAX_SPAN))[0] == 12
    for n in (159, 160):
        W, table, _ = row_patterns(*smem_limit(n))
        assert (W, len(table)) == (4, n)
        assert 8 * (2 * W * n + 2 * 1028) == (SMEM_MAX if n == 159 else SMEM_MAX + 64)


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
def check_windows(A, rp, ci, va, M, N, expect, seed):
    """image_windows as the model says, then the products: the pattern form's checks, the serial loop's bits on finite x
    (plain and with accumulate from -0.0), row ranges that start and end inside tiles, and x only 8-byte aligned."""
    import torch
    d = dev()
    A.set_image(3)
    pats = row_patterns(rp, ci, va)
    assert window_plan(pats) == expect
    assert A.info().image_windows == expect
    last = [ci[rp[r + 1] - 1] for r in range(M) if rp[r + 1] > rp[r]]
    x = special_x(N, last[::7], seed=seed)
    check_pattern_form(A, M, N, pats[0], len(pats[1]), x)

    xf = torch.nan_to_num(x, nan=0.5, posinf=3.0, neginf=-3.0)
    xh = xf.cpu().numpy()
    y0 = minus_zero_start(M)
    for start in (None, y0):
        y = torch.zeros(M, dtype=torch.float64, device="cuda") if start is None else start.clone()
        A.spmv(xf, y, accumulate=start is not None, algo=d.ALGO_ROW_IMAGE)
        ref = serial(rp, ci, va, xh, None if start is None else start.cpu().numpy())
        assert np.array_equal(bits(y.cpu().numpy()), bits(ref)), f"accumulate={start is not None}"

    ref = torch.zeros(M, dtype=torch.float64, device="cuda")
    A.spmv(x, ref, algo=d.ALGO_ROW)
    for lo, hi in ((0, M), (5, min(M, 1030)), (min(1000, M - 1), M - min(700, M // 4)), (M - 1, M), (1023, min(M, 2049))):
        if hi <= lo:
            continue
        y = torch.full((M,), 7.0, dtype=torch.float64, device="cuda")
        A.spmv_rows(lo, hi, x, y)
        torch.cuda.synchronize()
        assert same_bits_up_to_nan_payload(y[lo:hi], ref[lo:hi]), (lo, hi)
        assert bool((y[:lo] == 7.0).all()) and bool((y[hi:] == 7.0).all()), (lo, hi)

    buf = torch.empty(N + 1, dtype=torch.float64, device="cuda")
    buf[1:] = xf
    x8 = buf[1:]  # 8 bytes past a 16-byte boundary
    assert x8.data_ptr() % 16 == 8
    for algo in (d.ALGO_AUTO, d.ALGO_ROW_IMAGE):
        y = torch.zeros(M, dtype=torch.float64, device="cuda")
        A.spmv(x8, y, algo=algo)
        r = torch.zeros(M, dtype=torch.float64, device="cuda")
        A.spmv(xf, r, algo=d.ALGO_ROW)
        torch.cuda.synchronize()
        assert torch.equal(tbits(y), tbits(r)), f"algo {algo} on x + 1"


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n,expect", [("lap2d", 64, 3), ("lap2d", 300, 3), ("lap3d", 24, 0)])
def test_windows_on_stencils(kind, n, expect):
    """Tiles of 1024 rows: lap2d 300^2 ends in a partial tile, and its first and last tiles clamp the windows at x[0] and
    x[N - 1]; lap3d gathers."""
    d = dev()
    A = d.DeviceCSR.synth(d.SYNTH_LAP2D if kind == "lap2d" else d.SYNTH_LAP3D, n)
    rp, ci, va = A.download()
    i = A.info()
    check_windows(A, rp, ci, va, i.M, i.N, expect, seed=n)
    A.close()


@pytest.mark.gpu
@pytest.mark.parametrize("M,N", [(3000, 2500), (2500, 3100), (900, 900), (4097, 4000)])
def test_windows_on_pattern_pools(M, N):
    """One window over rows from a pool of deltas in [-40, 40]: M > N and M < N, empty rows, stored +-0.0, fewer rows
    than a tile and one row past four tiles."""
    d = dev()
    rp, ci, va = banded_pool(M, N, make_pool(30, M), M + N)
    A = d.DeviceCSR.upload(M, N, rp, ci, va)
    check_windows(A, rp, ci, va, M, N, 1, seed=M)
    A.close()


LIMITS = {"scattered": (scattered, (), 0), "count3": (count_limit, (3,), 3), "count3-W2": (count_limit, (3, 2), 0),
          "count2-W5": (count_limit, (2, 5), 2), "count4-W6": (count_limit, (4, 6), 0), "span256": (span_limit, (256,), 1),
          "span257": (span_limit, (257,), 0), "smem159": (smem_limit, (159,), 2), "smem160": (smem_limit, (160,), 0)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(LIMITS))
def test_windows_at_the_limits(name):
    """The library's plan is the model's exactly at each limit and one past it; both paths keep the bits."""
    d = dev()
    make, args, expect = LIMITS[name]
    rp, ci, va = make(*args)
    M, N = len(rp) - 1, int(ci.max()) + 1
    A = d.DeviceCSR.upload(M, N, rp, ci, va)
    check_windows(A, rp, ci, va, M, N, expect, seed=len(name))
    A.close()


@pytest.mark.gpu
def test_windows_only_on_the_pattern_form():
    d = dev()
    A = d.DeviceCSR.synth(d.SYNTH_LAP2D, 64)
    assert A.info().image_windows == 0
    A.set_image(1)
    assert A.info().image_windows == 0
    A.set_image(3)
    assert A.info().image_windows == 3
    A.set_image(0)
    assert A.info().image_windows == 0
    A.close()
