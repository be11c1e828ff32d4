"""Host-buffer multi-vector products Y = A X (spmv_b200_{csr,hll}_spmm_host[_f32], DeviceCSR / DeviceHLL.spmm_host).

Contract (include/spmv_b200.h, next to the device SpMM): every column of Y has the bits of the device SpMM on the same
handle for the same X, whatever k, ldx, ldy, window count, column-block width, pinned or pageable buffers, zero-copy or
staged Y, and long rows; only rows < M and columns < k of Y are written.  The reference of every case is the device
SpMM on the same handle (bitwise) and, on rows up to the long-row threshold, the oracle's serial loop per column.
The gaps of ld > k layouts hold a NaN sentinel whose bits must come back unchanged.
"""
import ctypes as C
import subprocess
from pathlib import Path

import numpy as np
import pytest

from conftest import golden_names, load_golden
from test_gpu_spmm import bits, hack_runs, hll_of, random_csr

ROOT = Path(__file__).resolve().parents[1]
KS = (1, 2, 3, 8, 31, 32, 33, 65)
SENT64 = np.array([0x7FF8DEADBEEF0001], np.uint64).view(np.float64)[0]
SENT32 = np.array([0x7FC0BEEF], np.uint32).view(np.float32)[0]


def test_bad_arguments_without_a_device():
    """A NULL handle or array, a negative k and a leading dimension below k are refused before anything is touched (the
    dummy addresses below are never dereferenced)."""
    from sparsematrixvectormultiplication_b200 import _native as N
    lib = N.lib()
    h, p = C.c_void_p(64), C.c_void_p(4096)
    invalid = -1  # SPMV_B200_ERR_INVALID
    for fn, extra in ((lib.spmv_b200_csr_spmm_host, (0,)), (lib.spmv_b200_hll_spmm_host, ()),
                      (lib.spmv_b200_csr_spmm_host_f32, (0,)), (lib.spmv_b200_hll_spmm_host_f32, ())):
        assert fn(None, 4, p, 4, p, 4, *extra) == invalid
        assert fn(h, -1, p, 4, p, 4, *extra) == invalid
        assert fn(h, 4, p, 3, p, 4, *extra) == invalid
        assert fn(h, 4, p, 4, p, 3, *extra) == invalid
        assert fn(h, 4, None, 4, p, 4, *extra) == invalid
        assert fn(h, 4, p, 4, None, 4, *extra) == invalid


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


def host_block(src, k, wide, pinned, sentinel):
    """Columns [0, k) of src as a host block: a fresh (rows, k) buffer, or columns 1..k of a (rows, k + 3) buffer whose
    other columns hold the sentinel.  Returns (buffer, block) as CPU torch tensors, pinned or pageable."""
    import torch
    rows = src.shape[0]
    buf = np.full((rows, k + 3 if wide else k), sentinel, src.dtype)
    lo = 1 if wide else 0
    buf[:, lo:lo + k] = src[:, :k]
    t = torch.from_numpy(buf)
    if pinned:
        t = t.pin_memory()
    return t, t[:, lo:lo + k]


def gaps_unchanged(buf, k, wide, sentinel, what):
    if wide:
        b = buf.numpy()
        outside = np.concatenate([b[:, :1], b[:, 1 + k:]], axis=1)
        want = np.full(outside.shape, sentinel, b.dtype)
        assert np.array_equal(outside.view(np.uint8), want.view(np.uint8)), f"{what}: wrote outside the M x k block"


def assert_bitwise(got, want, what):
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert got.shape == want.shape, f"{what}: shapes {got.shape} and {want.shape}"
    if got.size == 0:
        return
    bad = np.argwhere(got.view(np.uint8).reshape(got.shape[0], -1) != want.view(np.uint8).reshape(want.shape[0], -1))
    assert bad.size == 0, f"{what}: elements differ, first (row, byte) {bad[:4].tolist()}"


def device_spmm(A, X, k, Y0=None, accumulate=False, f32=False):
    """The device SpMM on the same handle: the bitwise reference."""
    import torch
    dt = torch.float32 if f32 else torch.float64
    Xd = torch.from_numpy(np.ascontiguousarray(X[:, :k])).cuda()
    M, N = A.info().M, A.info().N
    if M == 0:
        return np.zeros((0, k), X.dtype)
    if N == 0:  # an empty X has no device address to pass: A X is zero
        return (Y0[:, :k] if accumulate else np.zeros((M, k), X.dtype)).copy()
    Yd = torch.from_numpy(np.ascontiguousarray(Y0[:, :k])).cuda() if Y0 is not None else torch.zeros((M, k), dtype=dt, device="cuda")
    if f32:
        A.spmm_f32(Xd, Yd, accumulate=accumulate) if accumulate else A.spmm_f32(Xd, Yd)
    else:
        A.spmm(Xd, Yd, accumulate=accumulate) if accumulate else A.spmm(Xd, Yd)
    return Yd.cpu().numpy()


def check_host(A, X, k, wide, pinned, Y0=None, accumulate=False, f32=False, what=""):
    """One host-buffer product against the device SpMM; returns the host result."""
    sentinel = SENT32 if f32 else SENT64
    M = A.info().M
    Xbuf, Xh = host_block(X, k, wide, pinned, sentinel)
    Ybuf, Yh = host_block(Y0 if Y0 is not None else np.full((M, k), np.nan, X.dtype), k, wide, pinned, sentinel)
    fn = A.spmm_host_f32 if f32 else A.spmm_host
    out = fn(Xh, Yh, accumulate=accumulate) if accumulate else fn(Xh, Yh)
    assert out is Yh
    tag = f"{what} k={k} wide={wide} pinned={pinned} acc={accumulate}"
    gaps_unchanged(Ybuf, k, wide, sentinel, tag)
    got = Yh.numpy().copy()
    assert_bitwise(got, device_spmm(A, X, k, Y0, accumulate, f32), tag)
    return got


def oracle_columns(port, rp, ci, va, X, cols, Y0=None):
    out = []
    for c in cols:
        y = None if Y0 is None else Y0[:, c].astype(np.float64).copy()
        out.append(port.spmv_csr_serial(rp, ci, va, np.ascontiguousarray(X[:, c], np.float64), y=y))
    return np.column_stack(out)


def csr_case(name):
    rng = np.random.default_rng(sum(map(ord, name)))
    if name.startswith("golden:"):
        g = load_golden(name[7:])
        return int(g["M"]), int(g["N"]), g["row_ptr"].astype(np.int32), g["col_idx"].astype(np.int32), g["values"]
    if name == "short":
        M, N, lengths = 3000, 2500, rng.integers(0, 6, 3000)
    elif name == "uniform":
        M, N, lengths = 2048, 4000, np.full(2048, 16)
    elif name == "long":
        M, N = 96, 24000
        lengths = rng.integers(0, 60, M)
        lengths[[3, 10, 40, 95]] = [513, 8193, 20000, 900]
    elif name == "empty_rows":
        M, N = 1500, 900
        lengths = rng.integers(0, 5, M) * (rng.random(M) < 0.4)
    elif name == "unreferenced_columns":  # every row within the first half of the columns
        M, N = 1200, 4000
        lengths = rng.integers(1, 8, M)
        rp, ci, va = random_csr(rng, M, N // 2, lengths)
        return M, N, rp, ci, va
    elif name == "N0":
        return 7, 0, np.zeros(8, np.int32), np.zeros(0, np.int32), np.zeros(0)
    elif name == "M0":
        return 0, 9, np.zeros(1, np.int32), np.zeros(0, np.int32), np.zeros(0)
    elif name == "nnz0":
        M, N, lengths = 100, 80, np.zeros(100, np.int64)
    rp, ci, va = random_csr(rng, M, N, lengths)
    return M, N, rp, ci, va


CSR_CASES = [f"golden:{n}" for n in golden_names()] + ["short", "uniform", "long", "empty_rows", "unreferenced_columns",
                                                      "N0", "M0", "nnz0"]


@pytest.mark.gpu
@pytest.mark.parametrize("case", CSR_CASES)
def test_csr_bitwise(dev, port, monkeypatch, case):
    """Every k, ld = k and ld > k, pinned and pageable, zero-copy left automatic and forced off, with and without
    accumulate: bitwise the device SpMM, and the oracle's serial loop on rows up to the long-row threshold."""
    M, N, rp, ci, va = csr_case(case)
    rng = np.random.default_rng(5)
    X = rng.standard_normal((N, max(KS)))
    Y0 = rng.standard_normal((M, max(KS)))
    A = dev.DeviceCSR.upload(M, N, rp, ci, va)
    short = np.diff(rp) <= (A.info().long_threshold if M else 0)
    ocols = [0, 2, 30, 64]
    ref = oracle_columns(port, rp, ci, va, X, ocols) if M else None
    ref_acc = oracle_columns(port, rp, ci, va, X, ocols, Y0) if M else None
    for zero_copy in (None, "0"):
        if zero_copy is None:
            monkeypatch.delenv("SPMV_B200_HOST_ZEROCOPY", raising=False)
        else:
            monkeypatch.setenv("SPMV_B200_HOST_ZEROCOPY", zero_copy)
        for k in KS:
            for wide in (False, True):
                for pinned in (False, True):
                    if zero_copy == "0" and not pinned:
                        continue
                    for acc in (False, True):
                        got = check_host(A, X, k, wide, pinned, Y0[:, :k] if acc else None, acc, what=case)
                        cols = [i for i, c in enumerate(ocols) if c < k]
                        if M and cols:
                            want = (ref_acc if acc else ref)[:, cols]
                            assert_bitwise(got[short][:, [ocols[i] for i in cols]], want[short], f"{case} k={k} oracle")


@pytest.mark.gpu
@pytest.mark.parametrize("image", ["lap2d", "runs7", "tail"])
def test_hll_bitwise(dev, checker, image):
    """lap2d, runs of hack widths and M off a multiple of 32: bitwise the device SpMM and spmv_hll_serial per column."""
    from sparsematrixvectormultiplication_b200 import synth
    rng = np.random.default_rng(sum(map(ord, image)))
    if image == "lap2d":
        rp, ci, va = synth.lap2d_csr(48)
        M = N = 48 * 48
    else:
        lengths = hack_runs(rng, [3, 5, 2, 7, 4, 6, 1], 3, 32) if image == "runs7" else rng.integers(0, 20, 32 * 9 + 13)
        M, N = len(lengths), 700
        rp, ci, va = random_csr(rng, M, N, lengths)
    rp, ci = np.asarray(rp, np.int32), np.asarray(ci, np.int32)
    X = rng.standard_normal((N, max(KS)))
    h = hll_of(checker, M, N, rp, ci, va)
    H = dev.DeviceCSR.upload(M, N, rp, ci, va).to_hll()
    for k in KS:
        for wide in (False, True):
            for pinned in (False, True):
                got = check_host(H, X, k, wide, pinned, what=image)
                assert_bitwise(got[:, 0], checker.spmv_hll_serial(h, X[:, 0], M), f"{image} k={k} serial")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["csr", "hll"])
def test_f32_twins(dev, fmt):
    """The fp32 forms enable the float copy themselves and give the bits of spmm_f32, long rows included (CSR)."""
    rng = np.random.default_rng(32)
    M, N = 700, 9000
    lengths = rng.integers(0, 40, M)
    if fmt == "csr":
        lengths[[5, 300]] = [600, 8500]
    rp, ci, va = random_csr(rng, M, N, lengths)
    X = rng.standard_normal((N, max(KS))).astype(np.float32)
    Y0 = rng.standard_normal((M, max(KS))).astype(np.float32)
    A = dev.DeviceCSR.upload(M, N, rp, ci, va)
    T = A if fmt == "csr" else A.to_hll()
    for k in KS:
        for wide in (False, True):
            for pinned in (False, True):
                check_host(T, X, k, wide, pinned, f32=True, what=f"{fmt} f32")
                if fmt == "csr":
                    check_host(T, X, k, wide, pinned, Y0[:, :k], True, f32=True, what="csr f32")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["csr", "hll"])
def test_f32_after_f64_on_one_handle(dev, fmt):
    """spmm_host, then spmm_host_f32 on the same handle, whose float copy the second call makes: a matrix with long rows
    (CSR) or wide hacks (HLL), too small for plan-time timing, so that enable_f32 only queues the conversion.  The fp32
    result is bitwise spmm_f32 on the same handle, the fp64 one spmm before and after."""
    rng = np.random.default_rng(7)
    M, N = 300, 20000
    lengths = rng.integers(0, 30, M)
    lengths[[4, 150]] = [9000, 700]
    rp, ci, va = random_csr(rng, M, N, lengths)
    A = dev.DeviceCSR.upload(M, N, rp, ci, va)
    T = A if fmt == "csr" else A.to_hll()
    X = rng.standard_normal((N, 9))
    for pinned in (False, True):
        check_host(T, X, 9, False, pinned, what=f"{fmt} fp64 first")
    check_host(T, X.astype(np.float32), 9, False, True, f32=True, what=f"{fmt} fp32 after fp64")
    check_host(T, X.astype(np.float32), 9, True, False, f32=True, what=f"{fmt} fp32 again")
    check_host(T, X, 9, True, True, what=f"{fmt} fp64 after fp32")


@pytest.mark.gpu
@pytest.mark.parametrize("windows", ["1", "3", "64"])
@pytest.mark.parametrize("cols", [None, "1", "5"])
def test_windows_and_column_blocks(dev, monkeypatch, windows, cols):
    """Forced window counts and column-block widths, each on a fresh handle: the same bits as one call on defaults."""
    rng = np.random.default_rng(64)
    M, N = 5000, 30000
    lengths = rng.integers(0, 12, M)
    lengths[[7, 2500, 4999]] = [700, 9000, 520]
    rp, ci, va = random_csr(rng, M, N, lengths)
    X = rng.standard_normal((N, 33))
    Y0 = rng.standard_normal((M, 33))
    monkeypatch.setenv("SPMV_B200_HOST_WINDOWS", windows)
    if cols is None:
        monkeypatch.delenv("SPMV_B200_HOST_SPMM_COLS", raising=False)
    else:
        monkeypatch.setenv("SPMV_B200_HOST_SPMM_COLS", cols)
    A = dev.DeviceCSR.upload(M, N, rp, ci, va)
    H = A.to_hll()
    for k in (1, 8, 33):
        for wide in (False, True):
            for pinned in (False, True):
                check_host(A, X, k, wide, pinned, what=f"csr W={windows} kc={cols}")
                check_host(A, X, k, wide, pinned, Y0[:, :k], True, what=f"csr acc W={windows} kc={cols}")
                check_host(H, X, k, wide, pinned, what=f"hll W={windows} kc={cols}")


@pytest.mark.gpu
def test_alternating_with_the_single_vector_call(dev):
    """spmv_host, spmm_host, spmv_host on one handle: each bitwise what a fresh handle gives."""
    from sparsematrixvectormultiplication_b200 import synth
    rp, ci, va = synth.lap2d_csr(300)
    M = N = 300 * 300
    rng = np.random.default_rng(3)
    x = rng.standard_normal(N)
    X = rng.standard_normal((N, 5))
    for fmt in ("csr", "hll"):
        def fresh():
            A = dev.DeviceCSR.upload(M, N, rp, ci, va)
            return A if fmt == "csr" else A.to_hll()
        want_y, want_Y = fresh().spmv_host(x), fresh().spmm_host(X)
        T = fresh()
        assert_bitwise(T.spmv_host(x), want_y, f"{fmt} spmv_host first")
        assert_bitwise(T.spmm_host(X), want_Y, f"{fmt} spmm_host")
        assert_bitwise(T.spmv_host(x), want_y, f"{fmt} spmv_host again")
        assert_bitwise(T.spmm_host(X), want_Y, f"{fmt} spmm_host again")


@pytest.mark.gpu
def test_x_past_2_31_bytes(dev):
    """lap2d 1448^2 with k = 130: X is 2.18e9 bytes.  Sampled rows at both ends and in the middle, bitwise the device
    SpMM on the same handle."""
    import torch
    from sparsematrixvectormultiplication_b200 import synth
    n, k = 1448, 130
    rp, ci, va = synth.lap2d_csr(n)
    M = N = n * n
    assert N * k * 8 > 2 ** 31
    X = torch.empty((N, k), dtype=torch.float64).uniform_(-1.0, 1.0, generator=torch.Generator().manual_seed(1))
    A = dev.DeviceCSR.upload(M, N, rp, ci, va)
    Y = A.spmm_host(X)
    Yd = torch.empty((M, k), dtype=torch.float64, device="cuda")
    A.spmm(X.cuda(), Yd)
    rows = np.r_[0:64, M // 2 - 32:M // 2 + 32, M - 64:M]
    assert_bitwise(Y[rows].numpy(), Yd[torch.from_numpy(rows).cuda()].cpu().numpy(), "X past 2^31 bytes")


@pytest.mark.gpu
def test_python_argument_errors(dev):
    import torch
    A = dev.DeviceCSR.upload(3, 4, np.array([0, 1, 2, 3], np.int32), np.array([0, 1, 3], np.int32), np.ones(3))
    H = A.to_hll()
    X = np.ones((4, 2))
    for T in (A, H):
        with pytest.raises(ValueError):
            T.spmm_host(np.ones((5, 2)))                       # rows != N
        with pytest.raises(ValueError):
            T.spmm_host(X.astype(np.float32))                  # dtype
        with pytest.raises(ValueError):
            T.spmm_host(np.ones((4, 4))[:, ::2])               # column stride
        with pytest.raises(ValueError):
            T.spmm_host(X, np.zeros((3, 3)))                   # k of Y
        with pytest.raises(ValueError):
            T.spmm_host(X, np.zeros((2, 2)))                   # rows != M
        with pytest.raises(ValueError):
            T.spmm_host(torch.ones((4, 2), device="cuda", dtype=torch.float64))
        with pytest.raises(ValueError):
            T.spmm_host_f32(X)
        ro = np.zeros((3, 2))
        ro.flags.writeable = False
        with pytest.raises(ValueError):
            T.spmm_host(X, ro)
        big = np.zeros((8, 8))
        with pytest.raises(ValueError):
            T.spmm_host(big[:4, :2], big[1:4, :2])             # Y overlaps X
        T.spmm_host(big[:4, :2], big[4:7, :2])                 # adjacent, no overlap
        assert isinstance(T.spmm_host(torch.ones((4, 2), dtype=torch.float64)), torch.Tensor)


C_PROGRAM = r"""
#include <stdio.h>
#include <stdlib.h>
#include "spmv_b200.h"

static void *slurp(const char *path, long *bytes) {
    FILE *f = fopen(path, "rb");
    if (!f) return NULL;
    fseek(f, 0, SEEK_END);
    *bytes = ftell(f);
    fseek(f, 0, SEEK_SET);
    void *p = malloc(*bytes > 0 ? *bytes : 1);
    if (fread(p, 1, *bytes, f) != (size_t)*bytes) { fclose(f); return NULL; }
    fclose(f);
    return p;
}

int main(int argc, char **argv) {
    /* argv: dir M N nnz k ldx ldy; dir holds row_ptr.bin col_idx.bin values.bin X.bin, writes Y.bin */
    if (argc != 8) return 2;
    char path[4096];
    long b;
    int M = atoi(argv[2]), N = atoi(argv[3]), k = atoi(argv[5]);
    long long nnz = atoll(argv[4]), ldx = atoll(argv[6]), ldy = atoll(argv[7]);
    snprintf(path, sizeof path, "%s/row_ptr.bin", argv[1]); int *rp = slurp(path, &b);
    snprintf(path, sizeof path, "%s/col_idx.bin", argv[1]); int *ci = slurp(path, &b);
    snprintf(path, sizeof path, "%s/values.bin", argv[1]); double *va = slurp(path, &b);
    snprintf(path, sizeof path, "%s/X.bin", argv[1]); double *X = slurp(path, &b);
    snprintf(path, sizeof path, "%s/Y.bin", argv[1]); double *Y = slurp(path, &b);
    if (!rp || !ci || !va || !X || !Y) return 3;
    spmv_b200_csr *A = NULL;
    if (spmv_b200_csr_upload(M, N, nnz, rp, ci, va, &A) != SPMV_B200_OK) { fprintf(stderr, "%s\n", spmv_b200_last_error()); return 4; }
    if (spmv_b200_csr_spmm_host(A, k, X, ldx, Y, ldy, 0) != SPMV_B200_OK) { fprintf(stderr, "%s\n", spmv_b200_last_error()); return 5; }
    if (spmv_b200_csr_spmm_host(A, -1, X, ldx, Y, ldy, 0) != SPMV_B200_ERR_INVALID) return 6;
    if (spmv_b200_csr_spmm_host(A, k, X, k - 1, Y, ldy, 0) != SPMV_B200_ERR_INVALID) return 7;
    spmv_b200_csr_free(A);
    snprintf(path, sizeof path, "%s/Y.bin", argv[1]);
    FILE *f = fopen(path, "wb");
    fwrite(Y, sizeof(double), (size_t)M * ldy, f);
    fclose(f);
    printf("SPMM_HOST_C OK\n");
    return 0;
}
"""


@pytest.mark.gpu
def test_plain_c_caller(port, tmp_path):
    """A C program built against the library and its header only (no CUDA runtime header or library of its own) calls
    spmv_b200_csr_spmm_host on a golden fixture at ldx, ldy > k; every column equals the oracle's serial loop and the
    gaps of Y keep their sentinel bits."""
    import sparsematrixvectormultiplication_b200 as pkg
    lib = Path(pkg.LIB_PATH)
    src = tmp_path / "spmm_host_c.c"
    src.write_text(C_PROGRAM)
    exe = tmp_path / "spmm_host_c"
    subprocess.run(["gcc", "-std=c11", "-O1", f"-I{ROOT / 'include'}", str(src), "-o", str(exe), f"-L{lib.parent}",
                    "-lspmv_b200", f"-Wl,-rpath,{lib.parent}"], check=True)
    g = load_golden("rand_general_97x61")
    M, N = int(g["M"]), int(g["N"])
    rp, ci, va = g["row_ptr"].astype(np.int32), g["col_idx"].astype(np.int32), g["values"].astype(np.float64)
    k, ldx, ldy = 6, 9, 8
    X = np.random.default_rng(11).standard_normal((N, ldx))
    Y = np.full((M, ldy), SENT64)
    for name, a in (("row_ptr", rp), ("col_idx", ci), ("values", va), ("X", X), ("Y", Y)):
        a.tofile(tmp_path / f"{name}.bin")
    out = subprocess.run([str(exe), str(tmp_path), str(M), str(N), str(len(ci)), str(k), str(ldx), str(ldy)],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "SPMM_HOST_C OK" in out.stdout, (out.returncode, out.stdout, out.stderr)
    got = np.fromfile(tmp_path / "Y.bin", np.float64).reshape(M, ldy)
    assert np.all(bits(got[:, k:]) == bits(np.full((M, ldy - k), SENT64))), "wrote into the ldy gap"
    assert_bitwise(got[:, :k], oracle_columns(port, rp, ci, va, X, range(k)), "C caller against the oracle")
