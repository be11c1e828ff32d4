"""Drop-in host API (libspmv_b200.so) vs the reference: golden vectors + the oracle on random COO.
Bit-exact for every index and value array (SURVEY.md section 3.3 / 3.4)."""
import json
import os

import numpy as np
import pytest
from hypothesis import given, settings, strategies as st

from conftest import GOLDEN, golden_names, load_golden, random_coo
from sparsematrixvectormultiplication_b200 import host

THREADS = (1, 2, 3, 4, 8, 40)


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


@pytest.mark.parametrize("name", golden_names())
def test_parser_and_builders_match_golden(name):
    g = load_golden(name)
    pre = host.read_matrix_market(GOLDEN / "mtx" / f"{name}.mtx")
    assert (pre.M, pre.N, pre.nz) == (int(g["M"]), int(g["N"]), int(g["nz"]))
    assert pre.type == bytes(g["type"]).decode()
    assert np.array_equal(pre.I, g["I"]) and np.array_equal(pre.J, g["J"])
    assert np.array_equal(bits(pre.val), bits(g["val"]))
    csr = host.convert_in_csr(pre, name)
    assert (csr.M, csr.N, csr.nz) == (pre.M, pre.N, pre.nz)
    assert np.array_equal(csr.row_ptr, g["row_ptr"]) and np.array_equal(csr.col_idx, g["col_idx"])
    assert np.array_equal(bits(csr.values), bits(g["values"]))
    hll = host.convert_to_hll(pre)
    rows, maxnz, offset, JA, AS = hll.flat()
    assert np.array_equal(rows, g["hll_rows"]) and np.array_equal(maxnz, g["hll_maxnz"])
    assert np.array_equal(JA, g["hll_JA"]) and np.array_equal(bits(AS), bits(g["hll_AS"]))
    for b in range(hll.num_blocks):  # empty block: NULL arrays like the reference
        blk = hll.c.blocks[b]
        assert blk.N == pre.N
        assert (blk.MAXNZ == 0) == (not blk.JA) == (not blk.AS)
    for T in THREADS:
        s, e = host.prepare_thread_distribution(csr.M, csr.row_ptr, T, csr.nz)
        assert np.array_equal(np.stack([s, e]).reshape(2, -1), g[f"part_rows_{T}"]), T
        s, e = host.prepare_thread_distribution_hll(hll, T)
        assert np.array_equal(np.stack([s, e]).reshape(2, -1), g[f"part_hll_{T}"]), T


def test_parser_rejects_what_the_reference_rejects(capfd):
    for name in json.loads((GOLDEN / "errors.json").read_text()):
        with pytest.raises(host.HostApiError):
            host.read_matrix_market(GOLDEN / "mtx" / name)
    with pytest.raises(host.HostApiError):
        host.read_matrix_market(GOLDEN / "mtx" / "does_not_exist.mtx")


@settings(max_examples=120, deadline=None)
@given(st.integers(1, 140), st.integers(1, 70), st.integers(0, 700), st.booleans(), st.integers(0, 2**31))
def test_builders_match_oracle_on_random_coo(M, N, nz, dup, seed):
    from oracle import oracle as O
    chk = O.best_available()
    rng = np.random.default_rng(seed)
    coo = random_coo(rng, M, N, nz, dup=dup)
    pre = host.PreMatrix(coo.M, coo.N, coo.I, coo.J, coo.val)
    csr = host.convert_in_csr(pre)
    rp, ci, va = chk.coo_to_csr(coo)
    assert np.array_equal(csr.row_ptr, rp) and np.array_equal(csr.col_idx, ci) and np.array_equal(bits(csr.values), bits(va))
    hll = host.convert_to_hll(pre)
    h = chk.coo_to_hll(coo)
    rows, maxnz, offset, JA, AS = hll.flat()
    assert np.array_equal(rows, h.rows) and np.array_equal(maxnz, h.maxnz)
    assert np.array_equal(JA, h.JA) and np.array_equal(bits(AS), bits(h.AS))
    for T in (1, 2, 7, 33):
        s, e = host.prepare_thread_distribution(csr.M, csr.row_ptr, T, csr.nz)
        so, eo = chk.partition_rows(rp, T)
        assert np.array_equal(s, so) and np.array_equal(e, eo)
        s, e = host.prepare_thread_distribution_hll(hll, T)
        so, eo = chk.partition_hll(h, N, T)
        assert np.array_equal(s, so) and np.array_equal(e, eo)


def test_long_rows_with_and_without_duplicates(checker):
    """Rows above the builder's short-row threshold: merge-sort fast path (unique) and the
    reference-equivalent quicksort (duplicates), incl. sorted / reversed input."""
    rng = np.random.default_rng(11)
    for case in range(12):
        M, N, nz = 5, 4000, 3000
        coo = random_coo(rng, M, N, nz, dup=bool(case % 2))
        if case % 3 == 0:    # already sorted by (row, col)
            o = np.lexsort((coo.J, coo.I))
        elif case % 3 == 1:  # reverse sorted
            o = np.lexsort((coo.J, coo.I))[::-1]
        else:
            o = np.arange(coo.nz)
        coo.I, coo.J, coo.val = coo.I[o].copy(), coo.J[o].copy(), coo.val[o].copy()
        pre = host.PreMatrix(M, N, coo.I, coo.J, coo.val)
        csr = host.convert_in_csr(pre)
        rp, ci, va = checker.coo_to_csr(coo)
        assert np.array_equal(csr.col_idx, ci) and np.array_equal(bits(csr.values), bits(va)), case
        h = checker.coo_to_hll(coo)
        rows, maxnz, offset, JA, AS = host.convert_to_hll(pre).flat()
        assert np.array_equal(JA, h.JA) and np.array_equal(bits(AS), bits(h.AS)), case


def test_sort_row_is_the_reference_quicksort(checker):
    """The checker's CSR builder keeps file order inside a row and then runs the reference's quicksort on it, so a
    one-row matrix yields exactly what sort_row leaves (duplicates make the unstable order observable)."""
    from oracle import oracle as O
    rng = np.random.default_rng(5)
    for n in (2, 3, 17, 200):
        c = rng.integers(0, 6, n).astype(np.int32)  # many duplicates
        v = rng.standard_normal(n)
        c1, v1 = c.copy(), v.copy()
        host.sort_row(c1, v1, 0, n - 1)
        _, c2, v2 = checker.coo_to_csr(O.Coo(1, 6, n, np.zeros(n, np.int32), c.copy(), v.copy()))
        assert np.array_equal(c1, c2) and np.array_equal(bits(v1), bits(v2))


def test_partitioner_edge_cases(checker):
    rp = np.zeros(6, np.int32)  # five empty rows
    s, e = host.prepare_thread_distribution(5, rp, 3, 0)
    so, eo = checker.partition_rows(rp, 3)
    assert len(s) == len(so) == 0
    assert host.prepare_thread_distribution(0, np.zeros(1, np.int32), 4, 0)[0].size == 0
    rp = np.array([0, 10, 10, 10, 11], np.int32)  # trailing light rows
    for T in (1, 2, 3, 4, 9):
        s, e = host.prepare_thread_distribution(4, rp, T, 11)
        so, eo = checker.partition_rows(rp, T)
        assert np.array_equal(s, so) and np.array_equal(e, eo), T


def test_harness_matches_oracle(checker, port):
    rng = np.random.default_rng(9)
    a = rng.standard_normal(800)
    b = a + rng.standard_normal(800) * (rng.random(800) < 0.3) * 1e-3
    mean_abs, mean_rel, sig = host.computeDifferenceMetrics(a, b)
    sig_o, rel_o = checker.diff_metrics_c(a, b)
    assert (sig, mean_rel, mean_abs) == (sig_o, rel_o, 0.0)
    assert host.calculate_flops(83869696, 2.5e-4) == port.calculate_flops(83869696, 2.5e-4)
    host.initialize_metrics()
    for t in (3.0, 1.0, 2.0, 6.0):
        host.update_medium_metric(host.B200_CSR_TIME, t)
    assert host.get_metric_value(host.B200_CSR_TIME) == 3.0
    assert host.get_metric_min(host.B200_CSR_TIME) == 1.0 and host.get_metric_median(host.B200_CSR_TIME) == 2.5
    host.accumulateErrors(0.5, 0.25, host.B200_CSR_TIME)
    ma, mr = host.computeAverageErrors(host.B200_CSR_TIME)
    assert (ma, mr) == (0.5 / (4 + host.ITERATION_SKIP), 0.25 / (4 + host.ITERATION_SKIP))
    host.reset_medium_time_metrics()
    assert host.get_metric_value(host.B200_CSR_TIME) == 0.0
    host.cleanup_metrics()
    # algorithmic bytes of BASELINE.md section 3: lap2d 4096^2 -> 1.342 GB
    M, nnz = 4096 * 4096, 83869696
    assert host.calculate_csr_bytes(M, M, nnz) == nnz * 12 + 4 * (M + 1) + 16 * M
    assert abs(host.calculate_csr_bytes(M, M, nnz) / 1e9 - 1.342) < 1e-3
    v = np.zeros(7)
    assert (host.init_vector_at_one(v) == 1.0).all()


def test_driver_fails_loudly_without_a_gpu(tmp_path):
    """tools/spmv_driver.c (the main()-style driver) has no CPU fallback: on a machine without a CUDA device it must
    stop with exit status 3 and say why; on a GPU box the same command is covered by tests/test_gpu_parity.py."""
    import subprocess
    import sparsematrixvectormultiplication_b200 as pkg
    try:
        import torch
        if torch.cuda.is_available():
            pytest.skip("CUDA device present")
    except ImportError:
        pass
    exe = pkg.LIB_PATH.parent / "spmv_driver"
    if not exe.exists():
        pkg.build()
    out = subprocess.run([str(exe), "--csv", str(tmp_path / "r.csv"), str(GOLDEN / "mtx" / "general_matrix.mtx")],
                         capture_output=True, text=True)
    assert out.returncode == 3, out.stdout + out.stderr
    assert "no CUDA device" in out.stderr and "no CPU fallback" in out.stderr
    assert not (tmp_path / "r.csv").exists()


# ---------------------------------------------------------------------------------------------------
# parallel tokenizer of read_matrix_market (SURVEY.md section 8(f).4): same bits as the serial path
# ---------------------------------------------------------------------------------------------------
def _same_pre(a, b):
    return (a.M, a.N, a.nz) == (b.M, b.N, b.nz) and np.array_equal(a.I, b.I) and np.array_equal(a.J, b.J) \
        and np.array_equal(a.val.view(np.uint64), b.val.view(np.uint64)) and bytes(a.c.type) == bytes(b.c.type)


@pytest.mark.parametrize("name", golden_names())
def test_parallel_parser_equals_serial_on_fixtures(name, monkeypatch):
    path = GOLDEN / "mtx" / f"{name}.mtx"
    monkeypatch.setenv("SPMV_B200_PARSER_PARALLEL_MIN_BYTES", str(1 << 40))
    serial = host.read_matrix_market(path)
    monkeypatch.setenv("SPMV_B200_PARSER_PARALLEL_MIN_BYTES", "0")
    import ctypes
    gomp = ctypes.CDLL("libgomp.so.1")            # OMP_NUM_THREADS is only read when the runtime starts
    before = gomp.omp_get_max_threads()
    try:
        for threads in (2, 3, 16):
            gomp.omp_set_num_threads(threads)
            assert _same_pre(host.read_matrix_market(path), serial), f"{name} with {threads} threads"
    finally:
        gomp.omp_set_num_threads(before)


@pytest.mark.parametrize("kind,field", [("general", "real"), ("symmetric", "real"), ("general", "pattern"),
                                        ("symmetric", "pattern"), ("general", "integer"), ("skew-symmetric", "real")])
def test_parallel_parser_on_a_large_file(tmp_path, checker, kind, field):
    """A 300k-entry file (3-9 MB; the parallel pass is forced, and the default path is checked too) with ragged white space, entries spanning lines and
    exponents: default (parallel) parse == forced-serial parse == the checker's fscanf parser."""
    rng = np.random.default_rng(len(kind) * 31 + len(field))
    M, N, nz = 5000, 4000 if kind == "general" else 5000, 300_000
    I = rng.integers(1, M + 1, nz)
    J = rng.integers(1, N + 1, nz)
    if kind != "general":
        I, J = np.maximum(I, J), np.minimum(I, J)
    lines = [f"%%MatrixMarket matrix coordinate {field} {kind}", "% generated by the test", f"{M} {N} {nz}"]
    vals = rng.standard_normal(nz) * 10.0 ** rng.integers(-8, 9, nz)
    seps = ["  ", "\t", " ", "\n", " \t "]
    for k in range(nz):
        sep = seps[k % len(seps)]
        if field == "pattern":
            lines.append(f"{I[k]}{sep}{J[k]}")
        elif field == "integer":
            lines.append(f"{I[k]}{sep}{J[k]} {int(vals[k]) % 1000 - 500}")
        else:
            lines.append(f"{I[k]}{sep}{J[k]} {vals[k]:.17e}" if k % 3 else f"{I[k]} {J[k]}\n{float(vals[k])!r}")
    path = tmp_path / "big.mtx"
    path.write_text("\n".join(lines) + "\n")
    default = host.read_matrix_market(path)            # parallel above 4 MB (the real / integer files), serial below
    try:
        os.environ["SPMV_B200_PARSER_PARALLEL_MIN_BYTES"] = "0"
        fast = host.read_matrix_market(path)
        os.environ["SPMV_B200_PARSER_PARALLEL_MIN_BYTES"] = str(1 << 40)
        slow = host.read_matrix_market(path)
    finally:
        del os.environ["SPMV_B200_PARSER_PARALLEL_MIN_BYTES"]
    assert _same_pre(default, slow)
    assert _same_pre(fast, slow)
    ref = checker.read_matrix_market(path)
    assert (ref.M, ref.N, ref.nz) == (fast.M, fast.N, fast.nz)
    assert np.array_equal(ref.I, fast.I) and np.array_equal(ref.J, fast.J)
    assert np.array_equal(np.asarray(ref.val).view(np.uint64), fast.val.view(np.uint64))


@pytest.mark.parametrize("damage", ["truncated", "out_of_range", "junk_index", "glued_value"])
def test_parallel_parser_falls_back_on_irregular_bodies(tmp_path, monkeypatch, capfd, damage):
    """Whatever the parallel pass cannot vouch for is re-parsed by the serial loop, so errors (and the odd accepted
    input, e.g. '7abc' = index 7 followed by a token the NEXT field chokes on) behave as without it."""
    body = [f"{1 + k % 50} {1 + (7 * k) % 40} {k * 0.5}" for k in range(2000)]
    if damage == "truncated":
        body = body[:1500]
    elif damage == "out_of_range":
        body[1234] = "51 3 1.0"
    elif damage == "junk_index":
        body[777] = "x7 3 1.0"
    else:
        body[999] = "7 3 1.5abc"
    path = tmp_path / "bad.mtx"
    path.write_text("%%MatrixMarket matrix coordinate real general\n50 40 2000\n" + "\n".join(body) + "\n")
    results = []
    for threshold in ("0", str(1 << 40)):
        monkeypatch.setenv("SPMV_B200_PARSER_PARALLEL_MIN_BYTES", threshold)
        try:
            pre = host.read_matrix_market(path)
            results.append(("ok", pre.nz, pre.I.copy(), pre.J.copy(), pre.val.copy()))
        except host.HostApiError:
            results.append(("error",))
        results[-1] = results[-1] + (capfd.readouterr().out,)
    assert results[0][0] == results[1][0]
    assert results[0][-1] == results[1][-1], "same message on stdout"
    if results[0][0] == "ok":
        assert all(np.array_equal(a, b) for a, b in zip(results[0][1:-1], results[1][1:-1]))


@pytest.mark.parametrize("dup", [False, True])
def test_large_inputs_take_the_parallel_scatter(checker, dup, monkeypatch):
    """Above 2^20 entries convert_in_csr / convert_to_hll spread the counting scatter over the OpenMP threads (every
    thread owns a range of rows and scans the whole COO list): same arrays as the checker, bit for bit, for any
    thread count, duplicates included."""
    rng = np.random.default_rng(99 + dup)
    M, N, nz = 70_001, 50_000, 1_300_000
    coo = random_coo(rng, M, N, nz, dup=dup)
    rp, ci, va = checker.coo_to_csr(coo)
    h = checker.coo_to_hll(coo)
    import ctypes
    gomp = ctypes.CDLL("libgomp.so.1")            # the OpenMP runtime the library is linked against
    before = gomp.omp_get_max_threads()
    for threads in (1, 3, 8):
        gomp.omp_set_num_threads(threads)          # (OMP_NUM_THREADS is only read when the runtime starts)
        assert gomp.omp_get_max_threads() == threads
        pre = host.PreMatrix(M, N, coo.I, coo.J, coo.val)
        csr = host.convert_in_csr(pre)
        assert np.array_equal(csr.row_ptr, rp) and np.array_equal(csr.col_idx, ci)
        assert np.array_equal(csr.values.view(np.uint64), va.view(np.uint64)), f"{threads} threads"
        rows, maxnz, offset, JA, AS = host.convert_to_hll(pre).flat()
        assert np.array_equal(maxnz, h.maxnz) and np.array_equal(JA, h.JA)
        assert np.array_equal(AS.view(np.uint64), h.AS.view(np.uint64)), f"{threads} threads"
    gomp.omp_set_num_threads(before)


def test_parser_speed_report(tmp_path, checker, capsys):
    """Not a pass/fail bar (shared CPUs are noisy): prints the time of the checker's fscanf parser and of this repo's
    read_matrix_market on the same 400k-entry file, and checks they return the same COO.  Larger runs: tools/bench_parser.py."""
    import time
    rng = np.random.default_rng(3)
    M = N = 300_000
    nz = 400_000
    I, J, V = rng.integers(1, M + 1, nz), rng.integers(1, N + 1, nz), rng.standard_normal(nz)
    path = tmp_path / "speed.mtx"
    with open(path, "w") as f:
        f.write(f"%%MatrixMarket matrix coordinate real general\n{M} {N} {nz}\n")
        np.savetxt(f, np.column_stack([I, J, V]), fmt="%d %d %.17g")
    t0 = time.perf_counter()
    ours = host.read_matrix_market(path)
    t1 = time.perf_counter()
    ref = checker.read_matrix_market(path)
    t2 = time.perf_counter()
    assert np.array_equal(ref.I, ours.I) and np.array_equal(ref.J, ours.J)
    assert np.array_equal(np.asarray(ref.val).view(np.uint64), ours.val.view(np.uint64))
    with capsys.disabled():
        print(f"\n[parser] {nz} entries, {path.stat().st_size / 1e6:.0f} MB: this repo {t1 - t0:.3f} s, {checker.kind} fscanf loop {t2 - t1:.3f} s")
