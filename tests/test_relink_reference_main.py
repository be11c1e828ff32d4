"""Link-level drop-in, proven: the reference's OWN OpenMP driver (main.c, unmodified, compiled where it lies under
/root/reference) builds against include/*.h and links against libspmv_b200.so with nothing from src/*.c.

CPU container only (the reference tree is not on the GPU box).  The executable is only RUN when a GPU is present --
its products go through the CUDA path and there is no CPU fallback -- otherwise the test stops after checking that
the link has no undefined symbol and that the helper functions main.c needs behave."""
import ctypes as C
import os
import shutil
import subprocess
from pathlib import Path

import pytest

from sparsematrixvectormultiplication_b200 import _native as N

ROOT = Path(__file__).resolve().parents[1]
REF = Path("/root/reference")
PKG = ROOT / "sparsematrixvectormultiplication_b200"


@pytest.fixture(scope="module")
def relinked(tmp_path_factory):
    try:
        present = (REF / "main.c").is_file()
    except OSError:                      # a tree this user may not enter counts as absent
        present = False
    if not present:
        pytest.skip("reference tree not present")
    N.lib()
    build = tmp_path_factory.mktemp("relink") / "build"
    build.mkdir()
    exe = build / "SpMV_OpenMP"
    cmd = ["/usr/bin/gcc", "-std=c17", "-O2", "-fopenmp", f"-I{ROOT / 'include'}", str(REF / "main.c"), "-o", str(exe),
           f"-L{PKG}", "-lspmv_b200", f"-Wl,-rpath,{PKG}", "-Wl,--no-undefined", "-lm"]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    assert "implicit declaration" not in out.stderr, out.stderr   # every function main.c calls is declared in include/
    return exe


def test_reference_main_links_against_the_library(relinked):
    needed = subprocess.run(["nm", "-u", str(relinked)], capture_output=True, text=True).stdout
    for symbol in ("create_directory", "write_results_to_csv", "spvm_csr_parallel", "spmv_hll_simd", "convert_to_hll"):
        assert symbol in needed          # resolved at load time from libspmv_b200.so, not compiled in
    ldd = subprocess.run(["ldd", str(relinked)], capture_output=True, text=True).stdout
    assert "libspmv_b200.so" in ldd and "not found" not in ldd


PREBUILT = ROOT / "oracle" / "_ref" / "ref_main_relinked"   # oracle/Makefile target ref_main: travels to the GPU box


@pytest.mark.gpu
def test_reference_main_runs_on_the_fixture(tmp_path):
    """The unmodified reference driver, relinked, runs BASELINE config 1 end to end on the GPU box and writes its CSV;
    its own self-check columns (error_* vs the serial CSR product, main.c:145-362) must be zero."""
    if not PREBUILT.exists():
        pytest.skip("oracle/_ref/ref_main_relinked was not built (reference tree absent at build time)")
    relinked = PREBUILT
    # main.c reads ../matrix_for_test/ and writes ../result/ relative to its working directory
    (tmp_path / "matrix_for_test").mkdir()
    shutil.copy(ROOT / "tests" / "golden" / "mtx" / "general_matrix.mtx", tmp_path / "matrix_for_test")
    run = tmp_path / "run"
    run.mkdir()
    out = subprocess.run([str(relinked)], cwd=run, capture_output=True, text=True, timeout=600,
                         env={**os.environ, "SPMV_B200_RESIDENT": "1"})
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    rows = (tmp_path / "result" / "spmv_results_openmp.csv").read_text().splitlines()
    assert rows[0].startswith("matrix_name,rows,cols,nonzeros,num_threads,time_serial,")
    assert len(rows) >= 2 and rows[1].startswith("general_matrix.mtx,10,10,5,")
    header = rows[0].split(",")
    for row in rows[1:]:
        cells = dict(zip(header, row.split(",")))
        for name in header:
            if name.startswith("error_"):
                assert float(cells[name]) == 0.0, (name, cells[name])


def test_csv_row_has_the_reference_columns(tmp_path):
    lib = N.lib()
    target = tmp_path / "out.csv"
    d = N.DiffMetricsStruct(0.5, 0.25, 3)
    for _ in range(2):
        lib.write_results_to_csv(b"m.mtx", 10, 11, 5, 4, *[float(i) for i in range(1, 7)], d, d, d, d,
                                 *[float(i) for i in range(7, 21)], str(target).encode())
    lines = target.read_text().splitlines()
    assert len(lines) == 3                                   # header once, then one row per call
    header = lines[0].split(",")
    assert len(header) == 33 and header[:6] == ["matrix_name", "rows", "cols", "nonzeros", "num_threads", "time_serial"]
    assert header[11:13] == ["error_csr_relative", "error_csr_absolute"] and header[-1] == "efficiency_hll_simd"
    cells = lines[1].split(",")
    assert cells[:5] == ["m.mtx", "10", "11", "5", "4"] and cells[5] == "1.000000000000000"
    assert cells[11] == "0.250000000000000" and cells[12] == "0.500000000000000"   # relative first, then absolute
    # reference argument order (libs/utility.h:17-23): speedups, efficiencies, THEN flops -- the file has flops first
    assert cells[19] == "15.000000000000000" and cells[25] == "7.000000000000000" and cells[32] == "14.000000000000000"


def test_create_directory_never_wipes_by_default(tmp_path, monkeypatch):
    lib = N.lib()
    target = tmp_path / "result"
    lib.create_directory(str(target).encode())
    assert target.is_dir()
    (target / "keep.csv").write_text("x")
    monkeypatch.delenv("SPMV_B200_WIPE_RESULT_DIR", raising=False)
    lib.create_directory(str(target).encode())
    assert (target / "keep.csv").exists()
    monkeypatch.setenv("SPMV_B200_WIPE_RESULT_DIR", "1")
    (target / "sub").mkdir()
    lib.create_directory(str(target).encode())
    assert not (target / "keep.csv").exists() and (target / "sub").is_dir()
