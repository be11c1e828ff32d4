#!/usr/bin/env python
"""Round-2 single-GPU diagnostics (one gpurun call): fused-kernel batches on lap3d 512^3, R-MAT launch shapes,
aligned-group loads on uniform 32/row, the PCIe floor of the host-buffer call and its window sweep."""
import os
import sys
import time
from pathlib import Path

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
import torch  # noqa: E402

from sparsematrixvectormultiplication_b200 import device, synth  # noqa: E402

torch.cuda.set_device(0)


def timeit(fn, reps=20, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def section(name):
    print(f"\n== {name}", flush=True)


what = set(sys.argv[1:]) or {"lap3d", "rmat", "uniform", "pcie", "e2e"}

if "lap3d" in what:
    section("lap3d 512^3 on one GPU: plain / fused per batch")
    n = int(os.environ.get("DIAG_LAP3D_N", "512"))
    A = device.DeviceCSR.synth(synth.SYNTH_LAP3D, n)
    i = A.info()
    print(f"auto_algo {device.ALGO_NAMES[i.auto_algo]} row_batch {i.row_batch} fused_batch {i.fused_batch}")
    x = torch.ones(i.N, dtype=torch.float64, device="cuda")
    y = torch.empty(i.M, dtype=torch.float64, device="cuda")
    part = torch.zeros(A.partials_count(), dtype=torch.float64, device="cuda")
    ss = torch.ones(1, dtype=torch.float64, device="cuda")
    gb = i.algorithmic_bytes / 1e6
    for rnd in range(2):
        t = timeit(lambda: A.spmv(x, y))
        print(f"round {rnd}: plain auto {t*1e3:.1f} us {gb/t:.0f} GB/s")
        for batch in (0, 2, 3, 4, 5, 6, 7):
            os.environ["SPMV_B200_FUSED_BATCH"] = str(batch)
            t = timeit(lambda: A.spmv_fused(x, y, prev_sumsq=ss, partials=part))
            print(f"round {rnd}: fused batch {batch} {t*1e3:.1f} us {gb/t:.0f} GB/s")
        os.environ.pop("SPMV_B200_FUSED_BATCH")
        t = timeit(lambda: A.spmv_fused(x, y, prev_sumsq=ss, partials=part))
        print(f"round {rnd}: fused (plan choice {i.fused_batch}) {t*1e3:.1f} us {gb/t:.0f} GB/s")
    H = A.to_hll()
    hi = H.info()
    hp = torch.zeros(H.partials_count(), dtype=torch.float64, device="cuda")
    t = timeit(lambda: H.spmv(x, y))
    print(f"hll plain auto {t*1e3:.1f} us; fused {timeit(lambda: H.spmv_fused(x, y, prev_sumsq=ss, partials=hp))*1e3:.1f} us (row_batch {hi.row_batch})")
    for batch in (2, 3, 4, 5, 6, 7):
        os.environ["SPMV_B200_HLL_FUSED_BATCH"] = str(batch)
        t = timeit(lambda: H.spmv_fused(x, y, prev_sumsq=ss, partials=hp))
        print(f"hll fused batch {batch} {t*1e3:.1f} us")
    os.environ.pop("SPMV_B200_HLL_FUSED_BATCH")
    H.close()
    A.close()
    del x, y
    from sparsematrixvectormultiplication_b200.distributed import FusedPowerIteration
    F = FusedPowerIteration(synth.SYNTH_LAP3D, n, mailbox=True)
    print(f"FusedPowerIteration mailbox step {timeit(F.step)*1e3:.1f} us (fused_batch {F.A.info().fused_batch})")
    F.close()
    del F
    torch.cuda.empty_cache()

if "fusedgrid" in what:
    section("lap3d: plain row kernel vs the persistent fused row kernel, grid = CTAs per SM x 148")
    n = int(os.environ.get("DIAG_LAP3D_N", "512"))
    for ctas in (8, 16, 32, 64):
        os.environ["SPMV_B200_FUSED_CTAS_PER_SM"] = str(ctas)
        A = device.DeviceCSR.synth(synth.SYNTH_LAP3D, n)
        i = A.info()
        x = torch.ones(i.N, dtype=torch.float64, device="cuda")
        y = torch.empty(i.M, dtype=torch.float64, device="cuda")
        part = torch.zeros(A.partials_count(), dtype=torch.float64, device="cuda")
        ss = torch.ones(1, dtype=torch.float64, device="cuda")
        print(f"ctas/SM {ctas}: plan row_batch {i.row_batch} fused_batch {i.fused_batch}, partials {A.partials_count()}")
        if ctas == 8:
            for batch in (2, 4, 5):
                os.environ["SPMV_B200_ROW_BATCH"] = str(batch)
                A.replan()
                print(f"  plain row kernel batch {batch}: {timeit(lambda: A.spmv(x, y, algo=device.ALGO_ROW))*1e3:.1f} us")
            os.environ.pop("SPMV_B200_ROW_BATCH")
        for batch in (2, 4, 5):
            os.environ["SPMV_B200_FUSED_BATCH"] = str(batch)
            a = timeit(lambda: A.spmv_fused(x, y))
            b = timeit(lambda: A.spmv_fused(x, y, prev_sumsq=ss, partials=part))
            print(f"  fused row kernel batch {batch}: loop only {a*1e3:.1f} us, with scale + partials {b*1e3:.1f} us")
        os.environ.pop("SPMV_B200_FUSED_BATCH")
        H = A.to_hll()
        hp = torch.zeros(H.partials_count(), dtype=torch.float64, device="cuda")
        print(f"  hll: plain rows {timeit(lambda: H.spmv(x, y))*1e3:.1f} us, fused {timeit(lambda: H.spmv_fused(x, y, prev_sumsq=ss, partials=hp))*1e3:.1f} us")
        H.close()
        A.close()
        del x, y
        torch.cuda.empty_cache()
    os.environ.pop("SPMV_B200_FUSED_CTAS_PER_SM")

if "flatpick" in what:
    section("FLAT fused kernels: plan-time choice and every candidate, lap3d 512^3 and the 8-GPU rank size (512^3 / 8 rows)")
    for n, rows in ((512, None), (512, 512 ** 3 // 8)):
        A = device.DeviceCSR.synth(synth.SYNTH_LAP3D, n, row_begin=0, row_end=rows)
        i = A.info()
        H = A.to_hll()
        hi = H.info()
        print(f"rows {i.M}: CSR plan fused_batch {i.fused_batch} flat_batch {i.flat_batch}; HLL plan row_batch {hi.row_batch} fused_batch {hi.fused_batch} flat_batch {hi.flat_batch}")
        x = torch.ones(i.N, dtype=torch.float64, device="cuda")
        y = torch.empty(i.M, dtype=torch.float64, device="cuda")
        ss = torch.ones(1, dtype=torch.float64, device="cuda")
        part = torch.zeros((i.M + 255) // 256, dtype=torch.float64, device="cuda")
        print(f"  plain: CSR {timeit(lambda: A.spmv(x, y))*1e3:.1f} us, HLL {timeit(lambda: H.spmv(x, y))*1e3:.1f} us; "
              f"grid-stride fused: CSR {timeit(lambda: A.spmv_fused(x, y, prev_sumsq=ss, partials=part))*1e3:.1f} us, HLL {timeit(lambda: H.spmv_fused(x, y, prev_sumsq=ss, partials=part))*1e3:.1f} us")
        for batch in (2, 3, 4, 5, 6, 7):
            os.environ["SPMV_B200_FLAT_BATCH"] = os.environ["SPMV_B200_HLL_FLAT_BATCH"] = str(batch)
            a = timeit(lambda: A.spmv_fused_flat(x, y, inv_norm=ss, partials=part))
            b = timeit(lambda: H.spmv_fused_flat(x, y, inv_norm=ss, partials=part))
            print(f"  batch {batch}: CSR {a*1e3:.1f} HLL {b*1e3:.1f}", flush=True)
        for k in ("SPMV_B200_FLAT_BATCH", "SPMV_B200_HLL_FLAT_BATCH"):
            os.environ.pop(k, None)
        H.close()
        A.close()
        del x, y
        torch.cuda.empty_cache()

if "rmat" in what:
    section("R-MAT 24/16: binned kernel launch shapes")
    rp, ci, va = synth.rmat_csr_device(24, 16)
    M = 1 << 24
    A = device.DeviceCSR.wrap(M, M, rp, ci, va)
    x = torch.empty(M, dtype=torch.float64, device="cuda")
    device.synth_vector(x, 777)
    y = torch.empty(M, dtype=torch.float64, device="cuda")
    A.spmv(x, y, algo=device.ALGO_BINNED)
    y0 = y.clone()
    for rnd in range(3):
        for split in ("0", "1"):
            for vec4 in ("0", "2"):
                os.environ["SPMV_B200_BINNED_SPLIT"], os.environ["SPMV_B200_VEC4"] = split, vec4
                t = timeit(lambda: A.spmv(x, y, algo=device.ALGO_BINNED))
                err = float(((y - y0).abs() / y0.clamp_min(1e-300)).max())
                print(f"round {rnd}: split {split} vec4 {vec4}: {t*1e3:.1f} us  (max rel diff vs first {err:.1e})")
    os.environ.pop("SPMV_B200_BINNED_SPLIT")
    os.environ.pop("SPMV_B200_VEC4")
    A.close()
    del rp, ci, va, x, y, y0
    torch.cuda.empty_cache()

if "uniform" in what:
    section("uniform 8M x 32: scalar vs aligned-group vector kernel")
    M = 1 << 23
    A = device.DeviceCSR.synth(synth.SYNTH_UNIFORM, M, M, 32)
    H = A.to_hll()
    x = torch.empty(M, dtype=torch.float64, device="cuda")
    device.synth_vector(x, 4242)
    y = torch.empty(M, dtype=torch.float64, device="cuda")
    os.environ["SPMV_B200_VEC4"] = "0"
    A.spmv(x, y, algo=device.ALGO_VECTOR)
    y0 = y.clone()
    for rnd in range(3):
        for vec4 in ("0", "1", "2"):
            for width in ("0", "4", "8", "16"):
                os.environ["SPMV_B200_VEC4"], os.environ["SPMV_B200_VECTOR_WIDTH"] = vec4, width
                t = timeit(lambda: A.spmv(x, y, algo=device.ALGO_VECTOR))
                err = float(((y - y0).abs() / y0).max())
                print(f"round {rnd}: vec4 {vec4} width {width}: vector {t*1e3:.1f} us (diff {err:.1e})")
        os.environ.pop("SPMV_B200_VECTOR_WIDTH")
        for vec4 in ("0", "2"):
            os.environ["SPMV_B200_VEC4"] = vec4
            print(f"round {rnd}: vec4 {vec4}: binned {timeit(lambda: A.spmv(x, y, algo=device.ALGO_BINNED))*1e3:.1f} us")
        print(f"round {rnd}: hll slice {timeit(lambda: H.spmv(x, y, slice_kernel=True))*1e3:.1f} us")
    os.environ.pop("SPMV_B200_VEC4")
    H.close()
    A.close()
    del x, y, y0
    torch.cuda.empty_cache()

if "pcie" in what:
    section("PCIe floor: 128 MiB pinned, one direction and both at once")
    nbytes = 1 << 27
    h1, h2 = torch.empty(nbytes, dtype=torch.uint8).pin_memory(), torch.empty(nbytes, dtype=torch.uint8).pin_memory()
    d1, d2 = torch.empty(nbytes, dtype=torch.uint8, device="cuda"), torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

    def wall(fn, reps=10):
        fn()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) / reps

    def up():
        with torch.cuda.stream(s1):
            d1.copy_(h1, non_blocking=True)

    def down():
        with torch.cuda.stream(s2):
            h2.copy_(d2, non_blocking=True)

    def both():
        up()
        down()

    def both_chunked(k=16):
        c = nbytes // k
        for j in range(k):
            with torch.cuda.stream(s1):
                d1[j * c:(j + 1) * c].copy_(h1[j * c:(j + 1) * c], non_blocking=True)
            with torch.cuda.stream(s2):
                h2[j * c:(j + 1) * c].copy_(d2[j * c:(j + 1) * c], non_blocking=True)
    for name, fn in (("H2D alone", up), ("D2H alone", down), ("both at once", both), ("both, 16 chunks each", both_chunked)):
        t = wall(fn)
        print(f"{name}: {t*1e3:.3f} ms  ({nbytes/t/1e9:.1f} GB/s per direction)")
    try:
        print("numa:", open("/sys/bus/pci/devices/" + torch.cuda.get_device_properties(0).pci_bus_id.lower() + "/numa_node").read().strip()
              if hasattr(torch.cuda.get_device_properties(0), "pci_bus_id") else "n/a", "cpus allowed:", len(os.sched_getaffinity(0)))
    except Exception as e:
        print("numa probe failed:", e)

if "e2e" in what:
    section("host-buffer call on lap2d 4096^2: window sweep")
    n = 4096
    A = device.DeviceCSR.synth(synth.SYNTH_LAP2D, n)
    M = n * n
    xh = torch.empty(M, dtype=torch.float64).pin_memory()
    xh.copy_(1.0 + (torch.arange(M) % 7).double() / 8.0)
    yh = torch.empty(M, dtype=torch.float64).pin_memory()
    for rnd in range(2):
        for taper in ("0", "2"):
            for zero in ("1", "0"):
                os.environ["SPMV_B200_HOST_TAPER"], os.environ["SPMV_B200_HOST_ZEROCOPY"] = taper, zero
                os.environ.pop("SPMV_B200_HOST_WINDOWS", None)
                A.replan()
                for _ in range(2):
                    A.spmv_host_ptr(xh.data_ptr(), yh.data_ptr())
                t0 = time.perf_counter()
                for _ in range(10):
                    A.spmv_host_ptr(xh.data_ptr(), yh.data_ptr())
                print(f"round {rnd}: taper {taper} zero-copy {zero}: {(time.perf_counter() - t0) / 10 * 1e3:.3f} ms")
        os.environ.pop("SPMV_B200_HOST_TAPER", None)
        for zero in ("1",):
            os.environ["SPMV_B200_HOST_ZEROCOPY"] = zero
            for windows in (12, 16, 24, 32):
                if windows:
                    os.environ["SPMV_B200_HOST_WINDOWS"] = str(windows)
                else:
                    os.environ.pop("SPMV_B200_HOST_WINDOWS", None)
                A.replan()
                for _ in range(2):
                    A.spmv_host_ptr(xh.data_ptr(), yh.data_ptr())
                t0 = time.perf_counter()
                for _ in range(10):
                    A.spmv_host_ptr(xh.data_ptr(), yh.data_ptr())
                dt = (time.perf_counter() - t0) / 10
                print(f"round {rnd}: zero-copy y {zero} windows {windows or 'auto (tapered)'}: {dt*1e3:.3f} ms")
    os.environ.pop("SPMV_B200_HOST_ZEROCOPY", None)
    os.environ.pop("SPMV_B200_HOST_WINDOWS", None)
    A.close()
