#!/usr/bin/env python
"""bench.py -- SpMV GFLOPS and HBM GB/s for CSR and HLL on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--quick] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

N = 1  workload "lap2d_4096_csr" (BASELINE.json configs[1]): fp64 CSR product of the 2-D 5-point
       Laplacian on a 4096 x 4096 grid (16.8 M rows, 83.9 M nnz, 1.34 GB streamed per product).
       A step is ONE product y = A x with the matrix resident in HBM.  The other single-GPU configs
       (HLL of the same matrix, uniform 8M x 8M x 32 CSR/HLL, R-MAT, the 512^3 power iteration on one
       GPU) are measured too and reported under "others" -- they are not the headline.
N > 1  workload "lap3d_512_power" (configs[4]): power iteration on the 512^3 7-point Laplacian,
       rows partitioned by nnz over the N ranks, x refreshed every iteration.  Headline = "fused_split": boundary
       rows stored into the neighbours over NVLink by the product kernel, |w|^2 through peer mailboxes, two
       launches per iteration, no collective call.  Every other exchange is timed beside it under
       "exchange_modes" (halo-only and whole-vector refreshes: "allgather" = one ncclAllGather, "allgather_peer"
       = the same data movement written against peer memory; HLL twins; the one-launch forms) and every one of
       them is parity-checked against the single-GPU iteration inside the run ("parity").  A step is one
       iteration (product + norm + scale + exchange); value = 2 * nnz_global / t, strong scaling; "e2e" = the
       same loop with lambda read back on the host after every iteration.

--impl reference times the reference's own CPU implementation (oracle/_ref, built from the unmodified
reference sources; the oracle port if that .so is absent) on the host cores, same workload and metric.

One JSON line on stdout (rank 0).  Everything else goes to stderr.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402

HBM_NOMINAL_GBS = 8000.0   # BASELINE.json quotes fractions of 8 TB/s
FALLBACK_PEAK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


def ncu_traffic(workload: str, kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` on `workload` from the committed ncu --set full
    captures: profiles/ncu_traffic.json, keyed "<workload>|<kernel incl. template arguments>" (written by
    tools/ncu_summary.py --traffic-json).  None when that exact kernel (e.g. another plan-time batch) was never captured."""
    try:
        table = json.loads((ROOT / "profiles" / "ncu_traffic.json").read_text())
    except (OSError, ValueError):
        return None, None
    hit = table.get(f"{workload}|{kernel}")
    if not hit:
        return None, None
    return int(hit["dram_bytes"]), hit.get("source")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


_REAL_STDOUT = None


def capture_stdout():
    """Everything that libraries print on fd 1 (NCCL's version banner, the reference's printf()s) goes to
    stderr; the one JSON line is written to the real stdout by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    sys.stdout.flush()
    data = (json.dumps(line) + "\n").encode()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, data)


def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return FALLBACK_PEAK_GBS, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------------
# clocks: NVML sampled in a thread while the GPU is busy
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}

    def __init__(self, index=0, period=0.004):
        self.samples = []   # (t, sm_mhz, reasons_bitmask, power_w)
        self.windows = []
        self.period = period
        self._stop = threading.Event()
        self._thread = None
        self.max_sm = None
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    index = int(vis.split(",")[index])
                except (ValueError, IndexError):
                    pass
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # pragma: no cover
            log(f"[clocks] NVML unavailable: {e}")

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                try:
                    power = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                except Exception:
                    power = None
                self.samples.append((time.perf_counter(), sm, reasons, power))
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.ok:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=1.0)

    def window(self, t0, t1):
        self.windows.append((t0, t1))

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_sm, "reasons": [], "samples": 0, "source": "unavailable"}
        inside = [s for s in self.samples if any(a <= s[0] <= b for a, b in self.windows)]
        src = "nvml, sampled during the timed regions"
        if len(inside) < 3:  # a very short timed region: use every sample taken while the bench kept the GPU busy
            inside, src = self.samples, "nvml, sampled during the whole GPU-busy phase (timed region too short)"
        mask = 0
        for s in inside:
            mask |= s[2]
        reasons = sorted({name for bit, name in self.REASONS.items() if mask & bit})
        powers = [s[3] for s in inside if s[3] is not None]
        return {"sm_mhz": statistics.median(s[1] for s in inside), "sm_max_mhz": self.max_sm, "reasons": reasons,
                "samples": len(inside), "power_w_max": max(powers) if powers else None, "source": src}


# ---------------------------------------------------------------------------------------------------
# timing helpers
# ---------------------------------------------------------------------------------------------------
def time_device(fn, steps, warmup, sampler=None, world=1):
    """W untimed + exactly K timed calls; CUDA events on the current (launching) stream, barrier and
    synchronize on both sides, MAX over ranks.  Returns (ms_per_step, per_step_ms_list)."""
    import torch
    import torch.distributed as dist
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    t0 = time.perf_counter()
    marks[0].record()
    for i in range(steps):
        fn()
        marks[i + 1].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    t1 = time.perf_counter()
    if sampler:
        sampler.window(t0, t1)
    total = marks[0].elapsed_time(marks[steps])
    per = [marks[i].elapsed_time(marks[i + 1]) for i in range(steps)]
    if world > 1:
        t = torch.tensor([total], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total = float(t.item())
    return total / steps, per


def spmv_stats(nnz, bytes_alg, ms, peak):
    s = ms * 1e-3
    gbs = bytes_alg / s / 1e9
    return {"gflops": 2.0 * nnz / s / 1e9, "ms": ms, "gbs": gbs, "frac_of_measured_peak": gbs / peak,
            "frac_of_8tbs": gbs / HBM_NOMINAL_GBS, "algorithmic_bytes": int(bytes_alg)}


def ramp_vector(n, device):
    import torch
    return 1.0 + (torch.arange(n, device=device, dtype=torch.int64) % 7).to(torch.float64) / 8.0


DUMP_ROWS = 1 << 21   # 16 MiB of values + 16 MiB of row indices: the whole headline y (134 MB) exceeds a dump's 64 MB
DUMP_SEED = 20261020


def dump_outputs(out_dir, y):
    """What the caller of the timed product receives, y, at a fixed seeded sample of rows, so that two builds can be
    compared output for output: DIR/y_sample.npy (float64) and DIR/y_sample_rows.npy (its row indices, float64)."""
    import torch
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(y.numel(), size=min(DUMP_ROWS, y.numel()), replace=False))
    values = y[torch.from_numpy(rows).to(y.device)].cpu().numpy()
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "y_sample.npy", values.astype(np.float64))
    np.save(out / "y_sample_rows.npy", rows.astype(np.float64))
    log(f"[bench] wrote {len(rows)} sampled rows of y to {out}")


# ---------------------------------------------------------------------------------------------------
# CPU baseline (the reference's own CPU path on the host cores)
# ---------------------------------------------------------------------------------------------------
def cpu_baseline_lap2d(n, rp, ci, va, budget_s=20.0, hll_budget_s=5.0):
    """oracle/_ref (kind 'reference') or the oracle port, OpenMP over all host cores + the serial loop,
    on the full workload matrix; a bounded number of products."""
    from oracle import oracle as O
    chk = O.best_available()
    cores = os.cpu_count() or 1
    N = n * n
    x = 1.0 + (np.arange(N) % 7) / 8.0
    nnz = int(rp[-1])
    t0 = time.perf_counter()
    chk.spmv_csr_serial(rp, ci, va, x)
    serial_s = time.perf_counter() - t0
    starts, ends = chk.partition_rows(rp, cores)
    y = np.zeros(N)
    chk.spmv_csr_parallel(rp, ci, va, x, starts, ends, y=y)  # warm-up
    times = []
    t_begin = time.perf_counter()
    while len(times) < 95 and (time.perf_counter() - t_begin) < budget_s:
        t0 = time.perf_counter()
        chk.spmv_csr_parallel(rp, ci, va, x, starts, ends, y=y)
        times.append(time.perf_counter() - t0)
    mean_s = sum(times) / len(times)
    out = {"value": 2.0 * nnz / mean_s / 1e9, "unit": "GFLOP/s", "cores": len(starts), "kind": chk.kind,
           "sample": f"full lap2d_{n} matrix ({nnz} nnz), {len(times)} timed OpenMP CSR products (spvm_csr_parallel) "
                     f"after 1 warm-up, mean; host has {cores} logical cores",
           "serial_gflops": 2.0 * nnz / serial_s / 1e9, "best_gflops": 2.0 * nnz / min(times) / 1e9, "cpu_model": cpu_model()}
    # thread sweep of the OpenMP CSR product (the reference sweeps {2,4,8,16,32,40}, main.c:18) and the HLL paths
    try:
        sweep = {}
        t = 1
        while t <= cores:
            st, en = chk.partition_rows(rp, t)
            chk.spmv_csr_parallel(rp, ci, va, x, st, en, y=y)
            reps = []
            for _ in range(3):
                t0 = time.perf_counter()
                chk.spmv_csr_parallel(rp, ci, va, x, st, en, y=y)
                reps.append(time.perf_counter() - t0)
            sweep[str(len(st))] = 2.0 * nnz / min(reps) / 1e9
            t *= 2
        out["csr_openmp_gflops_by_threads"] = sweep
        if hll_budget_s > 0:
            out.update(cpu_baseline_hll(chk, n, rp, ci, va, x, nnz, cores, hll_budget_s))
    except Exception as e:  # pragma: no cover
        out["sweep_error"] = repr(e)
    return out


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def cpu_baseline_hll(chk, n, rp, ci, va, x, nnz, cores, budget_s):
    """The reference's spmv_hll_serial and spmv_hll (OpenMP over its own block partition) on the same matrix.  The HLL
    blocks are built by this repo's host converter (bit-identical to the reference's, tests/test_host_api.py)."""
    import ctypes as C
    from sparsematrixvectormultiplication_b200 import host
    N = n * n
    rows = np.repeat(np.arange(N, dtype=np.int32), np.diff(rp))
    hll = host.convert_to_hll(host.PreMatrix(N, N, rows, ci, va))
    del rows
    xs = np.ascontiguousarray(x, np.float64)
    y = np.zeros(hll.num_blocks * 32, np.float64)
    xp, yp = xs.ctypes.data_as(C.POINTER(C.c_double)), y.ctypes.data_as(C.POINTER(C.c_double))
    lib = chk.lib                                   # the checker's library: the reference .so when it was built
    blocks = C.cast(hll.c.blocks, C.c_void_p)       # same struct layout as the reference's ELLPACKBlock
    lib.spmv_hll_serial.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    lib.spmv_hll_serial.restype = None
    t0 = time.perf_counter()
    lib.spmv_hll_serial(hll.num_blocks, blocks, xp, yp)
    serial_s = time.perf_counter() - t0
    bs, be = host.prepare_thread_distribution_hll(hll, cores)
    bs, be = np.ascontiguousarray(bs, np.int32), np.ascontiguousarray(be, np.int32)
    lib.spmv_hll.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_int, C.c_void_p, C.c_void_p]
    lib.spmv_hll.restype = None
    call = lambda: lib.spmv_hll(blocks, xp, yp, len(bs), bs.ctypes.data_as(C.c_void_p), be.ctypes.data_as(C.c_void_p))  # noqa: E731
    call()
    times, t_begin = [], time.perf_counter()
    while len(times) < 30 and (time.perf_counter() - t_begin) < budget_s:
        t0 = time.perf_counter()
        call()
        times.append(time.perf_counter() - t0)
    return {"hll_serial_gflops": 2.0 * nnz / serial_s / 1e9, "hll_openmp_gflops": 2.0 * nnz / (sum(times) / len(times)) / 1e9,
            "hll_openmp_threads": len(bs), "hll_sample": f"{len(times)} timed spmv_hll products on {len(bs)} block ranges"}


# ---------------------------------------------------------------------------------------------------
# arms
# ---------------------------------------------------------------------------------------------------
def workload_config(n_gpus, lap3d_n=512):
    """The `config` object BOTH arms print (same keys, same values: the driver compares them)."""
    if n_gpus == 1:
        n = 4096
        return {"workload": "lap2d_4096_csr", "rows": n * n, "cols": n * n, "nnz": 5 * n * n - 4 * n, "format": "csr",
                "x": "1+(i mod 7)/8", "step": "one product y = A x, matrix resident",
                "l2": "inputs_exceed_l2 (1.34 GB streamed per product vs 126 MB L2)"}
    n = lap3d_n
    return {"workload": f"lap3d_{n}_power", "rows": n ** 3, "cols": n ** 3, "nnz": 7 * n ** 3 - 6 * n * n, "format": "csr",
            "x": "x0 = ones", "step": "one power iteration: y = A x; lambda = |y|_2; x = y / lambda",
            "l2": "inputs_exceed_l2"}


def run_reference(args):
    """The reference's CPU implementation of the path on the host cores, on our arm's config/metric: at N = 1 one OpenMP
    CSR product of the full lap2d matrix per step; at N > 1 one power iteration on the FULL lap3d matrix per step
    (reference spvm_csr_parallel for the product, norm + scale in an OpenMP region of the oracle)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from sparsematrixvectormultiplication_b200 import synth
    from oracle import oracle as O
    chk = O.best_available()
    cores = os.cpu_count() or 1
    config = workload_config(args.gpus, args.lap3d_n)
    if args.gpus == 1:
        n = 4096
        log("[reference] generating lap2d 4096^2 on the host (numpy twin) ...")
        rp, ci, va = synth.lap2d_csr(n)
        x = 1.0 + (np.arange(n * n) % 7) / 8.0
        nnz = int(rp[-1])
        starts, ends = chk.partition_rows(rp, cores)
        y = np.zeros(n * n)

        def step():
            chk.spmv_csr_parallel(rp, ci, va, x, starts, ends, y=y)
        sample = f"full lap2d_4096 matrix, one OpenMP CSR product (spvm_csr_parallel) per step on {len(starts)} threads"
        scaling = "weak"
    else:
        n = args.lap3d_n
        log(f"[reference] generating the full lap3d {n}^3 matrix on the host (OpenMP generator of the oracle) ...")
        t0 = time.perf_counter()
        rp, ci, va = O.lap3d_csr_host(n)
        nnz = int(rp[-1])
        log(f"[reference] {nnz} nnz in {time.perf_counter() - t0:.1f} s")
        starts, ends = chk.partition_rows(rp, cores)
        x = np.ones(n ** 3)
        y = np.zeros(n ** 3)
        lam = [0.0]

        def step():
            chk.spmv_csr_parallel(rp, ci, va, x, starts, ends, y=y)
            lam[0] = O.norm_scale(y, x, len(starts))
        sample = (f"FULL {n}^3 7-point Laplacian ({nnz} nnz), one power iteration per step: reference spvm_csr_parallel on "
                  f"{len(starts)} threads + norm and scale in an OpenMP region (oracle.c orc_norm_scale)")
        scaling = "strong"
    assert nnz == config["nnz"], (nnz, config["nnz"])
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    value = 2.0 * nnz / dt / 1e9
    line = {"impl": "reference", "metric": "spmv_gflops", "value": value, "unit": "GFLOP/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
            "cpu_baseline": {"value": value, "unit": "GFLOP/s", "cores": len(starts), "kind": chk.kind, "sample": sample},
            "e2e": {"value": value, "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if args.gpus > 1:
        line["lambda"] = lam[0]
    emit(line)


def bench_single_gpu(args):
    import torch
    from sparsematrixvectormultiplication_b200 import device, synth
    torch.cuda.set_device(0)
    peak, peak_src = measured_peak()
    sampler = ClockSampler(0)
    sampler.start()
    n = 4096
    workload = "lap2d_4096_csr"
    log(f"[bench] {device.device_info()}")
    A = device.DeviceCSR.synth(synth.SYNTH_LAP2D, n)
    info = A.info()
    M, nnz, bytes_alg = info.M, info.nnz, info.algorithmic_bytes
    x = ramp_vector(M, "cuda")
    y = torch.empty(M, dtype=torch.float64, device="cuda")
    launches_per_step = 1 + (2 if info.num_long_rows else 0)

    ms, per = time_device(lambda: A.spmv(x, y), args.steps, args.warmup, sampler)
    head = spmv_stats(nnz, bytes_alg, ms, peak)
    log(f"[bench] {workload}: {head['gflops']:.1f} GFLOP/s, {head['gbs']:.0f} GB/s, {ms*1e3:.1f} us/product "
        f"(min {min(per)*1e3:.1f}, median {statistics.median(per)*1e3:.1f})")
    if args.dump_outputs:   # before the legs below reuse y
        dump_outputs(args.dump_outputs, y)

    # ---- end to end through the C-ABI host call: pinned host x -> H2D, product, D2H -> pinned host y ----
    xh = torch.empty(M, dtype=torch.float64).pin_memory()
    xh.copy_(x.cpu())
    yh = torch.empty(M, dtype=torch.float64).pin_memory()
    e2e_steps = max(3, min(args.steps, 30))
    for _ in range(2):
        A.spmv_host_ptr(xh.data_ptr(), yh.data_ptr())
    t0 = time.perf_counter()
    e2e_each = []
    for _ in range(e2e_steps):          # every call is synchronous: per-call times for the spread, the mean for the value
        t_call = time.perf_counter()
        A.spmv_host_ptr(xh.data_ptr(), yh.data_ptr())
        e2e_each.append(time.perf_counter() - t_call)
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    sampler.window(t0, time.perf_counter())
    torch.cuda.synchronize()
    assert torch.equal(yh.cuda(), y), "end-to-end result differs from the resident product"
    e2e = {"value": 2.0 * nnz / e2e_s / 1e9, "unit": "GFLOP/s", "h2d_bytes_per_step": 8 * info.N, "d2h_bytes_per_step": 8 * M,
           "ms_per_step": e2e_s * 1e3, "steps": e2e_steps, "ms_min": min(e2e_each) * 1e3, "ms_median": statistics.median(e2e_each) * 1e3,
           "api": "spmv_b200_csr_spmv_host (one synchronous C-ABI call: pinned host x -> device, product, device -> pinned host y; upload, product and download pipelined over row windows on three streams)"}
    log(f"[bench] e2e: {e2e['value']:.1f} GFLOP/s ({e2e_s*1e3:.2f} ms/step)")

    others = {}
    if not args.quick:
        others = measure_others(args, A, x, y, peak, sampler, head)

    # ---- CPU baseline on the host cores (bounded) ----
    cpu = None
    if not args.no_cpu:
        try:
            rp, ci, va = A.download()
            cpu = cpu_baseline_lap2d(n, rp, ci, va, budget_s=args.cpu_budget)
            log(f"[bench] cpu_baseline: {cpu['value']:.2f} GFLOP/s on {cpu['cores']} threads ({cpu['kind']}), serial {cpu['serial_gflops']:.2f}")
            del rp, ci, va
        except Exception as e:  # pragma: no cover
            log(f"[bench] cpu baseline failed: {e!r}")
    sampler.stop()

    config = workload_config(1)
    assert (config["rows"], config["cols"], config["nnz"]) == (M, info.N, nnz)
    kernel_name = (f"csr_row_kernel<{info.row_batch},double>" if info.auto_algo == device.ALGO_ROW
                   else device.ALGO_NAMES[info.auto_algo])
    traffic, traffic_src = ncu_traffic(workload, kernel_name)
    line = {"metric": "spmv_gflops", "value": head["gflops"], "unit": "GFLOP/s", "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": config,
            "implementation": {"kernel": device.ALGO_NAMES[info.auto_algo] + " (automatic choice)", "kernel_symbol": kernel_name,
                               "row_batch": info.row_batch, "max_row_nnz": info.max_row_nnz, "tiles": info.num_tiles},
            "roofline": {"bound": "hbm", "achieved": head["gbs"], "peak": peak, "unit": "GB/s", "frac": head["gbs"] / peak,
                         "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "kernel": kernel_name,
                         "algorithmic_bytes_per_launch": int(bytes_alg), "frac_of_8tbs": head["frac_of_8tbs"],
                         "kernel_ms_min": min(per), "kernel_ms_median": statistics.median(per)},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches_per_step * args.steps,
            "clocks": sampler.summary(), "others": others}
    emit(line)


def measure_others(args, A2d, x2d, y2d, peak, sampler, head):
    """The remaining single-GPU configs of BASELINE.json -- reported, not the headline."""
    import torch
    from sparsematrixvectormultiplication_b200 import device, synth
    out = {"lap2d_4096_csr": dict(head, kernel="the headline product (automatic choice), repeated here for the ratios below")}
    steps, warm = max(5, min(args.steps, 100)), max(3, min(args.warmup, 10))

    def run(name, fn, nnz, bytes_alg, extra=None):
        try:
            ms, per = time_device(fn, steps, warm, sampler)
            out[name] = spmv_stats(nnz, bytes_alg, ms, peak)
            out[name]["ms_min"] = min(per)
            if extra:
                out[name].update(extra)
            log(f"[bench] {name}: {out[name]['gflops']:.1f} GFLOP/s, {out[name]['gbs']:.0f} GB/s ({ms*1e3:.1f} us)")
        except Exception as e:  # pragma: no cover
            out[name] = {"error": repr(e)}
            log(f"[bench] {name} failed: {e!r}")

    def csr_variants(name, A, x, y, with_auto=True):
        ia = A.info()
        if with_auto:
            run(f"{name}_csr", lambda: A.spmv(x, y), ia.nnz, ia.algorithmic_bytes, {"kernel": "automatic choice"})
        run(f"{name}_csr_stream_kernel", lambda: A.spmv(x, y, algo=device.ALGO_STREAM), ia.nnz, ia.algorithmic_bytes)
        run(f"{name}_csr_vector_kernel", lambda: A.spmv(x, y, algo=device.ALGO_VECTOR), ia.nnz, ia.algorithmic_bytes)
        run(f"{name}_csr_binned_kernel", lambda: A.spmv(x, y, algo=device.ALGO_BINNED), ia.nnz, ia.algorithmic_bytes)
        if ia.max_row_nnz <= 64:  # one thread per row is only meaningful without long rows
            run(f"{name}_csr_row_kernel", lambda: A.spmv(x, y, algo=device.ALGO_ROW), ia.nnz, ia.algorithmic_bytes, {"row_batch": ia.row_batch})
        if f"{name}_csr" in out and "error" not in out[f"{name}_csr"]:
            out[f"{name}_csr"]["kernel"] = "automatic choice: " + device.ALGO_NAMES[ia.auto_algo]

    def hll_variants(name, A, x, y):
        ia = A.info()
        H = A.to_hll()
        hi = H.info()
        run(f"{name}_hll", lambda: H.spmv(x, y), ia.nnz, hi.algorithmic_bytes, {"slots": hi.slots, "kernel": "automatic choice"})
        run(f"{name}_hll_stream_kernel", lambda: H.spmv(x, y, slice_kernel=False), ia.nnz, hi.algorithmic_bytes)
        run(f"{name}_hll_slice_kernel", lambda: H.spmv(x, y, slice_kernel=True), ia.nnz, hi.algorithmic_bytes)
        if hi.max_maxnz <= 64:
            run(f"{name}_hll_row_kernel", lambda: H.spmv(x, y, slice_kernel="rows"), ia.nnz, hi.algorithmic_bytes,
                {"row_batch": hi.row_batch, "kernel": H.row_form()})
        if f"{name}_hll" in out and "error" not in out[f"{name}_hll"]:
            out[f"{name}_hll"]["kernel"] = "automatic choice: " + device.HLL_KERNEL_NAMES[hi.auto_kernel]
            if hi.auto_kernel == 2:  # the lane-per-row path: which of its kernels the plan-time timing chose
                out[f"{name}_hll"]["kernel_symbol"] = H.row_form()
        H.close()

    try:
        csr_variants("lap2d_4096", A2d, x2d, y2d, with_auto=False)
        hll_variants("lap2d_4096", A2d, x2d, y2d)
    except Exception as e:  # pragma: no cover
        out["lap2d_4096_variants"] = {"error": repr(e)}

    # fp32 storage / fp64 arithmetic on the headline matrix (SURVEY.md section 8(f).3): reported, never the headline
    try:
        A2d.enable_f32()
        x32, y32 = x2d.to(torch.float32), torch.empty(y2d.numel(), dtype=torch.float32, device="cuda")
        ia = A2d.info()
        run("lap2d_4096_csr_f32", lambda: A2d.spmv_f32(x32, y32), ia.nnz, A2d.algorithmic_bytes_f32(),
            {"dtype": "f32 storage (values, x, y), f64 arithmetic", "bytes_formula": "8 nnz + 4 (M+1) + 4 M + 4 N",
             "kernel": A2d.row_form_f32()})
        A2d.spmv(x2d, y2d)
        out["lap2d_4096_csr_f32"]["max_rel_diff_vs_f64"] = float(((y32.double() - y2d).abs() / (8.0 * 1.75)).max().item())
        y32_multi = y32.clone()
        H32 = A2d.to_hll().enable_f32()
        run("lap2d_4096_hll_f32", lambda: H32.spmv_f32(x32, y32), ia.nnz, H32.algorithmic_bytes_f32(),
            {"dtype": "f32 storage (values, x, y), f64 arithmetic", "kernel": H32.row_form_f32()})
        # the same with the plan-time choice restricted to the one-row-per-thread forms (the round-1 / 2d kernels): what
        # the multi-row forms buy, on the same box in the same run; results must be bitwise equal
        os.environ["SPMV_B200_ROW_MULTI_TUNE"] = "0"
        try:
            A1 = device.DeviceCSR.synth(synth.SYNTH_LAP2D, 4096).enable_f32()
            run("lap2d_4096_csr_f32_one_row_forms", lambda: A1.spmv_f32(x32, y32), ia.nnz, A1.algorithmic_bytes_f32(),
                {"kernel": A1.row_form_f32()})
            out["lap2d_4096_csr_f32"]["bitwise_equal_to_one_row_form"] = bool(torch.equal(y32, y32_multi))
            H1 = A1.to_hll().enable_f32()
            run("lap2d_4096_hll_f32_one_row_forms", lambda: H1.spmv_f32(x32, y32), ia.nnz, H1.algorithmic_bytes_f32(),
                {"kernel": H1.row_form_f32()})
            H1.close()
            A1.close()
        finally:
            del os.environ["SPMV_B200_ROW_MULTI_TUNE"]
        H32.close()
        del x32, y32, y32_multi
    except Exception as e:  # pragma: no cover
        out["lap2d_4096_csr_f32"] = {"error": repr(e)}
        log(f"[bench] fp32 leg failed: {e!r}")

    # the reference's own GPU kernels, recompiled unmodified for sm_100a ("existing kernel" bar), on every single-GPU shape
    def reference_kernels(name, A, x, y, with_hll=True):
        try:
            from oracle import oracle as O
            if not O.reference_cuda_available():
                out[f"{name}_reference_kernels"] = {"skipped": "oracle/_ref/libspmv_ref_cuda.so not present"}
                return
            import ctypes as C
            from sparsematrixvectormultiplication_b200 import _native as N
            ref = O.ReferenceCuda()
            ia = A.info()
            ptrs = [C.c_void_p() for _ in range(3)]
            N.check(N.lib().spmv_b200_csr_device_arrays(A._h, *[C.byref(p) for p in ptrs]))

            class _Raw:
                def __init__(self, p):
                    self.p = p

                def data_ptr(self):
                    return self.p
            rp, ci, va = (_Raw(p.value) for p in ptrs)
            yr = torch.empty_like(y)
            A.spmv(x, y)
            scale = float(y.abs().max().item()) or 1.0
            best = None
            for which, kname in enumerate(O.ReferenceCuda.CSR_KERNELS):
                key = f"{name}_reference_{kname}"
                run(key, lambda: ref.csr_spmv(which, ia.M, ia.N, rp, ci, va, x, yr), ia.nnz, ia.algorithmic_bytes,
                    {"kernel": f"reference {kname}, unmodified, recompiled for sm_100a (cuda_src/csr_matrix_cuda.cu)"})
                if "error" not in out[key]:
                    out[key]["max_rel_diff_vs_ours"] = float((yr - y).abs().max().item()) / scale
                    best = min(best, out[key]["ms"]) if best else out[key]["ms"]
            if best and f"{name}_csr" in out and "ms" in out[f"{name}_csr"]:
                out[f"{name}_csr"]["speedup_vs_best_reference_csr_kernel"] = best / out[f"{name}_csr"]["ms"]
            if with_hll:
                H = A.to_hll()
                hi = H.info()
                host_hll = H.download()
                handle = ref.hll_upload(C.byref(host_hll.c), ia.M)
                best = None
                for which, kname in enumerate(O.ReferenceCuda.HLL_KERNELS):
                    key = f"{name}_reference_{kname}"
                    run(key, lambda: ref.hll_spmv(handle, which, x, yr), ia.nnz, hi.algorithmic_bytes,
                        {"kernel": f"reference {kname}, unmodified, recompiled for sm_100a (cuda_src/hll_matrix.cu); reference row-major block layout in one arena"})
                    if "error" not in out[key]:
                        out[key]["max_rel_diff_vs_ours"] = float((yr - y).abs().max().item()) / scale
                        best = min(best, out[key]["ms"]) if best else out[key]["ms"]
                if best and f"{name}_hll" in out and "ms" in out[f"{name}_hll"]:
                    out[f"{name}_hll"]["speedup_vs_best_reference_hll_kernel"] = best / out[f"{name}_hll"]["ms"]
                ref.hll_free(handle)
                H.close()
                del host_hll
            del yr
        except Exception as e:  # pragma: no cover
            out[f"{name}_reference_kernels"] = {"error": repr(e)}
            log(f"[bench] reference CUDA kernels on {name} failed: {e!r}")

    def e2e_host(name, A, x):
        """The C-ABI host call (pinned host x -> device, product, device -> pinned host y) on another shape."""
        try:
            ia = A.info()
            xh = torch.empty(ia.N, dtype=torch.float64).pin_memory()
            xh.copy_(x.cpu())
            yh = torch.empty(ia.M, dtype=torch.float64).pin_memory()
            for _ in range(2):
                A.spmv_host_ptr(xh.data_ptr(), yh.data_ptr())
            t0 = time.perf_counter()
            reps = 5
            for _ in range(reps):
                A.spmv_host_ptr(xh.data_ptr(), yh.data_ptr())
            dt = (time.perf_counter() - t0) / reps
            out[f"{name}_csr_e2e_host"] = {"gflops": 2.0 * ia.nnz / dt / 1e9, "ms": dt * 1e3, "h2d_bytes": 8 * ia.N, "d2h_bytes": 8 * ia.M,
                                          "api": "spmv_b200_csr_spmv_host"}
            log(f"[bench] {name} e2e host call: {out[f'{name}_csr_e2e_host']['gflops']:.1f} GFLOP/s ({dt*1e3:.2f} ms)")
        except Exception as e:  # pragma: no cover
            out[f"{name}_csr_e2e_host"] = {"error": repr(e)}

    reference_kernels("lap2d_4096", A2d, x2d, y2d)

    # config 3: uniform 8M x 8M, 32 nnz/row, CSR vs HLL hack 32
    try:
        M = 1 << 23
        A = device.DeviceCSR.synth(synth.SYNTH_UNIFORM, M, M, 32)
        x = torch.empty(M, dtype=torch.float64, device="cuda")
        device.synth_vector(x, 4242)
        y = torch.empty(M, dtype=torch.float64, device="cuda")
        csr_variants("uniform_8m_32", A, x, y)
        hll_variants("uniform_8m_32", A, x, y)
        Hp = A.to_hll()
        for knob in ("0", "1"):   # persisting-L2 window on x (SPMV_B200_L2_PERSIST) off / on, same kernels
            os.environ["SPMV_B200_L2_PERSIST"] = knob
            ia = A.info()
            run(f"uniform_8m_32_csr_vector_kernel_l2persist{knob}", lambda: A.spmv(x, y, algo=device.ALGO_VECTOR), ia.nnz, ia.algorithmic_bytes)
            run(f"uniform_8m_32_hll_slice_kernel_l2persist{knob}", lambda: Hp.spmv(x, y, slice_kernel=True), ia.nnz, Hp.info().algorithmic_bytes)
        os.environ.pop("SPMV_B200_L2_PERSIST", None)
        Hp.close()
        reference_kernels("uniform_8m_32", A, x, y)
        e2e_host("uniform_8m_32", A, x)
        A.close()
        del x, y
    except Exception as e:  # pragma: no cover
        out["uniform_8m_32"] = {"error": repr(e)}
        log(f"[bench] uniform failed: {e!r}")

    # config 4: R-MAT scale 24, 16 edges/row, skewed rows
    try:
        torch.cuda.empty_cache()
        rp, ci, va = synth.rmat_csr_device(24, 16)
        Mr = (1 << 24)
        A = device.DeviceCSR.wrap(Mr, Mr, rp, ci, va)
        ia = A.info()
        max_row = int((rp[1:] - rp[:-1]).max().item())
        x = torch.empty(Mr, dtype=torch.float64, device="cuda")
        device.synth_vector(x, 777)
        y = torch.empty(Mr, dtype=torch.float64, device="cuda")
        csr_variants("rmat_24_16", A, x, y)
        for knob, miss in (("0", "0"), ("1", "0"), ("1", "1")):   # x (128 MiB) exceeds the carve-out: hitRatio < 1
            os.environ["SPMV_B200_L2_PERSIST"], os.environ["SPMV_B200_L2_MISS_NORMAL"] = knob, miss
            run(f"rmat_24_16_csr_binned_kernel_l2persist{knob}_missnormal{miss}", lambda: A.spmv(x, y, algo=device.ALGO_BINNED), ia.nnz, ia.algorithmic_bytes)
        os.environ.pop("SPMV_B200_L2_PERSIST", None)
        os.environ.pop("SPMV_B200_L2_MISS_NORMAL", None)
        reference_kernels("rmat_24_16", A, x, y, with_hll=False)
        if "rmat_24_16_csr" in out and "error" not in out["rmat_24_16_csr"]:
            out["rmat_24_16_csr"].update({"max_row_nnz": max_row, "long_rows": ia.num_long_rows,
                                          "fragments": ia.num_fragments, "tiles": ia.num_tiles})
        A.close()
        del rp, ci, va, x, y
        torch.cuda.empty_cache()
    except Exception as e:  # pragma: no cover
        out["rmat_24_16_csr"] = {"error": repr(e)}
        log(f"[bench] rmat failed: {e!r}")

    # config 5 on ONE GPU: T1 of the multi-GPU scaling series
    try:
        from sparsematrixvectormultiplication_b200.distributed import FusedPowerIteration, PowerIteration
        for key, kwargs, what in (
                ("lap3d_512_power_1gpu", {"split": True}, "two launches: FLAT fused product (lazy normalisation, |w|^2 partials) + one-CTA exchange kernel"),
                ("lap3d_512_power_1gpu_one_launch", {"mailbox": True}, "one launch: grid-stride fused product + lazy normalisation + |w|^2 (mailbox)"),
                ("lap3d_512_power_1gpu_hll", {"split": True, "fmt": "hll"}, "HLL image, two launches"),
                ("lap3d_512_power_1gpu_hll_one_launch", {"mailbox": True, "fmt": "hll"}, "HLL image, one launch")):
            F = FusedPowerIteration(synth.SYNTH_LAP3D, 512, **kwargs)
            ms, per = time_device(F.step, steps, warm, sampler)
            fi = F.A.info()
            out[key] = {"gflops": 2.0 * F.nnz_global / (ms * 1e-3) / 1e9, "ms_per_iteration": ms, "nnz": F.nnz_global,
                        "launches_per_step": F.launches_per_step, "kernel": what,
                        "plan": {"fused_batch": fi.fused_batch, "flat_batch": fi.flat_batch, "flat_chunks": fi.flat_chunks}}
            F.close()
            log(f"[bench] {key}: {out[key]['gflops']:.1f} GFLOP/s ({ms:.3f} ms/iteration)")
            del F
            torch.cuda.empty_cache()
        P = PowerIteration(synth.SYNTH_LAP3D, 512)
        ms, per = time_device(P.step, steps, warm, sampler)
        out["lap3d_512_power_1gpu_unfused"] = {"gflops": 2.0 * P.nnz_global / (ms * 1e-3) / 1e9, "ms_per_iteration": ms,
                                               "nnz": P.nnz_global, "launches_per_step": P.launches_per_step}
        A3 = P.A
        i3 = A3.info()
        run("lap3d_512_csr_product_only", lambda: A3.spmv(P.x, P.y), i3.nnz, i3.algorithmic_bytes)
        log(f"[bench] lap3d_512_power_1gpu_unfused: {out['lap3d_512_power_1gpu_unfused']['gflops']:.1f} GFLOP/s ({ms:.3f} ms/iteration)")
        del P
        torch.cuda.empty_cache()
    except Exception as e:  # pragma: no cover
        out["lap3d_512_power_1gpu"] = {"error": repr(e)}
        log(f"[bench] lap3d failed: {e!r}")
    return out


HEAD_MODE = "fused_split"   # the headline exchange of the N > 1 line (fastest measured: profiles/r02*_bench_n*.json)
PARITY_ITERS = 12
PARITY_TOL = 1e-12   # tools/dist_check.py: x and lambda of every exchange mode vs the single-GPU iteration


def bench_multi_gpu(args):
    import torch
    import torch.distributed as dist
    from sparsematrixvectormultiplication_b200 import device, synth
    from sparsematrixvectormultiplication_b200.distributed import (AllgatherPowerIteration, AsyncPowerIteration,
                                                                   FusedPowerIteration, PeerAllgatherPowerIteration,
                                                                   PowerIteration)
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    cu = torch.device("cuda", local)
    peak, peak_src = measured_peak()
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    n = args.lap3d_n
    N_rows = n ** 3
    results = {}
    # ---- rank 0 alone on the WHOLE matrix (11.8 GB at 512^3: fits one GPU): (1) T1 of the strong-scaling series,
    # measured in the same run; (2) the parity reference: x and lambda after PARITY_ITERS iterations of the single-GPU
    # iteration, which every exchange mode below must reproduce on its owned + referenced rows.
    t1 = None
    x_ref = torch.empty(N_rows if not args.no_parity else 1, dtype=torch.float64, device=cu)
    lam_ref = torch.zeros(1, dtype=torch.float64, device=cu)
    if rank == 0 and not (args.no_t1 and args.no_parity):
        try:
            F1 = FusedPowerIteration(synth.SYNTH_LAP3D, n, single=True, split=True)   # the headline's kernels, whole matrix
            if not args.no_parity:
                for _ in range(PARITY_ITERS):
                    F1.step()
                lam_ref[0] = F1.eigenvalue_estimate()
                x_ref.copy_(F1.normalized_x())
                F1.reset(1.0)
            if not args.no_t1:
                ms1, _ = time_device(F1.step, max(5, min(args.steps, 30)), args.warmup, None, 1)
                t1 = {"ms_per_step": ms1, "gflops": 2.0 * F1.nnz_global / (ms1 * 1e-3) / 1e9, "launches_per_step": F1.launches_per_step,
                      "note": "same workload and kernel on ONE GPU (rank 0 alone, whole matrix), measured in this run"}
                log(f"[bench] 1 GPU same workload: {t1['gflops']:.1f} GFLOP/s, {ms1:.3f} ms/iteration")
            F1.close()
            del F1
            torch.cuda.empty_cache()
        except Exception as e:  # pragma: no cover
            log(f"[bench] single-GPU leg failed: {e!r}")
            lam_ref[0] = float("nan")
    dist.barrier()
    if not args.no_parity:
        dist.broadcast(x_ref, src=0)
        dist.broadcast(lam_ref, src=0)
    lam_ref_v = float(lam_ref.item())
    x_scale = float(x_ref.abs().max().item()) if not args.no_parity else 1.0

    def parity_of(P, mode):
        """PARITY_ITERS iterations from x0 = 1; x on the owned + referenced rows and lambda against the single-GPU leg."""
        P.reset(1.0)
        for _ in range(PARITY_ITERS):
            P.step()
        lam = P.eigenvalue_estimate()
        v = P.normalized_x() if hasattr(P, "normalized_x") else P.x
        lo = min([P.row_begin] + [a_ for _, a_, _ in P.plan.recvs])
        hi = max([P.row_end] + [b_ for _, _, b_ in P.plan.recvs])
        if mode.startswith("allgather"):
            lo, hi = 0, N_rows            # the whole replica is refreshed
        err = torch.tensor([float((v[lo:hi] - x_ref[lo:hi]).abs().max().item()) / x_scale,
                            abs(lam - lam_ref_v) / abs(lam_ref_v)], dtype=torch.float64, device=cu)
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        x_err, lam_err = float(err[0].item()), float(err[1].item())
        ok = bool(x_err <= PARITY_TOL and lam_err <= PARITY_TOL)   # NaN compares false
        P.reset(1.0)
        return {"x_err": x_err, "lambda_err": lam_err, "lambda": lam, "ok": ok}

    modes = ("fused_mailbox", "fused_split", "fused_split_hll", "fused_mailbox_hll", "fused_mailbox_csr_hack_aligned", "fused_async", "fused_peer_stores",
             "fused_nccl_halo", "halo", "allgather_peer", "allgather_peer_2streams", "allgather_peer_hybrid", "allgather_peer_kernel", "allgather", "allgather_broadcasts")
    extra_only = ("allgather_peer_2streams", "allgather_peer_hybrid")   # measured variants that lost (DESIGN.md section 4): on request only
    if args.modes:
        modes = tuple(m for m in modes if m in args.modes.split(",") or m == HEAD_MODE)
    else:
        modes = tuple(m for m in modes if m not in extra_only)
    parity = {}
    for mode in modes:
        if mode == "fused_async":
            P = AsyncPowerIteration(synth.SYNTH_LAP3D, n)
        elif mode == "fused_mailbox":
            P = FusedPowerIteration(synth.SYNTH_LAP3D, n, mailbox=True)
        elif mode == "fused_split":
            P = FusedPowerIteration(synth.SYNTH_LAP3D, n, split=True)
        elif mode == "fused_split_hll":
            P = FusedPowerIteration(synth.SYNTH_LAP3D, n, split=True, fmt="hll")
        elif mode == "fused_mailbox_hll":
            P = FusedPowerIteration(synth.SYNTH_LAP3D, n, mailbox=True, fmt="hll")
        elif mode == "fused_mailbox_csr_hack_aligned":
            # the CSR twin of the HLL mode on the same 32-row-aligned partition, forced onto the fused ROW kernel (the
            # plan-time choice may be the fused stream kernel, which groups the partial sums differently)
            os.environ["SPMV_B200_FUSED_BATCH"] = os.environ.get("SPMV_B200_FUSED_BATCH", "5")
            P = FusedPowerIteration(synth.SYNTH_LAP3D, n, mailbox=True, hack_aligned=True)
        elif mode == "fused_peer_stores":
            P = FusedPowerIteration(synth.SYNTH_LAP3D, n, peer_stores=True)
        elif mode == "fused_nccl_halo":
            P = FusedPowerIteration(synth.SYNTH_LAP3D, n, peer_stores=False)
        elif mode == "allgather":
            P = AllgatherPowerIteration(synth.SYNTH_LAP3D, n)
        elif mode == "allgather_peer":
            P = PeerAllgatherPowerIteration(synth.SYNTH_LAP3D, n, copy_streams=int(os.environ.get("SPMV_B200_PUSH_STREAMS", "1")))
        elif mode == "allgather_peer_2streams":
            P = PeerAllgatherPowerIteration(synth.SYNTH_LAP3D, n, copy_streams=int(os.environ.get("SPMV_B200_PUSH_STREAMS2", "2")))
        elif mode == "allgather_peer_hybrid":     # copy engines + push kernel at the same time
            P = PeerAllgatherPowerIteration(synth.SYNTH_LAP3D, n, kernel_peers=int(os.environ.get("SPMV_B200_PUSH_KERNEL_PEERS", str(max(1, (world - 1) // 3)))),
                                            push_ctas=int(os.environ.get("SPMV_B200_PUSH_CTAS", "0")))
        elif mode == "allgather_peer_kernel":
            P = PeerAllgatherPowerIteration(synth.SYNTH_LAP3D, n, copy_engine=False, push_ctas=int(os.environ.get("SPMV_B200_PUSH_CTAS", "0")))
        elif mode == "allgather_broadcasts":
            P = PowerIteration(synth.SYNTH_LAP3D, n, exchange="allgather")
        else:
            P = PowerIteration(synth.SYNTH_LAP3D, n, exchange=mode)
        if not args.no_parity:
            parity[mode] = parity_of(P, mode)
            if rank == 0:
                log(f"[bench] {world} GPUs {mode}: parity after {PARITY_ITERS} iterations: x {parity[mode]['x_err']:.2e}, "
                    f"lambda {parity[mode]['lambda_err']:.2e} -> {'ok' if parity[mode]['ok'] else 'FAIL'}")
        P.reset(1.0)
        head = mode == HEAD_MODE
        steps = args.steps if head else max(3, min(args.steps, 20))
        ms, per = time_device(P.step, steps, args.warmup, sampler if head else None, world)
        lam = P.eigenvalue_estimate()
        if hasattr(P, "recv_bytes"):
            recv = P.recv_bytes // 8
        else:
            recv = P.plan.allgather_doubles_received() if mode.startswith("allgather") else P.plan.halo_doubles_received()
        results[mode] = {"ms_per_step": ms, "gflops": 2.0 * P.nnz_global / (ms * 1e-3) / 1e9, "steps": steps,
                         "lambda": lam, "rows_local": P.rows, "nnz_local": P.nnz_local, "recv_bytes_per_step": 8 * recv,
                         "launches_per_step": P.launches_per_step, "nnz_global": P.nnz_global,
                         "bytes_local": P.algorithmic_bytes_local}
        if mode.startswith("allgather"):   # the whole-vector refresh is NVLink bound: say how fast the links ran
            results[mode]["nvlink_ingress_gbs_if_all_of_the_step"] = 8 * recv / (ms * 1e-3) / 1e9
        if mode.startswith("allgather_peer"):
            results[mode]["collective"] = (
                "no library call: every rank stores its slice into all replicas over NVLink peer memory ("
                + (f"one cudaMemcpyAsync per peer on {len(P.copy_streams)} stream(s), copy engines" + (f"; the last {P.kernel_peers} peer(s) of the rotation by spmv_b200_vec_push at the same time" if P.kernel_peers else "") if P.copy_engine else "spmv_b200_vec_push: one kernel, 256-bit loads and peer stores")
                + f"), then tags through peer mailboxes; interior rows [{P.interior[0]},{P.interior[1]}) of {P.rows} multiplied while it is in flight")
            try:   # the push + tags alone, same buffers
                def push_only():
                    P.ev_own.record(torch.cuda.current_stream())
                    P._push(0)
                    torch.cuda.current_stream().wait_event(P.ev_landed)
                    P.k += 1
                ams, _ = time_device(push_only, 10, 3, None, world)
                results[mode]["allgather_alone_ms"] = ams
                results[mode]["allgather_alone_ingress_gbs"] = 8 * recv / (ams * 1e-3) / 1e9
            except Exception as e:  # pragma: no cover
                results[mode]["allgather_alone_error"] = repr(e)
        if mode == "allgather":
            results[mode]["collective"] = ("ONE in-place ncclAllGather (dist.all_gather_into_tensor) over a padded rank-major x, "
                                           f"stride {P.stride} doubles; interior rows [{P.interior[0]},{P.interior[1]}) of {P.rows} multiplied while it is in flight")
            try:   # the collective alone, same buffers
                ams, _ = time_device(lambda: dist.all_gather_into_tensor(P.xg, P.own, group=P.ag_group), 10, 3, None, world)
                results[mode]["allgather_alone_ms"] = ams
                results[mode]["allgather_alone_ingress_gbs"] = 8 * recv / (ams * 1e-3) / 1e9
            except Exception as e:  # pragma: no cover
                results[mode]["allgather_alone_error"] = repr(e)
        if rank == 0:
            log(f"[bench] {world} GPUs {mode}: {results[mode]['gflops']:.1f} GFLOP/s, {ms:.3f} ms/iteration, lambda={lam:.12g}")
        if head:  # kernel-only product time on this rank (roofline of the dominant kernel)
            xs, row_begin = P.xs, P.row_begin
            product = P.A.spmv_fused_flat if getattr(P, "split", False) else P.A.spmv_fused
            kms, kper = time_device(lambda: product(xs[0].data_ptr(), xs[1].data_ptr() + 8 * row_begin, partials=P.partials),
                                    max(5, min(args.steps, 50)), 3, None, world)
            results["product_only_ms"] = kms
            pi = P.A.info()
            results["product_kernel"] = (f"csr_row_flat_kernel<{pi.flat_batch}>" if getattr(P, "split", False)
                                         else ("csr_stream_kernel (fused)" if pi.fused_batch == 0 else f"csr_row_fused_kernel<{pi.fused_batch}>"))
            if getattr(P, "peers", None) and P.peers[1] is not None:   # the same launch with the NVLink peer stores of the boundary rows
                pms, _ = time_device(lambda: product(xs[0].data_ptr(), xs[1].data_ptr() + 8 * row_begin, partials=P.partials,
                                                     peers=P.peers[1]), max(5, min(args.steps, 50)), 3, None, world)
                results["product_with_peer_stores_ms"] = pms
                if rank == 0:
                    log(f"[bench] {world} GPUs local fused product alone {kms:.3f} ms, with peer stores {pms:.3f} ms")
            # end to end as a caller that monitors convergence sees it: lambda read back on the HOST after every iteration
            # (an 8-byte device->host copy that synchronises the stream: no launch is queued ahead of the device)
            if getattr(P, "split", False):
                P.reset(1.0)
                lam_host = []

                def step_and_read():
                    P.step()
                    lam_host.append(float(P.scale[0].item()) ** 0.5)
                ems, _ = time_device(step_and_read, max(5, min(args.steps, 50)), 3, None, world)
                results["e2e_ms"] = ems
                results["e2e_lambda_last"] = lam_host[-1]
                if rank == 0:
                    log(f"[bench] {world} GPUs {mode} with lambda read back on the host every iteration: {ems:.3f} ms/iteration")
        if hasattr(P, "close"):
            P.close()
        del P
        if mode == "fused_mailbox_csr_hack_aligned":
            os.environ.pop("SPMV_B200_FUSED_BATCH", None)
        torch.cuda.empty_cache()
    del x_ref
    torch.cuda.empty_cache()
    # HLL and CSR iterations on the same hack-aligned partition must agree bit for bit (lambda after the timed run too)
    if "fused_mailbox_hll" in parity and "fused_mailbox_csr_hack_aligned" in parity:
        same = parity["fused_mailbox_hll"]["lambda"] == parity["fused_mailbox_csr_hack_aligned"]["lambda"]
        parity["fused_mailbox_hll"]["lambda_bitwise_equal_to_csr_on_the_same_partition"] = bool(same)
        parity["fused_mailbox_hll"]["ok"] = parity["fused_mailbox_hll"]["ok"] and bool(same)
    # ---- the plain product y = A x, row-partitioned (no exchange: x is replicated), CSR and HLL, for the other
    # single-GPU shapes: every rank owns an nnz-balanced row range (HLL: cut on 32-row hack boundaries, as the
    # reference cuts HLL work, src/hll_matrix.c:471-498); a step is one product on every rank, time = max over ranks.
    partitioned = {}
    try:
        from sparsematrixvectormultiplication_b200 import partition
        for name, kind, p0 in (("lap2d_4096", synth.SYNTH_LAP2D, 4096), (f"lap3d_{n}", synth.SYNTH_LAP3D, n)):
            parts = partition.hack_aligned(partition.synth_partition(kind, p0, 0, 0, world),
                                           p0 * p0 if kind == synth.SYNTH_LAP2D else p0 ** 3)
            if len(parts) != world:
                continue
            lo, hi = parts[rank]
            A = device.DeviceCSR.synth(kind, p0, row_begin=lo, row_end=hi)
            ia = A.info()
            x = torch.ones(ia.N, dtype=torch.float64, device="cuda")
            y = torch.empty(ia.M, dtype=torch.float64, device="cuda")
            nnz_global = synth.row_offset(kind, p0, 0, 0, parts[-1][1])
            steps = max(5, min(args.steps, 50))
            ms, _ = time_device(lambda: A.spmv(x, y), steps, args.warmup, None, world)
            H = A.to_hll()
            hi_ = H.info()
            ms_h, _ = time_device(lambda: H.spmv(x, y), steps, args.warmup, None, world)
            # bytes a rank really streams: its rows + the referenced part of x (about rows + 2 halo planes)
            local_csr = 12 * ia.nnz + 4 * (ia.M + 1) + 8 * ia.M + 8 * min(ia.N, ia.M + 2 * (p0 if kind == synth.SYNTH_LAP2D else p0 * p0))
            local_hll = local_csr - 12 * ia.nnz - 4 * (ia.M + 1) + 12 * hi_.slots + 8 * (hi_.num_hacks + 1)
            partitioned[name] = {
                "csr": {"ms_per_product": ms, "gflops": 2.0 * nnz_global / (ms * 1e-3) / 1e9, "rank0_gbs": local_csr / (ms * 1e-3) / 1e9,
                        "kernel": device.ALGO_NAMES[ia.auto_algo]},
                "hll": {"ms_per_product": ms_h, "gflops": 2.0 * nnz_global / (ms_h * 1e-3) / 1e9, "rank0_gbs": local_hll / (ms_h * 1e-3) / 1e9,
                        "kernel": device.HLL_KERNEL_NAMES[hi_.auto_kernel]},
                "rows_rank0": ia.M, "nnz_global": nnz_global}
            if rank == 0:
                log(f"[bench] {world} GPUs {name} row-partitioned product: CSR {partitioned[name]['csr']['gflops']:.0f} GFLOP/s ({ms*1e3:.1f} us), "
                    f"HLL {partitioned[name]['hll']['gflops']:.0f} GFLOP/s ({ms_h*1e3:.1f} us)")
            H.close()
            A.close()
            del x, y
            torch.cuda.empty_cache()
    except Exception as e:  # pragma: no cover
        partitioned["error"] = repr(e)
        if rank == 0:
            log(f"[bench] partitioned products failed: {e!r}")
    if sampler:
        sampler.stop()
    parity_ok = all(v["ok"] for v in parity.values()) if parity else None
    if rank == 0:
        h = results[HEAD_MODE]
        gbs = h["bytes_local"] / (results["product_only_ms"] * 1e-3) / 1e9
        traffic, traffic_src = ncu_traffic(f"lap3d_{n}_power_rank_of_{world}", results.get("product_kernel", ""))
        eff = (t1["ms_per_step"] / (world * h["ms_per_step"])) if t1 else None
        line = {"metric": "spmv_gflops", "value": h["gflops"], "unit": "GFLOP/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": h["ms_per_step"], "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(world, n),
                "implementation": {
                    "mode": HEAD_MODE,
                    "partition": "contiguous rows balanced by nnz (reference greedy rule)",
                    "exchange": "boundary rows stored into the peers' buffers over NVLink peer memory by the product kernel, |w|^2 through peer mailboxes; no collective call in the loop",
                    "step": "one power iteration = TWO launches: (1) FLAT fused product, grid as large as the matrix, never waits: w=(A w_prev)/|w_prev|, per-CTA |w|^2 partials, peer stores of boundary rows; (2) one-CTA exchange kernel: fixed-order sum of the partials, publish |w|^2 + tag into every rank's mailbox, wait for all ranks' tags (their boundary rows have landed), leave 1/|w| for the next launch"},
                # T1 / (N * T_N) with T1 = the SAME workload and kernel on one GPU, measured in this run (the driver's own
                # curve divides by the N=1 line of `bench.py --gpus 1`, which is another workload: lap2d single product)
                "efficiency_same_workload": eff,
                "parity": {"ok": parity_ok, "iters": PARITY_ITERS, "tolerance": PARITY_TOL,
                           "reference": "single-GPU fused iteration on rank 0 (whole matrix), x on every rank's owned + referenced rows (max abs error / max |x|) and lambda (relative), max over ranks",
                           "modes": parity},
                "roofline": {"bound": "hbm", "achieved": gbs, "peak": peak, "unit": "GB/s", "frac": gbs / peak,
                             "traffic": traffic, "traffic_source": traffic_src, "kernel": results.get("product_kernel"),
                             "peak_source": peak_src, "note": "rank 0's local CSR product alone (max over ranks); algorithmic bytes of its row slice = 12 nnz_local + 4 (rows+1) + 8 rows + 8 x (referenced columns of x)",
                             "algorithmic_bytes_per_launch": int(h["bytes_local"])},
                "cpu_baseline": None,
                "e2e": ({"value": 2.0 * h["nnz_global"] / (results["e2e_ms"] * 1e-3) / 1e9, "unit": "GFLOP/s", "h2d_bytes_per_step": 0,
                         "d2h_bytes_per_step": 8, "ms_per_step": results["e2e_ms"],
                         "note": "the iterated product with its per-iteration result (lambda = |A v|, 8 bytes) read back on the host after EVERY iteration, "
                                 "as a caller monitoring convergence does: the read synchronises the stream, so no launch is queued ahead of the device. "
                                 "x is device state and never crosses PCIe between iterations (h2d 0); see the N=1 line for the host-buffer product"}
                        if "e2e_ms" in results else
                        {"value": h["gflops"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                         "note": "iterated product: x and y never leave the devices between iterations; see the N=1 line for the host-buffer path"}),
                "gpu_launches": h["launches_per_step"] * args.steps, "clocks": sampler.summary() if sampler else None,
                "single_gpu_same_workload": t1,
                "partitioned_products": partitioned,
                "exchange_modes": {k: v for k, v in results.items() if isinstance(v, dict)}}
        emit(line)
    dist.barrier()
    dist.destroy_process_group()
    if parity_ok is False:
        log("[bench] PARITY FAILED: a multi-GPU exchange mode does not reproduce the single-GPU iteration")
        sys.exit(1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--quick", action="store_true", help="headline only: skip the other single-GPU configs")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--cpu-budget", type=float, default=20.0)
    ap.add_argument("--lap3d-n", type=int, default=512)
    ap.add_argument("--no-t1", action="store_true", help="multi-GPU: skip the single-GPU leg of the same workload")
    ap.add_argument("--no-parity", action="store_true", help="multi-GPU: skip the parity check of every exchange mode against the single-GPU iteration")
    ap.add_argument("--modes", default="", help="multi-GPU: comma-separated subset of the exchange modes (fused_mailbox always runs)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="single GPU: after the timed steps, write a fixed seeded sample of the headline product's y as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.impl != "ours" or world > 1 or args.gpus > 1):
        ap.error("--dump-outputs is implemented for the single-GPU run of this implementation (--gpus 1)")
    capture_stdout()
    if args.impl == "reference":
        return run_reference(args)
    if world > 1 or args.gpus > 1:
        if world == 1:
            log("bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
            sys.exit(2)
        return bench_multi_gpu(args)
    return bench_single_gpu(args)


if __name__ == "__main__":
    main()
