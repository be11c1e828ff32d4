"""One multi-vector product Y = A X (SpMM) against k single-vector products on the same matrix, in the same run.

    python tools/spmm_bench.py --out DIR [--ks 1,2,4,8,16,32] [--reps 10] [--warmup 3] [--workloads ...] [--batches 2,4,8]

Workloads: lap2d 4096^2 (CSR and HLL), uniform 8M x 32 per row (CSR and HLL), R-MAT scale 24 (CSR).  For each k the
two arms alternate: one SpMM over X (N x k, ld = k), then k automatic single-vector products (spmv_b200_csr_spmv /
spmv_b200_hll_spmv) on the k columns held as contiguous vectors; CUDA events around each arm, warm-up first, mean and
minimum over the timed repetitions.  Every working set exceeds the 126 MB L2 (the matrices are 1-3 GB).

Reported per case: time per call, speed-up over the k single-vector products (mean / mean), GFLOP/s = 2 nnz k / t,
algorithmic bytes (CSR 12 nnz + 4 (M+1) + 8 k (M+N); HLL 12 slots + 8 (hacks+1) + 8 k (M+N)) and their share of
8 TB/s, and a bitwise check of sampled rows against the per-column single-vector product in the serial order
(ALGO_ROW / the HLL lane-per-row kernel; CSR rows above the long-row threshold are summed in fragments and skipped).
The device name and power limit are read in the same run.  --batches repeats the SpMM arm under
SPMV_B200_SPMM_BATCH = each value (column / value loads in flight per lane).  JSON goes to DIR/spmm_bench.json.

--f32 measures the products on the float copy of enable_f32 instead (JSON: DIR/spmm_bench_f32.json).  Three arms
alternate: one spmv_b200_{csr,hll}_spmm_f32 (or one per batch with --batches), k automatic spmv_b200_{csr,hll}_spmv_f32
on the k float columns, and the fp64 SpMM of the same k.  Reported besides the above: the speed-up over the k fp32
products, the ratio of the fp64 SpMM time to the fp32 one, and fp32 algorithmic bytes (CSR 8 nnz + 4 (M+1) + 4 k (M+N);
HLL 8 slots + 8 (hacks+1) + 4 k (M+N)).  The bitwise check compares sampled rows with spmv_f32(ALGO_ROW) on the CSR
handle per column -- the exact reference of the fp32 contract; for HLL the same bits, since padding slots add +-0.0.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

PEAK_BYTES_PER_S = 8e12


def log(msg):
    print(msg, flush=True)


def card():
    import torch
    out = {"torch_name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        out["nvidia_smi"] = q.stdout.strip()
    except Exception as e:  # the numbers stay valid; the card line says why it is missing
        out["nvidia_smi"] = f"unavailable: {e!r}"
    return out


def build_workloads(names):
    """name -> (format, handle, M, N, nnz, matrix bytes of the algorithmic count, long threshold) built lazily."""
    from sparsematrixvectormultiplication_b200 import device, synth

    def lap2d():
        return device.DeviceCSR.synth(device.SYNTH_LAP2D, 4096)

    def uniform():
        return device.DeviceCSR.synth(device.SYNTH_UNIFORM, 1 << 23, 1 << 23, 32)

    def rmat():
        rp, ci, va = synth.rmat_csr_device(24, 16)
        return device.DeviceCSR.wrap(1 << 24, 1 << 24, rp, ci, va)

    makers = {"lap2d_4096": (lap2d, ("csr", "hll")), "uniform_8m_32": (uniform, ("csr", "hll")), "rmat_24_16": (rmat, ("csr",))}
    for name in names:
        make, formats = makers[name]
        yield name, make, formats


def time_case(A, fmt, k, X, Y, xs, ys, reps, warmup, batch_env, f64=None):
    """Alternating SpMM / k single-vector products; returns per-arm lists of ms.  X, Y, xs, ys float32 and f64 = (X, Y)
    in float64: the fp32 products and the fp64 SpMM as a third arm."""
    import torch
    from sparsematrixvectormultiplication_b200 import _native as N
    lib = N.lib()
    s = torch.cuda.current_stream()
    sp = C.c_void_p(s.cuda_stream)
    h = A._h
    f32 = f64 is not None
    px, py = C.c_void_p(X.data_ptr()), C.c_void_p(Y.data_ptr())
    vec = [(C.c_void_p(xs[c].data_ptr()), C.c_void_p(ys[c].data_ptr())) for c in range(k)]
    ld = X.stride(0) if X.shape[0] > 1 else k
    csr_spmm, hll_spmm = (lib.spmv_b200_csr_spmm_f32, lib.spmv_b200_hll_spmm_f32) if f32 else (lib.spmv_b200_csr_spmm, lib.spmv_b200_hll_spmm)

    def spmm(px=px, py=py, csr_spmm=csr_spmm, hll_spmm=hll_spmm):
        if fmt == "csr":
            N.check(csr_spmm(h, k, px, ld, py, k, 0, sp))
        else:
            N.check(hll_spmm(h, k, px, ld, py, k, sp))

    def singles():
        for x, y in vec:
            if fmt == "csr":
                N.check((lib.spmv_b200_csr_spmv_f32 if f32 else lib.spmv_b200_csr_spmv)(h, x, y, 0, 0, sp))
            else:
                N.check((lib.spmv_b200_hll_spmv_f32 if f32 else lib.spmv_b200_hll_spmv)(h, x, y, sp))

    arms = {"spmm": spmm, "singles": singles}
    if batch_env:
        arms = {f"spmm_batch{b}": (lambda b=b: (os.environ.__setitem__("SPMV_B200_SPMM_BATCH", str(b)), spmm())) for b in batch_env}
        arms["singles"] = singles
    if f32:
        p64 = (C.c_void_p(f64[0].data_ptr()), C.c_void_p(f64[1].data_ptr()))
        arms["spmm_f64"] = lambda: (os.environ.pop("SPMV_B200_SPMM_BATCH", None),
                                    spmm(*p64, lib.spmv_b200_csr_spmm, lib.spmv_b200_hll_spmm))
    times = {a: [] for a in arms}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for rep in range(warmup + reps):
        for a, fn in arms.items():
            ev[0].record(s)
            fn()
            ev[1].record(s)
            ev[1].synchronize()
            if rep >= warmup:
                times[a].append(ev[0].elapsed_time(ev[1]))
    os.environ.pop("SPMV_B200_SPMM_BATCH", None)
    return times


def bitwise_check(A, fmt, k, X, Y, long_threshold, rp_host, samples, seed):
    """Sampled rows of Y (the last SpMM) against the serial-order single-vector product of each column.  float32 X / Y:
    A is the CSR handle (also for an HLL product) and the reference is its spmv_f32(ALGO_ROW)."""
    import numpy as np
    import torch
    from sparsematrixvectormultiplication_b200 import device
    M = Y.shape[0]
    rng = np.random.default_rng(seed)
    rows = np.unique(np.concatenate([rng.integers(0, M, samples), [0, M - 1]]))
    f32 = X.dtype == torch.float32
    if fmt == "csr":
        lens = rp_host[rows + 1] - rp_host[rows]
        rows = rows[lens <= long_threshold]
    rows_d = torch.from_numpy(rows).cuda()
    Ys = Y[rows_d].cpu().numpy()
    y = torch.empty(M, dtype=X.dtype, device="cuda")
    bad = 0
    for c in range(k):
        x = X[:, c].contiguous()
        if f32:
            A.spmv_f32(x, y, algo=device.ALGO_ROW)
        elif fmt == "csr":
            A.spmv(x, y, algo=device.ALGO_ROW)
        else:
            A.spmv(x, y, slice_kernel="rows")
        want = y[rows_d].cpu().numpy()
        word = np.uint32 if f32 else np.uint64
        bad += int(np.count_nonzero(Ys[:, c].view(word) != want.view(word)))
    return {"rows_checked": int(len(rows)), "columns": k, "mismatches": bad}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--ks", default="1,2,4,8,16,32")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workloads", default="lap2d_4096,uniform_8m_32,rmat_24_16")
    ap.add_argument("--batches", default="", help="comma list: also time the SpMM arm under SPMV_B200_SPMM_BATCH = each")
    ap.add_argument("--samples", type=int, default=4096)
    ap.add_argument("--f32", action="store_true", help="the fp32-storage products (float X, Y, values), fp64 SpMM as a third arm")
    args = ap.parse_args()
    ks = [int(v) for v in args.ks.split(",") if v]
    batches = [int(v) for v in args.batches.split(",") if v]
    if args.reps < 1 or not ks or min(ks) < 1:
        ap.error("--reps and every k must be >= 1")
    out_dir = Path(args.out)
    out_dir.mkdir(parents=True, exist_ok=True)

    import numpy as np
    import torch
    from sparsematrixvectormultiplication_b200 import device
    if not torch.cuda.is_available():
        raise SystemExit("spmm_bench needs a CUDA device: nothing is measured without one")
    torch.cuda.set_device(0)
    result = {"card": card(), "device_info": device.device_info(), "ks": ks, "reps": args.reps, "warmup": args.warmup,
              "peak_bytes_per_s": PEAK_BYTES_PER_S, "batches": batches, "cases": []}
    log(f"[spmm_bench] {result['card']}")
    kmax = max(ks)
    for name, make, formats in build_workloads([w for w in args.workloads.split(",") if w]):
        t0 = time.perf_counter()
        A = make()
        ia = A.info()
        M, N_ = ia.M, ia.N
        rp_host = None
        gen = torch.Generator(device="cuda")
        gen.manual_seed(1234)
        Xfull = torch.rand((N_, kmax), dtype=torch.float64, device="cuda", generator=gen) + 0.5
        log(f"[spmm_bench] {name}: M={M} N={N_} nnz={ia.nnz} long rows={ia.num_long_rows} (built in {time.perf_counter() - t0:.1f} s)")
        if args.f32:
            A.enable_f32()
        dtype, size = (torch.float32, 4) if args.f32 else (torch.float64, 8)
        for fmt in formats:
            Mat = A if fmt == "csr" else A.to_hll()
            if fmt == "csr":
                matrix_bytes = (size + 4) * ia.nnz + 4 * (M + 1)
                rp_host = A.download()[0]
            else:
                if args.f32:
                    Mat.enable_f32()
                ih = Mat.info()
                matrix_bytes = (size + 4) * ih.slots + 8 * (ih.num_hacks + 1)
            for k in ks:
                X = Xfull[:, :k].to(dtype).contiguous()
                Y = torch.empty((M, k), dtype=dtype, device="cuda")
                xs = [X[:, c].contiguous() for c in range(k)]
                ys = [torch.empty(M, dtype=dtype, device="cuda") for _ in range(k)]
                f64 = (Xfull[:, :k].contiguous(), torch.empty((M, k), dtype=torch.float64, device="cuda")) if args.f32 else None
                times = time_case(Mat, fmt, k, X, Y, xs, ys, args.reps, args.warmup, batches, f64)
                if batches:  # leave Y from the default batch for the check
                    time_case(Mat, fmt, k, X, Y, xs, ys, 1, 0, [], f64)
                torch.cuda.synchronize()
                alg = matrix_bytes + size * k * (M + N_)
                case = {"workload": name, "format": fmt, "k": k, "M": M, "N": N_, "nnz": ia.nnz, "algorithmic_bytes": alg}
                for arm, ts in times.items():
                    mean, best = float(np.mean(ts)), float(np.min(ts))
                    case[arm] = {"mean_ms": mean, "min_ms": best, "ms": ts}
                    if arm.startswith("spmm") and arm != "spmm_f64":
                        case[arm].update({"gflops": 2.0 * ia.nnz * k / (mean * 1e-3) / 1e9,
                                          "bytes_per_s": alg / (mean * 1e-3),
                                          "fraction_of_8tbs": alg / (mean * 1e-3) / PEAK_BYTES_PER_S})
                default_batch = (2 if args.f32 else 4) if fmt == "csr" else 8
                spmm_arm = "spmm" if "spmm" in times else f"spmm_batch{default_batch if default_batch in batches else batches[0]}"
                case["speedup_mean"] = case["singles"]["mean_ms"] / case[spmm_arm]["mean_ms"]
                case["speedup_min"] = case["singles"]["min_ms"] / case[spmm_arm]["min_ms"]
                if args.f32:  # > 1: the fp32 SpMM is faster than the fp64 one
                    case["f64_over_f32_mean"] = case["spmm_f64"]["mean_ms"] / case[spmm_arm]["mean_ms"]
                    case["f64_over_f32_min"] = case["spmm_f64"]["min_ms"] / case[spmm_arm]["min_ms"]
                case["bitwise"] = bitwise_check(A if args.f32 else Mat, fmt, k, X, Y, ia.long_threshold, rp_host, args.samples, k)
                result["cases"].append(case)
                extra = " ".join(f"{a}={case[a]['mean_ms']:.3f}" for a in times if a.startswith("spmm_batch"))
                if args.f32:
                    extra += f" fp64 spmm {case['spmm_f64']['mean_ms']:.3f} ms (fp64/fp32 x{case['f64_over_f32_mean']:.2f})"
                log(f"[spmm_bench] {name} {fmt} k={k:2d}: spmm {case[spmm_arm]['mean_ms']:.3f} ms (min {case[spmm_arm]['min_ms']:.3f}) "
                    f"vs {k} x spmv {case['singles']['mean_ms']:.3f} ms -> x{case['speedup_mean']:.2f}; "
                    f"{case[spmm_arm]['gflops']:.0f} GFLOP/s, {case[spmm_arm]['fraction_of_8tbs'] * 100:.0f} % of 8 TB/s; "
                    f"bitwise {case['bitwise']['mismatches']} bad of {case['bitwise']['rows_checked']}x{k} {extra}")
                del X, Y, xs, ys, f64
            if fmt != "csr":
                Mat.close()
        A.close()
        del Xfull
        torch.cuda.empty_cache()
    result["card_after"] = card()
    result["storage"] = "float32" if args.f32 else "float64"
    out = out_dir / ("spmm_bench_f32.json" if args.f32 else "spmm_bench.json")
    out.write_text(json.dumps(result, indent=1))
    log(f"[spmm_bench] wrote {out}")


if __name__ == "__main__":
    main()
