"""Host-buffer multi-vector products Y = A X (spmv_b200_{csr,hll}_spmm_host) against the other ways to get there.

    python tools/spmm_host_bench.py --out DIR [--ks 1,2,4,8,16,32] [--reps 5] [--warmup 1] [--workloads ...]
                                      [--sweep-only] [--label NAME]

Workloads: lap2d 4096^2 (CSR and HLL), uniform 8M x 32 per row (CSR), R-MAT scale 24 (CSR).  For each k four arms
alternate, each a synchronous call timed with the host clock:
  pinned    spmm_host on pinned X and Y (ld = k)
  pageable  spmm_host on pageable X and Y
  singles   k spmv_host calls on k pinned column vectors
  manual    one upload of X, the device SpMM, one download of Y (pinned buffers, one stream)
Then the Y sweep that the zero-copy rule rests on, at ldy = k and ldy = k + 3 (pinned): spmm_host with the automatic
choice and with SPMV_B200_HOST_ZEROCOPY=0 (staged Y), and the device SpMM storing Y straight into pinned host memory
against the same product into device memory (CUDA events; the difference is what the stores over PCIe cost); and the
2-D copy rate of the column blocks: spmm_host on X of ld = 32 with SPMV_B200_HOST_SPMM_COLS = 8 (pieces as 2-D copies).
Reported: ms per call, ms per column, PCIe GB/s = 8 k (N + M) / t, and a bitwise sample of rows against the device SpMM.
The device name and power limit are read in the same run.  JSON goes to DIR/spmm_host_bench.json (with --label NAME:
DIR/spmm_host_bench_NAME.json, NAME also recorded in it).

--sweep-only runs the Y sweep alone.  The automatic arm of the sweep stores Y the way the rule in hostpath.cu
(spmm_zero_copy) decides, so in the cells where the rule stages it compares staged with staged.  Both strategies in
every cell come from a build whose spmm_zero_copy returns true: there the automatic arm is zero-copy wherever the buffer
is pinned, and SPMV_B200_HOST_ZEROCOPY=0 stages.  That is how the rule was measured (DESIGN.md section 3, "Host
buffers").
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tools"))

from spmm_bench import build_workloads, card, log  # noqa: E402


def timed(fn):
    t0 = time.perf_counter()
    fn()
    return (time.perf_counter() - t0) * 1e3


def summary(ms, k, M, N):
    best = min(ms)
    mean = sum(ms) / len(ms)
    return {"mean_ms": round(mean, 3), "min_ms": round(best, 3), "ms_per_column": round(mean / k, 3),
            "pcie_GBps": round(8 * k * (N + M) / (mean * 1e-3) / 1e9, 2)}


def env_arm(name, value, fn):
    old = os.environ.get(name)
    os.environ[name] = value
    try:
        return fn()
    finally:
        if old is None:
            del os.environ[name]
        else:
            os.environ[name] = old


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--ks", default="1,2,4,8,16,32")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--workloads", default="lap2d_4096,uniform_8m_32,rmat_24_16")
    ap.add_argument("--sweep-only", action="store_true", help="the Y sweep alone")
    ap.add_argument("--label", default="", help="names the JSON file and is recorded in it")
    args = ap.parse_args()
    import numpy as np
    import torch
    from sparsematrixvectormultiplication_b200 import _native as NL
    ks = [int(k) for k in args.ks.split(",")]
    kmax = max(ks)
    result = {"label": args.label, "sweep_only": args.sweep_only, "card": card(), "ks": ks, "reps": args.reps, "warmup": args.warmup, "cases": [], "y_sweep": [], "blocks_2d": []}
    log(f"[spmm_host_bench] {result['card']}")
    lib = NL.lib()
    formats_of = {"lap2d_4096": ("csr", "hll"), "uniform_8m_32": ("csr",), "rmat_24_16": ("csr",)}
    for name, make, _ in build_workloads([w for w in args.workloads.split(",") if w]):
        A = make()
        ia = A.info()
        M, N_ = ia.M, ia.N
        gen = torch.Generator().manual_seed(7)
        Xp = torch.empty(N_ * kmax, dtype=torch.float64).uniform_(0.5, 1.5, generator=gen).pin_memory()
        Yp = torch.empty(M * (kmax + 3), dtype=torch.float64).pin_memory()
        Xq = Xp.clone()                      # pageable
        Yq = torch.empty(M * kmax, dtype=torch.float64)
        Xd = torch.empty(N_ * kmax, dtype=torch.float64, device="cuda")
        Yd = torch.empty(M * (kmax + 3), dtype=torch.float64, device="cuda")
        log(f"[spmm_host_bench] {name}: M={M} N={N_} nnz={ia.nnz} long rows={ia.num_long_rows}")
        for fmt in formats_of[name]:
            T = A if fmt == "csr" else A.to_hll()
            for k in ks:
                X = Xp[:N_ * k].view(N_, k)
                Y = Yp[:M * k].view(M, k)
                Xpg, Ypg = Xq[:N_ * k].view(N_, k), Yq[:M * k].view(M, k)
                Xdev, Ydev = Xd[:N_ * k].view(N_, k), Yd[:M * k].view(M, k)
                cols = [(Xp[c * N_:(c + 1) * N_], Yp[c * M:(c + 1) * M]) for c in range(k)]

                def manual():
                    Xdev.copy_(X, non_blocking=True)
                    T.spmm(Xdev, Ydev)
                    Y.copy_(Ydev, non_blocking=True)
                    torch.cuda.synchronize()

                arms = {"pinned": lambda: T.spmm_host(X, Y), "pageable": lambda: T.spmm_host(Xpg, Ypg),
                        "singles": lambda: [T.spmv_host_ptr(x.data_ptr(), y.data_ptr()) for x, y in cols],
                        "manual": manual}
                times = {a: [] for a in arms}
                for rep in range(0 if args.sweep_only else args.warmup + args.reps):
                    for a, fn in arms.items():
                        ms = timed(fn)
                        if rep >= args.warmup:
                            times[a].append(ms)
                # bitwise sample: pinned arm against the device SpMM on the same handle
                T.spmm_host(X, Y)
                if args.sweep_only:
                    arms = {}
                Xdev.copy_(X)
                T.spmm(Xdev, Ydev)
                rows = torch.from_numpy(np.unique(np.random.default_rng(k).integers(0, M, 4096)))
                same = bool(torch.equal(Y[rows].view(torch.int64), Ydev.cpu()[rows].view(torch.int64)))
                case = {"workload": name, "format": fmt, "k": k, "M": M, "N": N_, "nnz": ia.nnz, "bitwise_sample": same}
                for a in arms:
                    case[a] = summary(times[a], k, M, N_)
                result["cases"].append(case)
                log(f"[spmm_host_bench] {name} {fmt} k={k}: " + "  ".join(
                    f"{a} {case[a]['mean_ms']:.2f} ms ({case[a]['pcie_GBps']:.1f} GB/s)" for a in arms) + f"  bitwise {same}")
                # the Y sweep (pinned)
                for ldy in (k, k + 3):
                    Yw = Yp[:M * ldy].view(M, ldy)[:, :k]
                    Ywd = Yd[:M * ldy].view(M, ldy)[:, :k]
                    sweep = {"workload": name, "format": fmt, "k": k, "ldy": ldy}
                    t_auto, t_staged = [], []
                    for rep in range(args.warmup + args.reps):
                        a = timed(lambda: T.spmm_host(X, Yw))
                        b = env_arm("SPMV_B200_HOST_ZEROCOPY", "0", lambda: timed(lambda: T.spmm_host(X, Yw)))
                        if rep >= args.warmup:
                            t_auto.append(a)
                            t_staged.append(b)
                    sweep["host_call_auto"] = summary(t_auto, k, M, N_)
                    sweep["host_call_staged"] = summary(t_staged, k, M, N_)
                    # the device product storing into host memory vs into device memory
                    Xdev.copy_(X)
                    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
                    fn = lib.spmv_b200_csr_spmm if fmt == "csr" else lib.spmv_b200_hll_spmm
                    extra = (0,) if fmt == "csr" else ()
                    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
                    dev_ms, host_ms = [], []
                    for rep in range(args.warmup + args.reps):
                        ev[0].record()
                        NL.check(fn(T._h, k, C.c_void_p(Xdev.data_ptr()), k, C.c_void_p(Ywd.data_ptr()), ldy, *extra, st))
                        ev[1].record()
                        NL.check(fn(T._h, k, C.c_void_p(Xdev.data_ptr()), k, C.c_void_p(Yw.data_ptr()), ldy, *extra, st))
                        ev[2].record()
                        torch.cuda.synchronize()
                        if rep >= args.warmup:
                            dev_ms.append(ev[0].elapsed_time(ev[1]))
                            host_ms.append(ev[1].elapsed_time(ev[2]))
                    sweep["device_spmm_into_device_ms"] = round(sum(dev_ms) / len(dev_ms), 3)
                    sweep["device_spmm_into_pinned_host_ms"] = round(sum(host_ms) / len(host_ms), 3)
                    sweep["zero_copy_store_GBps"] = round(8 * k * M / (sum(host_ms) / len(host_ms) * 1e-3) / 1e9, 2)
                    result["y_sweep"].append(sweep)
                    log(f"[spmm_host_bench]   Y sweep k={k} ldy={ldy}: auto {sweep['host_call_auto']['mean_ms']:.2f} ms, "
                        f"staged {sweep['host_call_staged']['mean_ms']:.2f} ms; device SpMM into device "
                        f"{sweep['device_spmm_into_device_ms']:.2f} ms, into pinned host {sweep['device_spmm_into_pinned_host_ms']:.2f} ms")
            if kmax >= 32 and not args.sweep_only:  # the 2-D copies of column blocks: X of ld 32, blocks of 8 columns
                k = 32
                X = Xp[:N_ * k].view(N_, k)
                Y = Yp[:M * k].view(M, k)
                t_one, t_blk = [], []
                for rep in range(args.warmup + args.reps):
                    a = timed(lambda: T.spmm_host(X, Y))
                    b = env_arm("SPMV_B200_HOST_SPMM_COLS", "8", lambda: timed(lambda: T.spmm_host(X, Y)))
                    if rep >= args.warmup:
                        t_one.append(a)
                        t_blk.append(b)
                blk = {"workload": name, "format": fmt, "k": k, "one_block": summary(t_one, k, M, N_),
                       "blocks_of_8_2d": summary(t_blk, k, M, N_)}
                result["blocks_2d"].append(blk)
                log(f"[spmm_host_bench]   k=32 one block {blk['one_block']['mean_ms']:.2f} ms, blocks of 8 (2-D pieces) "
                    f"{blk['blocks_of_8_2d']['mean_ms']:.2f} ms")
            if T is not A:
                T.close()
        del Xp, Yp, Xq, Yq, Xd, Yd
        A.close()
        torch.cuda.empty_cache()
    result["card_after"] = card()
    out = Path(args.out)
    out.mkdir(parents=True, exist_ok=True)
    path = out / (f"spmm_host_bench_{args.label}.json" if args.label else "spmm_host_bench.json")
    path.write_text(json.dumps(result, indent=1))
    log(f"[spmm_host_bench] wrote {path}")


if __name__ == "__main__":
    main()
