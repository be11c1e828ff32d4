"""The private image of a CSR handle against its fp64 form and csr_row_kernel, alternating in one process.

    python tools/csr_image_bench.py --out FILE [--reps 12] [--launches 50] [--workloads lap2d_4096,lap3d_384,...]

For each workload the handle is built as a user builds it (synth: owned arrays, plan-time timing on), so AUTO is whatever
the plan chose -- the private image (SPMV_B200_ALGO_ROW_IMAGE) where it timed fastest, with fp64 values or 1-byte value
codes, or in the pattern form (one byte per row).  Further handles of the same matrix hold the image with fp64 values
(set_image(1)), with value codes (set_image(2)) and in the pattern form (set_image(3)), each where the matrix qualifies.
Then ALGO_ROW (csr_row_kernel, the plan's batch), AUTO and ROW_IMAGE on each of those handles alternate: per repetition
`launches` back-to-back products of each arm between CUDA events, after a warm-up of all.  Every working set exceeds the 126 MB L2.  Reported per workload: mean / min / max microseconds per
product of each arm, the speed-up (ROW mean / AUTO mean), the chosen kernel, plan time (the synth call, timing included),
the image's device bytes and value bytes, the algorithmic bytes of the CSR product (12 nnz + 4 (M+1) + 8 M + 8 N) and the
bytes each image kernel actually reads (image_device_bytes + 8 M + 8 N, no row_ptr; 2 or 4 bytes of column field and 8 or 1
of value per slot, or 1 byte per row), each over its time, and whether AUTO and each image give ALGO_ROW's bits (it must wherever AUTO is a
serial-order kernel: the image, ROW, STREAM; uniform 32 per row is too long for the image and stays on the vector kernel,
whose shuffle sums differ in the last bits).  The device name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))


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


def makers():
    from sparsematrixvectormultiplication_b200 import device as d
    return {
        "lap2d_4096": lambda: d.DeviceCSR.synth(d.SYNTH_LAP2D, 4096),
        "lap3d_384": lambda: d.DeviceCSR.synth(d.SYNTH_LAP3D, 384),
        "lap3d_512": lambda: d.DeviceCSR.synth(d.SYNTH_LAP3D, 512),
        "uniform_8m_32": lambda: d.DeviceCSR.synth(d.SYNTH_UNIFORM, 1 << 23, 1 << 23, 32),
    }


def arm_ms(A, x, y, algo, launches):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(launches):
        A.spmv(x, y, algo=algo)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / launches


def run(name, make, reps, launches):
    import torch
    from sparsematrixvectormultiplication_b200 import device as d
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    A = make()
    torch.cuda.synchronize()
    plan_s = time.perf_counter() - t0
    i = A.info()
    images = {}  # the image in each form, whatever the plan chose
    for form, mode in (("f64", 1), ("coded", 2), ("patterns", 3)):
        H = make()
        try:
            H.set_image(mode)
            images[form] = H
        except Exception:  # the matrix does not qualify for this form
            H.close()
    g = torch.Generator(device="cuda").manual_seed(11)
    x = torch.randn(i.N, dtype=torch.float64, device="cuda", generator=g)
    y_row = torch.empty(i.M, dtype=torch.float64, device="cuda")
    y_auto = torch.empty(i.M, dtype=torch.float64, device="cuda")
    arms = [(A, d.ALGO_ROW, y_row), (A, d.ALGO_AUTO, y_auto)]
    arms += [(H, d.ALGO_ROW_IMAGE, torch.empty(i.M, dtype=torch.float64, device="cuda")) for H in images.values()]
    for H, algo, y in arms:
        arm_ms(H, x, y, algo, launches)
    torch.cuda.synchronize()
    bitwise = bool(torch.equal(y_row.view(torch.int64), y_auto.view(torch.int64)))
    times = [[] for _ in arms]
    for _ in range(reps):
        for (H, algo, y), ts in zip(arms, times):
            ts.append(arm_ms(H, x, y, algo, launches))
    t_row, t_auto = times[0], times[1]
    on_image = i.auto_algo == d.ALGO_ROW_IMAGE
    alg = i.algorithmic_bytes
    read = (i.image_device_bytes + 8 * i.M + 8 * i.N) if on_image else alg
    auto_kernel = A.image_form() if on_image else (f"csr_row_kernel<{i.row_batch},double>" if i.auto_algo == d.ALGO_ROW
                                                   else d.ALGO_NAMES[i.auto_algo])

    def stats(ts):
        return {"mean_us": 1e3 * statistics.mean(ts), "min_us": 1e3 * min(ts), "max_us": 1e3 * max(ts),
                "spread_us": 1e3 * (max(ts) - min(ts))}
    out = {"M": i.M, "N": i.N, "nnz": i.nnz, "max_row_nnz": i.max_row_nnz, "plan_s": plan_s,
           "row_kernel": f"csr_row_kernel<{i.row_batch},double>", "auto_algo": i.auto_algo, "auto_kernel": auto_kernel,
           "image_bytes": i.image_bytes, "image_device_bytes": i.image_device_bytes, "image_index_bytes": i.image_index_bytes,
           "image_value_bytes": i.image_value_bytes, "csr_array_bytes": 12 * i.nnz + 4 * (i.M + 1),
           "algorithmic_bytes": alg, "read_bytes_auto": read,
           "row": stats(t_row), "auto": stats(t_auto), "speedup_row_over_auto": statistics.mean(t_row) / statistics.mean(t_auto),
           "algorithmic_TBps_auto": alg / (1e-3 * statistics.mean(t_auto)) / 1e12,
           "read_TBps_auto": read / (1e-3 * statistics.mean(t_auto)) / 1e12,
           "auto_bitwise_equal_row": bitwise}
    line = f"[csr_image] {name}: row {out['row']['mean_us']:.1f} us, auto {out['auto']['mean_us']:.1f} us ({auto_kernel})"
    for (form, H), (_, _, y), ts in zip(images.items(), arms[2:], times[2:]):
        ih = H.info()
        rd = ih.image_device_bytes + 8 * i.M + 8 * i.N
        out[f"image_{form}"] = {"kernel": H.image_form(), "image_device_bytes": ih.image_device_bytes, "read_bytes": rd,
                                **stats(ts), "read_TBps": rd / (1e-3 * statistics.mean(ts)) / 1e12,
                                "speedup_over_auto": statistics.mean(ts) / statistics.mean(t_auto),
                                "bitwise_equal_row": bool(torch.equal(y_row.view(torch.int64), y.view(torch.int64)))}
        line += f", {form} {1e3 * statistics.mean(ts):.1f} us ({H.image_form()})"
        H.close()
    print(line + f", x{out['speedup_row_over_auto']:.3f}, bitwise {bitwise}, plan {plan_s:.2f} s", flush=True)
    A.close()
    del x, y_row, y_auto, arms
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=12)
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--workloads", default="lap2d_4096,lap3d_384,lap3d_512,uniform_8m_32")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("csr_image_bench: no CUDA device")
    mk = makers()
    result = {"card": card(), "reps": args.reps, "launches_per_rep": args.launches, "workloads": {}}
    for name in args.workloads.split(","):
        result["workloads"][name] = run(name, mk[name], args.reps, args.launches)
    result["card_after"] = card()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
