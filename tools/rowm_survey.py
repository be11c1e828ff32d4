"""Survey of the multi-row forms of the row kernels (csr_rowm_kernel / hll_rowm_kernel) in the built library, and of the
one-row kernels including the masked forms that multiply a CSR handle's private image (accumulate or not, 4-byte `int` or
narrow 2-byte `u16` column field, fp64 values or 1-byte `u8` value codes): registers,
spill bytes (csrc/build/*.ptxas.log) and how many of a step's loads ptxas issues ahead of the first multiply (cuobjdump
-sass).  A form whose loads are split by a DMUL stalls on its first gather before the rest is requested.  Then the
same for csr_pattern_kernel<W, ACCUM> (the pattern form of the private image): its W gathers (64-bit LDGs) against the
first DMUL.  And for csr_pattern_tile_kernel<W, ACCUM> (its tiled kernel): the global loads (LDG and the LDGSTS of
cp.async) ptxas places ahead of the tile's one BAR.SYNC, which should be all of them, and the shared-memory loads of
the rows after it.  No GPU needed.

    python tools/rowm_survey.py            # every rowm instantiation and, for comparison, the one-row kernels
"""
import re
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "sparsematrixvectormultiplication_b200"


def ptxas_info():
    info, cur = {}, None
    for log in (PKG / "csrc" / "build").glob("cuda_*.ptxas.log"):
        for line in log.read_text().splitlines():
            m = re.search(r"Compiling entry function '(\S+)'", line)
            if m:
                cur = m.group(1)
            m = re.search(r"(\d+) bytes spill stores", line)
            if m and cur:
                info.setdefault(cur, {})["spill"] = int(m.group(1))
            m = re.search(r"Used (\d+) registers", line)
            if m and cur:
                info.setdefault(cur, {})["regs"] = int(m.group(1))
    return info


def main():
    info = ptxas_info()
    sass = subprocess.run(["cuobjdump", "-sass", str(PKG / "libspmv_b200.so")], capture_output=True, text=True).stdout
    rows, patterns, tiles = [], [], []
    for body in re.split(r"Function : ", sass)[1:]:
        name = body.split()[0]
        t = re.search(r"csr_pattern_tile_kernelILi(\d+)ELb([01])E", name)
        if t:
            ops = re.findall(r"(?<!@!PT )\b(LDGSTS|LDG|BAR\.SYNC|LDS)\b", body)  # @!PT LDS: never-issued padding
            bar = ops.index("BAR.SYNC") if "BAR.SYNC" in ops else len(ops)
            loads = sum(op in ("LDG", "LDGSTS") for op in ops)
            rec = info.get(name, {})
            tiles.append((int(t.group(1)), int(t.group(2)), rec.get("regs"), rec.get("spill"),
                          sum(op in ("LDG", "LDGSTS") for op in ops[:bar]), loads, ops.count("LDS")))
            continue
        p = re.search(r"csr_pattern_kernelILi(\d+)ELb([01])E", name)
        if p:
            ops = re.findall(r"\b(LDG\.E\.64|DMUL)\b", body)
            first = ops.index("DMUL") if "DMUL" in ops else len(ops)
            rec = info.get(name, {})
            patterns.append((int(p.group(1)), int(p.group(2)), rec.get("regs"), rec.get("spill"), first, ops.count("LDG.E.64")))
            continue
        m = re.search(r"(csr|hll)_row(m|u?)_kernelILi(\d)E(?:Li(\d)ELi(\d)E)?([fd])(?:Lb([01])E)?(?:Lb([01])E)?([it])?([dfh])?", name)
        if not m:
            continue
        fmt, multi, batch, rows_per, ctas, v, masked, accum, index, stored = m.groups()
        ops = re.findall(r"\b(LDG|DMUL)\b", body)
        ahead = 0
        for op in ops:
            if op == "DMUL":
                break
            ahead += 1
        total = ops.count("LDG")
        # the most loads any path issues between two multiplies: the straight-line step of hll_rowu_kernel (width equal
        # to the batch) may sit after the predicated loop in the code, where the first DMUL above finds the loop's
        most, run = 0, 0
        for op in ops:
            run = 0 if op == "DMUL" else run + 1
            most = max(most, run)
        rec = info.get(name, {})
        rows.append((fmt, v, int(rows_per or 1), int(batch), int(ctas or 8), rec.get("regs"), rec.get("spill"), ahead, most, total,
                     "row" + multi + (" masked" if masked == "1" else "") + (" accum" if accum == "1" else "")
                     + (" u16" if index == "t" else "") + (" u8" if stored == "h" else "")))
    print("format storage rows batch ctas/SM regs spill_bytes loads_ahead_of_first_DMUL/loads most_loads_between_DMULs "
          "rows_in_flight/SM kernel")
    for r in sorted(rows):
        fmt, v, rp, b, c, regs, spill, ahead, most, total, kind = r
        print(f"{fmt} {'f32' if v == 'f' else 'f64'} {rp} {b} {c} {regs} {spill} {ahead}/{total} {most} {256 * c * rp} {kind}")
    print("\ncsr_pattern_kernel: W accum regs spill_bytes gathers_ahead_of_first_DMUL/gathers")
    for w, accum, regs, spill, ahead, total in sorted(patterns):
        print(f"csr_pattern_kernel {w} {accum} {regs} {spill} {ahead}/{total}")
    print("\ncsr_pattern_tile_kernel: W accum regs spill_bytes global_loads_ahead_of_BAR.SYNC/global_loads shared_loads")
    for w, accum, regs, spill, ahead, total, lds in sorted(tiles):
        print(f"csr_pattern_tile_kernel {w} {accum} {regs} {spill} {ahead}/{total} {lds}")


if __name__ == "__main__":
    sys.exit(main())
