#!/usr/bin/env python
"""Attributes an `ncu --set full --import-source on` capture of step_kernel to source lines / code regions.

ncu's CSV export of the source page only carries the SASS view, so this joins it with nvdisasm's line table of the SAME
library build (run it here, right after the capture came back, before rebuilding):

    python tools/sass_profile.py gpurun_out/prof.ncu-rep [--lib so100_mujoco_rl_b200/libso100_b200.so] [--top 25]

Prints executed warp instructions and stall samples per region (dynamics / solver / limit rows / sincos / servo+Euler /
task logic + I/O), the opcode histogram, and the hottest source lines.

    python tools/sass_profile.py --static [--lib ...] [--src CHECKOUT] [--func ...]

needs no capture and no GPU: the STATIC instruction count of the substep loop's body (the innermost backward branch whose
range holds every generated-dynamics instruction) per region, and its branch / reconvergence opcodes.  Regions come from
the source lines of --src (default: this checkout); a library built from another commit needs that commit's checkout.
"""
import argparse
import collections
import csv
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def line_table(lib: str, func_substr: str, labels: dict = None):
    """offset -> (file, line) of the innermost source line, from nvdisasm -gi of the cubin inside `lib`; an instruction
    of a helper inlined into the generated dynamics (so_fma, so_mul, ...) counts as the generated line that calls it.
    `labels`, if given, receives branch label -> offset."""
    tmp = tempfile.mkdtemp()
    subprocess.check_call(["cuobjdump", "-xelf", "all", os.path.abspath(lib)], cwd=tmp, stdout=subprocess.DEVNULL)
    cubin = [os.path.join(tmp, f) for f in os.listdir(tmp) if f.endswith(".cubin")][0]
    txt = subprocess.run(["nvdisasm", "-gi", "-c", cubin], capture_output=True, text=True).stdout
    table, cur, on, pending, innermost = {}, ("?", 0), False, [], True
    for ln in txt.splitlines():
        if ln.startswith("//---") and ".text." in ln:
            on = func_substr in ln
            continue
        if not on:
            continue
        m = re.search(r'//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?', ln)
        if m:  # the inline chain, innermost first
            if innermost:
                cur = (os.path.basename(m.group(1)), int(m.group(2)))
            if m.group(3) and os.path.basename(m.group(3)) == "so100_dyn_gen.cuh" and cur[0] != "so100_dyn_gen.cuh":
                cur = ("so100_dyn_gen.cuh", int(m.group(4)))
            innermost = False
            continue
        m = re.match(r"(\.L_x_\d+):", ln.strip())
        if m:
            pending.append(m.group(1))
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,6})\*/\s+(.*?);", ln)
        if m:
            table[int(m.group(1), 16)] = (cur, m.group(2).strip())
            innermost = True
            if labels is not None:
                labels.update((name, int(m.group(1), 16)) for name in pending)
            pending = []
    return table


def region_of(file: str, line: int, src_cache: dict, src: str = ROOT) -> str:
    """Region of a source line, read from the checkout `src` (the one the library was built from: line numbers move)."""
    if file == "so100_dyn_gen.cuh":
        return "dynamics (generated)"
    if file == "so100_dyn.cuh":
        lines = src_cache.setdefault(file, open(os.path.join(src, "so100_mujoco_rl_b200", "csrc", file)).read().splitlines())
        # walk up to the enclosing function header
        for k in range(min(line, len(lines)) - 1, -1, -1):
            m = re.match(r"SO_HD\s+\S+\s+(\w+)\(", lines[k])
            if m:
                fn = m.group(1)
                return {"solve_qacc": "solver sweeps + setup", "solve1": "solver sweeps + setup", "limit_row": "limit rows",
                        "impedance": "limit rows", "so_rcp": "solver sweeps + setup", "so_clamp": "solver sweeps + setup",
                        "so_sincos": "sincos", "task_kinematics": "task kinematics", "mat_vec": "task kinematics",
                        "mat_mul": "task kinematics"}.get(fn, "dyn.cuh:" + fn)
        return "dyn.cuh:?"
    if file == "so100_b200.cu":
        lines = src_cache.setdefault(file, open(os.path.join(src, "so100_mujoco_rl_b200", "csrc", file)).read().splitlines())
        for k in range(min(line, len(lines)) - 1, -1, -1):
            m = re.match(r"(?:__device__ __forceinline__|__global__)\s+.*?(\w+)\(", lines[k])
            if m:
                return {"physics": "servo + Euler + loop"}.get(m.group(1), "task logic + I/O (" + m.group(1) + ")")
        return "task logic + I/O"
    return "libdevice / intrinsics (" + file + ")"


def static_counts(lib: str, func: str, src: str) -> None:
    labels = {}
    table = line_table(lib, func, labels)
    offs = sorted(table)
    dyn = [o for o in offs if table[o][0][0] == "so100_dyn_gen.cuh"]
    if not dyn:
        sys.exit(f"no generated-dynamics instructions in {func}")
    loops = []  # (start, end) of backward branches spanning the generated dynamics
    for o in offs:
        m = re.match(r"(?:@!?U?P\w+\s+)?BRA\b.*`\((\.L_x_\d+)\)", table[o][1])
        if m and labels.get(m.group(1), o + 1) <= dyn[0] and o >= dyn[-1]:
            loops.append((labels[m.group(1)], o))
    if not loops:
        sys.exit("substep loop not found (no backward branch around the generated dynamics)")
    lo, hi = min(loops, key=lambda r: r[1] - r[0])
    body = [o for o in offs if lo <= o <= hi]
    reg, ops, cache = collections.Counter(), collections.Counter(), {}
    for o in body:
        (file, line), sass = table[o]
        reg[region_of(file, line, cache, src)] += 1
        op = sass.split()[1] if sass.startswith("@") else sass.split()[0]
        ops[op.split(".")[0]] += 1
    print(f"{func}: substep loop body [{lo:#x}, {hi:#x}]: {len(body)} static SASS instructions")
    for r, k in reg.most_common():
        print(f"  {r:42s} {k:6d}")
    print("  branch / reconvergence:", ", ".join(f"{o} {ops[o]}" for o in ("BSSY", "BSYNC", "BRA", "WARPSYNC", "VOTE", "VOTEU")))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("report", nargs="?")
    ap.add_argument("--static", action="store_true", help="static loop-body counts from the library alone (no capture)")
    ap.add_argument("--lib", default=os.path.join(ROOT, "so100_mujoco_rl_b200", "libso100_b200.so"))
    ap.add_argument("--src", default=ROOT, help="checkout the library was built from (its sources name the regions)")
    ap.add_argument("--func", default="step_kernelILi1ELb1E")
    ap.add_argument("--top", type=int, default=20)
    ap.add_argument("--substeps", type=int, default=16)
    args = ap.parse_args()
    if args.static:
        static_counts(args.lib, args.func, args.src)
        return
    if not args.report:
        ap.error("a report is needed unless --static")
    out = subprocess.run(["ncu", "-i", args.report, "--page", "source", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(out.splitlines()))
    hdr_i = next(i for i, r in enumerate(rows) if r and r[0] == "Address")
    hdr, data = rows[hdr_i], rows[hdr_i + 1:]
    iA, iS, iE, iN = hdr.index("Address"), hdr.index("Source"), hdr.index("Instructions Executed"), hdr.index("# Samples")
    stall_cols = [(k, h) for k, h in enumerate(hdr) if h.startswith("stall_") and "Not Issued" not in h]
    table = line_table(args.lib, args.func)
    base = int(data[0][iA], 16)
    reg_e, reg_s, line_e, ops = collections.Counter(), collections.Counter(), collections.Counter(), collections.Counter()
    stalls = collections.Counter()
    cache, total, mismatch = {}, 0, 0
    for r in data:
        off = int(r[iA], 16) - base
        e, ns = int(r[iE]), int(r[iN])
        (file, line), sass = table.get(off, (("?", 0), ""))
        op_ncu = r[iS].split()[1] if r[iS].strip().startswith("@") else r[iS].split()[0]
        if sass and op_ncu.split(".")[0] not in sass:
            mismatch += 1
        reg = region_of(file, line, cache, args.src)
        reg_e[reg] += e; reg_s[reg] += ns; line_e[(file, line)] += e; ops[op_ncu.split(".")[0]] += e
        total += e
        for k, h in stall_cols:
            stalls[h] += int(r[k] or 0)
    if mismatch > len(data) // 20:
        print(f"WARNING: {mismatch}/{len(data)} SASS lines do not match the library build - rebuild mismatch?", file=sys.stderr)
    warps = int(data[0][iE])  # the first instruction is executed once per warp
    per_sub = total / warps / args.substeps
    print(f"warp instructions {total}  per warp {total / warps:.0f}  per substep {per_sub:.0f}  ({len(data)} SASS lines)")
    print("\nregion                                    instr/substep   share   stall samples")
    tot_s = sum(reg_s.values()) or 1
    for reg, e in reg_e.most_common():
        print(f"{reg:42s} {e / warps / args.substeps:10.0f}   {100 * e / total:5.1f}%   {100 * reg_s[reg] / tot_s:5.1f}%")
    print("\nopcode histogram (executed):", ", ".join(f"{o} {100 * c / total:.1f}%" for o, c in ops.most_common(14)))
    ts = sum(stalls.values()) or 1
    print("stall samples:", ", ".join(f"{h[6:]} {100 * c / ts:.1f}%" for h, c in stalls.most_common(10)))
    print("\nhottest source lines (instr/substep):")
    for (file, line), e in line_e.most_common(args.top):
        print(f"  {file}:{line:<5d} {e / warps / args.substeps:8.1f}")


if __name__ == "__main__":
    main()
