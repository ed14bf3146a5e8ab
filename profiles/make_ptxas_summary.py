#!/usr/bin/env python
"""Registers / spills / shared memory of every kernel, from the `-Xptxas -v` logs the build leaves in
ctucopy_b200/csrc/ptxas_*.log (git-ignored), plus SASS excerpts that show the Blackwell-specific instructions of the
hot kernels.  Writes profiles/r02_ptxas.txt and profiles/r02_sass_excerpts.txt.
usage: python profiles/make_ptxas_summary.py"""
import glob
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "ctucopy_b200", "csrc")


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.split("\n")
    return [re.sub(r"\(.*", "", o).replace("void ", "").replace("ctu::", "") for o in out]


def main():
    rows = []
    for log in sorted(glob.glob(os.path.join(CSRC, "ptxas_*.log"))):
        cur = None
        for ln in open(log):
            m = re.search(r"Compiling entry function '(\S+)'", ln)
            if m:
                cur = {"tu": os.path.basename(log)[6:-4], "name": m.group(1), "spill_st": 0, "spill_ld": 0, "stack": 0, "regs": None, "smem": 0}
                rows.append(cur)
                continue
            if cur is None:
                continue
            m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", ln)
            if m:
                # an entry's own line and those of the device functions it calls (sqrt / division slow paths): keep the largest
                st, ss, sl = map(int, m.groups())
                cur["stack"], cur["spill_st"], cur["spill_ld"] = max(cur["stack"], st), max(cur["spill_st"], ss), max(cur["spill_ld"], sl)
            m = re.search(r"Used (\d+) registers", ln)
            if m:
                cur["regs"] = int(m.group(1))
                m2 = re.search(r"(\d+) bytes smem", ln)
                cur["smem"] = int(m2.group(1)) if m2 else 0
    names = demangle([r["name"] for r in rows])
    with open(os.path.join(ROOT, "profiles", "r02_ptxas.txt"), "w") as fh:
        fh.write("# nvcc 12.9 -gencode arch=compute_100a,code=sm_100a -O3 -Xptxas -v (ctucopy_b200/csrc/Makefile); static shared memory only\n")
        fh.write("# (dynamic shared memory is sized by the launchers).  %d kernels, %d with spills.\n" % (len(rows), sum(1 for r in rows if r["spill_st"] or r["spill_ld"])))
        fh.write("%-10s %-64s %5s %7s %9s %9s %6s\n" % ("unit", "kernel", "regs", "stack B", "spill st B", "spill ld B", "smem B"))
        for r, n in sorted(zip(rows, names), key=lambda x: (x[0]["tu"], x[1])):
            fh.write("%-10s %-64s %5s %7d %9d %9d %6d\n" % (r["tu"], n[:64], r["regs"], r["stack"], r["spill_st"], r["spill_ld"], r["smem"]))
    # ---- SASS excerpts
    so = os.path.join(ROOT, "ctucopy_b200", "libctucopy_b200.so")
    sass = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True).stdout.split("\n")
    funcs, cur = {}, None
    for ln in sass:
        m = re.search(r"Function : (\S+)", ln)
        if m:
            cur = m.group(1); funcs[cur] = []
        elif cur and re.match(r"\s+/\*[0-9a-f]{4,5}\*/", ln):
            funcs[cur].append(re.sub(r"/\* 0x[0-9a-f]+ \*/", "", ln).rstrip())
    want = [("k_frames2ILi400ELb0", ["FADD2", "FMUL2", "FFMA2", "LDGSTS", "SHFL", "STG", "LDS.64", "BAR"]),
            ("k_bankILi3ELi2ELb1", ["UBLKCP", "SYNCS", "FADD2", "FMUL2", "FFMA2", "LDS.64", "STS.64", "LDS.128", "MUFU", "BAR", "STG"]),
            ("k_bankILi3ELi2ELb0", ["UBLKCP", "SYNCS", "FFMA2", "LDS.128", "BAR", "STG"]),
            ("k_trapdctILi51ELi8", ["FFMA2", "FADD2", "LDCU.128", "LDS"]),
            ("k_frames256", ["FADD2", "FFMA2", "LDGSTS", "SHFL"]),
            ("k_tdiir_filter", ["DFMA", "DMUL", "I2F", "LDS.64", "BAR"]),
            ("k_nr_scan4ILi1ELi1", ["LDG.E.128", "STG.E.128", "MUFU"]),
            ("k_burgILi25ELb1ELi4ELb0", ["DFMA", "DADD", "DMUL", "SHFL", "WARPSYNC", "LDL", "STL", "BAR"]),
            ("k_synth_cILi512ELi256", ["LDG", "STG", "SHFL", "BAR"])]
    with open(os.path.join(ROOT, "profiles", "r02_sass_excerpts.txt"), "w") as fh:
        fh.write("# cuobjdump -sass ctucopy_b200/libctucopy_b200.so: instruction counts of the hot kernels and the first occurrences of the\n")
        fh.write("# instructions that matter (UBLKCP / SYNCS = cp.async.bulk + mbarrier, LDGSTS = cp.async, LDS.128 / LDG.E.128 = 16-byte accesses,\n# FADD2 / FMUL2 / FFMA2 = packed FP32 on register pairs with the .LO_HI swap, .NP sign and .F32 broadcast operand modifiers).\n")
        for key, pats in want:
            for fn, body in funcs.items():
                if key not in fn:
                    continue
                dm = demangle([fn])[0]
                fh.write("\n== %s: %d instructions\n" % (dm, len(body)))
                ops = {}
                for ln in body:
                    mm = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d\s+)?([A-Z0-9_.]+)", ln)
                    if mm:
                        op = mm.group(1)
                        ops[op.split(".")[0]] = ops.get(op.split(".")[0], 0) + 1
                fh.write("   opcode counts: " + ", ".join("%s %d" % kv for kv in sorted(ops.items(), key=lambda x: -x[1])[:24]) + "\n")
                for p_ in pats:
                    hits = [ln for ln in body if p_ in ln]
                    fh.write("   %-10s x%-4d %s\n" % (p_, len(hits), hits[0].strip()[:110] if hits else ""))
    print("wrote profiles/r02_ptxas.txt, profiles/r02_sass_excerpts.txt")


if __name__ == "__main__":
    main()
