#!/usr/bin/env python
"""Counts the SASS instructions of gang_fit_kernel's hot loop (the innermost loop that holds the VOTE
instructions: one trip = 4 nodes per lane x PODS_PER_WARP pods) and writes profiles/sass_ops_r2.json, the
op counts behind the decisions-only instruction roofline in bench.py (SURVEY 8(d) R2).

    python profiles/tools/sass_count.py [--lib batch-scheduler_b200/libbsched.so] [--kernel ILi0ELi3ELi2ELi0E]
                                        [--ppw 4] [--dump profiles/sass_gang_fit_r2.txt]

Pipe classes (sm_100a, as ncu groups them): the integer ALU pipe takes add/logic/shift/compare/select/
min-max/vote-free predicate ops at 64 lanes/clk/SM (16 per scheduler); IMAD* go to the FMA pipe; LDS/STS/
LDG/STG to the LSU; U* ops to the uniform datapath.  Every instruction costs one issue slot."""
import argparse, json, os, re, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

ALU = ("IADD3", "IADD", "LOP3", "SHF", "SHL", "SHR", "ISETP", "SEL", "VIMNMX", "VIMNMX3", "VIADDMNMX", "VIADD", "IMNMX",
       "PRMT", "MOV", "SGXT", "LEA", "PLOP3", "P2R", "R2P", "FSETP", "FSEL", "IABS", "BMSK", "POPC", "FLO", "CS2R", "S2R")
FMA = ("IMAD", "FFMA", "FMUL", "FADD", "HFMA2")
LSU = ("LDS", "STS", "LDG", "STG", "ATOMS", "ATOMG", "RED", "LDSM", "LD", "ST")


def classify(mn):
    base = mn.split(".")[0]
    if base.startswith("U") and base not in ("UNPACK",):
        return "uniform"
    if base in FMA:
        return "fma"
    if base in ALU:
        return "alu"
    if base in LSU:
        return "lsu"
    if base in ("VOTE", "VOTEU", "SHFL", "REDUX", "MATCH"):
        return "warp"
    if base in ("BRA", "WARPSYNC", "BSSY", "BSYNC", "NOP", "EXIT", "BAR", "CALL", "RET", "SYNCS", "ELECT", "FENCE", "MEMBAR"):
        return "ctrl"
    return "other"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", default=os.path.join(ROOT, "batch-scheduler_b200", "libbsched.so"))
    ap.add_argument("--kernel", default="ILi0ELi3ELi2ELi0E",
                    help="substring of the mangled gang_fit_kernel instance (default: <0,3,2,FIT_OUT_NONE>, the bench shape "
                         "in decisions-only mode)")
    ap.add_argument("--ppw", type=int, default=4)
    ap.add_argument("--marks-per-pair", type=int, default=4, help="VIADDMNMX per pair: (LN - 1) + LS, 4 for the bench shape (0,3,2)")
    ap.add_argument("--dump", default=None)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "sass_ops_r2.json"))
    a = ap.parse_args()
    txt = subprocess.run(["cuobjdump", "-sass", a.lib], capture_output=True, text=True, check=True).stdout
    # split into functions
    funcs = re.split(r"\n\s*Function : ", txt)
    body = None
    for f in funcs[1:]:
        name = f.split("\n", 1)[0].strip()
        if "gang_fit_kernel" in name and a.kernel in name:
            body, kname = f, name
            break
    if body is None:
        sys.exit(f"no gang_fit_kernel instance matching {a.kernel} in {a.lib}")
    ins = []   # (addr, mnemonic, text)
    for ln in body.splitlines():
        m = re.match(r"\s*/\*([0-9a-f]{4,5})\*/\s+(.*?);", ln)
        if not m:
            continue
        addr = int(m.group(1), 16)
        t = m.group(2).strip()
        t2 = re.sub(r"^@!?U?P\d+\s+", "", t)
        ins.append((addr, t2.split()[0], t))
    if a.dump:
        with open(a.dump, "w") as f:
            f.write(f"// cuobjdump -sass of {kname} ({os.path.basename(a.lib)})\n")
            for addr, mn, t in ins:
                f.write(f"/*{addr:05x}*/ {t}\n")
    # loops = backward branches; pick the innermost one that holds the lane arithmetic (VIADDMNMX)
    loops = []
    for addr, mn, t in ins:
        if mn.startswith("BRA"):
            m = re.search(r"0x([0-9a-f]+)", t)
            if m and int(m.group(1), 16) <= addr:
                loops.append((int(m.group(1), 16), addr))
    best = None
    for lo, hi in loops:
        inside = [x for x in ins if lo <= x[0] <= hi]
        marks = sum(1 for x in inside if x[1].startswith("VIADDMNMX"))
        if marks >= a.marks_per_pair * 4 and (best is None or len(inside) < len(best[2])):
            best = (lo, hi, inside, marks)
    if best is None:
        sys.exit("no loop with the lane arithmetic found")
    lo, hi, inside, marks = best
    pairs = 4 * a.ppw      # one trip = 4 nodes per lane x PODS_PER_WARP pods (the 4-word unrolled body)
    by_class, by_mn = {}, {}
    for addr, mn, t in inside:
        c = classify(mn)
        by_class[c] = by_class.get(c, 0) + 1
        by_mn[mn] = by_mn.get(mn, 0) + 1
    total = len(inside)
    out = {"kernel": kname, "lib": os.path.relpath(a.lib, ROOT), "loop": [hex(lo), hex(hi)], "instructions_in_loop": total,
           "pairs_per_trip": pairs, "issue_ops_per_pair": total / pairs,
           "alu_pipe_ops_per_pair": by_class.get("alu", 0) / pairs, "fma_pipe_ops_per_pair": by_class.get("fma", 0) / pairs,
           "lsu_ops_per_pair": by_class.get("lsu", 0) / pairs, "by_class": by_class,
           "by_mnemonic": dict(sorted(by_mn.items(), key=lambda kv: -kv[1])),
           "note": "static count of the innermost loop that holds the lane arithmetic (one trip = 4 nodes per lane x "
                   "PODS_PER_WARP pods); in score mode it includes the streaming score stores and their bounds checks; "
                   "per-tile / per-sweep instructions outside it are not counted"}
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("kernel", "instructions_in_loop", "pairs_per_trip", "issue_ops_per_pair",
                                          "alu_pipe_ops_per_pair", "fma_pipe_ops_per_pair", "lsu_ops_per_pair")}))


if __name__ == "__main__":
    main()
