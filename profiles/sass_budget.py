#!/usr/bin/env python3
"""Per-section instruction budget of the Newton loop of a solver kernel, from the SASS of the shipped
library with inline line info:

    cuobjdump -xelf all bayesian_inference_trpl_b200/libtrpl_b200.so
    nvdisasm -gi -c trpl_kernels.sm_100a.cubin > lined.sass
    python profiles/sass_budget.py lined.sass trpl_sim_kernelILi4ELb0 [--dump newton.sass]
    LOOP_MIN=300 LOOP_MAX=8000 python profiles/sass_budget.py lined.sass trpl_sim_cta_kernelILi4ELi8ELi1

The Newton loop is the FP64-densest loop of LOOP_MIN..LOOP_MAX instructions (default 400..1600, which
fits the warp kernel at M <= 4); LOOP_MIN=300 LOOP_MAX=8000 covers every trpl_sim_kernel and
trpl_sim_cta_kernel instantiation.

Every instruction of the innermost big loop (the Newton / Gauss-Seidel iteration) is attributed to
a section of csrc/trpl_solver.cuh through the source lines marked `// [sec:NAME]` there, and counted
by kind.  Code inlined from a helper (the species assembly, the tridiagonal solve) is named by its
call site plus the helper's own section, e.g. `N:surface` or `P-solve:pcr`.  Kinds:
  DFMA / DMUL / DADD      FP64 pipe, 2 issue cycles per warp instruction on an SMSP
  3reg                    DFMAs whose three sources are distinct vector registers without a .reuse
                          hit: 3 cycles (register-bank limit, profiles/r01_microbench.txt)
  SHFL, MUFU, ALU (FSEL/LOP3/ISETP/VIMNMX/SEL/IADD3...), MOV/IMAD, other
"""
import collections
import re
import sys

path, pat = sys.argv[1], sys.argv[2]
dump = sys.argv[sys.argv.index("--dump") + 1] if "--dump" in sys.argv else None
outer = "--outer" in sys.argv      # budget of the enclosing TIME loop minus the Newton loop (per-step code)
src_path = None

# ---- section map from the source: a line `// [sec:NAME]` opens NAME until the next marker
SOLVER = "trpl_solver.cuh"
sec_of_line = {}
import os
here = os.path.dirname(os.path.abspath(__file__))
src = open(os.path.join(here, "..", "bayesian_inference_trpl_b200", "csrc", SOLVER)).read().split("\n")
cur = None
for i, line in enumerate(src, 1):
    m = re.search(r"\[sec:([\w-]+)\]", line)
    if m:
        cur = m.group(1)
    sec_of_line[i] = cur

text = open(path).read().split("\n")
start = [i for i, l in enumerate(text) if l.startswith("_ZN") and pat in l and l.rstrip().endswith(":")][0]
ins = []          # (addr, text, chain)
chain = []
pending = []
for l in text[start + 1:]:
    if l.startswith("//---") and ins:
        break
    m = re.match(r'\s*//## File "([^"]+)", line (\d+)(?: inlined at "([^"]+)", line (\d+))?', l)
    if m:
        if not pending:
            pending = [(m.group(1), int(m.group(2)))]
        if m.group(3):
            pending.append((m.group(3), int(m.group(4))))
        continue
    m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?);", l)
    if m:
        if pending:
            chain, pending = pending, []
        ins.append((int(m.group(1), 16), m.group(2).strip(), chain))


def op(s):
    return re.sub(r"^@!?U?P\w+\s+", "", s).split()[0].split(".")[0]


loops = []
for a, s, _ in ins:
    if op(s) == "BRA":
        m = re.search(r"\(\.L_x_\d+\)", s)
        # branch targets are labels in nvdisasm output; fall back to address matching below
labels = {}
addr_of_label = {}
idx = 0
# second pass for labels
la = None
for l in text[start + 1:]:
    if l.startswith("//---") and idx > 0:
        break
    m = re.match(r"(\.L_x_\d+):", l)
    if m:
        la = m.group(1)
        continue
    m = re.match(r"\s*/\*([0-9a-f]{4,})\*/", l)
    if m:
        if la:
            addr_of_label[la] = int(m.group(1), 16)
            la = None
        idx += 1
for a, s, _ in ins:
    if op(s) == "BRA":
        m = re.search(r"`\((\.L_x_\d+)\)", s)
        if m and m.group(1) in addr_of_label and addr_of_label[m.group(1)] <= a:
            loops.append((addr_of_label[m.group(1)], a))
LO_, HI_ = (int(os.environ.get("LOOP_MIN", 400)), int(os.environ.get("LOOP_MAX", 1600)))
cands = [(lo, hi) for lo, hi in loops if LO_ <= sum(1 for a, _, _ in ins if lo <= a <= hi) <= HI_]
def _fp64_frac(c):
    body_ = [s_ for a_, s_, _ in ins if c[0] <= a_ <= c[1]]
    return sum(1 for s_ in body_ if op(s_) in ("DFMA", "DMUL", "DADD")) / float(len(body_))
lo, hi = sorted(cands, key=_fp64_frac)[-1]          # the Newton loop is the FP64-densest big loop
body = [(a, s, c) for a, s, c in ins if lo <= a <= hi]
if outer:
    enclosing = sorted([(l2, h2) for l2, h2 in loops if l2 < lo and h2 > hi], key=lambda c: c[1] - c[0])
    olo, ohi = enclosing[0]
    body = [(a, s, c) for a, s, c in ins if olo <= a <= ohi and not (lo <= a <= hi)]


def section(chain):
    # the outermost tagged frame (the call site in run_sim) names the row; the innermost one refines it
    secs = [sec_of_line.get(line) for f, line in chain if f.endswith(SOLVER)]
    secs = [s for s in secs if s and s not in ("kernel", "none")]
    if not secs:
        return "other"
    outer = secs[-1]
    inner = secs[0]
    return outer if inner == outer else outer + ":" + inner


ALU = {"FSEL", "LOP3", "ISETP", "VIMNMX", "SEL", "IADD3", "VIADD", "PLOP3", "SHF", "LEA", "ISCADD", "IABS",
       "VOTE", "VOTEU", "POPC", "FLO", "DSETP", "FSETP", "UISETP", "ULOP3", "UIADD3", "USEL", "R2UR", "FMNMX", "DMNMX"}
rows = collections.OrderedDict()
kinds = ["DFMA", "DMUL", "DADD", "3reg", "SHFL", "MUFU", "ALU", "MOV/IMAD", "other"]
for a, s, c in body:
    sec = section(c)
    r = rows.setdefault(sec, collections.Counter())
    o = op(s)
    if o in ("DFMA", "DMUL", "DADD"):
        r[o] += 1
        if o == "DFMA":
            srcs = [x.strip().lstrip("-|").rstrip("|") for x in s.split(o, 1)[1].split(",")[1:]]
            regs = [x.split(".")[0] for x in srcs if re.match(r"R\d+", x)]
            if len(set(regs)) == 3 and not any("reuse" in x for x in srcs):
                r["3reg"] += 1
    elif o == "SHFL":
        r["SHFL"] += 1
    elif o == "MUFU":
        r["MUFU"] += 1
    elif o in ALU:
        r["ALU"] += 1
    elif o in ("MOV", "IMAD", "UMOV", "CS2R", "UIMAD"):
        r["MOV/IMAD"] += 1
    else:
        r["other"] += 1
        r["_" + o] += 1

print("kernel %s   %s 0x%x-0x%x   %d instructions" % (pat, "time loop outside the Newton loop (static; the flush block runs once per 32 steps)"
                                                  if outer else "Newton loop", lo, hi, len(body)))
print("%-22s" % "section" + "".join("%9s" % k for k in kinds) + "%9s%9s" % ("FP64", "cycles*"))
tot = collections.Counter()
for sec, r in rows.items():
    fp = r["DFMA"] + r["DMUL"] + r["DADD"]
    cyc = 2.0 * fp + r["3reg"] + 0.85 * (r["SHFL"] + r["MUFU"] + r["ALU"] + r["MOV/IMAD"] + r["other"])
    print("%-22s" % sec + "".join("%9d" % r[k] for k in kinds) + "%9d%9.0f" % (fp, cyc))
    for k in kinds:
        tot[k] += r[k]
    tot["fp"] += fp
    tot["cyc"] += cyc
print("%-22s" % "TOTAL" + "".join("%9d" % tot[k] for k in kinds) + "%9d%9.0f" % (tot["fp"], tot["cyc"]))
others = collections.Counter()
for r in rows.values():
    for k, v in r.items():
        if k.startswith("_"):
            others[k[1:]] += v
print("other =", dict(others.most_common()))
print("* issue-time model of profiles/r01_microbench.txt: FP64 2 cycles, +1 for a 3-register DFMA, 0.85 per other instruction")
if dump:
    with open(dump, "w") as f:
        for a, s, c in body:
            f.write("%-24s /*%04x*/ %s\n" % (section(c), a, s))
