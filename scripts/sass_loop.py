"""Static look at the hot loop of exhaustive_all_kernel without a GPU: compiles only exhaustive_dev.cuh (a few seconds),
finds the innermost loops that hold the MUFU.RSQ64H of the bordered step and prints, per loop, the instruction count, the
sum of the stall counts the compiler encoded (= issue cycles of ONE warp running alone, scoreboard waits excluded), the
opcode mix and the local-memory traffic (spills).   python scripts/sass_loop.py [-DEXH_...=...] [--dump file] [--classes]
(--classes: the instantiation for the class-resolved store of PIPSORT_PRIOR_CLASSES instead of the default one; --counts: the one
for the store with the count table of PIPSORT_CAUSAL_COUNTS)"""
import os, re, subprocess, sys, tempfile
from collections import Counter
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TU = '#include "exhaustive_dev.cuh"\n'


def build(defs, out):
    src = os.path.join(tempfile.gettempdir(), "exh_tu_%d.cu" % os.getpid())
    open(src, "w").write(TU)
    cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-cubin", "-Xptxas", "-v",
           "-I", os.environ.get("PIPSORT_CSRC", os.path.join(ROOT, "pipsort_b200", "csrc")), "-I", os.path.join(ROOT, "include")] + defs + [src, "-o", out]
    r = subprocess.run(cmd, capture_output=True, text=True)
    os.unlink(src)
    if r.returncode:
        sys.exit(r.stderr)
    info = [l for l in r.stderr.split("\n") if "exhaustive_all" in l or "registers" in l or "spill" in l or "smem" in l]
    return info


def parse(cubin):
    txt = subprocess.run(["cuobjdump", "-sass", cubin], capture_output=True, text=True).stdout.split("\n")
    fns, cur, ins = {}, None, None
    for l in txt:
        if "Function :" in l:
            cur = l.split("Function :")[1].strip(); ins = []; fns[cur] = ins; last = None
            continue
        if cur is None:
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,5})\*/\s+(.*?);\s+/\* (0x[0-9a-f]+) \*/", l)
        if m:
            last = [int(m.group(1), 16), m.group(2).strip(), None]
            ins.append(last)
            continue
        m = re.match(r"\s+/\* (0x[0-9a-f]+) \*/", l)
        if m and last is not None and last[2] is None:
            last[2] = int(m.group(1), 16)
    return fns


def opname(t):
    p = t.split()
    op = p[1] if p[0].startswith("@") else p[0]
    return op.split(".")[0]


def main():
    defs = [a for a in sys.argv[1:] if a.startswith("-D") or a.startswith("--maxrreg")]
    dump = sys.argv[sys.argv.index("--dump") + 1] if "--dump" in sys.argv else None
    out = os.path.join(tempfile.gettempdir(), "exh_tu_%d.cubin" % os.getpid())
    for l in build(defs, out):
        print(l.strip())
    fns = parse(out)
    os.unlink(out)
    kind = 2 if "--counts" in sys.argv else (1 if "--classes" in sys.argv else 0)   # StoreKind (common.cuh)
    name = [k for k in fns if "exhaustive_all_kernel" in k and re.search(r"StoreKindE%dE" % kind, k)][0]
    ins = fns[name]
    print("kernel instructions:", len(ins))
    loops = []
    for a, t, w in ins:
        m = re.search(r"BRA\S*\s+(?:\S+,\s+)?(0x[0-9a-f]+)", t)
        if m and opname(t) == "BRA" and int(m.group(1), 16) <= a:
            loops.append((int(m.group(1), 16), a))
    rsq = [a for a, t, w in ins if "MUFU.RSQ64H" in t]
    seen = set()
    for r in rsq:
        inner = [lp for lp in loops if lp[0] <= r <= lp[1]]
        if not inner:
            continue
        lp = min(inner, key=lambda x: x[1] - x[0])
        if lp in seen:
            continue
        seen.add(lp)
        body = [(a, t, w) for a, t, w in ins if lp[0] <= a <= lp[1]]
        ops, st = Counter(), Counter()
        for a, t, w in body:
            ops[opname(t)] += 1; st[opname(t)] += (w >> 41) & 0xf
        n = len(body); stall = sum(st.values())
        f64 = sum(ops[o] for o in ("DFMA", "DADD", "DMUL", "DSETP"))
        print("loop %05x-%05x: %d instr, static %d cycles, fp64 %d (DFMA %d), MUFU %d, LDL %d STL %d LDC %d LDS %d SHFL %d LDG %d"
              % (lp[0], lp[1], n, stall, f64, ops["DFMA"], ops["MUFU"], ops["LDL"], ops["STL"], ops["LDC"] + ops["LDCU"], ops["LDS"], ops["SHFL"], ops["LDG"]))
        print("   ", " ".join("%s:%d/%d" % (o, c, st[o]) for o, c in ops.most_common(14)))
        if dump and ops["DFMA"] > 100 and ops["MUFU"] == 2:
            with open(dump, "w") as f:
                for a, t, w in body:
                    f.write("%05x s%2d %s wb%d wait%02x  %s\n" % (a, (w >> 41) & 0xf, "y" if (w >> 45) & 1 else " ", (w >> 46) & 7, (w >> 52) & 0x3f, t))


main()
