#!/usr/bin/env python
"""Static SASS of one k_scan instance, attributed to the kernel's source regions, and registers / spills of every instance:

    python profiles/scan_sass_regions.py [--instance 2,1,1,3,1] [--cubin metric.cubin] [--source hdp_b200/csrc/metric.cu]
                                         [--list REGION]

Without --cubin the source is compiled for sm_100a with the library's own nvcc flags (hdp_b200/build.py) plus -Xptxas -v into a
temporary directory (about a minute).  Each SASS instruction is attributed to the innermost source line of its
`nvdisasm -gi` annotation that lies in k_scan itself (an inlined helper counts where k_scan calls it); source lines map to regions by the lambdas of k_scan they sit in:
    flush     the season flush (`auto flush`)
    account   the accounting of a labelled run (`auto account` and its `spread`)
    phase_A   word extraction and the run filter (`auto extract_word`, `next_word`, `extract`)
    phase_B   the season loop from `---- phase B state ----` to the end of the kernel (queue pops, run decode, state machines)
    other     everything else (prologue, tables)
Per region: all instructions, and those of the integer ALU pipe (logic, shifts, compares, selects, byte permutes, min/max and the
three-input add) against those the FMA pipe can take (IMAD*, float add / multiply)."""
import argparse, collections, os, re, subprocess, sys, tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ALU = {"LOP3", "LOP", "SHF", "SHL", "SHR", "ISETP", "FSETP", "IADD3", "PRMT", "SEL", "FSEL", "VIMNMX", "IMNMX", "IABS", "PLOP3",
       "LEA", "BMSK", "SGXT", "P2R", "R2P", "FMNMX", "VIADD", "IADD"}
FMA = {"IMAD", "FADD", "FMUL", "FFMA", "IMUL"}


def regions_of(src):
    """line number -> region, from the lambda definitions inside k_scan"""
    lines = open(src).read().split("\n")
    start = next(i for i, l in enumerate(lines) if re.match(r"k_scan\(", l))
    end = next(i for i in range(start, len(lines)) if lines[i] == "}")
    reg = {}
    names = {"flush": "flush", "account": "account", "spread": "account", "extract_word": "phase_A", "next_word": "phase_A",
             "extract": "phase_A"}
    i = start
    while i < end:
        m = re.match(r"(\s*)auto (\w+) = \[", lines[i])
        if m and m.group(2) in names:
            close = m.group(1) + "};"
            j = next(k for k in range(i + 1, end) if lines[k] == close)
            for k in range(i, j + 1):
                reg[k + 1] = names[m.group(2)]
            i = j + 1
            continue
        i += 1
    b0 = next(i for i in range(start, end) if "---- phase B state ----" in lines[i])
    for k in range(b0, end + 1):
        reg.setdefault(k + 1, "phase_B")
    return reg, range(start + 1, end + 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--instance", default="2,1,1,3,1", help="NG,KS,kBytes,LMIN,BMAX")
    ap.add_argument("--cubin")
    ap.add_argument("--source", default=os.path.join(ROOT, "hdp_b200", "csrc", "metric.cu"))
    ap.add_argument("--list", metavar="REGION", help="also print the region's instructions with their source lines")
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    from hdp_b200 import build as b
    nvdis = os.path.join(os.path.dirname(b.nvcc()), "nvdisasm")
    tmp = tempfile.mkdtemp(prefix="scan_sass_")
    cubin = args.cubin
    if cubin is None:
        cubin = os.path.join(tmp, "metric.cubin")
        flags = [f for f in b.NVCC_FLAGS if not f.startswith("-Xcompiler") and not f.startswith("-fPIC")]
        r = subprocess.run([b.nvcc(), *flags, "-Xptxas=-v", "-I", os.path.join(ROOT, "include"), "-I", os.path.dirname(args.source),
                            "-cubin", "-o", cubin, args.source], capture_output=True, text=True)
        if r.returncode != 0:
            sys.exit(r.stdout + r.stderr)
        print("k_scan<NG,KS,kBytes,LMIN,BMAX>  registers  spill stores / loads (bytes)")
        cur = None
        for line in r.stderr.split("\n"):
            m = re.search(r"Compiling entry function '_ZN3hdp6k_scanILi(\d+)ELi(\d+)ELb([01])ELi(\d+)ELi(\d+)E", line)
            if m:
                cur = "<%s>" % ",".join(m.groups())
                spill = ""
            elif cur and "spill stores" in line:
                s = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
                spill = "%s / %s" % s.groups()
            elif cur and "Used" in line:
                print("  %-16s %4s  %s" % (cur, re.search(r"Used (\d+) registers", line).group(1), spill))
                cur = None
    ng, ks, by, lm, bm = args.instance.split(",")
    mangled = "_ZN3hdp6k_scanILi%sELi%sELb%sELi%sELi%sEEEv" % (ng, ks, by, lm, bm)
    syms = subprocess.run(["readelf", "-sW", cubin], capture_output=True, text=True).stdout
    idx = next(l.split(":")[0].strip() for l in syms.split("\n") if " FUNC " in l and l.split()[-1].startswith(mangled))
    sass = subprocess.run([nvdis, "-gi", "-c", "-fun", idx, cubin], capture_output=True, text=True, check=True).stdout
    reg, k_lines = regions_of(args.source)
    src_name = os.path.basename(args.source)
    total, alu, fma = collections.Counter(), collections.Counter(), collections.Counter()
    chain, fresh, line = [], True, None
    for l in sass.split("\n"):
        m = re.search(r'//## File "([^"]+)", line (\d+)', l)
        if m:
            if fresh:
                chain, fresh = [], False
            chain.append((os.path.basename(m.group(1)), int(m.group(2))))
            continue
        m = re.match(r"\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\w+\s+)?([A-Z][A-Z0-9_]*)", l)
        if not m:
            continue
        if not fresh:
            # innermost to outermost: the first location inside k_scan (helpers such as lds_u32 count where they are called)
            line = next((n for f, n in chain if f == src_name and n in k_lines), None)
            fresh = True
        r = reg.get(line, "other") if line is not None else "other"
        op = m.group(1)
        if r == args.list:
            print(line, l.strip())
        total[r] += 1
        alu[r] += op in ALU
        fma[r] += op in FMA
    print("k_scan<%s>: %d static instructions" % (args.instance, sum(total.values())))
    print("  %-8s %6s %6s %6s" % ("region", "all", "ALU", "FMA"))
    for r in ("flush", "account", "phase_A", "phase_B", "other"):
        print("  %-8s %6d %6d %6d" % (r, total[r], alu[r], fma[r]))


if __name__ == "__main__":
    main()
