"""Static code size of one kernel by enclosing source function: SASS instructions per function / per source line (nvdisasm -g line
table of an object built with -lineinfo). The step kernel's instruction-cache footprint matters (ncu: sm__icc_request_hit_rate 84 %,
'no_instructions' 18 % of the stall samples at 1 Mi games), so this shows where the bytes are.

With --json OUT it also sorts every function's instructions by the pipe that executes them (PIPES below) and writes the counts: the
deep step kernel is bound by instruction issue with the ALU pipe on top (LOP3 / ISETP / SEL / SHF / PRMT / VIMNMX, 2 cycles per warp
instruction and SMSP) while the FMA pipe, which takes IMAD at the same rate, has room, so the ALU column is the one to shrink. The
counts are static (instructions in the binary, not executed ones).
Usage: python tools/sass_size_by_function.py hex_gym_env_b200/build/step_11.o _Z16hexb_step_kernelILi11ELi1ELb0EEvN4hexb6ParamsE
           [top_lines] [--json OUT]"""
import collections, glob, json, os, re, subprocess, sys, tempfile

# opcode (without modifiers) -> pipe. Integer and logic work other than IMAD / IMUL is the ALU pipe's; IMAD / IMUL / FP32 the FMA
# pipe's; opcodes with a leading U run on the per-warp uniform datapath; POPC / FLO / BREV and conversions share the XU-rate pipe.
ALU = {"LOP3", "LOP", "ISETP", "SEL", "SHF", "SHL", "SHR", "PRMT", "VIMNMX", "VIMNMX3", "IMNMX", "IADD3", "IADD", "VIADD", "VIADDMNMX",
       "LEA", "PLOP3", "IABS", "BMSK", "SGXT", "MOV", "P2R", "R2P", "FSEL", "FSETP", "CSET", "CSETP", "ICMP", "IDP", "VOTE"}
FMA = {"IMAD", "IMUL", "IMADSP", "FFMA", "FMUL", "FADD", "HFMA2", "HMUL2", "HADD2", "FMNMX", "FSWZADD"}
XU = {"POPC", "FLO", "BREV", "I2F", "F2I", "F2F", "I2I", "F2FP", "MUFU", "I2FP", "F2IP"}
FP64 = {"DFMA", "DMUL", "DADD", "DSETP", "DMNMX"}
LSU = {"LD", "LDS", "LDG", "LDL", "LDC", "ST", "STS", "STG", "STL", "ATOM", "ATOMS", "ATOMG", "RED", "REDG", "REDUX", "SHFL",
       "MATCH", "LDSM", "CCTL", "MEMBAR", "FENCE", "ERRBAR", "SYNCS", "UBLKCP", "UTMACMDFLUSH", "LDCU"}
BRANCH = {"BRA", "BRX", "JMP", "JMX", "CALL", "RET", "EXIT", "BSSY", "BSYNC", "BREAK", "BPT", "WARPSYNC", "BAR", "YIELD", "KILL",
          "NANOSLEEP", "ACQBULK", "ELECT"}
PIPES = ("alu", "fma", "xu", "fp64", "lsu", "uniform", "branch", "other")


def pipe_of(op):
    base = op.split(".")[0]
    if base in LSU:           # (LDCU and the bulk-copy opcodes start with U but go through the memory pipes)
        return "lsu"
    if base in ALU:
        return "alu"
    if base in FMA:
        return "fma"
    if base in XU:
        return "xu"
    if base in FP64:
        return "fp64"
    if base in BRANCH:
        return "branch"
    if base.startswith("U") or base in ("R2UR", "S2UR"):
        return "uniform"
    return "other"


def disassemble(obj):
    with tempfile.TemporaryDirectory() as tmp:   # the host object embeds the cubin
        subprocess.run(["cuobjdump", "-xelf", "all", os.path.abspath(obj)], cwd=tmp, check=True, stdout=subprocess.DEVNULL)
        cubin = sorted(glob.glob(os.path.join(tmp, "*.cubin")))[0]
        return subprocess.run(["nvdisasm", "-g", "-c", cubin], stdout=subprocess.PIPE, text=True, check=True).stdout.split("\n")


def kernel_lines(dis, kernel):
    """{(file, line): [opcode, ...]} of one kernel (NOPs, the alignment padding after the last instruction, are left out)"""
    start = next(i for i, l in enumerate(dis) if l.startswith(kernel + ":"))
    loc, byline = None, collections.defaultdict(list)
    for l in dis[start + 1:]:
        if l.startswith("//--------------------- "):
            break
        m = re.match(r'\s*//## File "([^"]+)", line (\d+)', l)
        if m:
            loc = (os.path.basename(m.group(1)), int(m.group(2)))
            continue
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?);", l)
        if m:
            op = re.sub(r"^@!?U?P[T0-9]+\s+", "", m.group(2)).split()[0]
            if op != "NOP":
                byline[loc].append(op)
    return byline


def main():
    args = sys.argv[1:]
    out = None
    if "--json" in args:
        i = args.index("--json")
        out = args[i + 1]
        del args[i:i + 2]
    obj, kernel = args[:2]
    top = int(args[2]) if len(args) > 2 else 25
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    srcdir = os.path.join(root, "hex_gym_env_b200", "csrc")
    byline = kernel_lines(disassemble(obj), kernel)
    src = {f: open(os.path.join(srcdir, f)).read().split("\n") for f in os.listdir(srcdir) if f.endswith((".cu", ".cuh", ".h"))}

    def func_of(f, ln):
        if f not in src:
            return f
        L = src[f]
        for i in range(ln - 1, -1, -1):
            if re.match(r"^(HEXB_HD|__device__|__global__|static)", L[i]) and "(" in L[i]:
                m = re.search(r"(\w+)\s*\(", re.sub(r"__launch_bounds__\([^)]*\)+", "", L[i]))
                return m.group(1) if m else L[i]
        return "?"

    fn = collections.Counter()
    fpipes = collections.defaultdict(collections.Counter)
    for (f, ln), ops in byline.items():
        name = func_of(f, ln) if f is not None else "?"
        fn[name] += len(ops)
        for op in ops:
            fpipes[name][pipe_of(op)] += 1
    tot = sum(fn.values())
    alu = sum(p["alu"] for p in fpipes.values())
    if out:
        total = collections.Counter()
        for p in fpipes.values():
            total.update(p)
        opcodes = collections.Counter(op.split(".")[0] for ops in byline.values() for op in ops)
        doc = {"kernel": kernel, "object": os.path.basename(obj), "instructions": tot, "bytes": 16 * tot,
               "pipes": {p: total[p] for p in PIPES},
               "functions": {k: dict({"instructions": c}, **{p: fpipes[k][p] for p in PIPES if fpipes[k][p]}) for k, c in fn.most_common()},
               "opcodes": dict(opcodes.most_common())}
        with open(out, "w") as fh:
            json.dump(doc, fh, indent=1)
            fh.write("\n")
    print("%s: %d SASS instructions = %.1f KB, %d on the ALU pipe" % (kernel, tot, tot * 16 / 1024.0, alu))
    print("%6s  %5s  %5s  %s" % ("instr", "share", "alu", "function"))
    for k, c in fn.most_common():
        print("%6d  %5.1f%%  %5d  %s" % (c, 100.0 * c / tot, fpipes[k]["alu"], k))
    print("-- top lines")
    for (f, ln), ops in sorted(byline.items(), key=lambda kv: -len(kv[1]))[:top]:
        text = src[f][ln - 1].strip()[:100] if f in src and ln <= len(src[f]) else ""
        print("%6d  %s:%s  %s" % (len(ops), f, ln, text))


if __name__ == "__main__":
    main()
