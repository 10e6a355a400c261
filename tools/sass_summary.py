"""Static SASS summary of the hot kernels (no GPU needed): opcode histogram and instructions per source line.

usage: python tools/sass_summary.py [kernel-substring ...]   (default: the bench frame's k_shade / k_traverse instantiations)
Reads raytracer-server_b200/librtb200.so through cuobjdump / nvdisasm (-lineinfo build).  Counts are STATIC (every
instruction of the kernel once): the loop bodies of k_shade / k_traverse are straight-line code executed once per trip /
node step, so the per-line table is the cost model ncu's executed-instruction counts are checked against.
"""
import collections, os, re, subprocess, sys, tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "raytracer-server_b200", "librtb200.so")
KERNELS = sys.argv[1:] or ["k_shadeILi1ELi5ELi1ELb1ELi160", "k_traverseILb0E"]


def disassemble():
    d = tempfile.mkdtemp()
    subprocess.run(["cuobjdump", "-xelf", "all", LIB], cwd=d, check=True, capture_output=True)
    cubin = [f for f in os.listdir(d) if f.startswith("engine")][0]
    return subprocess.run(["nvdisasm", "-g", "-c", os.path.join(d, cubin)], check=True, capture_output=True, text=True).stdout


def main():
    asm = disassemble()
    for kern in KERNELS:
        ops, lines, total = collections.Counter(), collections.Counter(), 0
        infunc, cur = False, None
        for l in asm.splitlines():
            if l.startswith(".text.") or l.lstrip().startswith(".section\t.text."):
                infunc = kern in l
                continue
            if not infunc:
                continue
            m = re.search(r'//## File "([^"]+)", line (\d+)', l)
            if m:
                cur = (os.path.basename(m.group(1)), int(m.group(2)))
                continue
            m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", l)
            if m:
                op = m.group(1)
                base = op.split(".")[0]
                key = base
                if base in ("LDG", "STG", "LDS", "STS", "ATOMG", "RED", "LDGSTS", "MUFU", "LDL", "STL"):
                    key = ".".join(op.split(".")[:4]) if base in ("LDG", "RED", "ATOMG") else ".".join(op.split(".")[:2])
                ops[key] += 1
                lines[cur] += 1
                total += 1
        print(f"== {kern}: {total} SASS instructions")
        groups = collections.Counter()
        for k, v in ops.items():
            b = k.split(".")[0]
            g = ("fp32 fma/mul/add" if b in ("FFMA", "FMUL", "FADD", "FFMA2", "FMUL2", "FADD2") else
                 "fp32 min/max/cmp/select" if b in ("FMNMX", "FSETP", "FSEL", "FSET", "FCHK", "FMNMX3") else
                 "sfu (MUFU)" if b == "MUFU" else
                 "integer / logic / shift / permute" if b in ("IMAD", "IADD3", "IADD", "LOP3", "SHF", "PRMT", "LEA", "ISETP", "SEL", "IMNMX", "POPC", "FLO", "BREV", "I2F", "F2I", "I2FP", "F2FP", "VIADD", "VIMNMX", "IABS", "LOP", "UIADD3", "ULOP3", "UIMAD", "USHF", "ULEA", "UMOV", "USEL", "UISETP", "R2UR", "S2UR", "UPRMT", "UFLO", "UPOPC", "VIADDMNMX", "IMAD_WIDE") else
                 "memory" if b in ("LDG", "STG", "LDS", "STS", "ATOMG", "RED", "LDGSTS", "LDC", "LDCU", "LDL", "STL", "ATOMS", "LDSM", "CCTL", "MEMBAR", "LDGDEPBAR", "DEPBAR", "ERRBAR") else
                 "move" if b in ("MOV", "MOV64IUR", "CS2R", "S2R", "R2P", "P2R") else
                 "warp / control" if b in ("BRA", "BSSY", "BSYNC", "EXIT", "VOTE", "VOTEU", "SHFL", "BAR", "WARPSYNC", "MATCH", "NOP", "CALL", "RET", "BMOV", "BREAK", "PLOP3", "YIELD", "NANOSLEEP", "ELECT", "ENDCOLLECTIVE", "BPT", "REDUX", "CREDUX") else "other")
            groups[g] += v
        for g, v in groups.most_common():
            print(f"   {g:36s} {v:6d}  {100.0 * v / total:5.1f} %")
        print("   opcodes: " + "  ".join(f"{k} {v}" for k, v in ops.most_common(40)))
        print("   source lines with the most instructions:")
        for (f, ln), v in lines.most_common(28):
            print(f"      {f}:{ln:<5d} {v:5d}  {100.0 * v / total:4.1f} %")


if __name__ == "__main__":
    main()
