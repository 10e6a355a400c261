"""Registers, stack and spill bytes of every k_shade / k_traverse / k_generate instantiation (no GPU needed).

usage: python tools/shade_regs.py [engine.o]   (default: raytracer-server_b200/build/engine.o, as build.py leaves it)
REG and STACK come from `cuobjdump --dump-resource-usage`.  Spill bytes are the widths of the local-memory stores
(STL) and loads (LDL) in the kernel's SASS: for a kernel without a local array (STACK is then all spill area) this is
exactly what `ptxas -v` reports as spill stores / loads; k_traverse and the INLINE k_shade keep their traversal stack
in local memory, so their columns also count the stack's accesses.
"""
import os, re, shutil, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBJ = os.path.join(ROOT, "raytracer-server_b200", "build", "engine.o")
KERNELS = ("k_shade<", "k_traverse<", "k_generate<")
CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
WIDTH = {"U8": 1, "S8": 1, "U16": 2, "S16": 2, "64": 8, "128": 16}


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    return dict(zip(names, out.splitlines()))


def resource_usage(obj):
    text = subprocess.run([CUOBJDUMP, "--dump-resource-usage", obj], capture_output=True, text=True, check=True).stdout
    usage, fn = {}, None
    for line in text.splitlines():
        m = re.match(r"\s*Function (\S+):", line)
        if m:
            fn = m.group(1)
            continue
        m = re.search(r"REG:(\d+) STACK:(\d+)", line)
        if m and fn:
            usage[fn] = (int(m.group(1)), int(m.group(2)))
            fn = None
    return usage


def local_bytes(obj):
    text = subprocess.run([CUOBJDUMP, "-sass", obj], capture_output=True, text=True, check=True).stdout
    acc, fn = {}, None
    for line in text.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            fn = m.group(1)
            acc[fn] = [0, 0]
            continue
        m = re.search(r"\b(STL|LDL)((?:\.\w+)*)\s", line)
        if m and fn:
            w = next((WIDTH[s] for s in m.group(2).split(".") if s in WIDTH), 4)
            acc[fn][0 if m.group(1) == "STL" else 1] += w
    return acc


def table(obj=OBJ):
    """[(kernel, registers, stack bytes, spill store bytes, spill load bytes)], sorted by kernel"""
    usage, spills = resource_usage(obj), local_bytes(obj)
    names = demangle(list(usage))
    rows = []
    for fn, (reg, stack) in usage.items():
        name = names[fn].replace("rtb::", "").removeprefix("void ").split("(")[0]
        if name.startswith(KERNELS):
            st, ld = spills.get(fn, (0, 0))
            rows.append((name, reg, stack, st, ld))
    return sorted(rows)


def main():
    rows = table(sys.argv[1] if len(sys.argv) > 1 else OBJ)
    w = max(len(r[0]) for r in rows)
    print(f"{'kernel':<{w}}  {'regs':>4}  {'stack':>5}  {'spill st':>8}  {'spill ld':>8}")
    for name, reg, stack, st, ld in rows:
        print(f"{name:<{w}}  {reg:>4}  {stack:>5}  {st:>8}  {ld:>8}")


if __name__ == "__main__":
    main()
