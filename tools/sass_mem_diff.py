#!/usr/bin/env python
"""Compare two builds of one object file kernel by kernel (runs without a GPU):

    python tools/sass_mem_diff.py OLD.o NEW.o

Per kernel: registers (`cuobjdump -res-usage`), the total SASS instruction count, and the multiset of memory
instructions of `cuobjdump -sass`: every LDG*, STG*, RED* and ATOM* opcode with its modifiers and width (e.g.
LDG.E.128.CONSTANT, STG.E.U16).  Generic (LD / ST) and local (LDL / STL) accesses are counted too, so a parameter
read through a generic pointer or a spill shows up.  Constant-bank loads (LDC / LDCU) are left out: they move between
uniform and ordinary registers when the compiler re-allocates and are not memory traffic.

A refactor that keeps every kernel's memory traffic shows `memory same` for every kernel present in both builds.
Exit code 1 when a common kernel's memory multiset differs or it uses more registers.
"""
import collections
import re
import subprocess
import sys

MEM = re.compile(r"^(LDG|STG|REDG?|ATOMG?|LDL|STL|LD|ST)(\.|$)")


def cuobjdump(flag, obj):
    return subprocess.run(["cuobjdump", flag, obj], capture_output=True, text=True, check=True).stdout


def kernels(obj):
    """{mangled name: [Counter of memory opcodes, total instruction count, registers]}"""
    res, name = {}, None
    for line in cuobjdump("-sass", obj).splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            res[name] = [collections.Counter(), 0, 0]
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P[T0-9]+\s+)?([A-Z][A-Z0-9_.]*)", line)
        if name and m:
            if MEM.match(m.group(1)):
                res[name][0][m.group(1)] += 1
            res[name][1] += 1
    for fn, reg in re.findall(r"Function (\S+):\s*\n\s*REG:(\d+)", cuobjdump("-res-usage", obj)):
        res[fn][2] = int(reg)
    return res


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.split("\n")
    return [o.replace("void ", "").replace("mscs::", "") for o in out]


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    names = sorted(set(old) | set(new))
    bad = 0
    for name, pretty in zip(names, demangle(names)):
        if name not in new:
            print(f"{pretty}: removed ({old[name][1]} instructions)")
            continue
        if name not in old:
            print(f"{pretty}: new ({new[name][1]} instructions, {new[name][2]} registers)")
            continue
        (mo, to, ro), (mn, tn, rn) = old[name], new[name]
        same = mo == mn
        bad += not same or rn > ro
        print(f"{pretty}: registers {ro} -> {rn}, instructions {to} -> {tn}, memory {'same' if same else 'DIFFERENT'}")
        for op in sorted(set(mo) | set(mn)):
            print(f"    {op:28s} {mo[op]:4d} {mn[op]:4d}{'' if mo[op] == mn[op] else '   <--'}")
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
