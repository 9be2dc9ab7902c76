"""Compares the SASS of two builds of libpn12_b200.so kernel by kernel.

    python tools/sass_diff.py OLD.so NEW.so

For every kernel it compares the instruction stream (addresses, encodings and branch-target addresses removed, branch
labels renumbered in order of appearance) and the register / shared / stack / local usage.  It lists the kernels that
differ or exist in one build only and exits with 1 if there are any: a refactor of device code that claims to change
nothing can be checked without a GPU.
"""
from __future__ import annotations

import re
import subprocess
import sys

FUNC = re.compile(r"^\s*Function\s*:?\s*(\S+?):?\s*$")
INSN = re.compile(r"^\s*/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;")
TARGET = re.compile(r"\b(BRA|BRX|JMP|JMX|CALL|BSSY|SSY|PBK|PCNT)\b(.*?)(0x[0-9a-f]+|\.L_x_\d+)")
RES = re.compile(r"\b(REG|STACK|SHARED|LOCAL):(\d+)")


def cuobjdump(lib: str, flag: str) -> str:
    return subprocess.run(["cuobjdump", flag, lib], check=True, capture_output=True, text=True).stdout


def kernels(lib: str) -> dict[str, tuple[list[str], str]]:
    sass: dict[str, list[str]] = {}
    name = None
    for line in cuobjdump(lib, "-sass").splitlines():
        if m := FUNC.match(line):
            name = m.group(1)
            sass[name] = []
        elif name and (m := INSN.match(line)):
            sass[name].append(m.group(1))
    usage: dict[str, str] = {}
    name = None
    for line in cuobjdump(lib, "-res-usage").splitlines():
        if m := FUNC.match(line):
            name = m.group(1)
        elif name and RES.search(line):
            usage[name] = " ".join(f"{k}:{v}" for k, v in RES.findall(line))
            name = None
    return {k: (normalise(v), usage.get(k, "")) for k, v in sass.items()}


def normalise(insns: list[str]) -> list[str]:
    labels: dict[str, str] = {}

    def relabel(m: re.Match) -> str:
        return m.group(1) + m.group(2) + labels.setdefault(m.group(3), f"L{len(labels)}")
    return [re.sub(r"\s+", " ", TARGET.sub(relabel, i)) for i in insns]


def main(old_lib: str, new_lib: str) -> int:
    old, new = kernels(old_lib), kernels(new_lib)
    bad = []
    for name in sorted(old.keys() | new.keys()):
        if name not in old or name not in new:
            bad.append(f"only in {'old' if name in old else 'new'}: {name}")
            continue
        (a, a_use), (b, b_use) = old[name], new[name]
        if a_use != b_use:
            bad.append(f"resource usage differs: {name}: {a_use} -> {b_use}")
        if a != b:
            first = next((i for i, (x, y) in enumerate(zip(a, b)) if x != y), min(len(a), len(b)))
            bad.append(f"instructions differ: {name}: {len(a)} -> {len(b)} instructions, first difference at instruction {first}")
    for line in bad:
        print(line)
    same = sum(old[name] == new[name] for name in old.keys() & new.keys())
    print(f"{same} of {len(old.keys() | new.keys())} kernels identical")
    return 1 if bad else 0


if __name__ == "__main__":
    if len(sys.argv) != 3:
        sys.exit(__doc__)
    sys.exit(main(sys.argv[1], sys.argv[2]))
