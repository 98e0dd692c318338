#!/usr/bin/env python
"""Compare the machine code of two builds of the library, function by function.  A change that must leave the
generated code alone (a refactor, a new kernel next to untouched ones) is checked with it.

Usage: python profiles/sass_diff.py OLD.so NEW.so

Both libraries are disassembled with cuobjdump; instruction addresses and encodings are dropped, and the
anonymous-namespace tag of mangled names (a hash of the file contents) is replaced by the plain one.  For every
function the instruction sequence and the resource usage (registers, stack, shared and local memory: spills show
as stack / local) are compared.  Prints the functions that differ and exits non-zero if any does."""
import difflib
import re
import subprocess
import sys

ANON = re.compile(r"\d+_GLOBAL__N__[0-9a-f]+_\d+_\w+?_cu_[0-9a-f]{8}")
INSTR = re.compile(r"^\s+/\*[0-9a-f]+\*/\s+(.*?)\s*/\*\s*0x[0-9a-f]+\s*\*/\s*$")


def cuobjdump(flag, lib):
    out = subprocess.run(["cuobjdump", flag, lib], capture_output=True, text=True, check=True).stdout
    return ANON.sub("12_GLOBAL__N_1", out)


def functions(lib):
    """mangled name -> [resource line, instructions]"""
    funcs, cur = {}, None
    for ln in cuobjdump("-sass", lib).splitlines():
        m = re.search(r"Function : (\S+)", ln)
        if m:
            cur = funcs.setdefault(m.group(1), ["", []])[1]
        elif cur is not None and (m := INSTR.match(ln)):
            cur.append(m.group(1))
    name = None
    for ln in cuobjdump("-res-usage", lib).splitlines():
        m = re.match(r"\s*Function (\S+):$", ln)
        if m:
            name = m.group(1)
        elif name in funcs and "REG:" in ln:
            funcs[name][0] = ln.strip()
    return funcs


old, new = functions(sys.argv[1]), functions(sys.argv[2])
names = sorted(set(old) | set(new))
demangled = dict(zip(names, subprocess.run(["c++filt"], input="\n".join(names), capture_output=True,
                                           text=True).stdout.splitlines()))
bad = 0
for n in names:
    label = demangled.get(n, n).replace("(anonymous namespace)::", "").split("(")[0]
    if n not in old or n not in new:
        print(f"{label}: only in {'new' if n in new else 'old'}")
        bad += 1
        continue
    (ra, a), (rb, b) = old[n], new[n]
    if a != b:
        same = sum(blk.size for blk in difflib.SequenceMatcher(None, a, b, autojunk=False).get_matching_blocks())
        print(f"{label}: {len(a)} -> {len(b)} instructions, {max(len(a), len(b)) - same} changed")
    if ra != rb:
        print(f"{label}: {ra} -> {rb}")
    bad += a != b or ra != rb
print(f"{len(names)} functions, {len(names) - bad} identical")
sys.exit(1 if bad else 0)
