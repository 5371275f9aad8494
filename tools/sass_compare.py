#!/usr/bin/env python
"""Compare the SASS of two builds of libsbce.so function by function.

    python tools/sass_compare.py OLD.so NEW.so

Every function of OLD must exist in NEW (names demangled and normalised: see normalise) with the same instruction
listing: instruction text and encoding, addresses dropped.  Functions only in NEW are listed as added.  Exit code 0
when nothing of OLD changed.  Needs cuobjdump and cu++filt from the CUDA toolkit; no device."""
import os
import re
import shutil
import subprocess
import sys

CUDA_BIN = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin")


def tool(name):
    return shutil.which(name) or os.path.join(CUDA_BIN, name)


def functions(lib):
    """{demangled name: [instruction lines]} of every kernel in `lib`."""
    txt = subprocess.run([tool("cuobjdump"), "-sass", lib], capture_output=True, text=True, check=True).stdout
    funcs, cur = {}, None
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
            continue
        if cur is None:
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*)$", line)   # instruction: drop the address
        if m:
            funcs[cur].append(m.group(1).strip())
        elif re.match(r"\s*/\* 0x[0-9a-f]+ \*/\s*$", line):    # second half of the encoding
            funcs[cur].append(line.strip())
    names = subprocess.run([tool("cu++filt")], input="\n".join(funcs), capture_output=True, text=True,
                           check=True).stdout.splitlines()
    return {normalise(n): funcs[k] for n, k in zip(names, funcs)}


def normalise(name):
    """Kernel name without its parameter list, whitespace collapsed; an empty template parameter pack (which cu++filt
    prints as a trailing ", >" and which adds an empty pack to the parameter list) leaves no trace."""
    name = re.sub(r"\s+", " ", name.strip())
    name = re.sub(r"\((?:[^()]|\([^()]*\))*\)$", "", name)   # the trailing (balanced) parameter list
    return name.replace(", >", ">")


def main():
    old, new = functions(sys.argv[1]), functions(sys.argv[2])
    changed = [n for n in old if n in new and old[n] != new[n]]
    missing = [n for n in old if n not in new]
    added = sorted(n for n in new if n not in old)
    for n in missing:
        print("MISSING  %s" % n)
    for n in changed:
        print("CHANGED  %s (%d -> %d lines)" % (n, len(old[n]), len(new[n])))
    for n in added:
        print("added    %s (%d lines)" % (n, len(new[n])))
    same = len(old) - len(changed) - len(missing)
    print("%d of %d functions identical, %d changed, %d missing, %d added" % (same, len(old), len(changed),
                                                                             len(missing), len(added)))
    return 1 if changed or missing else 0


if __name__ == "__main__":
    sys.exit(main())
