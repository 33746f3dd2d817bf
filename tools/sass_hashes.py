"""Hash the SASS of every kernel of a built library, per mangled name, and compare two builds.

    python tools/sass_hashes.py LIB.so [--out hashes.json]
    python tools/sass_hashes.py NEW.so --against OLD.so      (or --against old_hashes.json)

A change that adds a value type or refactors host code should leave every existing kernel's machine code as
it was: with --against, every kernel of the old build must be present in the new one with the same SASS
(`cuobjdump -sass`, hashed with SHA-256).  Prints the counts and every kernel that changed or disappeared;
exits 1 if there is one.  Needs cuobjdump (CUDA toolkit), no GPU.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import re
import shutil
import subprocess
import sys

_FUNC = re.compile(r"^\s*Function : (\S+)\s*$")
_INSN = re.compile(r"^\s*/\*[0-9a-f]{4,}\*/|^\s*/\* 0x[0-9a-f]+ \*/")   # instruction and encoding lines
# anonymous namespaces are mangled with a hash of the file's contents: keep the file name only
_ANON = re.compile(r"_GLOBAL__N__[0-9a-f]+_\d+_(\w+?)_[0-9a-f]+(?=\d)")


def cuobjdump() -> str:
    for cand in (shutil.which("cuobjdump"), "/usr/local/cuda/bin/cuobjdump"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("cuobjdump not found")


def kernel_hashes(lib: str) -> dict[str, str]:
    out = subprocess.run([cuobjdump(), "-sass", lib], capture_output=True, text=True, check=True).stdout
    hashes: dict[str, str] = {}
    name, body = None, []

    def flush():
        if name is not None:
            h = hashlib.sha256("\n".join(body).encode()).hexdigest()
            if name in hashes and hashes[name] != h:   # (one kernel in two translation units with different code)
                h = hashes[name] + "|" + h
            hashes[name] = h

    for line in out.splitlines():
        m = _FUNC.match(line)
        if m:
            flush()
            name, body = _ANON.sub(r"_GLOBAL__N_\1_", m.group(1)), []
        elif name is not None and _INSN.match(line):
            body.append(" ".join(line.split()))   # (column padding follows the longest line of the module)
    flush()
    return hashes


def load(path: str) -> dict[str, str]:
    if path.endswith(".json"):
        with open(path) as f:
            return json.load(f)
    return kernel_hashes(path)


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("lib")
    ap.add_argument("--against", help="older build (.so) or its hashes (.json)")
    ap.add_argument("--out", help="write the hashes of LIB as JSON")
    a = ap.parse_args()
    new = load(a.lib)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(new, f, indent=1, sort_keys=True)
    if not a.against:
        print(f"{len(new)} kernels")
        return 0
    old = load(a.against)
    missing = sorted(k for k in old if k not in new)
    changed = sorted(k for k in old if k in new and new[k] != old[k])
    added = sorted(k for k in new if k not in old)
    print(f"old {len(old)} kernels, new {len(new)}: {len(old) - len(missing) - len(changed)} identical, "
          f"{len(changed)} changed, {len(missing)} missing, {len(added)} added")
    for k in changed:
        print("changed:", k)
    for k in missing:
        print("missing:", k)
    return 1 if (changed or missing) else 0


if __name__ == "__main__":
    sys.exit(main())
