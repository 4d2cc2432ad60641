#!/usr/bin/env python3
"""Fingerprint every device function of a CUDA library, or compare the functions of two builds.

A function's fingerprint is the SHA-256 of its SASS instruction lines (text and encoding, `cuobjdump -sass`) and of its
REG / SHARED / LOCAL / STACK usage (`cuobjdump -res-usage`).  Two builds whose fingerprints agree run the same device code.

    python tools/sass_fingerprint.py LIB              one line per function: fingerprint, mangled name
    python tools/sass_fingerprint.py OLD NEW          same-name functions whose fingerprint differs, and every function
                                                      present in one build only, matched by fingerprint to the other's
Exits 1 when the comparison finds a changed function or one without a counterpart.
"""
import hashlib
import re
import shutil
import subprocess
import sys

CUOBJDUMP = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"


def fingerprints(lib):
    sass = subprocess.run([CUOBJDUMP, "-sass", lib], check=True, capture_output=True, text=True).stdout
    res = subprocess.run([CUOBJDUMP, "-res-usage", lib], check=True, capture_output=True, text=True).stdout
    usage = dict(re.findall(r"Function (\S+):\n\s*(.*)", res))
    code, name = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            code[name] = []
        elif name and line.lstrip().startswith("/*"):
            code[name].append(line.strip())
    out = {}
    for name, lines in code.items():
        u = " ".join(re.findall(r"(?:REG|SHARED|LOCAL|STACK):\d+", usage.get(name, "")))
        out[name] = hashlib.sha256("\n".join(lines + [u]).encode()).hexdigest()[:16]
    return out


def demangle(names):
    filt = shutil.which("c++filt")
    if not filt or not names:
        return {n: n for n in names}
    r = subprocess.run([filt], input="\n".join(names), capture_output=True, text=True)
    return dict(zip(names, r.stdout.splitlines()))


def main(argv):
    if len(argv) == 1:
        for name, h in sorted(fingerprints(argv[0]).items()):
            print(h, name)
        return 0
    old, new = fingerprints(argv[0]), fingerprints(argv[1])
    print(f"# first build: {len(old)} functions, second build: {len(new)} functions")
    common = sorted(set(old) & set(new))
    changed = [n for n in common if old[n] != new[n]]
    print(f"# same name: {len(common)}, fingerprint differs: {len(changed)}")
    for n in changed:
        print(f"CHANGED {old[n]} -> {new[n]} {n}")
    only_old, only_new = sorted(set(old) - set(new)), sorted(set(new) - set(old))
    by_hash_new = {}
    for n in only_new:
        by_hash_new.setdefault(new[n], []).append(n)
    hashes_old = {old[n] for n in only_old}
    dm = demangle(only_old + only_new)
    unmatched = 0
    print(f"# only in the first build: {len(only_old)}, only in the second: {len(only_new)}")
    for n in only_old:
        match = by_hash_new.get(old[n], [])
        unmatched += not match
        print(f"{'RENAMED' if match else 'REMOVED'} {old[n]} {dm[n]}" + "".join(f"\n    -> {dm[m]}" for m in match))
    for n in only_new:
        if new[n] not in hashes_old:
            unmatched += 1
            print(f"ADDED {new[n]} {dm[n]}")
    print(f"# result: {'identical device code' if not changed and not unmatched else 'DIFFERENT'}"
          f" ({len(changed)} changed, {unmatched} without a counterpart)")
    return 1 if changed or unmatched else 0


if __name__ == "__main__":
    if len(sys.argv) not in (2, 3):
        sys.exit(__doc__)
    sys.exit(main(sys.argv[1:]))
