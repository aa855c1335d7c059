#!/usr/bin/env python3
"""Check that every kernel of an older build of libookd_gpu compiles to the same SASS in a newer one.

    python tools/sass_diff.py --rev HEAD~1                 # builds that revision's csrc/ in a temporary directory
    python tools/sass_diff.py OLD.o [NEW.o]                # NEW defaults to ookiedokie_b200/lib/ookd_gpu.o

A change that adds template parameters (e.g. the input format) renames the old instantiations, so kernels are matched
by their instructions: each old kernel's SASS (addresses and encodings stripped) must be the body of some new kernel,
preferably one with the same base name.  Prints one line per old kernel and exits 1 if any of them changed.
Needs cuobjdump (CUDA toolkit) and, with --rev, git, make and nvcc; no GPU.
"""
import argparse
import hashlib
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def cuobjdump():
    for c in ("cuobjdump", "/usr/local/cuda/bin/cuobjdump"):
        try:
            subprocess.run([c, "--version"], check=True, capture_output=True)
            return c
        except (OSError, subprocess.CalledProcessError):
            pass
    sys.exit("cuobjdump not found")


def kernels(path):
    """{mangled name: normalised SASS text} of every function in an object or shared library."""
    out = subprocess.run([cuobjdump(), "-sass", path], check=True, capture_output=True, text=True).stdout
    funcs, name, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                funcs[name] = "\n".join(body)
            name, body = m.group(1), []
            continue
        if name is None:
            continue
        ins = re.sub(r"/\*\s*[0-9a-fx]+\s*\*/", "", line)      # address column and encoding words
        ins = ins.strip()
        if ins and not ins.startswith(".") and not ins.startswith("Fatbin") and not ins.startswith("code for"):
            body.append(ins)
    if name:
        funcs[name] = "\n".join(body)
    return funcs


def demangle(names):
    try:
        r = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True)
        return dict(zip(names, r.stdout.splitlines()))
    except (OSError, subprocess.CalledProcessError):
        return {n: n for n in names}


def base_name(demangled):
    """Kernel name without return type, template arguments and parameters."""
    d = demangled[5:] if demangled.startswith("void ") else demangled
    return d.split("<")[0].split("(")[0]


def build_rev(rev, tmp):
    src = os.path.join(tmp, "src")
    os.makedirs(src)
    arch = subprocess.run(["git", "-C", ROOT, "archive", rev], check=True, capture_output=True).stdout
    subprocess.run(["tar", "-x", "-C", src], input=arch, check=True)
    # (the Makefile names its targets relative to csrc/)
    subprocess.run(["make", "-C", os.path.join(src, "ookiedokie_b200", "csrc"), "../lib/ookd_gpu.o"],
                   check=True, capture_output=True)
    return os.path.join(src, "ookiedokie_b200", "lib", "ookd_gpu.o")


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("old", nargs="?")
    ap.add_argument("new", nargs="?", default=os.path.join(ROOT, "ookiedokie_b200", "lib", "ookd_gpu.o"))
    ap.add_argument("--rev", help="git revision whose build is the old side")
    a = ap.parse_args()
    if not a.old and not a.rev:
        ap.error("give OLD or --rev")
    with tempfile.TemporaryDirectory() as tmp:
        old = kernels(build_rev(a.rev, tmp) if a.rev else a.old)
    new = kernels(a.new)
    by_body = {}
    for n, b in new.items():
        by_body.setdefault(hashlib.sha256(b.encode()).hexdigest(), []).append(n)
    dm = demangle(list(old) + list(new))
    bad = 0
    for n in sorted(old, key=lambda k: dm[k]):
        base = base_name(dm[n])
        hits = by_body.get(hashlib.sha256(old[n].encode()).hexdigest(), [])
        hits.sort(key=lambda k: base_name(dm[k]) != base)
        n_ins = old[n].count("\n") + 1
        if hits and base_name(dm[hits[0]]) == base:
            print(f"same     {n_ins:6d} instructions  {dm[n]}  ==  {dm[hits[0]]}")
        else:
            bad += 1
            print(f"CHANGED  {n_ins:6d} instructions  {dm[n]}")
    print(f"{len(old) - bad} of {len(old)} kernels of the old build unchanged; {len(new)} kernels in the new build")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
