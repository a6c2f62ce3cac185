"""Compares the SASS of every kernel of two builds of one csrc/*.cu file (instructions and encodings), instantiation by
instantiation.  Kernels are matched by name and template arguments, whatever their parameter lists; a kernel that
differs is listed with the opcodes whose counts differ.  Compiles both files with the library's flags for sm_100a;
needs nvcc, cuobjdump and cu++filt, no GPU.

    python profiles/tools/sass_compare.py OLD/csrc/FILE.cu [NEW/csrc/FILE.cu] [--prefix NAME]

NEW defaults to this repository's csrc/FILE.cu; --prefix keeps only the kernels whose name starts with NAME.
"""
import argparse
import collections
import os
import re
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, "probabilistic-self-update-line-vector-set-based-point-cloud-registration_b200", "csrc")
CUDA = "/usr/local/cuda/bin"
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-fmad=false", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler",
         "-fPIC"]


def kernel_key(mangled):
    """gnc_tls_kernel<(int)8, (int)512, (int)1>: the unqualified name and its template arguments, no parameters."""
    name = subprocess.run([os.path.join(CUDA, "cu++filt"), "-p", mangled], capture_output=True, text=True,
                          check=True).stdout.strip()
    return re.sub(r"^(?:\w+::|<unnamed>::)*", "", name)


def kernels(src, tmp, prefix):
    obj = os.path.join(tmp, f"{len(os.listdir(tmp))}.o")
    subprocess.check_call([os.path.join(CUDA, "nvcc"), *FLAGS, "-c", src, "-o", obj], cwd=os.path.dirname(src))
    sass = subprocess.run([os.path.join(CUDA, "cuobjdump"), "-sass", obj], capture_output=True, text=True,
                          check=True).stdout
    out, name = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = kernel_key(m.group(1))
            name = name if name.startswith(prefix) else None
            if name:
                out[name] = []
        elif name and re.search(r"/\*[0-9a-f]{4,}\*/|/\* 0x[0-9a-f]+ \*/", line):
            out[name].append(re.sub(r"\s+", " ", line.strip()))
    return out


def opcodes(lines):
    ops = collections.Counter()
    for line in lines:
        m = re.match(r"/\*[0-9a-f]{4,}\*/ (?:@!?U?P\w+ )?([A-Z][A-Z0-9_.]*)", line)
        if m:
            ops[m.group(1)] += 1
    return ops


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new", nargs="?")
    ap.add_argument("--prefix", default="")
    args = ap.parse_args()
    old = os.path.abspath(args.old)
    new = os.path.abspath(args.new) if args.new else os.path.join(CSRC, os.path.basename(old))
    with tempfile.TemporaryDirectory() as tmp:
        a, b = kernels(old, tmp, args.prefix), kernels(new, tmp, args.prefix)
    differ = 0
    for k in sorted(set(a) | set(b)):
        if k not in b:
            print(f"only in old  {k} ({len(a[k])} lines)")
        elif k not in a:
            print(f"only in new  {k} ({len(b[k])} lines)")
        elif a[k] == b[k]:
            print(f"identical    {k} ({len(a[k])} / {len(b[k])} lines)")
        else:
            differ += 1
            oa, ob = opcodes(a[k]), opcodes(b[k])
            delta = ", ".join(f"{op} {oa[op]} -> {ob[op]}" for op in sorted(set(oa) | set(ob)) if oa[op] != ob[op])
            print(f"DIFFERENT    {k} ({len(a[k])} / {len(b[k])} lines; {sum(oa.values())} / {sum(ob.values())} "
                  f"instructions; opcode counts: {delta or 'equal'})")
    sys.exit(1 if differ else 0)


if __name__ == "__main__":
    main()
