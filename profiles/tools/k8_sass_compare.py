"""Compares the SASS of every kernel of two builds of csrc/k8_features.cu (instructions and encodings), instantiation by
instantiation: a kernel that gained a template flag is matched with its flag false against the other build's kernel
without it.  Compiles both files with the library's flags for sm_100a; needs nvcc and cuobjdump, no GPU.

    python profiles/tools/k8_sass_compare.py OLD/csrc/k8_features.cu [NEW/csrc/k8_features.cu]
"""
import os
import re
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CUDA = "/usr/local/cuda/bin"
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "-fmad=false", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler",
         "-fPIC"]


def kernels(src, tmp):
    obj = os.path.join(tmp, f"{len(os.listdir(tmp))}.o")
    subprocess.check_call([os.path.join(CUDA, "nvcc"), *FLAGS, "-c", src, "-o", obj], cwd=os.path.dirname(src))
    sass = subprocess.run([os.path.join(CUDA, "cuobjdump"), "-sass", obj], capture_output=True, text=True,
                          check=True).stdout
    out, name = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            k = re.search(r"\d(k8_[a-z0-9_]+?)(I(?:Lb[01]E)+E|E)", m.group(1))
            # a trailing false flag (kCap = false) is the kernel as it was before the flag
            args = re.sub(r"(Lb[01]E)Lb0EE$", r"\1E", k.group(2))
            name = k.group(1) + args
            out[name] = []
        elif name and re.search(r"/\*[0-9a-f]{4}\*/|/\* 0x[0-9a-f]+ \*/", line):
            out[name].append(re.sub(r"\s+", " ", line.strip()))
    return out


def main():
    old = os.path.abspath(sys.argv[1])
    new = os.path.abspath(sys.argv[2]) if len(sys.argv) > 2 else os.path.join(
        ROOT, "probabilistic-self-update-line-vector-set-based-point-cloud-registration_b200", "csrc", "k8_features.cu")
    with tempfile.TemporaryDirectory() as tmp:
        a, b = kernels(old, tmp), kernels(new, tmp)
    differ = 0
    for k in sorted(set(a) | set(b)):
        if k not in b:
            print(f"only in old  {k}")
        elif k not in a:
            print(f"only in new  {k} ({len(b[k])} lines)")
        else:
            same = a[k] == b[k]
            differ += not same
            print(f"{'identical' if same else 'DIFFERENT'}    {k} ({len(a[k])} / {len(b[k])} lines)")
    sys.exit(1 if differ else 0)


if __name__ == "__main__":
    main()
