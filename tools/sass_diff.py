"""Compares the device code of two builds of libpioran_b200.so kernel by kernel.

`cuobjdump -sass` of each library is split at every `Function :` header.  A change to host code only must leave the set of
kernels and each kernel's SASS identical; the order of the kernels in the cubin may differ, so the whole dump is not compared.
Exit status 0 when every kernel matches.

    python tools/sass_diff.py OLD/libpioran_b200.so pioran.jl_b200/libpioran_b200.so
"""
import os
import shutil
import subprocess
import sys


def kernels(lib):
    exe = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    dump = subprocess.run([exe, "-sass", lib], check=True, capture_output=True, text=True).stdout
    out, name, body = {}, None, []
    for line in dump.splitlines():
        s = line.strip()
        if s.startswith("Function :"):
            name, body = s.split(":", 1)[1].strip(), []
            if name in out:
                raise SystemExit(f"{lib}: kernel {name} appears twice")
        elif name is not None and s and set(s) == {"."}:     # the dotted line that ends a function
            out[name] = "\n".join(body)
            name = None
        elif name is not None:
            body.append(line)
    return out


def main(old, new):
    a, b = kernels(old), kernels(new)
    only_old, only_new = sorted(set(a) - set(b)), sorted(set(b) - set(a))
    differ = sorted(k for k in set(a) & set(b) if a[k] != b[k])
    print(f"{os.path.basename(old)}: {len(a)} kernels; {os.path.basename(new)}: {len(b)} kernels")
    for label, names in (("only in the first", only_old), ("only in the second", only_new), ("different SASS", differ)):
        for k in names:
            print(f"{label}: {k}")
    ok = not (only_old or only_new or differ)
    print("identical" if ok else "DIFFERENT")
    return 0 if ok else 1


if __name__ == "__main__":
    if len(sys.argv) != 3:
        raise SystemExit(__doc__)
    sys.exit(main(sys.argv[1], sys.argv[2]))
