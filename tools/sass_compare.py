"""Compare the SASS of two builds of one CUDA source, kernel by kernel.

    python tools/sass_compare.py OLD.cu NEW.cu [--drop-template-arg false]

Compiles both files for sm_100a with the flags of pypevoc_b200/build.py (object files only),
disassembles them with cuobjdump -sass and compares every kernel present in both.  Kernel names are
matched after demangling, without their parameter lists; ``--drop-template-arg V`` first removes a
trailing template argument ``V`` from the NEW names, so that a kernel that gained a template flag
(``k<16, true, false>``) is matched with its old instantiation (``k<16, true>``), and ``k<false>``
with the untemplated ``k``.  Instruction lines that differ only in constant-bank offsets
(``c[0x0][0x...]``, where the kernel parameters live) are reported separately from real differences.
Exit status 1 when a matched kernel differs in anything else.
"""
import argparse
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from pypevoc_b200 import build  # noqa: E402

CBANK = re.compile(r"c\[0x0\]\[0x[0-9a-f]+\]")


def compile_sass(src, tmp, tag):
    obj = os.path.join(tmp, tag + ".o")
    flags = [f for f in build.NVCC_FLAGS if f != "-shared"]
    subprocess.check_call([build._nvcc()] + flags + ["-I", os.path.join(ROOT, "include"), "-I", build.CSRC, "-c",
                           src, "-o", obj])
    return subprocess.check_output(["cuobjdump", "-sass", obj], text=True)


def demangle(names):
    out = subprocess.run(["cu++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    return out.splitlines()


def kernels(sass):
    """{mangled name: [instruction text, without addresses and encodings]}"""
    funcs, cur = {}, None
    for line in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = funcs.setdefault(m.group(1), [])
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?)\s*;?\s*(/\*.*)?$", line)
        if cur is not None and m and m.group(1):
            cur.append(m.group(1))
    return funcs


def short_name(dem, drop=None):
    name = re.sub(r"^void ", "", dem)
    name = re.sub(r"\(bool\)0", "false", re.sub(r"\(bool\)1", "true", name))
    name = name.replace("(int)", "").split("(")[0]
    if drop is not None:
        name, k = re.subn(r", %s>$" % drop, ">", name)
        if not k:
            name = re.sub(r"<%s>$" % drop, "", name)
    return name


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--drop-template-arg", default=None)
    a = ap.parse_args()
    with tempfile.TemporaryDirectory() as tmp:
        old, new = kernels(compile_sass(a.old, tmp, "old")), kernels(compile_sass(a.new, tmp, "new"))
    om = dict(zip((short_name(d) for d in demangle(list(old))), old))
    nm = dict(zip((short_name(d, a.drop_template_arg) for d in demangle(list(new))), new))
    bad = 0
    for name in sorted(set(om) | set(nm)):
        if name not in om or name not in nm:
            print("%-60s only in %s" % (name, "old" if name in om else "new"))
            continue
        o, n = old[om[name]], new[nm[name]]
        if o == n:
            print("%-60s identical (%d instructions)" % (name, len(o)))
            continue
        if len(o) == len(n) and all(CBANK.sub("c[0x0][*]", x) == CBANK.sub("c[0x0][*]", y) for x, y in zip(o, n)):
            k = sum(x != y for x, y in zip(o, n))
            print("%-60s same but %d constant-bank offsets (%d instructions)" % (name, k, len(o)))
            continue
        bad += 1
        print("%-60s DIFFERS (%d vs %d instructions)" % (name, len(o), len(n)))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
