"""Compare the SASS of two builds of libbihrt.so function by function.

    python tools/sass_diff.py [--normalize] OLD/libbihrt.so NEW/libbihrt.so

Disassembles both with `cuobjdump -sass`, hashes the instruction text of every function and prints which functions are
identical, which differ and which exist in only one build.  A change that must not touch the code of existing kernels
(a new template instantiation, a new entry point) shows up as "identical" for all of them and "only in NEW" for the new
ones.  Exit code 1 if a function present in both builds differs.

--normalize compares the instructions without their encoding words, with the offsets of bank-0 constants (`c[0x0][...]`:
the kernel parameters) and the numbers of the registers (R, UR, P, UP) masked.  Opcodes, modifiers, immediates, memory
offsets and the order of the instructions are still compared.  A kernel parameter struct that loses or gains a field moves
the offsets of every later field, and register allocation may number the same registers differently: under --normalize
such kernels still compare identical.
"""
import argparse
import hashlib
import os
import re
import subprocess
import sys


def cuobjdump():
    for p in (os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump"), "cuobjdump"):
        if os.path.sep not in p or os.access(p, os.X_OK):
            return p
    return "cuobjdump"


_ENCODING = re.compile(r"/\*\s*0x[0-9a-f]{16}\s*\*/")
_MASKS = [(re.compile(r"c\[0x0\]\[[^\]]*\]"), "c[0x0][*]"),
          (re.compile(r"\b(U?R|U?P)\d+\b"), r"\1#")]


def normalized(line):
    """The instruction of one SASS line without its address and encoding, constant offsets and register numbers masked;
    None for a line that holds only an encoding word."""
    text = _ENCODING.sub("", line)
    text = re.sub(r"^\s*/\*[0-9a-f]+\*/", "", text).strip()
    if not text:
        return None
    for pat, repl in _MASKS:
        text = pat.sub(repl, text)
    return text


def functions(lib, normalize=False):
    """{mangled name: sha256 of its SASS text}.  Only the instruction lines count (the header of the section names the
    ELF it came from)."""
    out = subprocess.run([cuobjdump(), "-sass", lib], check=True, capture_output=True, text=True).stdout
    funcs, name, body = {}, None, []

    def close():
        if name is not None:
            funcs[name] = hashlib.sha256("\n".join(body).encode()).hexdigest()

    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            close()
            name, body = m.group(1), []
        elif name is not None and line.strip().startswith("/*"):
            if not normalize:
                body.append(line.strip())
            elif (text := normalized(line)) is not None:
                body.append(text)
    close()
    return funcs


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("-q", "--quiet", action="store_true", help="do not list the identical functions")
    ap.add_argument("--normalize", action="store_true",
                    help="ignore encoding words, bank-0 constant offsets and register numbers")
    args = ap.parse_args()
    a, b = functions(args.old, args.normalize), functions(args.new, args.normalize)
    same = sorted(k for k in a if k in b and a[k] == b[k])
    diff = sorted(k for k in a if k in b and a[k] != b[k])
    only_a, only_b = sorted(k for k in a if k not in b), sorted(k for k in b if k not in a)
    if not args.quiet:
        for k in same:
            print("identical   %s" % k)
    for k in diff:
        print("DIFFERENT   %s" % k)
    for k in only_a:
        print("only in OLD %s" % k)
    for k in only_b:
        print("only in NEW %s" % k)
    print("%d of %d functions of OLD identical in NEW; %d differ, %d only in OLD, %d only in NEW"
          % (len(same), len(a), len(diff), len(only_a), len(only_b)))
    return 1 if diff else 0


if __name__ == "__main__":
    sys.exit(main())
