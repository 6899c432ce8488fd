"""Compare the machine code of the conv / GEMM kernels of two builds of sed_conv.cu, kernel by kernel.

    nvcc <the Makefile's NVFLAGS> -c sed_conv.cu -o old.o      # at the old commit
    nvcc <the Makefile's NVFLAGS> -c sed_conv.cu -o new.o      # at the new commit
    python tools/sass_diff.py old.o new.o

`cuobjdump -sass` of each file is split into functions; addresses and encodings are dropped, the rest of every
instruction line is compared.  A differing pair is reported with the range of differing lines and whether both have the
same number of each opcode (a register-allocation or scheduling difference).  Kernels are matched by family and by the
template arguments both builds have: conv_umma_kernel lost <BRES, PATCH, EPI> (the kept instantiations are the GEMM:
false, false, EPI_LINEAR = 3) and conv_umma2_kernel lost <EG, FUSE1> (kept: 1, false).  Kernels of the old build without
a counterpart are listed as retired.  Exit status 1 if a matched pair differs or a kernel of the new build has no
counterpart."""
import argparse
import collections
import re
import subprocess
import sys

# family -> (indices of the template arguments the old build has and the new one does not, their kept values)
DROPPED = {
    "conv_umma_kernel": ((4, 5, 6), ("false", "false", "3")),
    "conv_umma2_kernel": ((9, 10), ("1", "false")),
}


def functions(path):
    """{demangled name: [normalised SASS lines]} of every function in `path`."""
    sass = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    names = [l.split(":", 1)[1].strip() for l in sass.splitlines() if l.strip().startswith("Function :")]
    demangled = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True,
                               check=True).stdout.splitlines()
    out, cur = {}, None
    for line in sass.splitlines():
        s = line.strip()
        if s.startswith("Function :"):
            cur = out.setdefault(demangled[len(out)], [])
            continue
        if cur is None:
            continue
        s = re.sub(r"/\*[^*]*\*/", "", s).strip()  # addresses and encodings
        if s and not s.startswith(".") and s != "..........":
            cur.append(s)
    return out


def opcode(line):
    """The opcode of a SASS line, without its predicate."""
    return re.sub(r"^@!?U?P\w+\s+", "", line).split()[0]


def split_args(s):
    """Top-level comma split of a template argument list."""
    args, depth, cur = [], 0, ""
    for ch in s:
        if ch == "," and depth == 0:
            args.append(cur.strip())
            cur = ""
            continue
        depth += ch in "<("
        depth -= ch in ">)"
        cur += ch
    return args + [cur.strip()]


def key(name, old):
    """(family, template arguments shared by both builds), or None for a retired instantiation of the old build."""
    m = re.match(r"void sed::(\w+)<(.*)>\(", name)
    if not m:
        return (name, ())
    family, args = m.group(1), split_args(m.group(2))
    if old and family in DROPPED:
        idx, kept = DROPPED[family]
        if tuple(args[i] for i in idx) != kept:
            return None
        args = [a for i, a in enumerate(args) if i not in idx]
    return (family, tuple(args))


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("old")
    ap.add_argument("new")
    args = ap.parse_args()
    old, new = functions(args.old), functions(args.new)
    old_by_key, retired = {}, []
    for name, body in old.items():
        k = key(name, True)
        if k is None:
            retired.append(name)
        else:
            old_by_key[k] = (name, body)
    bad = 0
    for name, body in sorted(new.items()):
        k = key(name, False)
        if k not in old_by_key:
            print("NO COUNTERPART  %s" % name)
            bad += 1
            continue
        oname, obody = old_by_key.pop(k)
        if obody == body:
            print("identical  %5d instructions  %s" % (len(body), name))
        else:
            idx = [i for i, (a, b) in enumerate(zip(obody, body)) if a != b]
            same_ops = collections.Counter(map(opcode, obody)) == collections.Counter(map(opcode, body))
            print("DIFFERENT  %5d vs %5d instructions, %d lines differ in [%d, %d], %s opcode counts  %s  <- %s" % (
                len(obody), len(body), len(idx), idx[0], idx[-1], "same" if same_ops else "DIFFERENT", name, oname))
            bad += 1
    for name in sorted(retired) + sorted(n for n, _ in old_by_key.values()):
        print("retired    %s" % name)
    print("%d kernels in the new build, %d identical to their counterpart, %d retired" %
          (len(new), len(new) - bad, len(old) - len(new)))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
