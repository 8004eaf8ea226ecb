"""Per-kernel comparison of two builds of csrc/: which functions' `cuobjdump -sass` listings differ, and which ptxas
register / spill lines (the `*.ptxas.log` files the Makefile writes) differ.  Anonymous-namespace hashes, which depend on
the build directory, are normalised away.

    python tools/sass_diff.py OLD_CSRC_DIR NEW_CSRC_DIR      (both built with `make`, e.g. a checkout of the parent)
"""
import re
import subprocess
import sys

OBJS = ("pde_tc", "pde_f32", "pde_f64", "pde_step", "pde_comm")


def _norm(name):
    name = re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__", name)
    # tc_kernel<D, ORDER, ACT, NDIR, NLAP>: NLAP defaults to NDIR, and such an instantiation pairs with the
    # four-argument tc_kernel<D, ORDER, ACT, NDIR> of builds from before that parameter existed
    return re.sub(r"(9tc_kernelILi\d+ELi\d+ELi\d+ELi(\d+)E)Li\2EE", r"\1E", name)


def _demangle(name):
    return subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()


def sass(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    res, name = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = _norm(m.group(1))
            res[name] = []
        elif name:
            res[name].append(line)
    return {k: "\n".join(v) for k, v in res.items()}


def ptxas(path):
    res, fn = {}, None
    for line in open(path):
        m = re.search(r"Compiling entry function '(\S+)'", line) or re.search(r"Function properties for (\S+)", line)
        if m:
            fn = _norm(m.group(1))
            res.setdefault(fn, [])
        elif fn and ("registers" in line or "spill" in line):
            res[fn].append(re.sub(r"^ptxas info\s*:\s*", "", line.strip()))
    return res


def main(old, new):
    for obj in OBJS:
        a, b = sass(f"{old}/{obj}.o"), sass(f"{new}/{obj}.o")
        diff = sorted(_demangle(n) for n in a if n in b and a[n] != b[n])
        only = sorted(_demangle(n) for n in set(a) ^ set(b))
        print(f"{obj}.o: {len(a)} functions, {len(a) - len(diff) - len(set(a) - set(b))} identical SASS")
        for n in diff:
            print("  SASS differs:", n)
        for n in only:
            print("  only in one build:", n)
        pa, pb = ptxas(f"{old}/{obj}.ptxas.log"), ptxas(f"{new}/{obj}.ptxas.log")
        for n in sorted(set(pa) | set(pb)):
            if pa.get(n) != pb.get(n):
                print("  ptxas differs:", _demangle(n), "|", " / ".join(pa.get(n, [])), "->", " / ".join(pb.get(n, [])))
            elif n in pb and any(re.search(r"[1-9]\d* bytes spill", l) for l in pb[n]):
                print("  spills (unchanged):", _demangle(n), "|", " / ".join(pb[n]))


if __name__ == "__main__":
    main(sys.argv[1], sys.argv[2])
