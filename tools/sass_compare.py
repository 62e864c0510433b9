"""Compare the kernels of two builds of libofspmm_b200.so: SASS per kernel (cuobjdump -sass, with
addresses and immediates masked) and ptxas registers / spills (the *.ptxas.log files the Makefile
writes next to the objects).  Kernels are matched by demangled name; a template argument a later
build added is removed before matching (the partition entry type `int2` of the narrow kernels, the
key type of the transpose kernels), and `> >` is matched with `>>` (c++filt closes a nested template
argument without the space when an empty trailing parameter pack follows it, as in the sampling
kernels' exclusion pack).

    python tools/sass_compare.py OLD_LIB NEW_LIB [--old-build DIR --new-build DIR]
"""
import argparse
import glob
import re
import subprocess


def sass(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            res[cur] = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s*(.*?);", line)
        if cur and m:
            res[cur].append(re.sub(r"0x[0-9a-f]+", "X", m.group(1)))
    return res


def ptxas(build_dir):
    res, cur = {}, None
    for f in glob.glob(build_dir + "/*.ptxas.log"):
        for line in open(f):
            m = re.search(r"Compiling entry function '(\S+)'", line)
            if m:
                cur = m.group(1)
            m = re.search(r"Used (\d+) registers", line)
            if m and cur:
                res.setdefault(cur, {})["regs"] = int(m.group(1))
            m = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", line)
            if m and cur:
                res.setdefault(cur, {})["spill"] = (int(m.group(1)), int(m.group(2)))
    return res


def demangle(names):
    out = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    return dict(zip(names, out))


def norm(d):
    d = d.replace("> >", ">>")
    d = d.replace(", int2>", ">").replace(", int2,", ",").replace("ofspmm::PartOf<int2>::Nz", "int")
    if "transpose_" in d:
        for a, b in (("<int, int>", "<int>"), ("<int, int, ", "<int, "), ("<long, long>", "<long>"),
                     ("<long, long, ", "<long, ")):
            d = d.replace(a, b)
    return d


def compare(old, new, what):
    do, dn = demangle(list(old)), demangle(list(new))
    by_name = {}
    for k in new:
        by_name.setdefault(norm(dn[k]), []).append(new[k])
    same, diff, missing = 0, [], []
    for k, v in old.items():
        cands = by_name.get(norm(do[k]))
        if cands is None:
            missing.append(do[k])
        elif any(c == v for c in cands):
            same += 1
        else:
            diff.append(do[k])
    print(f"{what}: {len(old)} kernels of the old build, {same} identical, {len(diff)} differ, {len(missing)} unmatched")
    for d in diff:
        print("  differs:", d[:200])
    for d in missing:
        print("  unmatched:", d[:200])
    print(f"{what}: {len(new) - same - len(diff)} kernels only in the new build")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old_lib")
    ap.add_argument("new_lib")
    ap.add_argument("--old-build")
    ap.add_argument("--new-build")
    a = ap.parse_args()
    compare(sass(a.old_lib), sass(a.new_lib), "SASS")
    if a.old_build and a.new_build:
        compare(ptxas(a.old_build), ptxas(a.new_build), "registers+spills")


if __name__ == "__main__":
    main()
