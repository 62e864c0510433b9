"""ptxas resources of the pattern-matrix (UnitVal) kernel instantiations against their weighted
twins: registers, spills and the shared-memory staging per CTA.  A twin is the same template with
the value type replaced by float or bf16 (every UnitVal kernel has at least one).  With --old-build
the weighted kernels are also compared with an earlier build (registers and spills).

    python tools/pattern_regs.py of-spmm_b200/build [--old-build DIR] [--md OUT.md]
"""
import argparse
import os
import re
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from sass_compare import demangle, ptxas  # noqa: E402

WARPS = 4


def stage_bytes(name):
    """Dynamic shared memory of a merge / atomic launch: WARPS TaskStage structs + WARPS mbarriers
    (fwd_launch.cuh, bwd.cu).  Mirrors the struct layout of spmm_kernels.cuh:TaskStage."""
    m = re.match(r"void ofspmm::(spmm_merge_kernel|bwd_atomic_kernel)<([^,]+), ([^,]+), (int|long), (.*)>", name)
    if not m:
        return None
    val, idx = m.group(3), m.group(4)
    items = int(m.group(5).split(", ")[-3])
    isz = 4 if idx == "int" else 8
    pad_i = 2 * (16 // isz)
    b = (items + pad_i) * isz + (items + 2 * pad_i) * isz
    if val != "ofspmm::UnitVal":
        vsz = 4 if val == "float" else 2
        b += (items + 2 * (16 // vsz)) * vsz
    b = (b + 15) // 16 * 16
    return WARPS * (b + 8)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("build")
    ap.add_argument("--old-build")
    ap.add_argument("--md")
    a = ap.parse_args()
    new = ptxas(a.build)
    dn = demangle(list(new))
    by = {dn[k]: v for k, v in new.items()}
    lines = ["| kernel (UnitVal) | regs | spill st/ld | twin regs (float / bf16 values) | stage bytes per CTA: unit / twin |",
             "|---|---|---|---|---|"]
    worse, spills, n_unit = [], [], 0
    for name, r in sorted(by.items()):
        if "ofspmm::UnitVal" not in name:
            continue
        n_unit += 1
        twins = [by.get(name.replace("ofspmm::UnitVal", t)) for t in ("float", "__nv_bfloat16")]
        twins_r = [t["regs"] if t else None for t in twins]
        present = [x for x in twins_r if x is not None]
        if r.get("spill", (0, 0)) != (0, 0):
            spills.append(name)
        if present and r["regs"] > min(present):
            worse.append((name, r["regs"], present))
        sb = stage_bytes(name)
        tw_name = name.replace("ofspmm::UnitVal", "float")
        tb = stage_bytes(tw_name) if sb is not None else None
        short = name.replace("void ofspmm::", "").replace("(ofspmm::FwdParams)", "").replace("(ofspmm::BwdAtomicParams)", "")
        lines.append(f"| `{short}` | {r['regs']} | {r.get('spill', (0, 0))[0]}/{r.get('spill', (0, 0))[1]} | "
                     f"{' / '.join('-' if x is None else str(x) for x in twins_r)} | "
                     f"{'-' if sb is None else f'{sb} / {tb}'} |")
    summary = [f"UnitVal instantiations: {n_unit}; with spills: {len(spills)}; "
               f"with more registers than the lighter weighted twin: {len(worse)}"]
    for w in worse:
        summary.append(f"  more registers: {w[0]} {w[1]} vs {w[2]}")
    if a.old_build:
        old = ptxas(a.old_build)
        do = demangle(list(old))
        ob = {do[k]: v for k, v in old.items()}
        changed = []
        for name, r in sorted(by.items()):
            o = ob.get(name.replace(", int2>", ">").replace(", int2,", ","), ob.get(name))
            if o is None:
                continue
            if o.get("regs") != r.get("regs") or o.get("spill", (0, 0)) != r.get("spill", (0, 0)):
                changed.append(f"  {name[:150]}: regs {o.get('regs')} -> {r.get('regs')}, "
                               f"spill {o.get('spill', (0, 0))} -> {r.get('spill', (0, 0))}")
        summary.append(f"kernels of the old build whose registers or spills changed: {len(changed)}")
        summary += changed
    print("\n".join(summary))
    if a.md:
        with open(a.md, "w") as f:
            f.write("\n".join(summary) + "\n\n" + "\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
