#!/usr/bin/env python
"""cuobjdump -sass multidimension_b200/libmdim_b200.so -> profiles/r2_sass_summary.md: per kernel family, the opcode counts
that show what the binary really does (256-bit global accesses, TMA, bulk copies, mbarriers, FFMA = 0 in the f32 hot paths)."""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "multidimension_b200", "libmdim_b200.so")
KEYS = ["LDG.E.256", "LDG.E.128", "LDG other", "STG.E.256", "STG.E.128", "STG other", "LTC64B", "UTMALDG", "UTMASTG", "UBLKCP", "SYNCS", "LDGSTS", "LDS", "STS", "BAR",
        "FFMA", "FMUL", "FADD", "IMAD", "LDC", "total"]


def demangle(names):
    p = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True)
    return p.stdout.split("\n")


def main():
    sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
    per = collections.OrderedDict()
    cur = None
    for ln in sass.split("\n"):
        m = re.match(r"\s*Function : (\S+)", ln)
        if m:
            cur = per.setdefault(m.group(1), collections.Counter())
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", ln)
        if not (m and cur is not None):
            continue
        op = m.group(1)
        cur["total"] += 1
        if op.startswith("LDG"):
            cur["LDG.E.256" if ".256" in op else "LDG.E.128" if ".128" in op else "LDG other"] += 1
            if "LTC64B" in op:
                cur["LTC64B"] += 1
        elif op.startswith("STG"):
            cur["STG.E.256" if ".256" in op else "STG.E.128" if ".128" in op else "STG other"] += 1
        else:
            for k in ("UTMALDG", "UTMASTG", "UBLKCP", "SYNCS", "LDGSTS", "LDS", "STS", "BAR", "FFMA", "FMUL", "FADD", "IMAD", "LDC"):
                if op.startswith(k):
                    cur[k] += 1
                    break
    names = demangle(list(per))
    rows = []
    for (mangled, c), name in zip(per.items(), names):
        name = re.sub(r"\(.*$", "", name.replace("(anonymous namespace)::", "")).replace("mdim::", "").replace("void ", "")
        rows.append((name, c))

    def pick(pred):
        return [(n, c) for n, c in rows if pred(n)]
    groups = [
        ("config 2: fused contiguous elementwise `k_eval<SigMulAddCF32, …, V=8, MAXR=1>` (256-bit accesses, no FFMA)", pick(lambda n: "SigMulAddCF32" in n and "8, 4, false, 1>" in n)),
        ("config 1: tensor-map TMA transpose `k_transpose_tma<ES, peers>`", pick(lambda n: n.startswith("k_transpose_tma"))),
        ("config 1 fallback: register-staged transpose `k_transpose<4, vec, peer>`", pick(lambda n: n.startswith("k_transpose<4, true,"))),
        ("config 3: gather `k_eval<SigGatherF32, u64 slots, V=4>` (LTC64B = the 64-byte L2 fetch flavour)", pick(lambda n: "SigGatherF32" in n and "4, 4, false, 1>" in n)),
        ("config 4: row folds `k_fold_rows<FAST>` (TMA bulk) and `k_fold_regs<L, FAST>`", pick(lambda n: n.startswith("k_fold_rows") or n.startswith("k_fold_regs<2,") or n.startswith("k_fold_regs<8,"))),
        ("sharded-axis fold: `k_fold_ring<S>` (TMA row tiles + peer-memory hand-off)", pick(lambda n: n.startswith("k_fold_ring") or "k_fold_ring" in n)),
        ("column walk `k_fold_xchg<S, DT, OP, ROWS, EXCHANGE>`: f32 / u64 sums, without (`k_fold_cols`, last argument false) and with the in-kernel all-reduce",
         pick(lambda n: "k_fold_xchg<unsigned int, 5, 0" in n or "k_fold_xchg<unsigned long, 4, 0" in n)),
        ("config 5 / 4b: pre-built rank-N signatures `k_eval<SigDiagMulAddCF32 / SigSubBcastF32, …, V=8>`", pick(lambda n: ("SigDiagMulAddCF32" in n or "SigSubBcastF32" in n) and "unsigned int, 8, 4, false" in n)),
    ]
    md = ["# Round 2 — SASS summary of `libmdim_b200.so` (sm_100a)", "",
          "`python scripts/sass_summary.py` (cuobjdump -sass of the built library; opcode counts per kernel, whole function).",
          f"{len(rows)} kernels in the library; the rows below are the ones the BASELINE configs run.  `FFMA` must be 0 in the f32 hot paths (Rust never",
          "contracts `x * y + 1.0`; the library is built with `--fmad=false`); the only FFMAs in the library sit inside `__fdiv_rn` / `sqrt` sequences.", ""]
    for title, sel in groups:
        md += [f"## {title}", "", "| kernel | " + " | ".join(KEYS) + " |", "|---|" + "---|" * len(KEYS)]
        for n, c in sel[:8]:
            md.append(f"| `{n[:110]}` | " + " | ".join(str(c.get(k, 0)) for k in KEYS) + " |")
        md.append("")
    tot = collections.Counter()
    for _, c in rows:
        tot.update(c)
    md += ["## Whole library", "", "| " + " | ".join(KEYS) + " |", "|" + "---|" * len(KEYS), "| " + " | ".join(str(tot.get(k, 0)) for k in KEYS) + " |", ""]
    hot_ffma = sum(c.get("FFMA", 0) for n, c in rows if ("SigMulAddCF32" in n or "SigDiagMulAddCF32" in n or "SigSubBcastF32" in n or n.startswith("k_fold_ring") or n.startswith("k_fold_xchg")))
    div_ffma = sum(c.get("FFMA", 0) for n, c in rows if n.startswith("k_fold_rows") or n.startswith("k_fold_regs"))
    md.append(f"FFMA in the f32 hot kernels without a division (MulAdd / DiagMulAdd / SubBcast signatures, the ring fold, the column walk): **{hot_ffma}**.")
    md.append(f"FFMA in `k_fold_rows` / `k_fold_regs` (all variants together): {div_ffma} — every one inside the IEEE division sequence of the fused epilogue's `fold / c`")
    md.append("(`__fdiv_rn`, Newton steps on the reciprocal: not a contraction of the expression's own multiply and add; the adds of the fold chain are `FADD`).")
    out = os.path.join(ROOT, "profiles", "r2_sass_summary.md")
    open(out, "w").write("\n".join(md) + "\n")
    print(out, len(rows), "kernels; hot FFMA:", hot_ffma)


if __name__ == "__main__":
    main()
