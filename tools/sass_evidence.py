#!/usr/bin/env python
"""Readable kernel evidence for profiles/ (VERDICT r1 item 8): per hot kernel a `cuobjdump -sass` excerpt with the
lines that prove the data path (UBLKCP = cp.async.bulk / TMA, SYNCS = mbarrier, UTC*MMA = tcgen05.mma, LDTM/STTM =
tcgen05.ld/st, HMMA = legacy mma.sync, DFMA/DADD = fp64 arithmetic) plus a mnemonic histogram, and one table of
`ptxas -v` facts (registers, static shared memory, stack frame, spills) from the build logs.

    python tools/sass_evidence.py            # writes profiles/sass_<tag>.txt and profiles/ptxas_table.md
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "iterativesolvers.jl_b200", "libb200krylov.so")
LOGS = os.path.join(ROOT, "iterativesolvers.jl_b200", "csrc", "build")
OUT = os.path.join(ROOT, "profiles")

# tag -> (substring of the mangled name that selects ONE instantiation, what to show)
HOT = {
    "cg_k2_spmv_dot_stream_f64": ("k_cg_spmv_dot_streamIdLi8E", "K2 of cg!: c = A u fused with dot(u, c); TMA-bulk streamed CSR"),
    "cg_persistent": ("k_cg_persistentIdLi8E", "cg! for small operators: the whole loop in one persistent cooperative kernel"),
    "cg_k1_update_u": ("k_cg_update_uId", "K1 of cg!: x += alpha u_old (deferred), u = r + beta u"),
    "cg_k3_update_r": ("k_cg_update_rId", "K3 of cg!: r -= alpha c fused with ||r||^2 (and the warp-parallel NVLink allreduce)"),
    "gmres_block_dots": ("k_block_dotsIdLi2E", "CGS/DGKS block of dots h = V' w (three-kernel path)"),
    "gmres_fused_orth": ("k_orth_fusedIdLi2E", "orthogonalize_and_normalize! CGS/DGKS in one cooperative launch + the GMRES scalar step"),
    "lobpcg_update_tc": ("k_update_tcILi1E", "LOBPCG update X, P, AX, AP, R (3xTF32 mma.sync)"),
    "lobpcg_gram_tcgen05": ("k_gram_umma", "LOBPCG Rayleigh-Ritz Gram products on tcgen05 (TMEM accumulators)"),
    "lobpcg_gram_legacy": ("k_gram_rr_tcILi2E", "LOBPCG Rayleigh-Ritz Gram products, legacy mma.sync path (kept for comparison)"),
    "pass_generic": ("k_passINS_8QmrWNextIdEE", "the fused-pass kernel of the general engines (one instantiation: QMR's w-recurrence pass)"),
    "spmv_stream_f64": ("k_spmv_streamIdLi8E", "mul!(y, A, x): TMA-bulk streamed CSR SpMV"),
    "cg_k2_spmv_dot_dia_f64": ("k_cg_spmv_dot_diaIdE", "K2 of cg! on the offset-diagonal copy: TMA-bulk streamed values + row masks"),
    "spmv_dia_f64": ("k_spmv_diaIdE", "mul!(y, A, x) on the offset-diagonal copy"),
}
KEY = re.compile(r"\b(UBLKCP|UTMALDG|UTMASTG|SYNCS|UTC[A-Z]*MMA|UTCBAR|UTCCP|LDTM|STTM|UTCALLOC|HMMA|DFMA|DADD|DMUL|FFMA|"
                 r"LDG|STG|LDS|STS|REDG|ATOMG|SHFL|BAR|ACQBULK|ELECT|LDGSTS|CCTL|MEMBAR|ERRBAR|FENCE)\b")


def dump_functions():
    txt = subprocess.run(["cuobjdump", "-sass", SO], stdout=subprocess.PIPE, text=True, check=True).stdout
    funcs, name, cur = {}, None, []
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                funcs[name] = cur
            name, cur = m.group(1), []
        elif name:
            cur.append(line)
    if name:
        funcs[name] = cur
    return funcs


def demangle(n):
    try:
        return subprocess.run(["c++filt", n], stdout=subprocess.PIPE, text=True).stdout.strip()
    except Exception:
        return n


def ptxas_table():
    rows = []
    for f in sorted(os.listdir(LOGS)):
        if not f.endswith(".ptxas.log"):
            continue
        txt = open(os.path.join(LOGS, f)).read()
        for m in re.finditer(r"Compiling entry function '(\S+)' for 'sm_100a'\n.*?\n\s*(\d+) bytes stack frame, (\d+) bytes "
                             r"spill stores, (\d+) bytes spill loads\n.*?Used (\d+) registers(?:, used (\d+) barriers)?"
                             r"(?:, (\d+) bytes smem)?", txt, re.S):
            rows.append((f.replace(".ptxas.log", ".cu"), m.group(1), int(m.group(5)), int(m.group(7) or 0), int(m.group(2)),
                         int(m.group(3)), int(m.group(4))))
    return rows


def main():
    funcs = dump_functions()
    os.makedirs(OUT, exist_ok=True)
    written = []
    for tag, (needle, what) in HOT.items():
        hits = [n for n in funcs if needle in n]
        if not hits:
            continue
        n = sorted(hits, key=len)[0]
        body = funcs[n]
        ins = [l for l in body if re.search(r"/\*[0-9a-f]{4}\*/", l)]
        hist = collections.Counter()
        for l in ins:
            m = re.search(r"/\*[0-9a-f]{4}\*/\s+(?:@!?U?P\d\s+)?([A-Z0-9_.]+)", l)
            if m:
                hist[m.group(1).split(".")[0]] += 1
        keyl = [l.rstrip() for l in ins if KEY.search(l) and re.search(r"UBLKCP|UTMA|SYNCS|UTC|LDTM|STTM|HMMA|DFMA|ACQBULK|ELECT|REDG|ERRBAR|MEMBAR", l)]
        path = os.path.join(OUT, f"sass_{tag}.txt")
        with open(path, "w") as f:
            f.write(f"# {what}\n# {demangle(n)}\n# cuobjdump -sass libb200krylov.so (sm_100a), {len(ins)} instructions\n")
            f.write("# mnemonic histogram: " + ", ".join(f"{k} {v}" for k, v in hist.most_common(40)) + "\n\n")
            f.write("# lines with TMA / mbarrier / tensor-core / fp64-FMA instructions (first 120):\n")
            f.write("\n".join(keyl[:120]) + "\n")
        written.append(path)
    rows = ptxas_table()
    hot_subs = [v[0].split("I")[0] if not v[0].startswith("k_pass") else v[0] for v in HOT.values()]
    with open(os.path.join(OUT, "ptxas_table.md"), "w") as f:
        f.write("# `ptxas -v` facts of the hot kernels (sm_100a; from iterativesolvers.jl_b200/csrc/build/*.ptxas.log)\n\n")
        f.write("| file | kernel | registers | static smem B | stack B | spill st B | spill ld B |\n|---|---|---|---|---|---|---|\n")
        for src, n, regs, smem, stack, ss, sl in rows:
            if any(h in n for h in hot_subs) or ss or sl:
                d = demangle(n)
                d = re.sub(r"\(anonymous namespace\)::", "", d).split("(")[0]
                f.write(f"| {src} | `{d}` | {regs} | {smem} | {stack} | {ss} | {sl} |\n")
        spills = [(n, ss, sl) for _, n, _, _, _, ss, sl in rows if ss or sl]
        f.write(f"\n{len(rows)} kernels compiled; {len(spills)} with register spills.\n")
    print("\n".join(written))


if __name__ == "__main__":
    main()
