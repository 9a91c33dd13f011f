#!/usr/bin/env python
"""SASS evidence of the Blackwell-native paths, taken from the built nerf_texture_b200/lib/libntx.so (no GPU needed):

    python tools/dump_sass.py            # writes profiles/r02_sass_{field,mlp,mlp_bwd,raymarch,grid,mesh}.txt
    python tools/dump_sass.py --round r03 texture_field     # profiles/r03_sass_texture_field.txt, with the kernels' ptxas report

For every kernel of the object: registers (from the ptxas log), and how often the tcgen05 / TMEM / TMA / mbarrier mnemonics occur
(`UTCHMMA` = tcgen05.mma — with `tmem[..]` as its first operand pair when A comes from tensor memory —, `LDTM`/`STTM` = tcgen05.ld/st,
`UTMALDG` = cp.async.bulk.tensor, `UTCBAR` = tcgen05.commit, `SYNCS` = mbarrier ops; /opt/skills/guides/B200_PROFILING.md), plus the
first occurrences verbatim."""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OBJ = os.path.join(ROOT, "nerf_texture_b200", "lib", "obj")
OUT = os.path.join(ROOT, "profiles")
PAT = ["UTCHMMA", "LDTM", "STTM", "UTMALDG", "UTCBAR", "SYNCS", "UTCATOMSWS", "HMMA", "RED", "ATOMS", "LDGSTS", "FMNMX3", "LDL", "STL", "LDG.E.128.CONSTANT"]


def demangle(names):
    r = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True)
    return r.stdout.splitlines() if r.returncode == 0 else names


def main():
    import argparse
    ap = argparse.ArgumentParser()
    ap.add_argument("--round", default="r02")
    ap.add_argument("units", nargs="*", default=["field", "mlp", "mlp_bwd", "raymarch", "grid", "mesh"])
    args = ap.parse_args()
    os.makedirs(OUT, exist_ok=True)
    for unit in args.units:
        obj = os.path.join(OBJ, unit + ".o")
        if not os.path.exists(obj):
            print("missing", obj, "(run python -m nerf_texture_b200.build first)")
            continue
        sass = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True).stdout
        kernels, cur = collections.OrderedDict(), None
        for line in sass.splitlines():
            m = re.match(r"\s*Function : (\S+)", line)
            if m:
                cur = m.group(1)
                kernels[cur] = []
            elif cur and "/*" in line and ";" in line:
                kernels[cur].append(line.strip())
        names = demangle(list(kernels))
        with open(os.path.join(OUT, "%s_sass_%s.txt" % (args.round, unit)), "w") as f:
            f.write("# cuobjdump -sass of nerf_texture_b200/lib/obj/%s.o (sm_100a) — mnemonic counts per kernel, tools/dump_sass.py\n" % unit)
            if args.round != "r02":                        # the round-2 files predate this: they carry no ptxas report
                log = obj + ".ptxas.log"
                f.write("\n# nvcc -Xptxas -v (%s)\n" % os.path.basename(log))
                for l in open(log).read().splitlines() if os.path.exists(log) else []:
                    if re.search(r"Compiling entry|registers|spill|smem", l):
                        f.write("# " + l.strip() + "\n")
            for (mangled, lines), name in zip(kernels.items(), names):
                counts = {p: sum(1 for l in lines if re.search(r"\b%s" % p, l)) for p in PAT}
                counts = {k: v for k, v in counts.items() if v}
                a_tmem = sum(1 for l in lines if re.search(r"UTCHMMA\s+tmem\[", l))
                f.write("\n== %s\n   %d SASS instructions; %s%s\n" % (name[:160], len(lines), ", ".join("%s x%d" % kv for kv in counts.items()) or "no tensor / TMA instructions",
                                                                   ("; UTCHMMA with the A operand in tensor memory x%d" % a_tmem) if a_tmem else ""))
                shown = collections.Counter()
                for l in lines:
                    for p in ("UTCHMMA", "LDTM", "STTM", "UTMALDG", "UTCBAR"):
                        if re.search(r"\b%s" % p, l) and shown[p] < 2:
                            shown[p] += 1
                            f.write("     " + re.sub(r"\s+/\* 0x[0-9a-f]+ \*/", "", l)[:150] + "\n")
        print("wrote profiles/%s_sass_%s.txt" % (args.round, unit))


if __name__ == "__main__":
    sys.exit(main())
