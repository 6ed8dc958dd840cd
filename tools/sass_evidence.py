"""Per-kernel SASS evidence of the built library (no GPU needed): for every kernel of libb2s.so the counts of the
Blackwell-specific instructions — UTCIMMA / UTCHMMA / UTCQMMA (tcgen05.mma), LDTM / STTM (tcgen05.ld / st), UTCBAR
(tcgen05.commit), UBLKCP (cp.async.bulk), UTMALDG (tensor-map TMA), SYNCS (mbarrier), POPC, REDUX, VIMNMX*,
DFMA, FFMA2 / FMUL2 (packed fma.rn.f32x2), FFMA — plus registers / spills from the ptxas logs.  Writes profiles/<round>_sass.md and a trimmed listing of
the shipped Hamming kernel's tcgen05 lines.   Usage: python tools/sass_evidence.py r02"""
import collections
import re
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]
LIB = ROOT / "monocular-visual-slam_b200" / "b200slam" / "libb2s.so"
OPS = ("UTCIMMA", "UTCHMMA", "UTCQMMA", "LDTM", "STTM", "UTCBAR", "UBLKCP", "UTMALDG", "SYNCS", "POPC", "REDUX", "VIMNMX3", "VIMNMX", "VIADDMNMX",
       "DFMA", "FFMA2", "FMUL2", "FFMA", "SHFL", "ATOMG", "LDS", "STS")


def kernels():
    """-> {demangled-ish name: [SASS lines]}"""
    txt = subprocess.run(["cuobjdump", "-sass", str(LIB)], capture_output=True, text=True, check=True).stdout
    out, cur = collections.OrderedDict(), None
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
        elif cur and re.match(r"\s+/\*[0-9a-f]{4}\*/", line):
            out[cur].append(line.rstrip())
    return out


def demangle(names):
    r = subprocess.run(["c++filt"] + list(names), capture_output=True, text=True)
    return r.stdout.splitlines() if r.returncode == 0 else list(names)


def counts(lines):
    c = collections.Counter()
    for l in lines:
        m = re.search(r"\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_]*)", l)
        if m:
            op = m.group(1)
            for o in OPS:
                if op == o or (o in ("VIMNMX", "FFMA", "DFMA", "LDS", "STS", "ATOMG", "SHFL", "REDUX", "POPC") and op.startswith(o) and not (o == "VIMNMX" and op.startswith("VIMNMX3"))):
                    c[o] += 1
                    break
            c["total"] += 1
    return c


def main():
    tag = sys.argv[1] if len(sys.argv) > 1 else "r02"
    ks = kernels()
    names = demangle(ks.keys())
    rows = []
    for (mangled, lines), name in zip(ks.items(), names):
        c = counts(lines)
        short = re.sub(r"\(.*", "", name).replace("void ", "").replace("b2s::", "")
        rows.append((short, c, mangled))
    md = [f"# {tag} — SASS evidence per kernel (`cuobjdump -sass libb2s.so`, sm_100a, built in the CPU container)", "",
          "Counts of static SASS instructions.  UTCIMMA / UTCHMMA = `tcgen05.mma` (int8 / tf32), LDTM = `tcgen05.ld`, UTCBAR = `tcgen05.commit`, "
          "UBLKCP = `cp.async.bulk` (TMA engine, 1-D), SYNCS = mbarrier ops.  No UTMALDG: operand tiles are contiguous 34 KB blocks, staged with 1-D bulk copies.", "",
          "| kernel | instr | " + " | ".join(OPS) + " |", "|---|---:|" + "---:|" * len(OPS)]
    for short, c, _ in sorted(rows, key=lambda r: -r[1]["total"]):
        md.append(f"| `{short}` | {c['total']} | " + " | ".join(str(c[o]) if c[o] else "" for o in OPS) + " |")
    # trimmed listing of the shipped Hamming kernel
    target = [r for r in rows if "hamming_knn2_i8s_kernel<true>" in r[0]]
    if target:
        _, _, mangled = target[0]
        md += ["", "## `hamming_knn2_i8s_kernel<true>` (shipped) — every tensor-core / TMEM / bulk-copy line", "", "```"]
        md += [l.split("*/", 1)[0].strip() + "*/ " + re.sub(r"\s*/\*.*", "", l.split("*/", 1)[1]).strip()
               for l in ks[mangled] if re.search(r"UTCIMMA|LDTM|UTCBAR|UBLKCP|UTCATOM|ELECT", l)]
        md += ["```"]
    (ROOT / "profiles" / f"{tag}_sass.md").write_text("\n".join(md) + "\n")
    print("wrote", ROOT / "profiles" / f"{tag}_sass.md", len(rows), "kernels")


if __name__ == "__main__":
    main()
