"""Per-kernel SASS instruction mix of libphotoverse_b200.so -> profiles/<argv[1]> (no GPU needed).
Counts the mnemonics that prove the Blackwell path (B200_PROFILING.md): UTCHMMA (tcgen05.mma), UTCBAR (tcgen05.commit),
LDTM / STTM (tcgen05.ld / st), UTMALDG / UTMASTG (TMA tensor load / store), UBLKCP (bulk copy), SYNCS (mbarrier),
and the legacy tensor path HMMA / LDSM (mma.sync / ldmatrix), plus the packed fp32x2 arithmetic FFMA2 / FADD2 / FMUL2."""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "photoverse_b200", "libphotoverse_b200.so")
OUT = os.path.join(ROOT, "profiles", sys.argv[1] if len(sys.argv) > 1 else "r02_sass_summary.txt")
MNEM = ["UTCHMMA", "UTCBAR", "LDTM", "STTM", "UTMALDG", "UTMASTG", "UBLKCP", "SYNCS", "HMMA", "LDSM", "FFMA2", "FADD2", "FMUL2", "MUFU"]

sass = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
counts = collections.OrderedDict()
cur = None
for line in sass.splitlines():
    m = re.match(r"\s*Function : (\S+)", line)
    if m:
        cur = m.group(1)
        counts[cur] = collections.Counter()
        continue
    if cur is None:
        continue
    m = re.search(r"/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d\s+)?([A-Z0-9_]+)", line)
    if m:
        op = m.group(1)
        counts[cur]["_total"] += 1
        for k in MNEM:
            if op.startswith(k):
                counts[cur][k] += 1
names = subprocess.run(["c++filt"], input="\n".join(counts), capture_output=True, text=True).stdout.splitlines()
rows = []
for mangled, dem in zip(counts, names):
    c = counts[mangled]
    short = re.sub(r"\(.*", "", dem.replace("void ", "").replace("pv::", ""))[:80]
    rows.append((short, c))
rows.sort(key=lambda r: (-r[1]["UTCHMMA"], -r[1]["HMMA"], r[0]))
with open(OUT, "w") as f:
    f.write("SASS instruction mix per kernel of photoverse_b200/libphotoverse_b200.so (cuobjdump -sass, sm_100a; tools/sass_summary.py)\n")
    f.write(f"{'kernel':82s}" + "".join(f"{k:>9s}" for k in MNEM) + f"{'instrs':>9s}\n")
    tot = collections.Counter()
    for short, c in rows:
        f.write(f"{short:82s}" + "".join(f"{c[k]:9d}" for k in MNEM) + f"{c['_total']:9d}\n")
        tot.update(c)
    f.write(f"{'TOTAL (' + str(len(rows)) + ' kernels)':82s}" + "".join(f"{tot[k]:9d}" for k in MNEM) + f"{tot['_total']:9d}\n")
print(open(OUT).read()[:6000])
