#!/bin/bash
# Per-kernel counts of the SASS mnemonics that prove the Blackwell-native paths (B200_PROFILING.md):
#   UTCHMMA = tcgen05.mma, LDTM / STTM = tcgen05.ld / .st, UTMALDG = TMA tensor load, UBLKCP = cp.async.bulk,
#   UTCBAR = tcgen05.commit, SYNCS = mbarrier ops, plus legacy HMMA (must be 0).
# Usage: profiles/sass_counts.sh [library.so] > profiles/r2_sass_counts.txt      (no GPU needed)
#   KEYS=DFMA,DADD,DMUL,MUFU FILTER='GaussianMixture, 2,' profiles/sass_counts.sh   other mnemonics; with FILTER, one
#   row per instantiation whose demangled name contains FILTER (instead of one row per kernel family)
LIB=${1:-kissmcmc.jl_b200/libkissmcmc_cuda.so}
export KEYS FILTER
echo "# $(basename $LIB)  sha256 $(sha256sum $LIB | cut -c1-16)  $(date -u +%F)"
cuobjdump -sass "$LIB" | python3 -c '
import re, subprocess, sys
import os
keys = os.environ.get("KEYS", "").split(",") if os.environ.get("KEYS") else \
    ["UTCHMMA", "LDTM", "STTM", "UTMALDG", "UBLKCP", "UTCBAR", "SYNCS", "HMMA"]
filt = os.environ.get("FILTER", "")
counts, cur = {}, None
for line in sys.stdin:
    m = re.match(r"\s*Function : (\S+)", line)
    if m:
        cur = m.group(1); counts.setdefault(cur, dict.fromkeys(keys, 0)); continue
    if cur is None: continue
    m = re.search(r"^\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
    if not m: continue
    op = m.group(1)
    for k in keys:
        if op == k or op.startswith(k + "."):
            counts[cur][k] += 1
names = list(counts)
dem = subprocess.run(["cu++filt"] + names, capture_output=True, text=True).stdout.splitlines() if names else []
rows = {}
for n, d in zip(names, dem):
    short = re.sub(r"\((int|bool)\)", "", d)
    short = re.sub(r"\(.*", "", short)
    if filt:
        if filt not in short: continue
    else:
        short = re.sub(r"<(kmc::\w+), \d+", r"<\1, D", short)   # one row per kernel family: max over the compiled d
    short = re.sub(r"^void ", "", short)
    c = counts[n]
    if not any(c[k] for k in keys): continue
    r = rows.setdefault(short, dict.fromkeys(keys, 0))
    for k in keys: r[k] = max(r[k], c[k])
print("%-90s " % "kernel (max over its instantiations / translation units)" + " ".join("%8s" % k for k in keys))
for short in sorted(rows):
    print("%-90s " % short[:90] + " ".join("%8d" % rows[short][k] for k in keys))
'
