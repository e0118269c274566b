#!/usr/bin/env python
"""SASS mnemonic counts per kernel of libmpcmmd.so (cuobjdump -sass): the proof lines for tcgen05 / TMEM / TMA / packed-FP32 use.  usage: sass_summary.py > profiles/r02_sass_summary.md"""
import re, subprocess, sys
from collections import Counter, OrderedDict
lib = sys.argv[1] if len(sys.argv) > 1 else "mpc-mmd_b200/mpcmmd_b200/libmpcmmd.so"
txt = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
cur, cnt = None, OrderedDict()
for ln in txt.splitlines():
    m = re.search(r"Function : (\S+)", ln)
    if m:
        cur = m.group(1); cnt[cur] = Counter(); continue
    m = re.search(r"^\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", ln)
    if m and cur:
        cnt[cur][m.group(1).split(".")[0]] += 1
keys = ["UTCHMMA", "UTCBAR", "LDTM", "UBLKCP", "SYNCS", "BAR", "FFMA2", "FFMA", "MUFU", "LDS", "STS", "LDG", "STG", "SHFL", "REDUX", "VIMNMX"]
print("# SASS summary of libmpcmmd.so (sm_100a), `python tools/sass_summary.py`\n")
print("UTCHMMA = tcgen05.mma, LDTM = tcgen05.ld (TMEM -> registers), UTCBAR = tcgen05.commit, UBLKCP = cp.async.bulk (TMA bulk copy), SYNCS = mbarrier operations,")
print("FFMA2 = packed FP32 (fma.rn.f32x2), REDUX = redux.sync, VIMNMX = integer min/max (top-k networks).  num_reduced = 5 instantiations; the others differ only in unroll counts.\n")
print("| kernel | SASS instructions | " + " | ".join(keys) + " |"); print("|---|---|" + "---|" * len(keys))
for k, c in cnt.items():
    name = subprocess.run(["c++filt", k], capture_output=True, text=True).stdout.strip()
    name = re.sub(r"\(DCfg.*|\(ValCfg.*|\(float const\*.*|\(unsigned.*", "", name).replace("void ", "").replace("(int)", "").replace("(bool)", "")
    if not re.match(r"k_(project|inner_cem|rollouts|opt_risk|select|noise|obs_sort|validate|init)", name):
        continue
    if re.search(r"<[234],|<[234]>|k_inner_cem<[6789]>|big<256>", name):
        continue
    print("| `%s` | %d | " % (name, sum(c.values())) + " | ".join(str(c.get(x, 0)) for x in keys) + " |")
