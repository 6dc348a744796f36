"""SASS evidence per hot kernel of liblavt_b200.so (CPU only, cuobjdump): counts of the tcgen05 (UTC*MMA), TMEM (LDTM / STTM), TMA (UTMALDG),
mma.sync (HMMA) and MUFU.EX2 mnemonics and the first tensor-core instruction.    python tools/sass_excerpts.py > profiles/r2_sass_excerpts.txt"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "lavt_rs_b200", "_lib", "liblavt_b200.so")
KERNELS = ("gemm_bf16_tc_kernel", "window_attn_tc2_kernel", "window_attn_tc3_kernel", "window_attn_bwd_tc_kernel", "window_attn_bwd_kernel", "window_attn_resident_kernel",
           "pwam_core")
out = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True).stdout
name, stats, first = None, collections.OrderedDict(), {}
pat = {"UTC*MMA (tcgen05.mma)": r"UTC[A-Z]*MMA", "of which .2CTA (cta_group::2)": r"UTC[A-Z]*MMA\.2CTA", "UTCBAR (tcgen05.commit)": r"UTCBAR", "LDTM (tcgen05.ld)": r"\bLDTM", "STTM (tcgen05.st)": r"\bSTTM",
       "UTMALDG (TMA load)": r"UTMALDG", "HMMA (mma.sync)": r"^\s*/\*[0-9a-f]+\*/\s+HMMA", "MUFU.EX2": r"MUFU\.EX2", "SYNCS (mbarrier)": r"\bSYNCS"}
for line in out.splitlines():
    m = re.search(r"Function : (\S+)", line)
    if m:
        name = m.group(1) if any(k in m.group(1) for k in KERNELS) else None
        if name:
            stats[name] = collections.Counter()
        continue
    if name and re.match(r"\s+/\*[0-9a-f]+\*/\s+\S", line):
        stats[name]["instructions"] += 1
        for k, p in pat.items():
            if re.search(p, line):
                stats[name][k] += 1
        if name not in first and re.search(r"UTC[A-Z]*MMA|HMMA", line):
            first[name] = re.sub(r"/\* 0x[0-9a-f]+ \*/", "", line).strip()
for nm, c in stats.items():
    dem = subprocess.run(["c++filt", nm], capture_output=True, text=True).stdout.strip()
    print(dem[:160])
    print("    " + "  ".join(f"{k} {c[k]}" for k in ["instructions", *pat]))
    print("    first tensor-core instruction: " + first.get(nm, "(none: bandwidth kernel)"))
