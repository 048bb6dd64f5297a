#!/usr/bin/env python3
"""SASS evidence per hot kernel of libdspfront.so: instruction totals and the counts of the mnemonics that prove the
design (tcgen05 = UTCHMMA / LDTM / UTCBAR, bulk TMA = UBLKCP, byte-plane dot products = IDP.4A, packed 16-bit compares =
VIADDMNMX / VIMNMX3, packed fp32 = FFMA2 / FADD2 / FMUL2, warp reductions = REDUX, mbarriers = SYNCS), with the first
occurrence of each as a sample line.  Usage: sass_excerpt.py [lib.so] > profiles/r02_sass_excerpt.txt"""
import collections, os, re, subprocess, sys
lib = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "dsp_audioreclabs_b200", "libdspfront.so")
HOT = ["frontend_pipe_kernelILb1", "frontend_pipe_kernelILb0", "knn_tc16_filter_kernelILi5E", "knn_dense_scan_kernel", "knn_scan_pair_kernel",
       "knn_refine_collect_kernel", "frontend_pcm_kernel", "frontend_exact_kernel", "dtw_kernel", "mfcc_kernel"]
KEYS = ["UTCHMMA", "LDTM", "UTCBAR", "UTCATOMSWS", "UBLKCP", "SYNCS", "IDP.4A", "VIADDMNMX", "VIMNMX3", "FFMA2", "FADD2", "FMUL2", "FFMA", "DFMA", "DADD",
        "REDUX", "SHFL", "POPC", "LDS", "STS", "LDG", "STG", "BAR", "USETMAXREG", "PRMT", "HMMA"]
out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
cur, seen = None, set()
cnt = collections.defaultdict(collections.Counter); first = collections.defaultdict(dict); total = collections.Counter()
for ln in out.splitlines():
    m = re.search(r"Function : (\S+)", ln)
    if m:
        cur = next((h for h in HOT if h in m.group(1)), None)
        if cur and cur in seen: cur = None          # first instantiation of a family only
        if cur: seen.add(cur); first[cur]["__name"] = m.group(1)
        continue
    if not cur: continue
    m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", ln)
    if not m: continue
    ins = m.group(2).strip()
    toks = ins.split()
    op = toks[1] if toks[0].startswith("@") else toks[0]
    total[cur] += 1
    for k in KEYS:
        if op == k or op.startswith(k + ".") or (k in ("IDP.4A",) and op.startswith(k)):
            cnt[cur][k] += 1
            first[cur].setdefault(k, f"/*{m.group(1)}*/ {ins}")
print(f"# cuobjdump -sass {os.path.basename(lib)} (sm_100a): hot kernels, instruction counts of the mnemonics that carry the design\n")
for h in HOT:
    if h not in total: continue
    print(f"== {first[h]['__name']}\n   {total[h]} SASS instructions")
    for k in KEYS:
        if cnt[h][k]:
            print(f"   {k:12s} x{cnt[h][k]:5d}   {first[h][k]}")
    print()
