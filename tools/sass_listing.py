#!/usr/bin/env python
"""Per-kernel SASS opcode counts of the tensor-core objects (cuobjdump -sass; runs on the CPU box after a build):
the evidence that k_xw_tc / k_dw_tc are tcgen05 (UTCHMMA), TMA (UTMALDG) and TMEM (LDTM) kernels.
Usage: python tools/sass_listing.py > profiles/sass_tc.txt"""
import collections
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEYS = ["UTCHMMA", "UTMALDG", "LDTM", "UTCBAR", "UTCATOMSWS", "SYNCS", "FENCE", "FFMA", "HMMA", "IMMA"]


def main():
    print("# SASS evidence for the tcgen05 / TMA / TMEM kernels (cuobjdump -sass of the objects linked into libbigcn_b200.so, sm_100a).")
    print("# UTCHMMA = tcgen05.mma (kind::tf32 here), UTMALDG = TMA tensor load (cp.async.bulk.tensor), LDTM = tcgen05.ld (TMEM -> registers),")
    print("# UTCBAR = tcgen05.commit -> mbarrier, UTCATOMSWS = TMEM allocation, SYNCS = mbarrier ops, FENCE = fence.proxy.async / tcgen05 fences.")
    for obj in ("bigcn_b200/csrc/gemm_tc.o",):
        txt = subprocess.run(["cuobjdump", "-sass", os.path.join(ROOT, obj)], capture_output=True, text=True).stdout
        cur, cnt = None, collections.OrderedDict()
        for line in txt.splitlines():
            m = re.search(r"Function : (\S+)", line)
            if m:
                cur = m.group(1)
                cnt[cur] = collections.Counter()
                continue
            if cur is None:
                continue
            m = re.search(r"^\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)", line)
            if m:
                cnt[cur][m.group(1).split(".")[0]] += 1
                cnt[cur]["__total"] += 1
        print("\n== " + obj)
        for f, c in cnt.items():
            name = subprocess.run(["c++filt", f], capture_output=True, text=True).stdout.strip()
            extra = [k for k in c if k.startswith("UT") and k not in KEYS]
            print(name[:140])
            print("    total %d  " % c["__total"] + "  ".join(f"{k}={c[k]}" for k in KEYS + extra if c[k]))


if __name__ == "__main__":
    main()
