"""Per-case instruction counts of the fp64 resident kernel's check pass, from the SASS (no GPU needed): the switch over check
groups compiles to one straight block per (weight, split) case; a block's MUFU.RCP64H count / 3 is its number of edges.
usage: sass_check_cases.py <binary> <substring-of-demangled-kernel-name>"""
import re, subprocess, sys
from collections import Counter
binary, pat = sys.argv[1], sys.argv[2]
out = subprocess.run(["cuobjdump", "-sass", binary], capture_output=True, text=True).stdout
FP64 = ("DFMA", "DADD", "DMUL", "DSETP")
for blk in re.split(r"\n\s*Function : ", out)[1:]:
    name = blk.split("\n", 1)[0].strip()
    dem = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()
    if pat not in dem:
        continue
    print("==", dem)
    ins = [m.group(1).strip() for m in re.finditer(r"/\*[0-9a-f]{4,}\*/\s+(.*?);", blk)]
    seg, tot = [], Counter()
    for t in ins + ["EXIT"]:
        seg.append(t)
        if not re.search(r"\b(BRA|EXIT|RET|BRX|JMX)\b", t) or t.startswith("@"):
            continue
        ops = Counter((p[1] if p[0].startswith("@") else p[0]).split(".")[0] for p in (s.split() for s in seg))
        if ops["MUFU"] >= 3 and ops["MUFU"] % 3 == 0:
            e = ops["MUFU"] // 3
            fp = sum(ops[k] for k in FP64)
            print(f"  edges={e:2d} len={len(seg):5d} per edge: all {len(seg) / e:6.1f}  FP64 {fp / e:5.1f}  other {(len(seg) - fp) / e:5.1f}"
                  f"   IMAD {ops['IMAD'] / e:4.1f} LOP3 {ops['LOP3'] / e:4.1f} FSEL {ops['FSEL'] / e:4.1f} FFMA {ops['FFMA'] / e:4.1f}")
        seg = []
