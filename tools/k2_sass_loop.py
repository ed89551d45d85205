#!/usr/bin/env python3
"""Static SASS summary of K2's bilinear sampling loops: for each instantiation of k2_kernel in an object or library, the
innermost loop around each group of 16 LDG.E.U8 (one group of four samples per thread), its instruction count, the
conversion-pipe instructions in it (I2F / F2I / FRND), reciprocals, reconvergence points, shared atomics, and where in the
loop the loads sit.  No GPU needed.

    python tools/k2_sass_loop.py aruco3_b200/csrc/build/k2_decode.o
"""
import re
import subprocess
import sys
from collections import Counter


def kernels(path):
    sass = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    out, cur = {}, None
    for ln in sass.splitlines():
        m = re.match(r"\s*Function : (\S+)", ln)
        if m:
            cur = m.group(1) if "k2_kernel" in m.group(1) else None
            if cur:
                out[cur] = []
            continue
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?);", ln)
        if m and cur:
            out[cur].append((int(m.group(1), 16), m.group(2).strip()))
    return out


def main():
    for name, ins in kernels(sys.argv[1]).items():
        form = "CTA per candidate (WIDE)" if "ILb1" in name else "warp per candidate"
        addr = {a: k for k, (a, _) in enumerate(ins)}
        ld = [k for k, (_, t) in enumerate(ins) if "LDG.E.U8" in t]
        print(f"k2_kernel, {form}: {len(ins)} SASS instructions, {len(ld)} LDG.E.U8")
        for g in range(0, len(ld), 16):
            cl, best = ld[g:g + 16], None
            for k, (_, t) in enumerate(ins):
                m = re.search(r"\bBRA\s+(?:`\()?0x([0-9a-f]+)", t)
                if m and not t.startswith("BRA.DIV"):
                    s = addr.get(int(m.group(1), 16))
                    if s is not None and s < cl[0] and k > cl[-1] and (best is None or k - s < best[1] - best[0]):
                        best = (s, k)
            if best is None:
                continue
            s, e = best
            body = [t for _, t in ins[s:e + 1]]
            ops = Counter(re.match(r"(?:@!?U?P\w+\s+)?([A-Z0-9_]+)", t).group(1) for t in body)
            print(f"  loop of {len(body)} instructions: conversions (I2F/F2I/FRND) {sum(ops[o] for o in ('I2F', 'F2I', 'FRND'))}, "
                  f"MUFU.RCP {sum(1 for t in body if 'MUFU.RCP' in t)}, BSSY {ops['BSSY']}, IMAD.WIDE {sum(1 for t in body if 'IMAD.WIDE' in t)}, "
                  f"ATOMS {ops['ATOMS']}, generic ATOM {ops['ATOM']}, LDG.E.U8 {len(cl)} at +{cl[0] - s} … +{cl[-1] - s}")


if __name__ == "__main__":
    main()
