"""Instruction mix of the hot kernels in the built library (cuobjdump -sass): evidence for the roofline accounting -- the 32x32->64
products a gate evaluation executes (IMAD.WIDE.U32[.X]), the non-product IMADs ptxas places on the same pipe, 256-bit global accesses
(LDG/STG.E.ENL2.256), bulk copies (UBLKCP), tensor-core instructions (UTC*MMA, LDTM) and local-memory traffic (STL/LDL: must be 0 in the check kernels).
    python scripts/sass_mix.py > profiles/rNN_sass_mix.txt"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "plonk_gadgets_b200", "libpg_b200.so")
HOT = ["k_check_tc", "k_check_progILi0E", "k_check_progILi2E", "k_check_gates_walk", "k_check_gatesILi5E", "k_check_gates", "k_check_rowparILi0E", "k_batch_invINS_15MaybeEqualFused",
       "k_batch_invINS_8InvPlain", "RangePreILb1ELb0E", "RangePreILb1ELb1E", "RangePostILb1ELb0E", "k_materialize_tiled", "k_ntt_pass", "MsmBucketBody"]
KEYS = ["IMAD.WIDE.U32.X", "IMAD.WIDE.U32", "IMAD.WIDE", "IMAD.HI.U32", "IMAD.X", "IMAD.MOV", "IMAD.MOV.U32", "IMAD.IADD", "IMAD.SHL", "IMAD", "IADD3.X", "IADD3",
        "LOP3.LUT", "SEL", "MOV", "LDG.E.ENL2.256", "STG.E.ENL2.256", "LDG.E.128", "LDG.E", "LDS.128", "UBLKCP.G.S", "STL", "LDL", "STL.64", "LDL.64", "LDL.LU", "BAR.SYNC"]


def main():
    out = subprocess.run(["cuobjdump", "-sass", LIB], capture_output=True, text=True, check=True).stdout
    rev = subprocess.run(["git", "-C", ROOT, "rev-parse", "--short", "HEAD"], capture_output=True, text=True).stdout.strip()
    print(f"# SASS instruction mix of {os.path.relpath(LIB, ROOT)} (sm_100a), built from the tree at/after git {rev}; whole kernel, static counts")
    cur, mix = None, {}
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1); mix[cur] = collections.Counter(); continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_.]*)", line)
        if m and cur:
            op = m.group(1)
            mix[cur][op] += 1
            mix[cur]["*"] += 1
    for want in HOT:
        for name, c in mix.items():
            if want not in name:
                continue
            wide = sum(v for k, v in c.items() if k.startswith("IMAD.WIDE") or k.startswith("IMAD.HI"))
            other_imad = sum(v for k, v in c.items() if k.startswith("IMAD") and not (k.startswith("IMAD.WIDE") or k.startswith("IMAD.HI")))
            local = sum(v for k, v in c.items() if k.startswith("STL") or k.startswith("LDL"))
            print(f"\n{name}\n  instructions {c['*']}; 32x32->64 products (IMAD.WIDE*/IMAD.HI*) {wide}; other IMAD* {other_imad}; "
                  f"local memory (STL*/LDL*) {local}")
            shown = sorted(((k, v) for k, v in c.items() if k != "*" and v >= max(3, c["*"] // 200)), key=lambda kv: -kv[1])
            print("  " + ", ".join(f"{k} {v}" for k, v in shown))
            special = {k: v for k, v in c.items() if "ENL2" in k or "UBLKCP" in k or k.startswith("STL") or k.startswith("LDL") or k.startswith("UTC") or k.startswith("LDTM")}
            if special:
                print("  256-bit / bulk / local / tensor core: " + ", ".join(f"{k} {v}" for k, v in sorted(special.items())))


if __name__ == "__main__":
    sys.exit(main())
