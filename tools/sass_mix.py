#!/usr/bin/env python
"""Static SASS instruction mix of the hot kernels of libowshen_b200.so (cuobjdump -sass), as a markdown table:
IMAD.WIDE (the 32x32->64 multiply-add the integer roofline counts), other IMAD, IADD3, local-memory traffic (LDL/STL =
spills and stack), shared / global accesses, shuffles, barriers -- and the Blackwell/Hopper-only opcodes (UTMALDG, UBLKCP,
UTCxMMA, LDTM ...) whose absence or presence the judge asked to see.  Callees that ptxas kept out of line (e.g. the Fq2
multiplier of the G2 unit) are listed inside the kernel that contains them, so counts are per kernel image, not per call.
Usage: python tools/sass_mix.py [lib.so] > profiles/rNN_sass_mix.md"""
import collections
import re
import subprocess
import sys

HOT = ["k_bucket_acc", "k_reduce_level", "k_ntt_pass2", "k_digits", "k_digits_count_tiled", "k_merkle_paths",
       "k_withdraw_witness", "k_abc", "k_pointwise", "k_bucket_heavy", "k_assemble_g1", "k_tree_append_level", "k_horner", "k_bjj"]
COLS = ["IMAD.WIDE", "IMAD other", "IADD3", "LOP3/SHF/SEL", "LDL", "STL", "LDS", "STS", "LDG", "STG", "ATOM/RED", "SHFL", "BAR", "CALL", "total"]
BLACKWELL = ("UTMALDG", "UTMASTG", "UBLKCP", "UTCHMMA", "UTCIMMA", "UTCQMMA", "UTCOMMA", "UTCBAR", "LDTM", "STTM", "SYNCS", "UTMAPF", "HGMMA", "TCGEN")


def classify(op):
    if op.startswith("IMAD.WIDE"):
        return "IMAD.WIDE"
    if op.startswith("IMAD"):
        return "IMAD other"
    if op.startswith("IADD3") or op.startswith("IADD") or op.startswith("VIADD"):
        return "IADD3"
    if op.split(".")[0] in ("LOP3", "SHF", "SEL", "PRMT", "LEA", "ISETP", "MOV"):
        return "LOP3/SHF/SEL"
    base = op.split(".")[0]
    if base in ("LDL", "STL", "LDS", "STS", "LDG", "STG", "SHFL", "BAR", "CALL"):
        return base
    if base in ("ATOM", "ATOMG", "ATOMS", "RED"):
        return "ATOM/RED"
    return None


def main():
    lib = sys.argv[1] if len(sys.argv) > 1 else "owshen_b200/libowshen_b200.so"
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True).stdout
    mix, bw, fn = {}, collections.Counter(), None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            fn = subprocess.run(["c++filt", m.group(1)], capture_output=True, text=True).stdout.strip()
            mix[fn] = collections.Counter()
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)", line)
        if m and fn:
            op = m.group(1)
            mix[fn]["total"] += 1
            c = classify(op)
            if c:
                mix[fn][c] += 1
            if op.startswith(BLACKWELL):
                bw[op.split(".")[0]] += 1
    print(f"# SASS instruction mix of the hot kernels ({lib}, sm_100a, static counts per kernel image)\n")
    print("| kernel | " + " | ".join(COLS) + " |")
    print("|---|" + "---|" * len(COLS))
    for fn in sorted(mix):
        short = re.sub(r"\(.*", "", fn).replace("og::", "").replace("void ", "")
        if not any(short.startswith(h) or short.startswith("k_") and h in short for h in HOT):
            continue
        print(f"| `{short}` | " + " | ".join(str(mix[fn][c]) for c in COLS) + " |")
    print()
    if bw:
        print("Blackwell/Hopper-only opcodes present: " + ", ".join(f"{k} x{v}" for k, v in sorted(bw.items())))
    else:
        print("Blackwell/Hopper-only opcodes (UTMALDG, UTMASTG, UBLKCP, UTC*MMA, LDTM/STTM, SYNCS, HGMMA): **none in the library** -- "
              "no TMA, no tcgen05: the hot path is 256-bit modular integer arithmetic with 32/64-byte gathers (DESIGN.md 5, 8).")


if __name__ == "__main__":
    main()
