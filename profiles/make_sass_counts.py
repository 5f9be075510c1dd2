#!/usr/bin/env python
"""Static SASS instruction counts of the Cornell warp-queue kernels, by opcode class, from `cuobjdump -sass` of the trimmed
build's object (vecchio_b200/csrc/vk_warpq_simple.o).  Static counts: every instruction of the kernel's code once, however
often it runs -- what the compiler made, before any GPU run.

    python profiles/make_sass_counts.py BEFORE.o AFTER.o > profiles/r3_cornell_warpq_sass_counts.md

BEFORE.o: vk_warpq_simple.o built from the parent commit; AFTER.o: the same object of this tree."""
import collections
import re
import subprocess
import sys

CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"
# (column, kernel symbol pattern): the single-frame instances only
KERNELS = [("k_warpq_flat", r"k_warpq_flatILb0E8OneFrame"), ("k_warpq_flat_static<Cornell>", r"k_warpq_flat_static.*8OneFrame")]
# classes the change is about, in the order of the table; everything else is summed under "other"
ROWS = ["BRA", "BSSY", "BSYNC", "NOP", "LDCU.U8", "LDCU", "LDC", "MOV", "UMOV", "IMAD.MOV", "ISETP", "UISETP", "FFMA", "FMUL", "FADD",
        "FSETP", "FSEL", "FMNMX", "MUFU", "LDS", "STS", "SHFL", "VOTE"]


def kernels(obj):
    text = subprocess.run([CUOBJDUMP, "-sass", obj], capture_output=True, text=True, check=True).stdout
    out, cur = {}, None
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if m and cur:
            ins = re.sub(r"^@!?U?P\w+\s+", "", m.group(1).strip())
            out[cur].append(ins.split()[0])
    return out


def classify(op):
    if op.startswith("LDCU.U8"):
        return "LDCU.U8"
    if op.startswith("IMAD.MOV"):
        return "IMAD.MOV"
    base = op.split(".")[0]
    return base if base in ROWS else "other"


def counts(obj, pat):
    ks = kernels(obj)
    hit = [k for k in ks if re.search(pat, k)]
    if not hit:
        return None
    c = collections.Counter(classify(op) for op in ks[hit[0]])
    c["total"] = len(ks[hit[0]])
    return c


def main():
    before, after = sys.argv[1], sys.argv[2]
    cols = [("before: " + KERNELS[0][0], counts(before, KERNELS[0][1]))]
    cols += [("after: " + name, counts(after, pat)) for name, pat in KERNELS]
    cols = [(n, c) for n, c in cols if c is not None]
    print("# Static SASS instruction counts of the Cornell warp-queue kernel (sm_100a, `cuobjdump -sass`)\n")
    print("Made by `profiles/make_sass_counts.py` from `vecchio_b200/csrc/vk_warpq_simple.o` of the parent commit (before) and of this")
    print("change (after), `OneFrame` instances.  Static counts: each instruction of the kernel's code once, not how often it runs.")
    print("`k_warpq_flat` is the generic kernel (`VECCHIO_NO_STATIC_FLAT=1`, and every simple scene without a compiled shape);")
    print("after the change both kernels shade each batch with its queue's class body.\n")
    print("| class | " + " | ".join(n for n, _ in cols) + " |")
    print("|---|" + "---|" * len(cols))
    for r in ROWS + ["other", "total"]:
        print(f"| `{r}` | " + " | ".join(str(c.get(r, 0)) for _, c in cols) + " |")
    print("| code KB | " + " | ".join(f"{c['total'] * 16 / 1024:.1f}" for _, c in cols) + " |")


if __name__ == "__main__":
    main()
