#!/usr/bin/env python3
"""Kernel-by-kernel comparison of two builds of libvecchio_gpu.so (`make gpu` in each tree, no GPU needed).

    python scripts/compare_kernels.py BASE_TREE HEAD_TREE [--changed KERNEL ..]

Reads each tree's vecchio_b200/csrc/ptxas_*.log (registers, stack frame, spill stores / loads) and the
`cuobjdump -sass` of vecchio_b200/lib/libvecchio_gpu.so.  Kernels are matched by demangled name and template
arguments, with the work domain (OneFrame / FrameArgs / ListArgs / FrameListArgs) as the last template argument; the older
form of a domain kernel, `X_frames<a..>` / `X_list<a..>`, maps to `X<a.., FrameArgs>` / `X<a.., ListArgs>`,
and any other kernel to itself with the domain OneFrame.  SASS verdicts:
    same          identical instructions
    local-slots   identical once the offsets of local loads / stores are masked (a different stack-slot assignment)
    same-ops      the same multiset of opcodes
    DIFF          anything else
A head kernel of a domain the base build has no kernel of at all is listed as NEW with its resources, beside those of
its ListArgs twin (the same kernel over a pixel list of one frame) when the head build has one.
Exit status 0 when every base kernel is in the head build and every head kernel either is in the base build or NEW,
every matched kernel keeps its resources, every single-frame kernel is `same` and every other one `same` or
`local-slots`.  A kernel named after --changed (its demangled name without namespace or arguments, e.g.
k_to_color) is one the change means to alter, add or remove: it is listed with its verdict, as NEW when the base
build lacks it or as REMOVED when the head build does, and does not fail the comparison."""
import collections, glob, os, re, shutil, subprocess, sys

DOMAINS = ("OneFrame", "FrameArgs", "ListArgs", "FrameListArgs")


def demangle(names):
    tool = shutil.which("c++filt") or shutil.which("cu++filt")
    out = subprocess.run([tool], input="\n".join(names), capture_output=True, text=True, check=True).stdout
    return dict(zip(names, out.splitlines()))


def key_of(dem):
    """'void ns::k<a, b, FrameArgs>(..)' or 'void ns::k_frames<a, b>(.., FrameArgs)' -> ('ns::k<a, b>', 'FrameArgs')"""
    depth, cut = 0, len(dem)
    for i, ch in enumerate(dem):
        depth += ch == "<"
        depth -= ch == ">"
        if ch == "(" and depth == 0:
            cut = i
            break
    head, params = dem[:cut].removeprefix("void "), dem[cut:]
    m = re.fullmatch(r"(.*)<(.*), (\w+)>", head)
    if m and m.group(3) in DOMAINS:
        return f"{m.group(1)}<{m.group(2)}>", m.group(3)
    m = re.fullmatch(r"(.*?)_(frames|list)(<.*)?", head)
    if m and re.search(r"(FrameArgs|ListArgs)\)$", params):
        return m.group(1) + (m.group(3) or ""), "FrameArgs" if m.group(2) == "frames" else "ListArgs"
    return head, "OneFrame"


def load(tree):
    res = {}
    for log in glob.glob(os.path.join(tree, "vecchio_b200/csrc/ptxas_*.log")):
        entry = None
        for line in open(log):
            if m := re.search(r"Compiling entry function '(\w+)'", line):
                entry = m.group(1)
            elif entry and (m := re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", line)):
                res.setdefault(entry, {}).update(stack=int(m[1]), st=int(m[2]), ld=int(m[3]))
            elif entry and (m := re.search(r"Used (\d+) registers", line)):
                res.setdefault(entry, {})["regs"] = int(m[1])
                entry = None
    so = os.path.join(tree, "vecchio_b200/lib/libvecchio_gpu.so")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    sass, cur = {}, None
    for line in subprocess.run([cuobjdump, "-sass", so], capture_output=True, text=True, check=True).stdout.splitlines():
        if m := re.match(r"\s+Function : (\S+)", line):
            cur = sass.setdefault(m.group(1), [])
        elif cur is not None and (m := re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)):
            cur.append(m.group(1))
    names = demangle(sorted(sass))
    kernels = {}
    for mangled, code in sass.items():
        k = key_of(names[mangled])
        if k in kernels:
            sys.exit(f"{tree}: two kernels map to {k}")
        kernels[k] = (mangled, code, res.get(mangled))
    return kernels


def verdict(a, b):
    if a == b:
        return "same"
    mask = lambda code: [re.sub(r"\[(R\d+)(\+0x[0-9a-f]+)?\]", r"[\1+off]", i) if re.match(r"(@!?U?P\w+ )?(LDL|STL)", i) else i for i in code]
    if mask(a) == mask(b):
        return "local-slots"
    ops = lambda code: collections.Counter(re.sub(r"^@!?U?P\w+ ", "", i).split(" ")[0] for i in code)
    return "same-ops" if ops(a) == ops(b) else "DIFF"


def main():
    args = sys.argv[1:]
    if len(args) < 2 or (len(args) > 2 and args[2] != "--changed"):
        sys.exit(__doc__)
    changed = set(args[3:])
    base, head = load(args[0]), load(args[1])
    ok = True
    fmt = lambda r: "-" if r is None else f"{r['regs']}r {r['stack']}s {r['st']}/{r['ld']}"
    base_domains = {d for _, d in base}
    short = lambda k: re.sub(r"<.*", "", k[0]).split("::")[-1]
    new = sorted(k for k in head.keys() - base.keys() if k[1] not in base_domains or short(k) in changed)
    removed = sorted(k for k in base.keys() - head.keys() if short(k) in changed)
    for k in sorted(base.keys() - head.keys() - set(removed)) + sorted(head.keys() - base.keys() - set(new)):
        print(f"UNMATCHED {'base' if k in base else 'head'}: {k[0]} [{k[1]}]")
        ok = False
    tally = collections.Counter()
    for k in removed:
        print(f"{k[0][:72]:<72} {k[1]:<13} {fmt(base[k][2]):>16}  REMOVED")
        tally[(k[1], "REMOVED")] += 1
    if new:
        print(f"{'new kernel':<72} {'domain':<13} {'head':>16} {'ListArgs twin':>16}")
    for k in new:
        twin = head.get((k[0], "ListArgs"))
        print(f"{k[0][:72]:<72} {k[1]:<13} {fmt(head[k][2]):>16} {fmt(twin[2]) if twin else '-':>16}  NEW")
        tally[(k[1], "NEW")] += 1
    print(f"{'kernel':<72} {'domain':<9} {'base':>16} {'head':>16}  sass")
    for k in sorted(base.keys() & head.keys()):
        (_, ca, ra), (_, cb, rb) = base[k], head[k]
        v = verdict(ca, cb)
        bad = ra != rb or v in ("same-ops", "DIFF") or (k[1] == "OneFrame" and v != "same")
        if bad and short(k) in changed:
            v, bad = v + " (changed on purpose)", False
        ok &= not bad
        tally[(k[1], v)] += 1
        print(f"{k[0][:72]:<72} {k[1]:<9} {fmt(ra):>16} {fmt(rb):>16}  {v}{'  <--' if bad else ''}")
    print("; ".join(f"{d} {v}: {n}" for (d, v), n in sorted(tally.items())), f"-> {'OK' if ok else 'FAIL'}")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
