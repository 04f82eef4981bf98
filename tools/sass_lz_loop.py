#!/usr/bin/env python3
"""Common-path instruction count of every k_inflate_lz instantiation, read from the SASS.

    python3 tools/sass_lz_loop.py [otezip_b200/csrc/otz_shim.o | otezip_b200/libotezip_b200.so]

Runs `cuobjdump -sass` on the built object or library and, in every k_inflate_lz function, looks at the loops
(backward branches) whose body shuffles a descriptor (SHFL.IDX) and both loads from and stores to shared memory: that
is the match loop of the LZ77 executor.  Along every path once around such a loop (forward branches taken or not,
inner loops not entered) it counts the instructions of the paths that make at least two shared loads and two shared
stores, i.e. that execute whole matches; one match is two loads and two stores per lane.  The figure printed is the
fewest instructions per match over those paths: the cost of a common-case record.  A predicated-off instruction
(@!PT) is not counted.
"""
import os
import re
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_FUNC = re.compile(r"^\s*Function : (\S+)")
_INSN = re.compile(r"^\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;")
_TARGET = re.compile(r"(0x[0-9a-f]+)\s*$")
_KIND = re.compile(r"k_inflate_lzILi(\d+)ELb(\d)ELb(\d)ELb(\d)E")


def cuobjdump():
    p = shutil.which("cuobjdump")
    if p:
        return p
    for c in (os.environ.get("CUDA_HOME", ""), "/usr/local/cuda"):
        if c and os.path.exists(os.path.join(c, "bin", "cuobjdump")):
            return os.path.join(c, "bin", "cuobjdump")
    sys.exit("cuobjdump not found (set CUDA_HOME)")


def functions(text):
    """{mangled name: [(address, predicate, opcode, operands)]}"""
    out, cur = {}, None
    for line in text.splitlines():
        m = _FUNC.match(line)
        if m:
            cur = out.setdefault(m.group(1), [])
            continue
        m = _INSN.match(line)
        if m and cur is not None:
            body = m.group(2)
            pred = ""
            if body.startswith("@"):
                pred, body = body.split(None, 1)
            op, _, rest = body.partition(" ")
            cur.append((int(m.group(1), 16), pred, op, rest))
    return out


def succs(ins, i, index):
    """indices that can follow instruction i (None = leaves the function)"""
    _, pred, op, rest = ins[i]
    if pred == "@!PT":
        return [i + 1]
    uncond = pred in ("", "@PT")
    base = op.split(".")[0]
    if base in ("EXIT", "RET", "BRX", "JMX", "JMP"):
        return [] if uncond else [i + 1]
    if base == "BRA":
        t = index.get(int(_TARGET.search(rest).group(1), 16))
        return [t] if uncond else [t, i + 1]
    return [i + 1]


def common_path(ins):
    """(instructions per match, instructions once around the loop, matches per trip) of the cheapest whole-match trip"""
    index = {a: i for i, (a, _, _, _) in enumerate(ins)}
    best = None
    for j, (_, pred, op, rest) in enumerate(ins):
        if op.split(".")[0] != "BRA" or pred == "@!PT":
            continue
        h = index.get(int(_TARGET.search(rest).group(1), 16))
        if h is None or h > j:
            continue
        body = ins[h:j + 1]
        if not any(o.startswith("SHFL.IDX") for _, _, o, _ in body):
            continue
        # the paths h -> j (the back edge) that stay in [h, j] and enter no inner loop only go forward: one pass in address
        # order keeps, per instruction and (loads, stores) made so far (capped), the fewest instructions to get there
        cost = {h: {(0, 0): 0}}
        for i in range(h, j + 1):
            states = cost.pop(i, None)
            if not states:
                continue
            _, p, o, _ = ins[i]
            live = p != "@!PT"
            dl, ds = int(live and o.startswith("LDS")), int(live and o.startswith("STS"))
            nxt = {}
            for (nl, ns), n in states.items():
                key = (min(nl + dl, _CAP), min(ns + ds, _CAP))
                if key not in nxt or n + live < nxt[key]:
                    nxt[key] = n + live
            if i == j:
                for (nl, ns), n in nxt.items():
                    m = min(nl, ns) // 2
                    if m >= 1 and (best is None or n / m < best[0]):
                        best = (n / m, n, m)
                continue
            for k in succs(ins, i, index):
                if k is None or k <= i or k > j:
                    continue   # leaves the loop, or an inner loop's back edge
                tgt = cost.setdefault(k, {})
                for key, n in nxt.items():
                    if key not in tgt or n < tgt[key]:
                        tgt[key] = n
    return best


_CAP = 8   # loads / stores counted per trip: four matches


def main():
    path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "otezip_b200", "csrc", "otz_shim.o")
    text = subprocess.run([cuobjdump(), "-sass", path], check=True, capture_output=True, text=True).stdout
    rows = []
    for name, ins in functions(text).items():
        m = _KIND.search(name)
        if not m:
            continue
        w, wide, seg, par = m.groups()
        label = "k_inflate_lz<%s, %s, %s, %s>" % (w, "true" if wide == "1" else "false", "true" if seg == "1" else "false",
                                                  "true" if par == "1" else "false")
        rows.append((label, common_path(ins)))
    if not rows:
        sys.exit("no k_inflate_lz function in %s" % path)
    for label, r in sorted(rows):
        if r is None:
            print("%-42s  no match loop found" % label)
        else:
            print("%-42s  %5.1f instructions per common-case match  (%d per trip, %d match%s)"
                  % (label, r[0], r[1], r[2], "" if r[2] == 1 else "es"))


if __name__ == "__main__":
    main()
