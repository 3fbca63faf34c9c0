"""Static size of a kernel's hot loop: disassembles <lib.so>, finds in kernel <symbol-substring> the smallest loop
(backward branch) that contains all of the given marker mnemonics, and prints its instruction count by mnemonic
plus the count outside side exits (blocks that end in CALL / EXIT / a jump out of the loop are listed separately).
No GPU needed: used to compare symbol-loop versions before spending GPU time (DESIGN.md section 7).
usage: sass_loop.py <lib.so> <kernel-substring> [marker ...]      (default markers: BREV POPC)"""
import re
import subprocess
import sys
from collections import Counter


def kernel_sass(so, sym):
    txt = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True, check=True).stdout
    ins, on = [], False
    for ln in txt.splitlines():
        if "Function :" in ln:
            on = sym in ln
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,})\*/\s+(.*?);", ln)
        if on and m:
            ins.append((int(m.group(1), 16), m.group(2).strip()))
    return ins


def hot_loop(ins, markers):
    best = None
    for a, t in ins:
        m = re.search(r"\bBRA\b.*?(0x[0-9a-f]+)\s*$", t)
        if not m:
            continue
        tgt = int(m.group(1), 16)
        if tgt >= a:
            continue
        body = [(x, y) for x, y in ins if tgt <= x <= a]
        if all(any(re.search(rf"\b{mk}\b", y) for _, y in body) for mk in markers):
            if best is None or len(body) < len(best):
                best = body
    return best


def main():
    so, sym = sys.argv[1], sys.argv[2]
    markers = sys.argv[3:] or ["BREV", "POPC"]
    best = hot_loop(kernel_sass(so, sym), markers)
    if best is None:
        sys.exit("no loop holds all markers")
    lo, hi = best[0][0], best[-1][0]
    # split into basic blocks at branch targets / after unconditional transfers
    targets = set()
    for a, t in best:
        m = re.search(r"(0x[0-9a-f]+)\s*$", t)
        if m and re.search(r"\b(BRA|BSSY|CALL)\b", t):
            targets.add(int(m.group(1), 16))
    blocks, cur = [], []
    for a, t in best:
        if a in targets and cur:
            blocks.append(cur)
            cur = []
        cur.append((a, t))
        if re.search(r"\b(BRA|EXIT|CALL|RET)\b", t) and not t.startswith("@"):
            blocks.append(cur)
            cur = []
    if cur:
        blocks.append(cur)
    side = 0
    for b in blocks:
        last = b[-1][1]
        m = re.search(r"\bBRA\b.*?(0x[0-9a-f]+)\s*$", last)
        out_jump = m and not (lo <= int(m.group(1), 16) <= hi) and not last.startswith("@")
        if re.search(r"\b(CALL|EXIT)\b", last) or out_jump:
            side += len(b)
    ops = Counter(re.sub(r"^@!?U?P\d+\s+", "", t).split()[0].split(".")[0] for _, t in best)
    print(f"{sym}: loop {lo:#x}..{hi:#x}: {len(best)} instructions, {side} in side-exit blocks, {len(best) - side} on the loop paths")
    print("  " + "  ".join(f"{k}:{v}" for k, v in ops.most_common(14)))


if __name__ == "__main__":
    try:
        main()
    except BrokenPipeError:  # output piped into head
        pass
