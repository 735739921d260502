"""Opcode histogram of the hot loop of a kernel from `cuobjdump -sass` output (no GPU needed).

usage: python profiles/tools/sass_loop.py <lib.so> <kernel-name-substring> [--dump] [--reuse]
The hot loop is taken as the innermost backward branch span that holds the most VIMNMX/FMNMX instructions.
"""
import collections
import re
import subprocess
import sys


def kernels(so):
    txt = subprocess.run(["cuobjdump", "-sass", so], capture_output=True, text=True).stdout
    cur, out = None, {}
    for ln in txt.splitlines():
        m = re.search(r"Function : (\S+)", ln)
        if m:
            cur = m.group(1)
            out[cur] = []
            continue
        m = re.match(r"\s+/\*([0-9a-f]{4,6})\*/\s+(.*?);", ln)
        if m and cur:
            out[cur].append((int(m.group(1), 16), m.group(2).strip()))
    return out


def opcode(ins):
    t = ins.split()
    if t[0].startswith("@"):
        t = t[1:]
    return t[0]


def hot_loop(ins, key=None):
    if key is None:  # the packed kernels are recognised by their int16x2 min/max, the others by any min/max
        key = (".S16x2", ".16x2") if any(".S16x2" in s for _, s in ins) else ("VIMNMX", "FMNMX", "VIADDMNMX")
    addr = [a for a, _ in ins]
    loops = []
    for i, (a, s) in enumerate(ins):
        m = re.search(r"BRA(?:\.\w+)* (?:`\(\.L_x_\d+\)|0x([0-9a-f]+))", s)
        if not m or not m.group(1):
            continue
        tgt = int(m.group(1), 16)
        if tgt >= a:
            continue
        j = addr.index(tgt) if tgt in addr else None
        if j is None:
            continue
        body = ins[j:i + 1]
        n = sum(1 for _, x in body if any(k in x for k in key))
        if n:
            loops.append((n, body))
    # the smallest loop that holds at least half of the min/max instructions of the richest one: the row loop, also
    # where the compiler has peeled a copy of its body into the enclosing task loop
    top = max((n for n, _ in loops), default=0)
    best = min((b for n, b in loops if 2 * n >= top), key=len, default=[])
    return best


def regs(tok, width):
    m = re.match(r"\[?-?R(\d+)", tok)
    return set(range(int(m.group(1)), int(m.group(1)) + width)) if m and m.group(1) else set()


def width(op, tok):
    if ".64" in tok or "WIDE" in op:
        return 2
    if "[" in tok:  # a 32-bit address (shared memory)
        return 1
    return 4 if op.endswith(".128") else (2 if op.endswith(".64") else 1)


def store_reuse(body):
    """Global stores / cp.async in the loop one of whose operand registers is written again before the loop's end."""
    out = []
    for k, (a, s) in enumerate(body):
        op = opcode(s)
        if not (op.startswith("STG") or op.startswith("LDGSTS")):
            continue
        ops = [t.strip() for t in s.split(None, 2 if s.startswith("@") else 1)[-1].split(",")]
        used = set().union(*(regs(t, width(op, t)) for t in ops))
        for b, t in body[k + 1:]:
            top = opcode(t)
            if top.startswith(("ST", "LDGSTS", "BRA", "BSSY", "BSYNC", "DEPBAR", "LDGDEPBAR", "CCTL", "ISETP", "UI", "UL", "UM", "US", "PLOP")):
                continue
            dst = t.split(None, 2 if t.startswith("@") else 1)[-1].split(",")[0].strip()
            hit = regs(dst, width(top, dst)) & used
            if hit:
                out.append((a, s, b, t))
                break
    return out


if __name__ == "__main__":
    so, pat = sys.argv[1], sys.argv[2]
    for name, ins in kernels(so).items():
        if pat not in name:
            continue
        body = hot_loop(ins)
        h = collections.Counter(opcode(s) for _, s in body)
        print(f"== {name}: {len(ins)} instr, hot loop {len(body)} instr [{body[0][0]:#x}..{body[-1][0]:#x}]" if body else f"== {name}: no loop")
        for k, v in h.most_common():
            print(f"   {v:5d} {k}")
        if "--reuse" in sys.argv:
            r = store_reuse(body)
            print(f"   stores whose operand registers are rewritten later in the step: {len(r)}")
            for a, s, b, t in r:
                print(f"     {a:06x} {s}  <-  {b:06x} {t}")
        if "--dump" in sys.argv:
            for a, s in body:
                print(f"  {a:06x} {s}")
