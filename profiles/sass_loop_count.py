"""Per-step SASS mnemonic counts of the tape kernel's main loop (the first loop of more than 100 instructions: the full-group
loop, unrolled TAPE_PF = 8 times), in total and without the reset path (the short forward branches around each CALL of
reset_f32_call).
usage: cuobjdump -sass -fun <kernel symbol> libcstr_b200.so > k.sass; python profiles/sass_loop_count.py k.sass [unroll]"""
import re
import sys
from collections import Counter

path = sys.argv[1]
unroll = int(sys.argv[2]) if len(sys.argv) > 2 else 8
ins = []  # (addr, pred, mnemonic, text)
pat = re.compile(r"/\*([0-9a-f]{4,})\*/\s+(.*?);")
for line in open(path):
    m = pat.search(line)
    if not m:
        continue
    addr = int(m.group(1), 16)
    text = m.group(2).strip()
    toks = text.split()
    pred = ""
    if toks[0].startswith("@"):
        pred = toks[0]
        toks = toks[1:]
    ins.append((addr, pred, toks[0], text))
addr_idx = {a: k for k, (a, _, _, _) in enumerate(ins)}
# backward branches -> loops
loops = []
for k, (a, p, mn, t) in enumerate(ins):
    if mn.startswith("BRA"):
        tgt = int(re.search(r"0x([0-9a-f]+)", t).group(1), 16)
        if tgt < a:
            loops.append((addr_idx[tgt], k))
lo, hi = [l for l in loops if l[1] - l[0] > 100][0]  # the first big loop: the full-group main loop
body = range(lo, hi + 1)
# reset regions: forward conditional branches whose skipped range contains a CALL
excl = set()
for k in body:
    a, p, mn, t = ins[k]
    if mn.startswith("BRA") and p:
        tgt = int(re.search(r"0x([0-9a-f]+)", t).group(1), 16)
        if tgt > a and tgt in addr_idx and addr_idx[tgt] <= hi:
            rng = range(k + 1, addr_idx[tgt])
            if any(ins[j][2].startswith("CALL") for j in rng) and len(rng) < 80:
                excl.update(rng)
allc = Counter(ins[k][2].split(".")[0] for k in body)
hot = Counter(ins[k][2].split(".")[0] for k in body if k not in excl)
print(f"loop {ins[lo][0]:#x}..{ins[hi][0]:#x}: {len(body)} instructions, {len(body) - len(excl)} outside the reset path; per step ({unroll} unrolled): "
      f"{len(body) / unroll:.1f} all, {(len(body) - len(excl)) / unroll:.1f} non-reset")
print("mnemonic  all/step  non-reset/step")
for mn, c in sorted(allc.items(), key=lambda x: -x[1]):
    print(f"{mn:10s} {c / unroll:6.2f} {hot[mn] / unroll:6.2f}")
