#!/usr/bin/env python
"""Static instruction count of the strip kernel's row loop (stage_rows, the FULL instance) in a SASS dump:

    cuobjdump -sass -fun <label_pass_fast instance> csrc/build/label_pass.o > x.sass; python scripts/sass_loop_count.py x.sass

The loop is [target, back edge] of the first unconditional backward branch whose range holds the first LDS.64."""
import re, sys
ins = []
for line in open(sys.argv[1]):
    m = re.match(r'\s+/\*([0-9a-f]{4,5})\*/\s+(.*?);', line)
    if m:
        ins.append((int(m.group(1), 16), m.group(2).strip()))
first_lds = next(a for a, t in ins if t.startswith('LDS.64'))
loop = None
for a, t in ins:
    m = re.search(r'BRA(?:\.U)?\s+(?:!?U?P\d,\s*)?0x([0-9a-f]+)', t)
    if m and not t.startswith('@') :
        tgt = int(m.group(1), 16)
        if tgt <= first_lds < a:
            loop = (tgt, a); break
lo, hi = loop
body = [(a, t) for a, t in ins if lo <= a <= hi]
op = lambda t: re.sub(r'^@!?U?P\w+\s+', '', t).split()[0]
print(f"{sys.argv[1]}: total {len(ins)}  loop [{lo:#x},{hi:#x}] {len(body)} instructions")
from collections import Counter
c = Counter(op(t).split('.')[0] for a, t in body)
print("  loop body by opcode:", dict(c.most_common(14)))
