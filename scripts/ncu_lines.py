#!/usr/bin/env python
"""Rank the source lines of the first kernel in an .ncu-rep by executed warp instructions (per CTA).
usage: python scripts/ncu_lines.py rep.ncu-rep [top_n]"""
import csv, io, re, subprocess, sys
rep = sys.argv[1]; top = int(sys.argv[2]) if len(sys.argv) > 2 else 60
src = subprocess.run(['ncu', '-i', rep, '--page', 'source', '--csv', '--print-source', 'cuda,sass'], capture_output=True, text=True).stdout
rows = list(csv.reader(io.StringIO(src)))
hi = [i for i, r in enumerate(rows) if r and r[0] == 'Line No']
names = [rows[h - 1][1] for h in hi]
def I(x):
    try: return int(x)
    except: return 0
per = []
first = names[0]
grid = None
for n, h0 in enumerate(hi):
    if n > 0 and rows[h0 - 2][0] == 'File Path' and re.search(r'csrc/marlnav_[a-z_]+\.cu$', rows[h0 - 2][1]) and n > 0 and per: break
    h = rows[h0]; ix = {nm: i for i, nm in enumerate(h)}
    end = hi[n + 1] - 2 if n + 1 < len(hi) else len(rows)
    fname = rows[h0 - 2][1].split('/')[-1].replace('marlnav_', '')
    for r in rows[h0 + 1:end]:
        if len(r) < 10 or r[0] == '': continue
        per.append((I(r[ix['Instructions Executed']]), I(r[ix['L1 Wavefronts Shared Excessive']]), I(r[ix['# Samples']]), fname + ':' + r[0], r[1][:100]))
raw = subprocess.run(['ncu', '-i', rep, '--page', 'raw', '--csv'], capture_output=True, text=True).stdout
rr = list(csv.reader(io.StringIO(raw)))
g = float(rr[2][rr[0].index('launch__grid_size')])
tot = sum(p[0] for p in per)
print(first[:100]); print('warp inst', tot, 'per CTA', round(tot / g, 1), 'excess smem wavefronts per CTA', round(sum(p[1] for p in per) / g, 1))
for p in sorted(per, key=lambda x: -x[0])[:top]:
    print(f'{p[0]/g:7.1f} {100*p[0]/tot:5.1f}% excwf={p[1]/g:6.1f} smp={p[2]:5d} {p[3]}: {p[4]}')
