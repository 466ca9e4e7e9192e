r"""Attribute the SASS of a render kernel to its device functions: walk the instructions in address order and assign each to
the function of the source file whose source line was seen last (inlined rt_math/rt_shade/rt_trace code inherits it).
usage: python profiles/ncu_body_breakdown.py file.ncu-rep [source-file-in-csrc function-regex start-body]
       (defaults: the USE_FP16 kernel, rt_half.cuh and its device functions)"""
import csv
import re
import subprocess
import sys

src = sys.argv[1]
SRC_FILE = sys.argv[2] if len(sys.argv) > 2 else 'rt_half.cuh'
FUNCS = sys.argv[3] if len(sys.argv) > 3 else r'coop_\w+|ref_line_test_h|sphere_test_h|scatter_h|camera_ray_h|hit_point_h|sky_h|random_in_unit_sphere_h|best_update'
START = sys.argv[4] if len(sys.argv) > 4 else 'k_render_h'
pool_src = open(__file__.rsplit('/', 2)[0] + '/dd2360-raytracing_b200/csrc/' + SRC_FILE).read().splitlines()
# line -> enclosing function name in SRC_FILE
func_of, cur = {}, 'header'
for i, l in enumerate(pool_src, 1):
    m = re.search(r'\b(' + FUNCS + r')\b\s*\(', l)
    if m and ('__device__' in l or '__global__' in l or l.startswith('template') or 'void' in l or 'bool' in l or 'Hit' in l) and ';' not in l.split('{')[0]:
        cur = m.group(1)
    func_of[i] = cur
txt = subprocess.run(['ncu', '-i', src, '--page', 'source', '--csv', '--print-source', 'cuda,sass'], capture_output=True, text=True).stdout
rows, fname, hdr, line = [], None, None, None
for r in csv.reader(txt.splitlines()):
    if not r:
        continue
    if r[0] == 'File Path':
        fname = r[1].split('/')[-1]
    elif r[0] == 'Line No':
        hdr = r
    elif hdr and r[0].isdigit():
        line = int(r[0])
    elif hdr and r[0] == '' and len(r) > 10 and r[2].startswith('0x'):
        try:
            rows.append((int(r[2], 16), fname, line, int(r[hdr.index('Instructions Executed')]), int(r[hdr.index('Thread Instructions Executed')]), r[3].strip()))
        except ValueError:
            pass
rows.sort()
seen = set()
agg, cur = {}, START
for addr, f, ln, wi, ti, sass in rows:
    if addr in seen:
        continue
    seen.add(addr)
    if f == SRC_FILE and ln in func_of:
        cur = func_of[ln]
    a = agg.setdefault(cur, [0, 0, 0])
    a[0] += wi; a[1] += ti; a[2] += 1
tw = sum(a[0] for a in agg.values()); tt = sum(a[1] for a in agg.values())
print(f'{"body":16s} {"sass":>6s} {"warp-inst %":>11s} {"thread-inst %":>13s} {"active":>7s}')
for k, a in sorted(agg.items(), key=lambda kv: -kv[1][0]):
    print(f'{k:16s} {a[2]:6d} {100*a[0]/tw:11.1f} {100*a[1]/tt:13.1f} {a[1]/max(a[0],1):7.1f}')
print('total warp instructions', tw, 'thread instructions', tt)
