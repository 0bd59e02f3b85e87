#!/usr/bin/env python
"""Per-kernel SASS instruction counts of the shipped library -> profiles/sass_summary.txt.

Evidence for which hardware paths each kernel uses (B200_PROFILING.md, "What proves a Blackwell-native
kernel"): UTC*MMA = tcgen05.mma, LDTM/STTM = tcgen05.ld/st, UTMALDG/UTMASTG = TMA tensor copies,
UBLKCP = cp.async.bulk, FFMA2/FMUL2 = packed fp32, RED/ATOM = reductions.  __graft_entry__.build() writes
the same summary to sevenn_b200/csrc/build/sass_summary.txt; runs without a GPU (cuobjdump needs none)."""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
WATCH = ['UTCHMMA', 'UTCQMMA', 'UTCIMMA', 'UTCMMA', 'LDTM', 'STTM', 'UTMALDG', 'UTMASTG', 'UBLKCP', 'UTCBAR', 'SYNCS',
         'FFMA2', 'FMUL2', 'FADD2', 'FFMA', 'HMMA', 'LDGSTS', 'RED', 'ATOM', 'LDG', 'STG', 'LDS', 'STS', 'SHFL']


def demangle(names):
    try:
        out = subprocess.run(['c++filt'], input='\n'.join(names), capture_output=True, text=True).stdout.splitlines()
        return dict(zip(names, out))
    except Exception:
        return {n: n for n in names}


def main(lib=None, out=None):
    lib = lib or os.path.join(ROOT, 'sevenn_b200', 'lib', 'libsevenn_b200.so')
    out = out or os.path.join(ROOT, 'profiles', 'sass_summary.txt')
    sass = subprocess.run(['cuobjdump', '-sass', lib], capture_output=True, text=True).stdout
    counts = collections.OrderedDict()
    cur = None
    for line in sass.splitlines():
        m = re.match(r'\s*Function : (\S+)', line)
        if m:
            cur = counts.setdefault(m.group(1), collections.Counter())
            continue
        if cur is None:
            continue
        m = re.match(r'\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z][A-Z0-9_]*)', line)
        if m:
            op = m.group(1)
            cur['_total'] += 1
            for w in WATCH:
                if op == w or (w in ('RED', 'ATOM') and op.startswith(w)) or (w.startswith('UTC') and op.startswith(w)):
                    cur[w] += 1
                    break
    names = demangle(list(counts))
    total = collections.Counter()
    lines = []
    for fn, c in counts.items():
        total.update(c)
        nm = re.sub(r'\(.*', '', names[fn])
        nm = nm.replace('s7b::', '')
        cols = ' '.join(f'{w}={c[w]}' for w in WATCH if c[w])
        lines.append(f'{nm[:110]:<110} n={c["_total"]:<6} {cols}')
    head = [f'# SASS instruction counts per kernel of {os.path.relpath(lib, ROOT)} (tools/sass_summary.py; cuobjdump -sass)',
            '# ' + ' '.join(f'{w}={total[w]}' for w in WATCH if total[w]) + f'  kernels={len(counts)}', '']
    with open(out, 'w') as f:
        f.write('\n'.join(head + sorted(lines)) + '\n')
    return total


if __name__ == '__main__':
    t = main(*(sys.argv[1:3]))
    print({k: v for k, v in t.items() if k != '_total'})
