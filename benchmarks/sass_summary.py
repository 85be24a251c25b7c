"""Per-kernel counts of the Blackwell-native SASS mnemonics in the built library (B200_PROFILING.md, "What proves a
Blackwell-native kernel"): tcgen05.mma -> UTC*MMA, tcgen05.ld/st -> LDTM/STTM, TMA -> UTMALDG/UTMASTG/UBLKCP, cp.async ->
LDGSTS; legacy tensor paths (HMMA/IMMA = mma.sync) listed so their absence is visible.  Runs where cuobjdump is (no GPU):

    python benchmarks/sass_summary.py [lbt_b200/liblbt_b200.so] > profiles/r2_sass_summary.txt

__graft_entry__.build() compares profiles/r2_sass_summary.txt with every build and says when it needs regenerating.
"""
import collections
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MNEMONICS = ['UTCIMMA', 'UTCHMMA', 'UTCQMMA', 'UTCBAR', 'LDTM', 'STTM', 'UTMALDG', 'UTMASTG', 'UBLKCP', 'UTMAPF', 'LDGSTS',
             'SYNCS', 'HMMA', 'IMMA', 'ATOMG', 'REDG', 'RED.']


def summarize(lib):
    cuobjdump = os.environ.get('CUOBJDUMP', '/usr/local/cuda/bin/cuobjdump')
    out = subprocess.run([cuobjdump, '-sass', lib], capture_output=True, text=True, check=True).stdout
    per = collections.OrderedDict()
    cur = None
    for line in out.splitlines():
        m = re.search(r'Function : (\S+)', line)
        if m:
            cur = m.group(1)
            per[cur] = collections.Counter()
            continue
        if cur is None or '/*' not in line:
            continue
        m = re.search(r'^\s*/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_.]+)', line)
        if not m:
            continue
        op = m.group(1)
        per[cur]['_total'] += 1
        for mn in MNEMONICS:
            if op.startswith(mn):
                key = mn.rstrip('.')
                per[cur][key] += 1
                if mn == 'UTCIMMA' and '.2CTA' in op:
                    per[cur]['UTCIMMA.2CTA'] += 1
                if mn == 'UTMALDG' and 'IM2COL' in op:
                    per[cur]['UTMALDG.IM2COL'] += 1
                break
    return per


def demangle(names):
    try:
        r = subprocess.run(['c++filt'], input='\n'.join(names), capture_output=True, text=True, check=True).stdout.splitlines()
        return dict(zip(names, r))
    except Exception:
        return {n: n for n in names}


def render(lib):
    per = summarize(lib)
    pretty = demangle(list(per))
    cols = ['UTCIMMA', 'UTCIMMA.2CTA', 'UTCBAR', 'LDTM', 'STTM', 'UTMALDG', 'UTMALDG.IM2COL', 'UTMASTG', 'LDGSTS', 'SYNCS', 'HMMA', 'IMMA',
            'ATOMG', 'RED', '_total']
    tot = collections.Counter()
    lines = ['# cuobjdump -sass %s : per-kernel instruction counts (sm_100a SASS)' % os.path.relpath(lib, ROOT),
             '# tcgen05.mma -> UTCIMMA (kind::i8), tcgen05.ld -> LDTM, cp.async.bulk.tensor -> UTMALDG, tcgen05.commit -> UTCBAR, '
             'cp.async -> LDGSTS, mbarrier -> SYNCS; HMMA/IMMA = legacy mma.sync (must be 0)',
             ','.join(['kernel'] + cols)]
    for k, c in per.items():
        name = re.sub(r'\(.*$', '', pretty[k].replace('(anonymous namespace)::', '').replace('void ', '')).replace('lbt::', '').replace(',', ';')
        lines.append(','.join([name] + [str(c.get(x, 0)) for x in cols]))
        tot.update(c)
    lines.append(','.join(['TOTAL'] + [str(tot.get(x, 0)) for x in cols]))
    return '\n'.join(lines) + '\n'


if __name__ == '__main__':
    sys.stdout.write(render(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, 'lbt_b200', 'liblbt_b200.so')))
