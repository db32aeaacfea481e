"""Per-kernel counts of the SASS mnemonics that prove a Blackwell-native kernel (B200_PROFILING.md): UTC*MMA = tcgen05.mma,
LDTM/STTM = tcgen05.ld/st, UTMALDG/UTMASTG = TMA tensor load/store (.MULTICAST = cluster multicast), UTCBAR = tcgen05.commit,
HMMA would be the legacy mma.sync path.  Written to profiles/sass_opcodes.txt when run as a script, and to
hawkeye_b200/build/sass_opcodes.txt by __graft_entry__.build()."""
import collections
import os
import re
import subprocess
import sys

PAT = re.compile(r'\b(UTC[A-Z]*MMA|LDTM|STTM|UTMALDG|UTMASTG|UBLKCP|UTCBAR|UTCCP|HMMA|HGMMA|SYNCS|MAPA|UCGABAR_ARV|LDGSTS)\b[.\w]*')


def summarize(so_path):
    out = subprocess.run(['cuobjdump', '-sass', so_path], capture_output=True, text=True, check=True).stdout
    arch = sorted(set(re.findall(r'arch = (sm_\w+)', out)))
    per, cur = collections.OrderedDict(), None
    for line in out.splitlines():
        m = re.search(r'Function : (\S+)', line)
        if m:
            cur = per.setdefault(m.group(1), collections.Counter())
            continue
        if cur is None:
            continue
        m = PAT.search(line)
        if m:
            op = m.group(0)
            key = op.split('.')[0]
            if key == 'UTMALDG' and 'MULTICAST' in op:
                key = 'UTMALDG.MULTICAST'
            if key == 'UTCBAR' and 'MULTICAST' in op:
                key = 'UTCBAR.MULTICAST'
            cur[key] += 1
    lines = [f'# cuobjdump -sass {os.path.basename(so_path)}   (architectures in the binary: {", ".join(arch)})',
             '# kernel: counts of tcgen05 / TMEM / TMA / legacy-MMA mnemonics; kernels without any are plain SIMT kernels']
    try:
        names = subprocess.run(['c++filt'], input='\n'.join(per), capture_output=True, text=True).stdout.splitlines()
    except Exception:
        names = list(per)
    simt = 0
    for (mangled, c), name in zip(per.items(), names):
        keys = [k for k in c if k not in ('SYNCS', 'LDGSTS')]
        if not keys:
            simt += 1
            continue
        short = re.sub(r'\(.*', '', name.replace('(anonymous namespace)::', '')).replace('void ', '').replace('hk::', '')
        lines.append(f'{short:60s} ' + ' '.join(f'{k}={c[k]}' for k in sorted(c)))
    lines.append(f'# + {simt} SIMT kernels (elementwise / reductions / layout) without tensor-core or TMA instructions')
    return '\n'.join(lines) + '\n'


if __name__ == '__main__':
    here = os.path.dirname(os.path.abspath(__file__))
    so = sys.argv[1] if len(sys.argv) > 1 else os.path.join(here, '..', 'hawkeye_b200', 'libhawkeye_b200.so')
    txt = summarize(so)
    open(os.path.join(here, 'sass_opcodes.txt'), 'w').write(txt)
    print(txt)
