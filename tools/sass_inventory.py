"""SASS inventory of the built library (cuobjdump -sass): the mnemonics that prove the Blackwell paths, per kernel.

    python tools/sass_inventory.py > profiles/r02_sass_inventory.md
"""
import collections
import re
import subprocess
import sys
from pathlib import Path

LIB = Path(__file__).resolve().parent.parent / 'nerficg_b200' / 'libnerf_b200.so'
COLS = ['UTCHMMA', 'LDTM', 'UBLKCP', 'LDGSTS', 'SYNCS', 'USETMAXREG', 'ELECT', 'RED+ATOMG', 'MEMBAR', 'SHFL', 'F2FP']


def main():
    sass = subprocess.run(['cuobjdump', '-sass', str(LIB)], capture_output=True, text=True, check=True).stdout
    names = subprocess.run(['c++filt'], input='\n'.join(re.findall(r'Function : (\S+)', sass)), capture_output=True, text=True).stdout.split('\n')
    kernels, cur, idx = collections.OrderedDict(), None, 0
    for line in sass.splitlines():
        m = re.search(r'Function : (\S+)', line)
        if m:
            cur = re.sub(r'\(.*', '', names[idx]).replace('nerf::', '').replace('void ', '').replace('(bool)', '').replace('(int)', '')
            idx += 1
            kernels[cur] = collections.Counter()
            continue
        m = re.match(r'\s+/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P\d+\s+)?([A-Z0-9_]+)', line)
        if m and cur:
            op = m.group(1)
            kernels[cur]['instr'] += 1
            kernels[cur][op] += 1
            if '.2CTA' in line and op == 'UTCHMMA':
                kernels[cur]['2CTA'] += 1
    # one row per kernel template family: K2 is instantiated per (keys per lane, padded cdf length)
    fam = collections.OrderedDict()
    for k, c in kernels.items():
        f = re.sub(r'<\d+, \d+>', '<K, pad>', k)
        fam.setdefault(f, []).append((k, c))
    print(f'# SASS inventory of `nerficg_b200/libnerf_b200.so` (final round-2 build, `cuobjdump -sass`, sm_100a; `python tools/sass_inventory.py`)\n')
    print('`UTCHMMA` = tcgen05.mma (last column: how many are `.2CTA` = cta_group::2 -- the chain kernels; wgrad is single-CTA), `LDTM` = tcgen05.ld, `UBLKCP` = cp.async.bulk')
    print('(TMA 1-D bulk copy), `SYNCS` = mbarrier ops, `USETMAXREG` = setmaxnreg, `RED`/`ATOMG` = global reductions. K2 is instantiated per')
    print('(keys per lane, padded cdf length): the row shows the range over its instances.\n')
    print('| kernel | instances | SASS instr | ' + ' | '.join(COLS) + ' | of which UTCHMMA.2CTA |')
    print('|---|---|---|' + '---|' * (len(COLS) + 1))
    def rng(vals):
        lo, hi = min(vals), max(vals)
        return str(lo) if lo == hi else f'{lo}–{hi}'
    for f, items in sorted(fam.items(), key=lambda kv: -max(c['instr'] for _, c in kv[1])):
        cells = []
        for col in COLS:
            cells.append(rng([c['RED'] + c['ATOMG'] + c['REDG'] if col == 'RED+ATOMG' else c[col] for _, c in items]))
        print(f'| `{f}` | {len(items)} | {rng([c["instr"] for _, c in items])} | ' + ' | '.join(cells) + f' | {rng([c["2CTA"] for _, c in items])} |')


if __name__ == '__main__':
    sys.exit(main())
