"""Counts the SASS mnemonics that prove which hardware path each hot kernel of libdiffsbdd_b200.so takes (tcgen05 MMAs incl. the
cta_group::2 form, TMEM loads/stores, bulk copies, multicast commits, cluster barriers, packed fp32, vector REDs).

    python profiles/sass_summary.py > profiles/r2e_sass.txt"""
import collections
import os
import re
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from diffsbdd_b200 import _build  # noqa: E402

KEYS = ['UTCHMMA.2CTA', 'UTCHMMA', 'UTCBAR.2CTA.MULTICAST', 'UTCBAR', 'LDTM', 'STTM', 'UBLKCP', 'UTMALDG', 'UCGABAR_ARV', 'SYNCS', 'FENCE.VIEW.ASYNC',
        'USETMAXREG', 'FHFMA', 'HADD2.F32', 'MUFU.EX2', 'MUFU.RCP', 'FFMA2', 'FADD2', 'FMUL2', 'F2FP', 'REDG.E.ADD.F32x4', 'REDG', 'LDG.E.128', 'STS.64', 'STS.128', 'LDS.128']
WANT = ['tc_edge_kernelILb0ELb1ELi256ELb0ELb1', 'tc_edge_kernelILb1ELb1ELi256ELb0ELb1', 'tc_edge_kernelILb0ELb1ELi256ELb0ELb0',
        'tc_node_block_kernelILi256', 'tc_node_gemm_kernelILb1ELi256', 'tc_node_mlp_kernelILb1ELi256']
out = subprocess.run(['cuobjdump', '-sass', _build.LIB_PATH], capture_output=True, text=True).stdout
cur, counts = None, collections.OrderedDict()
for line in out.splitlines():
    m = re.search(r'Function : (\S+)', line)
    if m:
        cur = next((w for w in WANT if w in m.group(1)), None)
        if cur:
            counts[cur] = collections.Counter()
        continue
    if cur:
        m = re.match(r'\s+/\*[0-9a-f]+\*/\s+(?:@!?U?P\d+\s+)?([A-Za-z0-9_.]+)', line)
        if m:
            op = m.group(1)
            counts[cur]['_total'] += 1
            for k in KEYS:
                if op.startswith(k):
                    counts[cur][k] += 1
print('# SASS mnemonic counts (cuobjdump -sass diffsbdd_b200/libdiffsbdd_b200.so); prefixes: UTCHMMA includes UTCHMMA.2CTA, REDG includes F32x4')
print('# kernels: <COORD, F16, H, TB, PAIR> = tc_edge_kernel template arguments')
for name, c in counts.items():
    print(f'\n{name}   ({c["_total"]} instructions)')
    print('   ' + '  '.join(f'{k}={c[k]}' for k in KEYS if c[k]))
