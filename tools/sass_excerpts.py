"""profiles/r02_sass_excerpts.txt: instruction census and excerpts of the shipped objects (dev tool; no GPU needed)."""
import collections, re, subprocess
def sass(obj):
    return subprocess.run(['cuobjdump', '-sass', obj], capture_output=True, text=True).stdout
def funcs(txt):
    out = {}; cur = None
    for l in txt.split('\n'):
        m = re.search(r'Function : (\S+)', l)
        if m: cur = m.group(1); out[cur] = []; continue
        if cur and re.match(r'\s+/\*[0-9a-f]{4,6}\*/', l): out[cur].append(l.rstrip())
    return out
SPECIAL = ('UTC', 'UTMA', 'LDTM', 'FADD2', 'FFMA2', 'FMUL2', 'CCTL', 'SYNCS', 'UCGABAR', 'MAPA', 'CGAERRBAR')
rep = []
B = 'thepayne_b200/csrc/_build/'
for obj, pat, marks in [(B + 'gemm_tu.o', 'tc_gemm_kernelILi128ELi2ELi0EE', ['UTCHMMA', 'UTMALDG', 'UTMASTG', 'LDTM']),
                        (B + 'gemm_tu.o', 'tc_gemm_kernelILi64ELi2ELi1EE', ['UTCHMMA', 'LDTM']),
                        (B + 'gemm_tu.o', 'tc_hidden_stack_kernel', ['UTCHMMA', 'UCGABAR_ARV', 'UTMALDG']),
                        (B + 'tail_fast_tu.o', 'tail_fast_kernelILi14ELb0ELNS_8FastBodyE0EE', ['FADD2', 'LDS.128', 'CCTL', 'CALL']),
                        (B + 'tail_cluster_tu.o', 'tail_cluster_kernelILi16E', ['UCGABAR_ARV', 'MAPA', 'ST.E.64', 'LD.E.64'])]:
    f = funcs(sass(obj))
    name = [k for k in f if pat in k][0]
    ins = f[name]
    ops = collections.Counter()
    for l in ins:
        m = re.search(r'\*/\s+(@!?U?P\d+\s+)?([A-Z0-9_.]+)', l)
        if m: ops[m.group(2) if m.group(2).startswith(SPECIAL) else m.group(2).split('.')[0]] += 1
    rep.append('== %s  (%s)\n   %d SASS instructions\n   mnemonic census: %s\n' % (
        name, obj.split('/')[-1], len(ins), ', '.join('%s %d' % kv for kv in ops.most_common(48))))
    for mk in marks:
        idx = [i for i, l in enumerate(ins) if re.search(r'\*/\s+(@!?U?P\d+\s+)?' + re.escape(mk), l)]
        if not idx: continue
        i = idx[0]
        rep.append('   -- first %s (%d in the function), lines %d..%d:\n%s\n' % (
            mk, len(idx), max(0, i - 6), i + 18, '\n'.join(ins[max(0, i - 6):i + 18])))
open('profiles/r02_sass_excerpts.txt', 'w').write(
    '# cuobjdump -sass of the shipped objects (sm_100a): instruction census and excerpts around the Blackwell-specific\n'
    '# instructions -- UTCHMMA = tcgen05.mma, UTMALDG / UTMASTG = TMA tensor load / store, LDTM = tcgen05.ld (TMEM), UTCBAR =\n'
    '# tcgen05.commit, SYNCS = mbarrier, FADD2 = packed fp32x2 add, CCTL.E.RML2 = discard.global.L2, UCGABAR_ARV / UCGABAR_WAIT =\n'
    '# barrier.cluster.arrive / wait, MAPA = mapa.shared::cluster, ST.E.64 / LD.E.64 in the cluster tail = st / ld.shared::cluster (DSMEM).\n\n' + '\n'.join(rep))
print('wrote profiles/r02_sass_excerpts.txt')
