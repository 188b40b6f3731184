"""Kernel-by-kernel comparison of two `cuobjdump -sass` listings (every instruction and encoding line).

    python scripts/sass_same.py OLD.sass NEW.sass

A kernel of OLD that NEW no longer has under the same name is looked up as stolt_col_kernel<S, R3, PF, false> (the
instantiations that gained the SPLIT template parameter and the unused `src` argument of the velocity scan).
"""
import re,sys
def funcs(path):
    d={}; cur=None
    for line in open(path):
        m=re.search(r'Function : (\S+)',line)
        if m: cur=m.group(1); d[cur]=[]; continue
        if cur: d[cur].append(line.rstrip())
    return d
a=funcs(sys.argv[1]); b=funcs(sys.argv[2])
seen = set()
for k in a:
    k2=k
    if k not in b:  # stolt_col_kernel<S, R3, PF> -> stolt_col_kernel<S, R3, PF, false>
        k2=k.replace('EEEvNS0_9ColParamsE','ELb0EEEvNS0_9ColParamsEPK6float2')
    seen.add(k2)
    print('%-75s %s' % (k[:75], 'same' if a[k]==b.get(k2) else ('DIFF' if k2 in b else 'MISSING')), '' if k2==k else '-> '+k2)
print('new only:', [k for k in b if k not in seen])
