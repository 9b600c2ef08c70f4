import re, subprocess, sys
def funcs(so):
    out = subprocess.run(['cuobjdump', '-sass', so], stdout=subprocess.PIPE, text=True, check=True).stdout
    d, cur = {}, None
    for line in out.splitlines():
        m = re.search(r'Function : (\S+)', line)
        if m:
            cur = re.sub(r'_GLOBAL__N__[0-9a-f]+_\d+_\w+?_cu_[0-9a-f]+', 'ANON', m.group(1)); d[cur] = []; continue
        if cur and re.search(r'/\*[0-9a-f]{4}\*/', line):
            ins = re.sub(r'/\*[0-9a-f]{4}\*/', '', line.split(';')[0]).strip()
            d[cur].append(ins)
    return d
a, b = funcs(sys.argv[1]), funcs(sys.argv[2])
same = [f for f in a if f in b and a[f] == b[f]]
diff = [f for f in a if f in b and a[f] != b[f]]
new = [f for f in b if f not in a]
gone = [f for f in a if f not in b]
dm = lambda f: subprocess.run(['c++filt', f], stdout=subprocess.PIPE, text=True).stdout.strip().split('(')[0]
print('kernels with identical SASS: %d' % len(same))
print('changed:'); [print('  ' + dm(f)) for f in diff]
print('new:'); [print('  ' + dm(f)) for f in new]
print('removed:'); [print('  ' + dm(f)) for f in gone]
