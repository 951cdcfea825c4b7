import re,subprocess,sys
def funcs(path):
    out={}; cur=None; buf=[]
    for line in open(path):
        m=re.match(r'\s*Function : (\S+)',line)
        if m:
            if cur: out[cur]=buf
            cur=m.group(1); buf=[]
        elif cur is not None:
            l=re.sub(r'/\*[0-9a-f]{4,}\*/','',line)
            l=' '.join(l.split())
            if l.startswith('/*') or not l: continue
            buf.append(l)
    if cur: out[cur]=buf
    return out
def normlabels(lines):
    m={}
    def rep(x):
        k=x.group(0)
        if k not in m: m[k]=f'.L{len(m)}'
        return m[k]
    return [re.sub(r'\.L_x_\d+',rep,l) for l in lines]
a=funcs(sys.argv[1]); b=funcs(sys.argv[2])
dem=lambda ns: dict(zip(ns, subprocess.run(['c++filt'],input='\n'.join(ns),capture_output=True,text=True).stdout.split('\n')))
da=dem(list(a)); db=dem(list(b))
bmap={v.replace(', pdsb::LoadedRows>','>').replace(', pdsb::LoadedRows)',')'):k for k,v in db.items()}
same=diff=0
for k,v in da.items():
    kb=bmap.get(v)
    if kb is None: print("MISSING",v); diff+=1; continue
    if normlabels(a[k])==normlabels(b[kb]): same+=1
    else: diff+=1; print("DIFF",v[:140])
print(f"pre-existing kernels: {len(a)}; identical SASS: {same}; different: {diff}; kernels added: {len(b)-len(a)}")
