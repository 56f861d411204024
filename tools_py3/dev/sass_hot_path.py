import re,subprocess,collections,sys
def funcs(cubin):
    out=subprocess.run(['cuobjdump','-sass',cubin],capture_output=True,text=True).stdout
    for f in re.split(r'\n\s+Function : ',out)[1:]:
        name=f.split('\n')[0]
        L=[]
        for l in f.split('\n'):
            m=re.match(r'\s+/\*([0-9a-f]{4})\*/\s+(.*?)\s*;',l)
            if m: L.append((int(m.group(1),16),m.group(2)))
        yield name,L
tgt=lambda s:int(re.search(r'0x([0-9a-f]+)$',s).group(1),16)
for cub in sys.argv[1:]:
    for name,L in funcs(cub):
        if 'k_push' not in name: continue
        first=next((a for a,s in L if 'LDG.E.128' in s),None)
        if first is None: continue
        br=[(a,tgt(s),s) for a,s in L if 'BRA' in s and re.search(r'0x[0-9a-f]+$',s)]
        end,head,_=[b for b in br if 0x200<b[1]<first and b[0]>first][-1]
        # forward branch with the largest span inside the loop = jump over the slow block
        fw=[b for b in br if head<=b[0]<end and b[1]>b[0] and b[1]<=end]
        ja,jt,_=max(fw,key=lambda b:b[1]-b[0])
        hot=[(a,s) for a,s in L if head<=a<=ja or jt<=a<=end]
        # drop retry loops (backward branches inside the hot range)
        for a,t,s in br:
            if head<=a<=ja and t<a and t>=head and a!=end:
                hot=[(x,y) for x,y in hot if not (t<=x<=a)]
        c=collections.Counter((s.split()[1] if s.startswith('@') else s.split()[0]).split('.')[0] for a,s in hot)
        dp=sum(v for k,v in c.items() if k in('DFMA','DMUL','DADD','DSETP'))
        print(name[17:44],'hot',len(hot),'dp',dp,'LDL/STL',c['LDL']+c['STL'],dict(c.most_common(10)))
