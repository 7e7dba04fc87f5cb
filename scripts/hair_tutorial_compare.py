import subprocess, numpy as np, os, time
ROOT='/root/repo'
for t in (0,1,2):
    out=f'/tmp/hair_{t}.raw'
    t0=time.time()
    r=subprocess.run([os.path.join(ROOT,'oracle/_ref/link_compat/embree_hair_geometry'),out,'96','72','4',str(t),'3000'],stdout=subprocess.PIPE,stderr=subprocess.STDOUT,text=True,timeout=600)
    dt=time.time()-t0
    print(r.returncode, r.stdout.strip()[-300:], "%.1fs"%dt)
    g=np.fromfile(out,np.uint32); w=np.fromfile(os.path.join(ROOT,f'tests/golden/hair_geometry_{t}_96x72.raw'),np.uint32)
    ch=lambda a: np.stack([a&255,(a>>8)&255,(a>>16)&255],-1).astype(np.int32)
    d=np.abs(ch(g)-ch(w)).max(-1)
    print("type",t,"pixels differing",(d>0).sum(),"of",len(d),"; >2 levels:",(d>2).sum(),"; >16:",(d>16).sum(),"mean colour",ch(g).mean(0),ch(w).mean(0))
