import sys, torch, ctypes as C
sys.path.insert(0,'/root/repo')
from rtucker_b200._lib import lib, ptr, stream_ptr, check
L = lib()
n=400
prof=torch.zeros(148*4,dtype=torch.int64,device='cuda')
X=torch.randn(n,4*n,dtype=torch.float64,device='cuda'); A=(X@X.T).contiguous()
ws=torch.zeros(L.rt_eigh_ws_bytes(n),dtype=torch.uint8,device='cuda')
w=torch.empty(n,dtype=torch.float64,device='cuda'); V=torch.empty(n,n,dtype=torch.float64,device='cuda')
check(L.rt_eigh(ptr(A.clone()),n,ptr(w),ptr(V),ptr(ws),stream_ptr()),'eigh'); torch.cuda.synchronize()
L.rt_eigh_set_profile(C.c_void_p(prof.data_ptr()))
check(L.rt_eigh(ptr(A.clone()),n,ptr(w),ptr(V),ptr(ws),stream_ptr()),'eigh'); torch.cuda.synchronize()
L.rt_eigh_set_profile(None)
p=prof.view(148,4).cpu().double()
for i,name in enumerate(['phaseA','sync1','phaseB','sync2']):
    v=p[:,i]; srt=v.sort().values
    print(f"{name}: min {srt[0]:.0f} p25 {srt[37]:.0f} median {srt[74]:.0f} p75 {srt[111]:.0f} max {srt[-1]:.0f}  argmax cta {int(v.argmax())}")
print('phaseB per cta (k):', [int(x/1000) for x in p[:,2].tolist()])
print('phaseA per cta (k):', [int(x/1000) for x in p[:,0].tolist()])
