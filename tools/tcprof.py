import sys, torch, ctypes as C
sys.path.insert(0,'/root/repo')
from rtucker_b200 import ops
from rtucker_b200._lib import lib
L=lib()
dev=torch.device('cuda'); N,B,r2=40943,512,200
q=torch.randn(B,r2,device=dev)/r2**0.5; O=torch.randn(N,r2,device=dev)
off=torch.arange(0,(B+1)*2,2,device=dev,dtype=torch.int32); idx=torch.randint(0,N,(B*2,),device=dev,dtype=torch.int32)
ops.score_bce_fwd_bwd(q,q,O,off,idx,0.1,variant=1); torch.cuda.synchronize()
prof=torch.zeros(148*12,dtype=torch.int64,device=dev); L.rt_score_tc_set_profile(C.c_void_p(prof.data_ptr()))
ops.score_bce_fwd_bwd(q,q,O,off,idx,0.1,variant=1); torch.cuda.synchronize()
L.rt_score_tc_set_profile(None)
p=prof.view(148,12).cpu().double()
names=['gemm1 stage+issue','mask','wait gemm1','epilogue1','gemm23 stage+issue','wait gemm23','epilogue2 (H)','tile epilogue (dO)','  g1: cp.async issue','  g1: cp.async wait','  g1: round in place','  g1: barrier']
tot=p.sum(1)
print('cycles per CTA: mean %.0f max %.0f' % (tot.mean(), tot.max()))
for i,n in enumerate(names): print(f'  {n:24s} mean {p[:,i].mean():10.0f}  ({100*p[:,i].mean()/tot.mean():.1f}%)')
