import sys, torch, ctypes as C
sys.path.insert(0,'/root/repo')
from rtucker_b200._lib import lib, ptr, stream_ptr, check
def al(x): return (x+255)//256*256
for n in (20, 400):
    dev=torch.device('cuda')
    X=torch.randn(n,4*n,dtype=torch.float64,device=dev); A=(X@X.T).contiguous()
    nb=(n+15)//16; nb+= nb&1; nb=max(nb,2); npad=nb*16; npairs=nb//2
    off_scal = al(npad*npad*8)*2 + al(npairs*1024*8) + al(npairs*4)
    ws=torch.zeros(lib().rt_eigh_ws_bytes(n),dtype=torch.uint8,device=dev)
    w=torch.empty(n,dtype=torch.float64,device=dev); V=torch.empty(n,n,dtype=torch.float64,device=dev)
    check(lib().rt_eigh(ptr(A.clone()),n,ptr(w),ptr(V),ptr(ws),stream_ptr()),'eigh')
    torch.cuda.synchronize()
    scal=ws[off_scal:off_scal+8*24].view(torch.float64).cpu()
    print(n,'norm2',scal[0].item(),'off per sweep',[f'{x:.1e}' for x in scal[1:21].tolist()],'scale',scal[21].item())
# per-phase cycle profile
L = lib()
for n in (20, 400):
    prof=torch.zeros(148*4,dtype=torch.int64,device='cuda')
    L.rt_eigh_set_profile(C.c_void_p(prof.data_ptr()))
    X=torch.randn(n,4*n,dtype=torch.float64,device='cuda'); A=(X@X.T).contiguous()
    ws=torch.zeros(L.rt_eigh_ws_bytes(n),dtype=torch.uint8,device='cuda')
    w=torch.empty(n,dtype=torch.float64,device='cuda'); V=torch.empty(n,n,dtype=torch.float64,device='cuda')
    check(L.rt_eigh(ptr(A.clone()),n,ptr(w),ptr(V),ptr(ws),stream_ptr()),'eigh'); torch.cuda.synchronize()
    p=prof.view(148,4).cpu()
    print(n,'CTA0 cycles A,sync,B,sync:',p[0].tolist(),' CTA5:',p[5].tolist(),' CTA100:',p[100].tolist())
L.rt_eigh_set_profile(None)
