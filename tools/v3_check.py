"""GPU check of the variant-2 score kernel (score_bce_v3.cu): fp16 tcgen05 building blocks, bulk reduce,
parity against the fp32 FFMA kernel, and timing.  python tools/v3_check.py [quick]"""
import sys, time, torch
sys.path.insert(0, '/root/repo')
from rtucker_b200 import ops
from rtucker_b200._lib import lib, ptr, stream_ptr, check
dev = torch.device('cuda'); torch.manual_seed(0)

def selftest(N, K, a_mn, b_mn, flags):
    A = torch.randint(-3, 4, (128, K), device=dev).float()
    B = torch.randint(-3, 4, (N, K), device=dev).float()
    Ain = A.t().contiguous() if a_mn else A
    Bin = B.t().contiguous() if b_mn else B
    D = torch.zeros(128, N, device=dev)
    check(lib().rt_tc_selftest16(ptr(Ain), ptr(Bin), ptr(D), N, K, a_mn, b_mn, flags, stream_ptr()), 'selftest16')
    torch.cuda.synchronize()
    ref = A @ B.t()
    return bool(torch.equal(D, ref)), float((D - ref).abs().max())

for a_mn in (0, 1):
    for b_mn in (0, 1):
        for flags in ((0,) if not (a_mn or b_mn) else (0, 3)):
            print(f"selftest16 N=208 K=128 a_mn={a_mn} b_mn={b_mn} flags={flags}:", selftest(208, 128, a_mn, b_mn, flags), flush=True)
print("selftest16 N=96 K=208 kk:", selftest(96, 208, 0, 0, 0))
a = torch.randn(2048, device=dev); b = torch.randn(2048, device=dev); o = torch.zeros(2048, device=dev)
check(lib().rt_bulk_reduce_selftest(ptr(a), ptr(b), ptr(o), 2048, stream_ptr()), 'bulk'); torch.cuda.synchronize()
print("bulk store+reduce exact:", bool(torch.equal(o, a + b)), flush=True)

def case(B, N, r2, nnz_per=2, zstd=4.0, o_absmax=None, seed=1):
    g = torch.Generator(device='cpu').manual_seed(seed)
    O = torch.linalg.qr(torch.randn(N, r2, generator=g))[0].contiguous().to(dev) if N >= r2 else torch.randn(N, r2, generator=g).to(dev)
    scale = zstd * (N / r2) ** 0.5
    q = (torch.randn(B, r2, generator=g) * scale).to(dev)
    off = torch.arange(0, (B + 1) * nnz_per, nnz_per).int().to(dev)
    idx = torch.randint(0, N, (B * nnz_per,), generator=g).int().to(dev)
    l0, H0, d0 = ops.score_bce_fwd_bwd(q, q, O, off, idx, 0.1, variant=0)
    l2, H2, d2 = ops.score_bce_fwd_bwd(q, None, O, off, idx, 0.1, variant=2, o_absmax=o_absmax)
    torch.cuda.synchronize()
    rel = lambda x, y: float((x.double() - y.double()).norm() / y.double().norm())
    return rel(l2, l0), rel(H2, H0), rel(d2, d0)

quick = len(sys.argv) > 1
shapes = [(128, 96, 16, 1, 4.0), (100, 1000, 20, 2, 4.0), (512, 5000, 200, 2, 4.0), (300, 777, 52, 3, 4.0),
          (512, 40943, 200, 2, 4.0), (512, 40943, 200, 2, 12.0), (64, 200, 176, 1, 4.0), (512, 3000, 208, 2, 4.0), (1, 5, 3, 1, 2.0),
          (130, 97, 7, 1, 3.0)]
for (B, N, r2, nn, zs) in shapes:
    e2 = case(B, N, r2, nn, zs)
    print(f"B={B} N={N} r2={r2} zstd={zs}: v2 rel err loss/H/dO =", ["%.2e" % e for e in e2], flush=True)
print("hint=1.0:", ["%.2e" % e for e in case(512, 40943, 200, 2, 4.0, o_absmax=1.0)])

def timeit(fn, n=20):
    for _ in range(3): fn()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    ts = []
    for _ in range(n):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    ts.sort(); return ts[len(ts) // 2]

for (B, N, r2) in [(512, 40943, 200)] + ([] if quick else [(512, 1000000, 200)]):
    g = torch.Generator().manual_seed(3)
    O = torch.linalg.qr(torch.randn(N, r2, generator=g))[0].contiguous().to(dev)
    q = (torch.randn(B, r2, generator=g) * 600).to(dev)
    off = torch.arange(0, (B + 1) * 2, 2).int().to(dev); idx = torch.randint(0, N, (B * 2,), generator=g).int().to(dev)
    outs = (torch.empty(1, dtype=torch.float64, device=dev), torch.empty(B, r2, device=dev), torch.empty(N, r2, device=dev))
    for v in (0, 2):
        ws = torch.empty(int(lib().rt_score_bce_ws_bytes(B, N, r2, v)) + 16, dtype=torch.uint8, device=dev)
        ms = timeit(lambda: ops.score_bce_fwd_bwd(q, None if v == 2 else q, O, off, idx, 0.1, variant=v, out=outs, ws=ws, o_absmax=1.0 if v == 2 else None))
        print(f"N={N} variant {v}: {ms*1e3:.1f} us  {6.0*B*N*r2/ms/1e9:.1f} TFLOP/s", flush=True)
