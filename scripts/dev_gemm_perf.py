import torch, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tokenhmr_b200._lib import lib, check
L = lib(); dev = torch.device("cuda:0"); torch.manual_seed(0)
st = lambda: torch.cuda.current_stream().cuda_stream
P = lambda t: None if t is None else t.data_ptr()
def gemm(A, B, bias, resid, act, o32, o16, bn):
    M, K = A.shape; N = B.shape[0]
    check(L.thmr_gemm_f16(A.data_ptr(), K, B.data_ptr(), K, M, N, K, P(bias), P(resid), N, act, P(o32), N, P(o16), N, bn, st()))
def timeit(fn, iters=50):
    for _ in range(5): fn()
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters
M = 12288
for (name, N, K, act, mode) in [("qkv", 3840, 1280, 0, "s16"), ("proj", 1280, 1280, 0, "add"), ("fc1", 5120, 1280, 1, "s16"), ("fc2", 1280, 5120, 0, "add")]:
    A = torch.randn(M, K, device=dev).half(); B = (torch.randn(N, K, device=dev) * 0.03).half()
    bias = torch.randn(N, device=dev)
    o16 = torch.empty(M, N, device=dev, dtype=torch.float16); x = torch.zeros(M, N, device=dev)
    tcb = timeit(lambda: torch.matmul(A, B.t()))
    line = f"{name} N={N} K={K}: cublas {tcb*1e3:.1f}us {2*M*N*K/tcb/1e9:.0f} TF |"
    for bn in (512, 256):
        if mode == "s16": fn = lambda: gemm(A, B, bias, None, act, None, o16, bn)
        else: fn = lambda: gemm(A, B, bias, x, 0, x, None, bn)
        t = timeit(fn)
        line += f" bn{bn} {t*1e3:.1f}us {2*M*N*K/t/1e9:.0f} TF |"
    print(line, flush=True)
