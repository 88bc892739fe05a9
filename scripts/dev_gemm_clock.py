import torch, subprocess, time, threading
from tokenhmr_b200._lib import lib, check
L = lib(); dev = torch.device("cuda:0"); torch.manual_seed(0)
st = lambda: torch.cuda.current_stream().cuda_stream
M, N, K = 12288, 3840, 1280
A = torch.randn(M, K, device=dev).half(); B = (torch.randn(N, K, device=dev) * 0.03).half()
bias = torch.randn(N, device=dev); o16 = torch.empty(M, N, device=dev, dtype=torch.float16)
def mine(bn): check(L.thmr_gemm_f16(A.data_ptr(), K, B.data_ptr(), K, M, N, K, bias.data_ptr(), None, N, 0, None, N, o16.data_ptr(), N, bn, st()))
def sample(fn, secs=2.5):
    rows = []
    p = subprocess.Popen(["nvidia-smi", "--query-gpu=clocks.sm,power.draw", "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
    th = threading.Thread(target=lambda: [rows.append(l) for l in p.stdout], daemon=True); th.start()
    for _ in range(20): fn()
    torch.cuda.synchronize(); time.sleep(0.3)
    n0 = len(rows); t0 = time.time(); it = 0
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True); e0.record()
    while time.time() - t0 < secs:
        for _ in range(50): fn()
        it += 50
        torch.cuda.synchronize()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / it
    p.terminate()
    vals = [tuple(float(x) for x in r.split(",")) for r in rows[n0+3:]]
    clk = sorted(v[0] for v in vals); pw = sorted(v[1] for v in vals)
    return ms, clk[len(clk)//2] if clk else 0, pw[len(pw)//2] if pw else 0
for name, fn in [("cublas", lambda: torch.matmul(A, B.t())), ("mine bn256", lambda: mine(256)), ("mine 2cta", lambda: mine(512))]:
    ms, clk, pw = sample(fn)
    print(f"{name}: {ms*1e3:.1f} us  {2*M*N*K/ms/1e9:.0f} TF  sm_clk {clk:.0f} MHz  power {pw:.0f} W  -> util {2*M*N*K/ms/1e9/(148*8192*clk*1e-6)*100:.0f}%", flush=True)
