"""GAE HBM sweep: achieved GB/s of crl_gae_raw at T=128 for several N."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from cleanrl_jl_b200 import _lib
lib = _lib.load()
T = 128
for N in (1 << 18, 1 << 20, 1 << 21):
    v = torch.randn((T, N), device="cuda"); r = torch.randn((T, N), device="cuda")
    d = (torch.rand((T, N), device="cuda") < 0.01).to(torch.uint8)
    adv = torch.empty((T, N), device="cuda"); ret = torch.empty((T, N), device="cuda")
    def launch():
        _lib.check(lib.crl_gae_raw(_lib.ptr(v), _lib.ptr(r), _lib.ptr(d), None, None, _lib.ptr(adv), _lib.ptr(ret), T, N, 0.99, 0.95, 0,
                                   torch.cuda.current_stream().cuda_stream))
    for _ in range(3): launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10): launch()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    print("N", N, "ms %.4f" % ms, "GB/s %.0f" % ((17 * T * N + 5 * N) / ms / 1e6))
    del v, r, d, adv, ret
