"""Prefill GEMM throughput (TFLOP/s) on the Llama-3-8B shapes for token counts 512 / 4096: token tile 128 / 256 x ring
depth.  Also a whole-model prefill estimate: sum over the four GEMMs x 32 layers."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bee2bee_b200 import ops
C = ops.native(); C.init_kernels(0)
dev = "cuda"
H, F, QKV = 4096, 14336, 6144
shapes = {"qkv": (QKV, H, ops.EPI_PLAIN), "o": (H, H, ops.EPI_RESIDUAL), "gate/up": (2 * F, H, ops.EPI_GLU), "down": (H, F, ops.EPI_RESIDUAL)}
ws = {k: [(torch.randn(n, kk, device=dev) * 0.02).bfloat16() for _ in range(3)] for k, (n, kk, _) in shapes.items()}

def timed(fn, reps=5):
    fn(); torch.cuda.synchronize()
    ts = []
    for i in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(i); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]

for T in (512, 4096):
    total = {}
    for name, (n, k, epi) in shapes.items():
        x = torch.randn(T, k, device=dev).bfloat16()
        res = torch.randn(T, n, device=dev).bfloat16() if epi == ops.EPI_RESIDUAL else None
        out = torch.empty(T, n // 2 if epi == ops.EPI_GLU else n, device=dev, dtype=torch.bfloat16)
        flops = 2.0 * T * n * k
        for bn, st in [(128, 0), (128, 3), (128, 2), (256, 0), (256, 3), (256, 2)]:
            def run(i=0):
                ops.gemm(ws[name][i % 3], x, out=out, epi=epi, residual=res, bn=bn, splitk=1, stages=st)
            try:
                us = timed(run)
            except Exception as e:
                print(f"T={T} {name} bn={bn} stages={st}: FAILED {e}")
                continue
            total.setdefault((bn, st), 0.0)
            total[(bn, st)] += us
            print(f"T={T:5d} {name:8s} bn={bn:3d} stages={st}: {us:8.1f} us  {flops / us / 1e6:7.1f} TFLOP/s", flush=True)
    for key, us in sorted(total.items()):
        print(f"T={T:5d} layer GEMMs bn={key[0]} stages={key[1]}: {us:8.1f} us -> 32 layers {us * 32 / 1e3:6.2f} ms ({2.0 * T * 7.0e9 / (us * 32) / 1e6:6.1f} TFLOP/s on the 7.0 G layer params)")
