"""Micro-benchmark of K1a engines on the shapes the hot path uses (CUDA events, L2 flushed between repeats)."""
import sys, os, json
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deeprecommendation_b200 import ops

SHAPES = [tuple(int(v) for v in a.split('x')) for a in sys.argv[1:]] or [(9447, 2094, 256), (9461, 2094, 256), (9600, 2094, 256), (162541, 128, 128), (62423, 128, 128), (512, 2094, 128), (512, 2094, 256), (100000, 2094, 128)]
flush = torch.empty(256 * 1024 * 1024 // 4, device='cuda')
out = {}
for M, K, N in SHAPES:
    x = torch.randn(M, K, device='cuda'); w = torch.randn(N, K, device='cuda') / K ** 0.5; b = torch.randn(N, device='cuda')
    for eng in ('simt', 'tf32x3', 'tf32x3!', 'tf32x3!narrow', 'bf16x3!', 'bf16!') + (('shortk!',) if K <= 128 else ()):
        if eng == 'tf32x3!narrow' and N <= 128:
            continue
        if eng == 'tf32x3!narrow':                      # the 128 x 128 tiles that the wide form replaces for 128 < N
            run = lambda: ops.linear_tc_batch([(x, w, b, None)], engine='tf32x3')
        else:
            run = lambda: ops.linear_raw(x, w, b, engine=eng)
        ts = []
        for r in range(7):
            flush.zero_()
            a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); run(); e.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(e))
        ms = sorted(ts)[len(ts) // 2]
        gb = 4.0 * (M * K + N * K + M * N) / 1e9
        out[f'{M}x{K}->{N} {eng}'] = {'ms': round(ms, 4), 'GB/s': round(gb / (ms * 1e-3), 1), 'TFLOP/s': round(2.0 * M * K * N / (ms * 1e-3) / 1e12, 2)}
        print(f'{M}x{K}->{N} {eng:8s} {ms:8.4f} ms  {gb / (ms * 1e-3):8.1f} GB/s  {2.0 * M * K * N / (ms * 1e-3) / 1e12:7.2f} TFLOP/s', flush=True)
json.dump(out, open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'gpurun_out', 'gemm_bench.json'), 'w'), indent=1)
