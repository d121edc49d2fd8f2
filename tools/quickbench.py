"""Kernel-only throughput of one resident document for several kernel organisations / tile shapes.

usage: python tools/quickbench.py [size_mib] ; env KERNELS=persistent,split NWS=8,16
"""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mojo_simdjson_b200 import device, synth
size = (int(sys.argv[1]) if len(sys.argv) > 1 else 1024) << 20
doc = synth.status_array(size)
d_in = torch.from_numpy(doc).cuda(); d_out = torch.empty(size // 3, dtype=torch.int32, device='cuda')
ctx = device.Stage1Context(0)
for kernel in os.environ.get('KERNELS', 'persistent,split').split(','):
    ctx.set_kernel(kernel)
    for nw in [int(x) for x in os.environ.get('NWS', '0').split(',')]:
        ctx.set_warps(nw)
        for _ in range(5): ctx.enqueue(d_in, d_out, 0)
        torch.cuda.synchronize()
        reps = max(10, min(200, (8 << 30) // size))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps): ctx.enqueue(d_in, d_out, 0)
        e1.record(); torch.cuda.synchronize()
        res = ctx.finish()
        ms = e0.elapsed_time(e1) / reps
        print(kernel, 'NW', nw, 'size_mib', size >> 20, 'ms %.4f' % ms, 'GB/s %.0f' % (size / ms / 1e6),
              'err', res.error, 'n', res.n, flush=True)
