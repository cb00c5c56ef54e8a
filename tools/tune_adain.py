"""Sweep the pipelined AdaIN kernel's knobs on one level of BASELINE configs[1] and print GB/s
(algorithmic bytes / CUDA-event time).  GPU box only:  python tools/tune_adain.py [batch] [channels]"""
import itertools
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rpst  # noqa: E402

batch = int(sys.argv[1]) if len(sys.argv) > 1 else 16
ch = int(sys.argv[2]) if len(sys.argv) > 2 else 256
H = W = 512
dev = torch.device("cuda")
c = torch.relu(torch.randn(batch, ch, H, W, device=dev) + 0.5)
s = torch.relu(torch.randn(batch, ch, H, W, device=dev) * 2 + 1)
p = torch.randn(batch, ch, H, W, device=dev)
out = torch.empty_like(c)
L = rpst._lib.lib()
ws = torch.empty(L.rpst_adain_workspace_bytes(batch, ch, H * W), dtype=torch.uint8, device=dev)
stream = torch.cuda.current_stream().cuda_stream


def run(prev):
    rpst._lib.check(L.rpst_adain_fwd(c.data_ptr(), s.data_ptr(), prev.data_ptr() if prev is not None else None,
                                     out.data_ptr(), batch, ch, H * W, ch * H * W, 1e-5, None, ws.data_ptr(), ws.numel(), stream))


def timeit(prev, iters=10):
    for _ in range(3):
        run(prev)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        run(prev)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


E = batch * ch * H * W * 4
# plain copy reference points on this very box
x = torch.empty_like(c)
for _ in range(3):
    x.copy_(c)
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(10):
    x.copy_(c)
b.record()
torch.cuda.synchronize()
print(json.dumps({"torch_copy_GBs": 2 * E * 10 / (a.elapsed_time(b) / 1e3) / 1e9}))
del x

rows = []
for lag_mb, hints in itertools.product([24, 32, 48, 64], [1, 0]):
    rpst.set_tuning("adain_lag_bytes", lag_mb << 20)
    rpst.set_tuning("adain_hints", hints)
    t_plain = timeit(None)
    t_blend = timeit(p)
    row = {"lag_mb": lag_mb, "hints": hints, "plain_ms": round(t_plain, 4),
           "plain_GBs": round(3 * E / (t_plain / 1e3) / 1e9, 1), "blend_ms": round(t_blend, 4),
           "blend_GBs": round(4 * E / (t_blend / 1e3) / 1e9, 1)}
    rows.append(row)
    print(json.dumps(row), flush=True)
best = max(rows, key=lambda r: r["blend_GBs"])
print("BEST", json.dumps(best))
