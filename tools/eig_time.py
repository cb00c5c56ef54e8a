"""Batched 256x256 matrix square roots at the automatic Jacobi block width: 16-column blocks (8-CTA clusters) up to
batch 20, 32-column blocks (4-CTA clusters) above.  GPU box only."""
import json, os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rpst
n = 256
def t(fn, it=5):
    for _ in range(2): fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(it): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / it
for batch in (1, 8, 12, 16, 32):
    g = torch.Generator(device="cuda").manual_seed(n)
    a = torch.randn(batch, n, 2 * n, device="cuda", dtype=torch.float64, generator=g)
    a = a @ a.transpose(1, 2) / (2 * n)
    print(json.dumps({"batch": batch, "block_cols": 32 if batch * (n // 32) > 160 else 16,
                      "ms": round(t(lambda: rpst.matrix_sqrt(a)), 3)}), flush=True)
