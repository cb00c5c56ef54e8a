"""Segment AdaIN backward at BASELINE configs[4] (1x256x1024x2048, 19 classes in 32x32 blocks, label seeds
4000/5000 as in tools/seg_time.py), in one process:
  (a) rpst_seg_adain_bwd alone, and segment AdaIN forward + backward through autograd;
  (b) the masked training transform: segment AdaIN (differentiable=True), calc_style_loss and
      calc_content_loss(norm=True), torch.autograd.grad w.r.t. content and style;
  (c) the same step with plain AdaIN (what bench.py's `train` leg times);
  (d) the reference arm: fp32 torch autograd of the reference's segment AdaIN op sequence (oracle.restate.seg_adain,
      restated without its detach) on the same GPU.
Gradients are first checked against fp64 autograd on two channels.  Each line is JSON; ms from CUDA events after
warm-up (the 2 GiB tensors are far larger than L2).  GB/s are over algorithmic bytes.  The first line records the
GPU, its power limit and max SM clock (nvidia-smi --query-gpu, read-only).
Usage: python tools/seg_train_time.py [--out FILE]"""
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import rpst  # noqa: E402
from oracle import restate as R  # noqa: E402

OUT = None


def emit(rec):
    line = json.dumps(rec)
    print(line, flush=True)
    if OUT:
        with open(OUT, "a") as f:
            f.write(line + "\n")


def dev_ms(fn, iters=10, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def seg_adain_ref(content, style, c_labels, s_labels, eps=1e-5):
    """oracle.restate.seg_adain_batch op for op, on the tensors' device and differentiable."""
    outs = []
    ch = content.shape[1]
    for i in range(content.shape[0]):
        cf, sf = content[i].reshape(ch, -1), style[i].reshape(ch, -1)
        cl, sl = c_labels[i].reshape(-1).long(), s_labels[i].reshape(-1).long()
        out = cf.clone()
        for lab, ok in R.segment_label_validity(cl.cpu(), sl.cpu()).items():
            if not ok:
                continue
            ci = torch.nonzero(cl == lab).reshape(-1)
            si = torch.nonzero(sl == lab).reshape(-1)
            mc, ms = cf[:, ci], sf[:, si]
            mu_c, sd_c = mc.mean(1, keepdim=True), torch.sqrt(mc.var(1, keepdim=True) + eps)
            mu_s, sd_s = ms.mean(1, keepdim=True), torch.sqrt(ms.var(1, keepdim=True) + eps)
            out = out.index_copy(1, ci, (mc - mu_c) / sd_c * sd_s + mu_s)
        outs.append(out.reshape(content.shape[1:]))
    return torch.stack(outs)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    idx = torch.cuda.current_device()
    name, power, clock = (x.strip() for x in q[idx].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock, "torch_name": torch.cuda.get_device_name()}


def main():
    global OUT
    if "--out" in sys.argv:
        OUT = sys.argv[sys.argv.index("--out") + 1]
    assert torch.cuda.is_available(), "needs a CUDA device"
    emit(gpu_info())
    n, ch, h, w = 1, 256, 1024, 2048
    c, s = R.synth_features((n, ch, h, w), cfg=5, device="cuda")
    cl = R.synth_labels(n, h, w, classes=19, block=32, seed=4000, device="cuda")
    sl = R.synth_labels(n, h, w, classes=19, block=32, seed=5000, device="cuda")
    g = torch.randn((n, ch, h, w), device="cuda", generator=torch.Generator(device="cuda").manual_seed(7))

    # ---- gradients against fp64 on a slice (two channels)
    cc, sc = c[:, :2].contiguous().requires_grad_(), s[:, :2].contiguous().requires_grad_()
    dc, ds = torch.autograd.grad(rpst.seg_adain_batch(cc, sc, cl, sl, differentiable=True), (cc, sc), g[:, :2])
    c64, s64 = c[:, :2].double().requires_grad_(), s[:, :2].double().requires_grad_()
    w_dc, w_ds = torch.autograd.grad(seg_adain_ref(c64, s64, cl, sl), (c64, s64), g[:, :2].double())
    err = {"check": "gradients vs fp64 autograd, channels 0-1", "rel_l2_dc": R.rel_l2(dc, w_dc),
           "rel_l2_ds": R.rel_l2(ds, w_ds)}
    emit(err)
    assert err["rel_l2_dc"] < 1e-4 and err["rel_l2_ds"] < 1e-4, err
    del cc, sc, dc, ds, c64, s64, w_dc, w_ds

    E = c.numel() * 4            # content and style planes have the same size here
    lab = 2 * h * w              # both label maps
    L = rpst._lib.lib()
    ws = torch.empty(L.rpst_seg_adain_bwd_workspace_bytes(n, ch, h * w, h * w), dtype=torch.uint8, device="cuda")
    dcb, dsb = torch.empty_like(c), torch.empty_like(s)

    def bwd():
        rpst._lib.check(L.rpst_seg_adain_bwd(g.data_ptr(), c.data_ptr(), s.data_ptr(), cl.data_ptr(), sl.data_ptr(),
                                             dcb.data_ptr(), dsb.data_ptr(), n, ch, h * w, h * w, 1e-5, ws.data_ptr(),
                                             ws.numel(), torch.cuda.current_stream().cuda_stream))

    # (a) backward alone: algorithmic 3E_c + 2E_s; the design reads g, c, s twice (reduce + apply) and writes dc, ds
    alg = 5 * E
    design = {"grad_out": 2.0, "content": 2.0, "style": 2.0, "grad_content": 1.0, "grad_style": 1.0}
    for _ in range(2):
        ms = dev_ms(bwd)
        emit({"arm": "a: seg_adain_bwd", "ms": ms, "GBs_alg": alg / ms / 1e6, "alg_bytes": alg,
              "design_bytes": 8 * E + 2 * lab, "bytes_moved_over_minimum_per_tensor": design,
              "workspace_bytes": ws.numel()})
    del dcb, dsb, ws
    cr, sr = c.clone().requires_grad_(), s.clone().requires_grad_()

    def fwd_bwd():
        out = rpst.seg_adain_batch(cr, sr, cl, sl, differentiable=True)
        torch.autograd.grad(out, (cr, sr), g)

    ms = dev_ms(fwd_bwd)
    emit({"arm": "a: seg_adain fwd+bwd (autograd)", "ms": ms, "GBs_alg": (3 * E + 5 * E) / ms / 1e6,
          "alg_bytes": 8 * E})

    # (b) / (c): the training transform; algorithmic bytes as bench.py's train leg: forward 3E, loss statistics
    # 2 x 2E, loss backward 2E + 3E, transform backward 5E
    step_alg = (3 + 4 + 5 + 5) * E

    def step(transform):
        def run():
            out = transform(cr, sr)
            loss = rpst.calc_style_loss(out, sr.detach()) + rpst.calc_content_loss(out, cr.detach(), norm=True)
            torch.autograd.grad(loss, (cr, sr))
        return run

    seg_step = step(lambda x, y: rpst.seg_adain_batch(x, y, cl, sl, differentiable=True))
    plain_step = step(rpst.adaptive_instance_normalization)
    for _ in range(2):   # alternated
        for name, fn in (("b: masked training transform (segment AdaIN)", seg_step),
                         ("c: training transform (plain AdaIN)", plain_step)):
            ms = dev_ms(fn, iters=6, warm=2)
            emit({"arm": name, "ms": ms, "GBs_alg": step_alg / ms / 1e6, "alg_bytes": step_alg})

    # (d) reference arm: the reference's op sequence in fp32 torch autograd, segment AdaIN fwd+bwd only
    def ref_fwd_bwd():
        out = seg_adain_ref(cr, sr, cl, sl)
        torch.autograd.grad(out, (cr, sr), g)

    ms = dev_ms(ref_fwd_bwd, iters=3, warm=1)
    emit({"arm": "d: reference op sequence fp32 autograd, seg_adain fwd+bwd", "ms": ms,
          "GBs_alg": 8 * E / ms / 1e6, "alg_bytes": 8 * E})


if __name__ == "__main__":
    main()
