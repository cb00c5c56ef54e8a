#!/usr/bin/env python
"""bench.py — headline benchmark: stylized images/s @512^2 for the multiscale RP-AdaIN transform
(BASELINE.json configs[1]: `run_deeper_multiscale_rp_adain`, batch 32 per GPU, levels
C = 16,32,64,128,256 at full 512x512 resolution; SURVEY.md §8d).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--scaling weak|strong] [--no-sustained] [--no-extra]
                    [--dump-outputs DIR]

A step = one pass of the hot path over one batch: AdaIN on the deepest level + `prev + AdaIN` on the
four shallower ones (network/adain_rp.py:286-302 with the decoder convolutions factored out), five
C-ABI calls into librpst.  One process per GPU (torchrun for N>1), batch sharded, no collective on the
data path (weak scaling: 32 images per GPU).  Prints ONE JSON line on rank 0.

Beside the headline the same line carries (all measured inside this run):
  sustained    the same step repeated for >= 2 s (power-capped clocks), next to the K-step burst figure
  e2e          host buffers in/out through rpst.hostpipe, with its PCIe roofline (measured pinned copy bandwidth)
  e2e_images   512^2 images in host memory -> stub RP encoder (cuDNN) -> rpst decode -> image back    [N = 1]
  configs      BASELINE configs #1, #3, #4, #5: device time, roofline fraction, tensor-pipe %, CPU baseline [N = 1]
  train        config-#5-shaped training transform (AdaIN fwd+bwd + loss statistics) with the 3.1 MB gradient
               all-reduce overlapped with the backward pass — the only collective of the path
  strong       32 images in total split over the N ranks (strong scaling of the headline step)

--dump-outputs DIR writes what rank 0's last timed step returned, one float32 file per level (DIR/out_c<C>.npy), so
that two builds run with the same arguments can be compared output for output (see dump_outputs).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LEVELS = [16, 32, 64, 128, 256]     # hidden_dim 16, rp_blocks 5, enc_stack_way deeper
H = W = 512
BATCH = 32
METRIC = "stylized images/sec @512^2 (multiscale RP-AdaIN transform)"
UNIT = "images/s"
WORKLOAD = ("configs[1]: multiscale RP-AdaIN (run_deeper_multiscale_rp_adain) transform, "
            "batch 32/GPU @512x512, levels C=16,32,64,128,256")


def algorithmic_bytes(batch: int) -> int:
    """SURVEY.md §8d: 3*E*4 for the plain AdaIN level, 4*E*4 for every blended level."""
    hw = H * W
    top = 3 * batch * LEVELS[-1] * hw * 4
    lower = sum(4 * batch * c * hw * 4 for c in LEVELS[:-1])
    return top + lower


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonHwPowerBrakeSlowdown: "hw_power_brake_slowdown"}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        med = statistics.median(self.samples) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def physical_gpu_index(local: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local])
        except Exception:
            return local
    return local


# ------------------------------------------------------------------------------- reference arm
def cpu_reference_images_per_s(images: int, repeats: int):
    """The reference's CPU path for this workload: ITS aten op sequence (`var`, `mean`, `sub`, `div`, `mul`, `add`,
    `add`; network/base.py:399-418, network/adain_rp.py:300-301) in eager torch on all host cores, restated in
    oracle/restate.py (`multiscale_transform_aten`) — the reference is Python and does not travel to the GPU box."""
    import torch
    from oracle import restate as R
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    g = torch.Generator().manual_seed(2002)
    feats = [(torch.relu(torch.randn(images, c, H, W, generator=g) + 0.5),
              torch.relu(torch.randn(images, c, H, W, generator=g) * 2 + 1)) for c in LEVELS]
    prevs = [torch.randn(images, c, H, W, generator=g) for c in LEVELS[:-1]]
    best = float("inf")
    times = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        R.multiscale_transform_aten([f[0] for f in feats], [f[1] for f in feats], prevs)
        dt = time.perf_counter() - t0
        times.append(dt)
        best = min(best, dt)
    return images / best, cores, times


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    # warm-up steps then K timed steps, each step = a bounded sample of the workload: 1 image through the five levels
    feats_per_step = 1
    for _ in range(max(args.warmup, 1)):
        cpu_reference_images_per_s(feats_per_step, 1)
    v, cores, times = cpu_reference_images_per_s(feats_per_step, args.steps)
    total = sum(times)
    value = feats_per_step * args.steps / total
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "sample": "each step = 1 image of the batch through all five levels (images are independent), "
                                 "reference aten op sequence in eager torch on the host cores"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{args.steps} steps x 1 image x 5 levels, torch {torch.__version__} CPU, {cores} threads"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------- B200 arm
def make_step(torch, rpst, dev, batch, seed):
    gen = torch.Generator(device=dev).manual_seed(seed)
    cs = [torch.relu(torch.randn(batch, c, H, W, device=dev, generator=gen) + 0.5) for c in LEVELS]
    ss = [torch.relu(torch.randn(batch, c, H, W, device=dev, generator=gen) * 2 + 1) for c in LEVELS]
    ps = [torch.randn(batch, c, H, W, device=dev, generator=gen) for c in LEVELS[:-1]]
    outs = [torch.empty_like(c) for c in cs]
    L = rpst._lib.lib()
    ws = torch.empty(max(L.rpst_adain_workspace_bytes(batch, c, H * W) for c in LEVELS), dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream
    top = len(LEVELS) - 1
    order = [top] + list(range(top - 1, -1, -1))

    def launch(l):
        prev = None if l == top else ps[l].data_ptr()
        rpst._lib.check(L.rpst_adain_fwd(cs[l].data_ptr(), ss[l].data_ptr(), prev, outs[l].data_ptr(), batch, LEVELS[l],
                                         H * W, LEVELS[l] * H * W, 1e-5, None, ws.data_ptr(), ws.numel(), stream))

    def step(events=None):
        for l in order:
            if events is not None:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                launch(l)
                b.record()
                events.append((l, a, b))
            else:
                launch(l)
    return step, (cs, ss, ps, outs)


DUMP_ELEMS = 1 << 21        # per level: 5 x 8 MiB of float32 stays under 64 MB in all
DUMP_SEED = 7


def dump_outputs(path, outs):
    """Write one output per level as <path>/out_c<C>.npy (float32, flattened NCHW order).  A level with more than
    DUMP_ELEMS elements is sampled at DUMP_ELEMS distinct element indices drawn with DUMP_SEED and sorted, so the
    sample depends only on the output's size and files of two runs with the same arguments line up."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    for c, out in zip(LEVELS, outs):
        flat = out.reshape(-1)
        if flat.numel() > DUMP_ELEMS:
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(flat.numel(), DUMP_ELEMS, replace=False))
            flat = flat[torch.from_numpy(idx).to(flat.device)]
        np.save(os.path.join(path, f"out_c{c}.npy"), flat.float().cpu().numpy())


def train_leg(torch, dist, rpst, dev, world, steps=6):
    """Config-#5-shaped training transform on every rank (one 1024x2048 image, C=256 level): AdaIN forward,
    loss statistics (style + normalised content loss, network/adain_rp.py:81-88), backward through both, and the
    decoder-gradient all-reduce (AdaINRPNet: 784 963 fp32 parameters = 3.1 MB, SURVEY §8e) issued on a side stream
    when the decoder gradients would be ready (before the transform's backward), so it overlaps the backward."""
    from rpst.dist import GradBucket
    from oracle import restate as R
    c, s = R.synth_features((1, 256, 1024, 2048), cfg=5, device=dev)
    c.requires_grad_()
    s.requires_grad_()
    params = [torch.nn.Parameter(torch.zeros(784963, device=dev))]
    params[0].grad = torch.randn(784963, device=dev)
    bucket = GradBucket(params)
    comm = torch.cuda.Stream(dev)
    ar_events = []

    def step(record):
        out = rpst.adaptive_instance_normalization(c, s)
        loss = rpst.calc_style_loss(out, s.detach()) + rpst.calc_content_loss(out, c.detach(), norm=True)
        ready = torch.cuda.Event()
        ready.record()                                   # decoder gradients exist from here on
        with torch.cuda.stream(comm):
            comm.wait_event(ready)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(comm)
            bucket.allreduce_mean({"loss": loss})
            b.record(comm)
            if record:
                ar_events.append((a, b))
        torch.autograd.grad(loss, (c, s))
        torch.cuda.current_stream().wait_stream(comm)

    for _ in range(2):
        step(False)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(steps):
        step(True)
    t1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / steps
    ar_us = statistics.median(a.elapsed_time(b) for a, b in ar_events) * 1e3
    # the collective alone (no bucket packing), same 3.1 MB buffer, back to back
    nccl_us = None
    if world > 1:
        flat = torch.zeros(784963 + 64, device=dev)
        for _ in range(5):
            dist.all_reduce(flat)
        torch.cuda.synchronize()
        dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(20):
            dist.all_reduce(flat)
        b.record()
        torch.cuda.synchronize()
        nccl_us = a.elapsed_time(b) / 20 * 1e3
    if world > 1:
        t = torch.tensor([ms, ar_us, nccl_us], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ar_us, nccl_us = float(t[0]), float(t[1]), float(t[2])
    E = c.numel() * 4
    # forward 3E, loss statistics 2 x 2E (two pairs), loss backward 2E + 3E, AdaIN backward 5E
    alg = (3 + 4 + 5 + 5) * E
    del c, s
    torch.cuda.empty_cache()
    return {"workload": "configs[4]-shaped training transform per GPU: 1x256x1024x2048 AdaIN fwd+bwd + style/content loss "
                        "statistics fwd+bwd + all-reduce of a 3.1 MB gradient bucket overlapped with the backward",
            "images_per_s": world / (ms / 1e3), "ms_per_step": ms, "allreduce_bucket_us": ar_us, "allreduce_nccl_us": nccl_us,
            "allreduce_bytes": 784963 * 4 + 256, "algorithmic_GBs_per_gpu": alg / (ms / 1e3) / 1e9, "scaling": "weak",
            "collective": "NCCL all-reduce (sum) on one flat fp32 bucket, side stream, waits only on the decoder-gradient event"}


def run_b200(args):
    import torch
    import torch.distributed as dist
    import rpst
    import bench_configs as BC
    from rpst.hostpipe import MultiscaleHostPipe

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = BC.bind_to_gpu_numa_node(local)       # before any pinned allocation: host buffers NUMA-local to the GPU
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world > 1:
            t = torch.tensor([x], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x

    strong = args.scaling == "strong"
    batch = args.batch if not strong else max(1, args.batch // world)
    step, (cs, ss, ps, outs) = make_step(torch, rpst, dev, batch, 2002 + rank)
    top = len(LEVELS) - 1

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(physical_gpu_index(local))
    sampler.start()
    events = []
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_start.record()
    for _ in range(args.steps):
        step(events)
    t_end.record()
    barrier()
    clocks = sampler.stop()
    elapsed_ms = max_over_ranks(t_start.elapsed_time(t_end))
    per_level_ms = {c: 0.0 for c in LEVELS}
    for l, a, b in events:
        per_level_ms[LEVELS[l]] += a.elapsed_time(b)
    kernel_ms = sum(per_level_ms.values())
    value = world * batch * args.steps / (elapsed_ms / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs)        # before the legs below run the step again

    # ---- sustained: the same step for >= 2 s (the burst above lasts ~0.3 s; the power cap settles later)
    sustained = None
    if not args.no_sustained:
        n_sus = max(args.steps, int(2200.0 / max(elapsed_ms / args.steps, 1e-3)))
        sampler2 = ClockSampler(physical_gpu_index(local))
        sampler2.start()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n_sus):
            step()
        b.record()
        barrier()
        clk2 = sampler2.stop()
        s_ms = max_over_ranks(a.elapsed_time(b))
        sustained = {"seconds": s_ms / 1e3, "steps": n_sus, "value": world * batch * n_sus / (s_ms / 1e3), "unit": UNIT,
                     "ms_per_step": s_ms / n_sus, "GBs_per_gpu": algorithmic_bytes(batch) * n_sus / (s_ms / 1e3) / 1e9,
                     "frac": algorithmic_bytes(batch) * n_sus / (s_ms / 1e3) / 1e9 / peaks()[0], "clocks": clk2}

    # ---- strong scaling of the same step: 32 images in total over the N ranks
    strong_leg = None
    if not strong and world > 1 and not args.no_extra:
        sb = max(1, BATCH // world)
        sstep, keep = make_step(torch, rpst, dev, sb, 4002 + rank)
        for _ in range(3):
            sstep()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(args.steps):
            sstep()
        b.record()
        barrier()
        s_ms = max_over_ranks(a.elapsed_time(b))
        strong_leg = {"scaling": "strong", "global_batch": sb * world, "batch_per_gpu": sb,
                      "value": world * sb * args.steps / (s_ms / 1e3), "unit": UNIT, "ms_per_step": s_ms / args.steps}
        del sstep, keep
        torch.cuda.empty_cache()

    # ---- e2e: same transform through the host-buffer front door (PCIe inside the timed region)
    e2e = None
    if not args.no_e2e:
        pipe = MultiscaleHostPipe(LEVELS, H, W, dev)
        pin = lambda c: torch.empty(1, c, H, W, dtype=torch.float32).pin_memory()
        hc = [pin(c).copy_(cs[i][:1].cpu()) for i, c in enumerate(LEVELS)]
        hs = [pin(c).copy_(ss[i][:1].cpu()) for i, c in enumerate(LEVELS)]
        hp = [pin(c).copy_(ps[i][:1].cpu()) for i, c in enumerate(LEVELS[:-1])]
        ho = [[pin(c) for c in LEVELS] for _ in range(2)]
        pipe.run(hc, hs, hp, ho, 4)
        barrier()
        e_imgs = args.e2e_images
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        pipe.run(hc, hs, hp, ho, e_imgs)
        b.record()
        barrier()
        e_ms = max_over_ranks(a.elapsed_time(b))
        # parity of what came back over PCIe against the resident path (same sample)
        chk = float((ho[(e_imgs - 1) & 1][top].cuda() - outs[top][:1]).abs().max())
        # PCIe roofline: pinned H2D and D2H running together on every rank at the same time (shared root complexes)
        barrier()
        bw = BC.pcie_bandwidth(dev)
        barrier()
        h2d_s = pipe.h2d_bytes_per_image / (bw["h2d_GBs"] * 1e9)
        d2h_s = pipe.d2h_bytes_per_image / (bw["d2h_GBs"] * 1e9)
        roof = 1.0 / max(h2d_s, d2h_s)                       # images/s per rank: full duplex, the slower direction bounds
        roof_all = -max_over_ranks(-roof) * world            # min over ranks x N
        e_val = world * e_imgs / (e_ms / 1e3)
        e2e = {"value": e_val, "unit": UNIT,
               "h2d_bytes_per_step": pipe.h2d_bytes_per_image * batch, "d2h_bytes_per_step": pipe.d2h_bytes_per_image * batch,
               "images_timed": e_imgs, "max_abs_diff_vs_resident": chk,
               "pcie_roofline": {"value": roof_all, "unit": UNIT, "h2d_GBs_rank0": bw["h2d_GBs"], "d2h_GBs_rank0": bw["d2h_GBs"],
                                 "how": bw["how"] + f", all {world} ranks at once; bound = slower direction, min over ranks x N"},
               "frac": e_val / roof_all, "numa": numa,
               "note": "pinned NUMA-local host buffers, per-image H2D/compute/D2H double-buffered on 3 streams; PCIe-bound: "
                       "1.29 GB of features in + 0.52 GB out per image"}
        del pipe, hc, hs, hp, ho

    # ---- training leg with the path's only collective (short; every N)
    train = None
    if not args.no_extra:
        del cs, ss, ps, outs, step
        torch.cuda.empty_cache()
        try:
            train = train_leg(torch, dist, rpst, dev, world)
        except Exception as e:
            train = {"error": repr(e)[:300]}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = peaks()
    alg = algorithmic_bytes(batch)
    achieved = alg * args.steps / (kernel_ms / 1e3) / 1e9
    traffic = None
    tp = os.path.join(ROOT, "profiles", "adain_traffic.json")
    if os.path.exists(tp):
        try:
            # ncu dram__bytes_read.sum + dram__bytes_write.sum, averaged over the step's 5 launches
            traffic = json.load(open(tp)).get("dram_bytes_per_launch_avg")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": "adain_tma_kernel<6> (5 launches/step: C=256 plain, C=128..16 blend; averaged over the launches)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "algorithmic_bytes_per_step": alg,
                "frac_of_nominal_8TBs": achieved / 8000.0,
                "per_level_GBs": {str(c): ((3 if c == LEVELS[-1] else 4) * batch * c * H * W * 4 * args.steps)
                                  / (per_level_ms[c] / 1e3) / 1e9 for c in LEVELS},
                "tensor_pipe": BC.tensor_pipe_summary() or None}

    cpu = None
    configs = None
    e2e_img = None
    if world == 1 and not args.no_cpu:
        v, cores, times = cpu_reference_images_per_s(2, 3)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": "2 images x 5 levels, best of 3, reference aten op sequence in eager torch CPU "
                         "(oracle/restate.py multiscale_transform_aten)"}
    if world == 1 and not args.no_extra:
        try:
            e2e_img = BC.e2e_images(dev, world, cpu=not args.no_cpu)
        except Exception as e:
            e2e_img = {"error": repr(e)[:300]}
        configs = BC.all_configs(dev, cpu=not args.no_cpu)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "batch_per_gpu": batch, "global_batch": batch * world, "parallelism": f"batch-sharded x{world}, no collective",
                       "l2": "inputs exceed L2 (54 GiB touched per step vs 126 MB L2); no explicit flush needed"},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "sustained": sustained, "e2e_images": e2e_img,
            "configs": configs, "train": train, "strong": strong_leg, "clocks": clocks,
            "gpu_launches": 5 * args.steps}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=BATCH, help="images per GPU (32 = BASELINE configs[1])")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="strong: --batch images in TOTAL over the ranks")
    ap.add_argument("--e2e-images", type=int, default=32)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sustained", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the configs / e2e_images / train / strong legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write rank 0's outputs of the last step as DIR/out_c<C>.npy "
                         "(float32, a fixed seeded sample of at most 2^21 elements per level)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
