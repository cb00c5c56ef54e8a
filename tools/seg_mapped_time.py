"""Segment AdaIN through plane maps and into a channel slice, timed against the copies it replaces.

  1. unmapped path: a second build of librpst.so (--prev-lib, e.g. the parent commit's) against this tree's, alternating,
     on BASELINE configs[4] (1x256x1024x2048, 19 classes in 32x32 tiles), plain and with prev; outputs must be
     bit-identical between the builds
  2. shuffled masked level (same shape, shuffle_map): gather + seg_adain_batch against the mapped seg_adain_batch
  3. concat level, LDMS4-shaped 1x(64+64)x1024x2048: torch.cat route against seg_adain_concat

Every tensor is larger than L2.  Each shape is warmed before it is timed and the arms alternate (--rounds, default 2).
Usage: python tools/seg_mapped_time.py [--prev-lib PATH] [--rounds R] [--bench] [--only-bench]
(--bench also runs bench.py for both builds, --only-bench runs nothing else)"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import rpst  # noqa: E402
from oracle import restate as R  # noqa: E402

ROUNDS = 2   # --rounds


def emit(**kw):
    print(json.dumps(kw), flush=True)


def device_line():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                        "-i", str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q}


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


def peak_extra(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    out = fn()
    torch.cuda.synchronize()
    extra = torch.cuda.max_memory_allocated() - base
    del out
    return extra


def load(path):
    lib = ctypes.CDLL(path)
    for name in ("rpst_seg_adain_workspace_bytes", "rpst_seg_adain_fwd"):
        res, args = rpst._lib.SIGNATURES[name]
        getattr(lib, name).restype = res
        getattr(lib, name).argtypes = args
    return lib


def unmapped_ab(prev_lib):
    n, ch, h, w = 1, 256, 1024, 2048
    c, s = R.synth_features((n, ch, h, w), cfg=5, device="cuda")
    cl = R.synth_labels(n, h, w, seed=4000, device="cuda")
    sl = R.synth_labels(n, h, w, seed=5000, device="cuda")
    prev = torch.randn_like(c)
    hw = h * w
    libs = {"parent": load(prev_lib), "branch": rpst._lib.lib()}
    outs = {k: torch.empty_like(c) for k in libs}
    ws = torch.empty(max(L.rpst_seg_adain_workspace_bytes(n, ch, hw, hw) for L in libs.values()), dtype=torch.uint8,
                     device="cuda")
    E = c.numel() * 4
    stream = torch.cuda.current_stream().cuda_stream

    def call(k, p):
        rc = libs[k].rpst_seg_adain_fwd(c.data_ptr(), s.data_ptr(), cl.data_ptr(), sl.data_ptr(),
                                        None if p is None else p.data_ptr(), outs[k].data_ptr(), n, ch, hw, hw, 1e-5,
                                        None, ws.data_ptr(), ws.numel(), stream)
        assert rc == 0, rc

    for p in (None, prev):
        for k in libs:
            call(k, p)
        torch.cuda.synchronize()
        emit(part=1, prev=p is not None, outputs_equal=torch.equal(outs["parent"], outs["branch"]))
    for r in range(ROUNDS):
        for p in (None, prev):
            alg = (4 if p is not None else 3) * E + 2 * hw
            for k in libs:
                ms = dev_ms(lambda: call(k, p), iters=30, warm=5)
                emit(part=1, round=r, build=k, prev=p is not None, ms=round(ms, 4), GBs=round(alg / ms / 1e6, 1))


def shuffled_level():
    n, ch, h, w = 1, 256, 1024, 2048
    c, s = R.synth_features((n, ch, h, w), cfg=5, device="cuda")
    cl = R.synth_labels(n, h, w, seed=4000, device="cuda")
    sl = R.synth_labels(n, h, w, seed=5000, device="cuda")
    m = rpst.shuffle_map(n, ch, 4, "cuda")
    alg = 3 * c.numel() * 4 + 2 * h * w

    def gathered():
        cg = c.flatten(0, 1)[m.long()].view_as(c)
        sg = s.flatten(0, 1)[m.long()].view_as(s)
        return rpst.seg_adain_batch(cg, sg, cl, sl)

    def mapped():
        return rpst.seg_adain_batch(c, s, cl, sl, content_map=m, style_map=m)

    arms = {"gather+seg_adain_batch": gathered, "mapped seg_adain_batch": mapped}
    with torch.no_grad():
        emit(part=2, outputs_equal=torch.equal(gathered(), mapped()))
        for k, fn in arms.items():
            emit(part=2, arm=k, peak_extra_GB=round(peak_extra(fn) / 1e9, 3))
        for r in range(ROUNDS):
            for k, fn in arms.items():
                ms = dev_ms(fn)
                emit(part=2, round=r, arm=k, ms=round(ms, 4), GBs_alg=round(alg / ms / 1e6, 1))


def concat_level():
    n, cp, ch, h, w = 1, 64, 64, 1024, 2048
    c, s = R.synth_features((n, ch, h, w), cfg=5, device="cuda")
    prev = torch.randn((n, cp, h, w), device="cuda")
    cl = R.synth_labels(n, h, w, seed=4000, device="cuda")
    sl = R.synth_labels(n, h, w, seed=5000, device="cuda")
    E = c.numel() * 4
    alg = 2 * prev.numel() * 4 + 3 * E + 2 * h * w   # prev read + written, segment AdaIN 3E, labels

    arms = {"torch.cat": lambda: torch.cat([prev, rpst.seg_adain_batch(c, s, cl, sl)], dim=1),
            "seg_adain_concat": lambda: rpst.seg_adain_concat(prev, c, s, cl, sl)}
    with torch.no_grad():
        a, b = (fn() for fn in arms.values())
        emit(part=3, outputs_equal=torch.equal(a, b))
        del a, b
        for k, fn in arms.items():
            emit(part=3, arm=k, peak_extra_GB=round(peak_extra(fn) / 1e9, 3))
        for r in range(ROUNDS):
            for k, fn in arms.items():
                ms = dev_ms(fn)
                emit(part=3, round=r, arm=k, ms=round(ms, 4), GBs_alg=round(alg / ms / 1e6, 1))


def bench_ab(prev_lib):
    for r in range(ROUNDS):
        for k, path in (("parent", prev_lib), ("branch", rpst._lib.LIB_PATH)):
            env = dict(os.environ, RPST_LIB=path)
            p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "30",
                                "--warmup", "5", "--no-cpu"], capture_output=True, text=True, env=env, cwd=ROOT)
            line = p.stdout.strip().splitlines()[-1] if p.stdout.strip() else p.stderr[-2000:]
            emit(part="bench", round=r, build=k, rc=p.returncode, result=line)


def main():
    global ROUNDS
    ap = argparse.ArgumentParser()
    ap.add_argument("--prev-lib", default=None, help="a second build of librpst.so for the unmapped-path A/B")
    ap.add_argument("--rounds", type=int, default=ROUNDS)
    ap.add_argument("--bench", action="store_true")
    ap.add_argument("--only-bench", action="store_true")
    args = ap.parse_args()
    ROUNDS = args.rounds
    if not torch.cuda.is_available():
        sys.exit("seg_mapped_time.py measures on the GPU; no CUDA device found")
    emit(**device_line())
    if not args.only_bench:
        if args.prev_lib:
            unmapped_ab(args.prev_lib)
            torch.cuda.empty_cache()
        shuffled_level()
        torch.cuda.empty_cache()
        concat_level()
    if args.prev_lib and (args.bench or args.only_bench):
        torch.cuda.empty_cache()
        bench_ab(args.prev_lib)
    emit(**device_line())


if __name__ == "__main__":
    main()
