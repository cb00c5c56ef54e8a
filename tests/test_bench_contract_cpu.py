"""bench.py's reference arm runs without a GPU: check the JSON line's contract keys here so that a change to
bench.py cannot silently break what the driver parses (the B200 arm is exercised on the GPU box)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("stylized images/sec") and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["steps"] == 1 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["scaling"] == "weak" and d["vs_baseline"] is None
    assert d["dtype"] == "f32" and d["data"] == "synthetic" and "workload" in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["unit"] == "images/s" and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_print_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_both_arms_name_the_same_workload():
    """VERDICT r1: `same_config` was false because the two arms spelled `config.workload` differently."""
    sys.path.insert(0, ROOT)
    import bench
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert src.count('"workload": WORKLOAD') == 2          # one per arm, both the module constant
    assert bench.WORKLOAD.startswith("configs[1]")
    assert bench.algorithmic_bytes(32) == 57982058496       # SURVEY §8d: 54 GiB per 32-image step


def test_dump_outputs_sample_is_fixed_and_bounded(tmp_path):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    outs = [torch.arange(n, dtype=torch.float64) for n in (3, 4, 5, 6, bench.DUMP_ELEMS + 1000)]
    bench.dump_outputs(str(tmp_path / "a"), outs)
    bench.dump_outputs(str(tmp_path / "b"), outs)
    for c, o in zip(bench.LEVELS, outs):
        a, b = np.load(tmp_path / "a" / f"out_c{c}.npy"), np.load(tmp_path / "b" / f"out_c{c}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, b)
        if o.numel() <= bench.DUMP_ELEMS:
            assert np.array_equal(a, o.numpy())
        else:       # distinct sorted element indices (arange: value == index)
            assert a.shape == (bench.DUMP_ELEMS,) and (np.diff(a) > 0).all() and a[-1] < o.numel()


def test_dump_outputs_rejected_for_the_reference_arm(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr


def test_stub_rp_network_cpu_leg_runs():
    """The CPU arm of the `e2e_images` leg: stub RP encoder/decoder + the reference's AdaIN op sequence."""
    import torch
    sys.path.insert(0, ROOT)
    import bench_configs as BC
    torch.manual_seed(0)
    net = BC.StubRPNet().eval()
    c, s = torch.rand(1, 3, 24, 24), torch.rand(1, 3, 24, 24)
    with torch.no_grad():
        feats = net.encode_rp_intermediate(c)
        assert [f.shape[1] for f in feats] == [16, 32, 64, 128, 256] and all(f.shape[2:] == (24, 24) for f in feats)
        out = BC.stylize_images(net, c, s, oracle=True)
    assert out.shape == (1, 3, 24, 24) and torch.isfinite(out).all()
