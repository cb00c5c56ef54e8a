"""bench.py --dump-outputs: the files hold the outputs of the headline step for bench's seeded inputs, so two builds
run with the same arguments can be compared file for file."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import restate as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_hold_the_last_timed_step(tmp_path):
    got_dir, want_dir = tmp_path / "got", tmp_path / "want"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--batch", "1", "--steps", "2", "--warmup", "1",
                          "--no-sustained", "--no-e2e", "--no-cpu", "--no-extra", "--dump-outputs", str(got_dir)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    sys.path.insert(0, ROOT)
    import bench
    import rpst
    names = sorted(f"out_c{c}.npy" for c in bench.LEVELS)
    assert sorted(os.listdir(got_dir)) == names
    assert sum(os.path.getsize(got_dir / n) for n in names) <= 64e6

    # the same inputs regenerated in this process (rank 0's seed), fp64 oracle (it copies them to the host), sampled by
    # the same rule
    _, (cs, ss, ps, _) = bench.make_step(torch, rpst, torch.device("cuda", 0), 1, 2002)
    top = len(bench.LEVELS) - 1
    want = [R.adain(cs[l], ss[l], dtype=torch.float64) if l == top else R.adain_blend(ps[l], cs[l], ss[l], dtype=torch.float64)
            for l in range(top + 1)]
    bench.dump_outputs(str(want_dir), want)
    for n in names:
        g, w = np.load(got_dir / n), np.load(want_dir / n)
        assert g.dtype == np.float32 and g.shape == (bench.DUMP_ELEMS,)
        assert R.rel_l2(torch.from_numpy(g), torch.from_numpy(w)) < 1e-5, n
