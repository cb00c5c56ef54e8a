#!/bin/bash
# same box, alternating builds: previous commit's library vs the working tree's
run() {
  RPST_LIB=$PWD/rp-style-transfer_b200/$1 python - <<'PY'
import json, os, subprocess, sys
sys.path.insert(0, os.getcwd())
sys.argv = ["bench.py", "--steps", "20", "--warmup", "5", "--no-e2e", "--no-cpu"]
import io, contextlib
buf = io.StringIO()
with contextlib.redirect_stdout(buf):
    import runpy; runpy.run_path("bench.py", run_name="__main__")
d = json.loads(buf.getvalue().strip().splitlines()[-1])
print(os.path.basename(os.environ["RPST_LIB"]), round(d["roofline"]["achieved"]), {k: round(v) for k, v in d["roofline"]["per_level_GBs"].items()}, d["clocks"]["sm_mhz"])
PY
}
for i in 1 2; do
  run librpst_prev.so
  run librpst.so

done
