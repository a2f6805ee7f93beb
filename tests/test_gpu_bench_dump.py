"""`bench.py --dump-outputs`: what the timed path returned is written as float arrays within 64 MiB, is the same from run
to run (whatever the number of timed steps), and `--steps` sets the number of timed steps."""
import json
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

READS = 100_000  # of the 100 bp headline workload: three blocks
ARGS = ["--gpus", "1", "--warmup", "3", "--reads", str(READS), "--no-extra-workloads", "--no-e2e", "--no-fastq", "--no-other-mode",
        "--no-cpu-baseline"]


def _bench(steps, out):
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), *ARGS, "--steps", str(steps), "--dump-outputs", str(out)],
                       capture_output=True, text=True, cwd=str(ROOT), timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_dump_outputs_and_steps(tmp_path):
    a, b = _bench(1, tmp_path / "a"), _bench(3, tmp_path / "b")
    assert a["steps"] == 1 and b["steps"] == 3 and a["verified_round_trip"] and b["verified_round_trip"]
    assert a["gpu_launches"] > 0 and b["gpu_launches"] == 3 * a["gpu_launches"]
    names = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert names == sorted(p.name for p in (tmp_path / "b").iterdir())
    assert names == sorted(f"{n}.npy" for n in ("block_offsets", "block_crc", "block_bytes_crc32", "container_sample",
                                                 "acids_sample", "quals_sample", "read_off_sample"))
    d = {n[:-4]: np.load(tmp_path / "a" / n) for n in names}
    for n in names:
        assert d[n[:-4]].dtype in (np.float32, np.float64) and np.array_equal(d[n[:-4]], np.load(tmp_path / "b" / n)), n
    assert sum(x.nbytes for x in d.values()) <= 64 << 20
    off = d["block_offsets"]
    assert len(off) == 4 and off[0] == 0 and (np.diff(off) > 8).all()
    assert len(d["block_crc"]) == len(d["block_bytes_crc32"]) == 3
    assert np.array_equal(d["read_off_sample"], np.arange(READS + 1) * 100.0)  # fewer than the sample size: all of them
    assert d["acids_sample"].max() <= 4 and d["quals_sample"].max() <= 93 and len(d["acids_sample"]) == len(d["quals_sample"])
