"""bench.py's JSON-line contract, checked on the CPU through the reference arm
(`--impl reference` times the C++ oracle port on the host cores; no GPU involved),
and its --dump-outputs on the GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2",
                        "--warmup", "1", "--cpu-sample-slots", "16384"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "slots/s" and line["higher_is_better"] is True
    assert line["metric"].startswith("committed slots/sec")
    assert line["value"] > 0 and line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"]


def test_product_paths_never_import_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's cpu legs may touch oracle/."""
    pkg = os.path.join(ROOT, "frankenpaxos_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".inc", ".c", ".h", ".hpp")):
                text = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "fpx_oracle" not in text and "from oracle" not in text and "import oracle" not in text, f


@pytest.mark.gpu
def test_dump_outputs_of_the_last_timed_step_are_reproducible(tmp_path):
    """--dump-outputs: the reply streams of the last timed step, float64, at most 64 MB, identical over two runs."""
    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-e2e",
                            "--no-extra", "--cpu-sample-slots", "16384", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
        assert sum(f.stat().st_size for f in d.iterdir()) <= 64 << 20
        dumps.append({f.name: np.load(f) for f in d.iterdir()})
    assert sorted(dumps[0]) == ["chosen.npy", "phase2b.npy", "sync.npy", "watermark.npy"]
    for name, a in dumps[0].items():
        assert a.dtype == np.float64 and a.size > 0 and np.array_equal(a, dumps[1][name]), name
    status, n_p2b, n_nack, n_chosen, wm = dumps[0]["sync.npy"]
    assert status == 0 and n_p2b == 3 << 20 and n_nack == 0 and n_chosen == 1 << 20
    assert wm == dumps[0]["watermark.npy"][0] == 5 << 20
    # 3 warm-up + 2 timed steps: the last timed step chose every slot of the fifth window, nothing else
    assert np.array_equal(np.sort(dumps[0]["chosen.npy"][:, 0]), np.arange(4 << 20, 5 << 20))
    assert len(dumps[0]["phase2b.npy"]) == 1 << 20 and np.all(dumps[0]["phase2b.npy"][:, 2] >= 4 << 20)
