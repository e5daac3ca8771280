"""bench.py --dump-outputs: every timed workload writes what its last timed step returned, in float32, within the size
bound, equal to the construction of its seeded inputs and identical from run to run; --steps sets the timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=1800)


def test_steps_must_be_positive():
    p = run_bench("--steps", "0")
    assert p.returncode == 2 and "--steps" in p.stderr


@pytest.mark.gpu
def test_dump_outputs_are_the_construction_and_repeat(tmp_path):
    import bench
    n, extra_n, steps = 4096, 16384, 2
    dumps = []
    for run in ("a", "b"):
        out = tmp_path / run
        p = run_bench("--n", str(n), "--extra-n", str(extra_n), "--steps", str(steps), "--warmup", "0", "--no-cpu",
                      "--dump-outputs", str(out))
        assert p.returncode == 0, p.stderr[-3000:]
        d = json.loads(p.stdout.strip().splitlines()[-1])
        assert d["steps"] == steps and all(rec["steps"] == steps for rec in d["extra"].values())
        files = sorted(os.listdir(out))
        assert files == sorted(f"{k}.npy" for k in ("verify_status", "proof_L10_R5_status", "proof_L32_R16_status",
                                                    "bn254_status", "sign_signatures", "sign_status", "rlc_verdict"))
        assert sum(os.path.getsize(out / f) for f in files) <= 64 << 20
        dumps.append({f[:-4]: np.load(out / f) for f in files})
    a, b = dumps
    for name, arr in a.items():
        assert arr.dtype == np.float32, name
        assert np.array_equal(arr, b[name]), name              # seeded inputs: the same outputs in every run

    def construction(size, first):
        want = np.ones(size, dtype=np.float32)
        want[first::16] = 0
        return want

    assert np.array_equal(a["verify_status"], construction(n, 3))
    for name in ("proof_L10_R5_status", "proof_L32_R16_status", "bn254_status"):
        assert np.array_equal(a[name], construction(extra_n, 5)), name
    assert np.array_equal(a["sign_status"], np.ones(extra_n, dtype=np.float32))
    assert a["rlc_verdict"].tolist() == [1.0]
    sig = a["sign_signatures"]                                # 16,384 x 80 bytes > DUMP_VALUES: a sample of rows
    assert sig.shape == (bench.DUMP_VALUES // bench.SIG_BYTES, bench.SIG_BYTES)
    assert sig.min() >= 0 and sig.max() <= 255 and np.array_equal(sig, np.round(sig))      # bytes, exactly
    assert len(np.unique(sig[:, :48], axis=0)) == len(sig)                                   # distinct rows: no repeats
