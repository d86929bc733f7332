"""-m gpu: bench.py --dump-outputs writes what the last timed step returned (entropy-coded segment, decoded planes) and
writes the same files in every run with the same arguments."""
import os
import subprocess
import sys

import numpy as np
import pytest

import jpezy_b200 as J

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# C1 (one 512x512 image per step), a ring of 4 frames: step 5, the last of 6, encodes and decodes frame 1
ARGS = ["--workload", "c1", "--steps", "6", "--warmup", "3", "--ring", "4", "--no-configs", "--no-e2e", "--no-cpu-baseline"]


def dump(out_dir):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *ARGS, "--dump-outputs", str(out_dir)], cwd=ROOT,
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    return {n: np.load(os.path.join(out_dir, n + ".npy")) for n in ("segments", "segment_bytes", "decoded")}


def test_dump_outputs_is_the_last_step_and_reproducible(tmp_path, oracle):
    a, b = dump(tmp_path / "a"), dump(tmp_path / "b")
    assert all(a[n].dtype in (np.float32, np.float64) for n in a)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 << 20
    assert all(np.array_equal(a[n], b[n]) for n in a)
    W = H = 512
    r, g, bl = J.synth.image(0, W, H, frame=1)
    scan = oracle.encode(r, g, bl, W, H, scan_only=True)
    assert a["segment_bytes"].tolist() == [len(scan)]
    assert a["segments"].astype(np.uint8).tobytes() == scan
    _, _, R0, G0, B0 = oracle.decode(oracle.header(W, H) + scan + b"\xff\xd9")
    planes = a["decoded"].reshape(3, -1)
    assert planes.shape[1] == R0.size
    assert max(int(np.abs(planes[k] - x.astype(np.float32)).max()) for k, x in enumerate((R0, G0, B0))) <= 1
