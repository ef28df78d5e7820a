"""bench.py --dump-outputs: the last timed step's frames (a seeded sample) and sizes, the same from run to run, and
frames that decode to whole chunks."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import helpers as H

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--nchunks", "256",
           "--no-secondary", "--no-cpu-baseline", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    return line, {f: np.load(os.path.join(out, f + ".npy")) for f in ("sizes", "frame_index", "frames")}


def test_bench_dump_outputs(tmp_path):
    line, a = _bench(tmp_path / "a")
    assert line["steps"] == 2 and line["config"]["chunks_per_gpu"] == 256
    assert sorted(os.listdir(tmp_path / "a")) == ["frame_index.npy", "frames.npy", "sizes.npy"]
    _, b = _bench(tmp_path / "b")
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.array_equal(a[k], b[k]), k
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    sizes, idx, frames = a["sizes"], a["frame_index"].astype(np.int64), a["frames"]
    assert sizes.shape == (256,) and (sizes > 0).all() and sizes.sum() / (256 * 65536) == pytest.approx(line["ratio"])
    assert len(idx) == frames.shape[0] == 64 and len(np.unique(idx)) == 64
    for i, row in zip(idx, frames):
        n = int(sizes[i])
        assert not row[n:].any()
        back = H.libzstd_decode(row[:n].astype(np.uint8).tobytes(), 65536)
        assert back is not None and len(back) == 65536, i
