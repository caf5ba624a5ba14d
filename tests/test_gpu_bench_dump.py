"""``bench.py --dump-outputs``: what it writes is what the timed path computed, in float32, within 64 MB."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from oracle import synth

pytestmark = pytest.mark.gpu

ROOT = Path(__file__).resolve().parent.parent


def test_dump_outputs_is_the_timed_steps_output(proj, tmp_path):
    out = tmp_path / "dump"
    run = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "2", "--warmup", "1", "--distinct", "1",
                          "--e2e-steps", "1", "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(out)],
                         capture_output=True, text=True, cwd=tmp_path)
    assert run.returncode == 0, run.stderr[-3000:]
    assert json.loads(run.stdout)["steps"] == 2
    assert sum(f.stat().st_size for f in out.iterdir()) <= 64 << 20
    views, yx = np.load(out / "views.npy"), np.load(out / "views_yx.npy")
    assert views.dtype == yx.dtype == np.float32
    assert views.shape == (32, 4, 3, 8192, 3) and yx.shape == (8192, 2)
    y, x = yx.astype(np.int64).T
    assert len(set(zip(y, x))) == 8192 and y.max() < 1080 and x.max() < 1920
    # with one distinct seed, image i of the batch is the seed-0 panorama rolled by 37 * i columns
    pano = synth.noise(8192, 4096, 0)
    for i in (0, 1, 31):
        want = proj.project_image(np.roll(pano, 37 * i, axis=1), [0, 90, 180, 270], [30, 60, 90], 1920, 1080, 120)
        assert np.array_equal(views[i], want[:, :, y, x].astype(np.float32)), i
