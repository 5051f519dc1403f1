"""bench.py --dump-outputs (-m gpu): the arrays written after the timed steps are what the public API returns for the
same seeded workload, so two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dumped_outputs_match_the_public_api(ctx, tmp_path):
    import lpvspectral_jl_b200 as lp
    from lpvspectral_jl_b200 import _lib as L

    import bench

    env = dict(os.environ, RANK="0", WORLD_SIZE="1", LOCAL_RANK="0")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-admm",
                          "--no-extra", "--cpu-windows", "1", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.strip()][-1])
    assert d["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["psd.npy", "window_sums.npy"]
    sums = np.load(tmp_path / "window_sums.npy")
    psd = np.load(tmp_path / "psd.npy")
    assert sums.dtype == psd.dtype == np.float64 and sums.shape == psd.shape == (bench.NF,)
    K = d["config"]["windows_per_gpu"]
    assert np.array_equal(psd, lp.window_finalize(L.WIN_PSD, sums, bench.NF, K))
    t, y, f, _ = bench.make_cfg2()
    ref, _ = lp.ls_windowpsd(y, t, f, nw=bench.NW, window_func=lp.hanning, ctx=ctx)
    assert np.linalg.norm(psd - ref) / np.linalg.norm(ref) < 1e-12
