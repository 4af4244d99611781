"""bench.py --dump-outputs on the GPU: the files hold what the timed device-resident step computed -- the same results
the host-buffer path gives for the same seeded bag, rendered again in this process."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_is_the_timed_steps_results(gpu_ctx, tmp_path):
    import bench
    from sonar_slam_b200 import _lib, pipeline, synth
    from sonar_slam_b200.bruce_slam.feature_extraction import FeatureExtraction

    F, out = 48, tmp_path / "outputs"
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), "--frames", str(F), "--steps", "2",
                        "--warmup", "1", "--pairs", "0", "--cpu-sample", "2", "--dump-outputs", str(out)],
                       capture_output=True, text=True, cwd=tmp_path, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    d = {p.stem: np.load(p) for p in out.glob("*.npy")}
    assert set(d) == {"frame_index", "T", "iterations", "inliers", "status", "cloud_count", "cloud_frame_index",
                      "cloud_xy"}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert np.array_equal(d["frame_index"], np.arange(F)) and np.array_equal(d["cloud_frame_index"], np.arange(F))

    bag = synth.make_trajectory_frames(F, seed=0, device="cuda")
    fx = FeatureExtraction()
    fx.generate_map_xy(synth.Ping(0, None, 30.0 / bench.R, bench.R, bag["bearings"]))
    maps = _lib.Maps(gpu_ctx, fx.map_x, fx.map_y, bench.R, bench.B, fx.width, fx.height)
    fe = pipeline.FrontEnd(gpu_ctx, maps, max_frames=F, tau=bench.TAU_SOCA,
                           icp=_lib.IcpParams(smooth_length=0, max_iterations=20))
    want = fe.run_host(bag["frames"].cpu().numpy(), bag["poses_odom"])
    assert (want["status"] == 0).any()
    assert np.array_equal(d["T"], want["T"])
    for k in ("iterations", "inliers", "status"):
        assert np.array_equal(d[k], want[k]), k
    assert np.array_equal(d["cloud_count"], want["npoints"])
    res = fe.results_dev()
    xy = gpu_ctx.to_host(res["cloud_xy"], (F, res["cloud_stride"], 2), np.float32)
    assert np.array_equal(d["cloud_xy"], np.concatenate([xy[f, :want["npoints"][f]] for f in range(F)]))
