"""CPU-only: the CPU legs of bench.py (cpu_baseline / --impl reference) run and speak the JSON contract."""
import json
import os
import subprocess
import sys

import numpy as np

BENCH = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "bench.py")


def test_cpu_pipeline_leg_runs_on_a_tiny_sample():
    import bench
    from sonar_slam_b200 import synth
    d = synth.make_trajectory_frames(6, seed=1)
    bench._cpu_init(d["bearings"])
    secs = bench.cpu_pipeline(d["frames"].numpy(), d["poses_odom"], d["bearings"])
    assert 0.0 < secs < 60.0


def test_reference_arm_prints_one_json_line(monkeypatch, capsys):
    import bench
    monkeypatch.setattr(bench, "host_cores", lambda: (2, 8))   # usable (affinity mask), reported by the OS
    monkeypatch.setattr(sys, "argv", ["bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0"])
    a = bench.parse()
    bench.run_reference(a)
    out = [l for l in capsys.readouterr().out.splitlines() if l.startswith("{")]
    assert len(out) == 1
    line = json.loads(out[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["unit"] == "frames/s" and line["value"] > 0
    assert line["cpu_baseline"]["cores"] == 2 and line["e2e"]["h2d_bytes_per_step"] == 0
    assert line["cpu_baseline"]["cores_reported_by_os"] == 8 and len(line["config"]["step_seconds"]) == 1


def test_host_cores_follow_the_affinity_mask():
    import os
    import bench
    usable, reported = bench.host_cores()
    assert 1 <= usable <= reported and usable == len(os.sched_getaffinity(0))


def test_bench_refuses_to_run_the_product_path_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, BENCH, "--steps", "1", "--warmup", "0"], capture_output=True, text=True)
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)


class _FakeDevice:
    """Stands in for the library context and front end: device memory is one host byte buffer, addresses are offsets
    into it (starting at 4096 so that no buffer sits at address 0)."""

    def __init__(self, F, stride, rng):
        self.mem = bytearray(4096)
        self.F, self.stride = F, stride
        self.T = rng.normal(size=(F, 3, 3)).astype(np.float32)
        self.ints = {k: rng.integers(0, 50, F).astype(np.int32) for k in ("iterations", "inliers", "status")}
        self.count = rng.integers(0, stride + 3, F).astype(np.int32)   # a few above the stride: truncated clouds
        self.xy = rng.normal(size=(F, stride, 2)).astype(np.float32)
        self.addr = {k: self._put(a) for k, a in
                     dict(T=self.T, cloud_count=self.count, cloud_xy=self.xy, **self.ints).items()}

    def _put(self, a):
        at = len(self.mem)
        self.mem += a.tobytes()
        return at

    def to_host(self, ptr, shape, dtype):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        return np.frombuffer(bytes(self.mem[ptr:ptr + n]), dtype).reshape(shape).copy()

    def results_dev(self):
        return dict(self.addr, cloud_stride=self.stride)


def test_dumped_outputs_sample_and_bound(tmp_path):
    """bench.py --dump-outputs: a step of up to DUMP_FRAMES frames is kept whole; a larger one is sampled with a fixed
    seed (the same frames every run); clouds are read at the library's stride and clipped to it; every file is
    float32 or float64 and the total stays under 64 MiB even for the largest clouds."""
    import bench
    rng = np.random.default_rng(3)
    small = _FakeDevice(40, 16, rng)
    out = bench.last_step_outputs(small, small, small.F)
    assert np.array_equal(out["frame_index"], np.arange(small.F)) and np.array_equal(out["T"], small.T)
    for k, v in small.ints.items():
        assert np.array_equal(out[k], v) and out[k].dtype == np.float64
    assert np.array_equal(out["cloud_count"], small.count)
    want = np.concatenate([small.xy[f, :min(small.count[f], small.stride)] for f in range(small.F)])
    assert np.array_equal(out["cloud_frame_index"], np.arange(small.F)) and np.array_equal(out["cloud_xy"], want)

    big = _FakeDevice(bench.DUMP_FRAMES + 500, 4, rng)
    a, b = bench.last_step_outputs(big, big, big.F), bench.last_step_outputs(big, big, big.F)
    assert all(np.array_equal(a[k], b[k]) for k in a)
    idx = a["frame_index"].astype(int)
    assert len(idx) == bench.DUMP_FRAMES and np.all(np.diff(idx) > 0) and idx[-1] < big.F
    assert np.array_equal(a["T"], big.T[idx]) and np.array_equal(a["status"], big.ints["status"][idx])
    cf = a["cloud_frame_index"].astype(int)
    assert len(cf) == bench.DUMP_CLOUDS and np.isin(cf, idx).all()
    assert np.array_equal(a["cloud_xy"], np.concatenate([big.xy[f, :min(big.count[f], big.stride)] for f in cf]))

    bench.dump_outputs(str(tmp_path / "d"), a)
    for k in a:
        assert np.load(tmp_path / "d" / f"{k}.npy").dtype in (np.float32, np.float64), k
    cap_points = 8192    # sfe_frontend_params_default
    worst = bench.DUMP_FRAMES * (9 * 4 + 5 * 8) + bench.DUMP_CLOUDS * (cap_points * 2 * 4 + 8)
    assert worst < 64 * 2**20


def test_clock_sampler_keeps_the_load_until_samples_arrive(tmp_path, monkeypatch):
    """nvidia-smi that starts slower than the timed region (eight of them at N = 8): the sampler keeps the workload
    running, untimed, until it has its samples instead of reporting none."""
    import stat
    import time
    import bench
    fake = tmp_path / "nvidia-smi"
    fake.write_text("#!/bin/bash\nsleep 0.4\nwhile true; do echo '0, 1965, 1965, 700.0, Not Active, Not Active, "
                    "Not Active, Active'; sleep 0.05; done\n")
    fake.chmod(fake.stat().st_mode | stat.S_IEXEC)
    monkeypatch.setenv("PATH", f"{tmp_path}:" + __import__("os").environ["PATH"])
    c = bench.ClockSampler(0)
    c.start()
    extra = c.keep_load_until(3, lambda: time.sleep(0.01))
    out = c.stop()
    assert extra > 0 and out["samples"] >= 3 and out["sm_mhz"] == 1965.0 and out["reasons"] == ["sw_power_cap"]


def test_clock_sampler_counts_only_lines_after_the_mark(tmp_path, monkeypatch):
    """The sampler is started before the data is rendered (nvidia-smi's start-up is over when the timed region
    begins); what it printed before mark() -- idle clocks -- is not part of the report."""
    import stat
    import time
    import bench
    fake = tmp_path / "nvidia-smi"
    fake.write_text("#!/bin/bash\nfor i in 1 2 3; do echo '0, 120, 1965, 90.0, Not Active, Not Active, Not Active, "
                    "Not Active'; sleep 0.03; done\nsleep 0.3\nwhile true; do echo '0, 1965, 1965, 700.0, Not Active, "
                    "Not Active, Not Active, Not Active'; sleep 0.03; done\n")
    fake.chmod(fake.stat().st_mode | stat.S_IEXEC)
    monkeypatch.setenv("PATH", f"{tmp_path}:" + __import__("os").environ["PATH"])
    c = bench.ClockSampler(0)
    c.start()
    time.sleep(0.25)          # "rendering + warm-up": the three idle lines arrive
    c.mark()
    c.keep_load_until(3, lambda: time.sleep(0.01))
    out = c.stop()
    assert out["lines_before_timed_region_not_counted"] == 3
    assert out["samples"] >= 3 and out["sm_mhz"] == 1965.0 and out["reasons"] == []


def test_rank_binding_near_its_gpu(tmp_path):
    """bench.py under torchrun: a rank restricts itself to its GPU's local CPUs (sysfs local_cpulist) before it pins
    host memory; without the entry, or when the list is not narrower than what it may use, nothing changes."""
    import os
    import bench
    assert bench.parse_cpulist("0-3,8,10-11\n") == [0, 1, 2, 3, 8, 10, 11] and bench.parse_cpulist("") == []
    before = os.sched_getaffinity(0)
    try:
        assert bench.bind_near_gpu(0, 0x1b, 0, sysfs=str(tmp_path))["bound"] is False          # no such device
        dev = tmp_path / "0000:1b:00.0"
        dev.mkdir()
        (dev / "local_cpulist").write_text(",".join(map(str, sorted(before))) + "\n")
        assert bench.bind_near_gpu(0, 0x1b, 0, sysfs=str(tmp_path))["bound"] is False          # not narrower
        if len(before) > 1:
            one = sorted(before)[0]
            (dev / "local_cpulist").write_text(f"{one},100000\n")
            r = bench.bind_near_gpu(0, 0x1b, 0, sysfs=str(tmp_path))
            assert r["bound"] and r["cpus"] == 1 and os.sched_getaffinity(0) == {one}
    finally:
        os.sched_setaffinity(0, before)
