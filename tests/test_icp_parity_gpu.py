"""GPU parity sweep of the scan matcher (SURVEY.md 8(c): libpointmatcher is not vendored, parity is UNPINNED; this is
what an unpinned stage can offer):

  * default mode (sequential float32 sums, the oracle's accumulation order): status, iteration count, inlier count
    and the 3x3 result are BIT-IDENTICAL to oracle/icp_ref.c on every problem -- far inside the north star's
    1e-3 m / 1e-3 rad;
  * float64-accumulation mode (sfe_icp_params.flags bit 1): same status, and where the iteration count agrees the same
    inlier count; its pose deviates from the float32 chain by what the float32 chain deviates from exact arithmetic;
  * a third, independent arm -- float64 numpy + scipy cKDTree -- shows where both sit: the float64-accumulating GPU
    mode is the closer one; the float32-sequential oracle (and with it the default mode) is within ~2e-3 m of it on
    the worst of 200 scans, 1e-5 m on the median one.

200 BASELINE-config-3 pairs (2 000 x 20 000 points, identity guess) x {fixed 20 iterations, shipped checkers} and
200 pipeline-sized problems (~350 x ~1 100 points, odometry-like guesses).  The deviation histograms are printed and,
when SFE_ICP_SWEEP_REPORT names a file, written there as JSON (profiles/r02_icp_parity_sweep.json is one)."""
import json
import os

import numpy as np
import pytest
import torch
from scipy.spatial import cKDTree

from oracle import oracle as orc
from sonar_slam_b200 import _lib, ops, synth

pytestmark = pytest.mark.gpu
N_SWEEP = int(os.environ.get("SFE_ICP_SWEEP", "200"))


def _pose(T):
    T = np.asarray(T, np.float64)
    return np.array([T[0, 2], T[1, 2], np.arctan2(T[1, 0], T[0, 0])], np.float64)


def _pack(clouds):
    off = np.zeros(len(clouds) + 1, np.int32)
    off[1:] = np.cumsum([len(c) for c in clouds])
    return torch.from_numpy(np.concatenate(clouds).astype(np.float32)).cuda(), torch.from_numpy(off).cuda()


def _gpu(pairs, guesses, **kw):
    sp, so = _pack([p[0] for p in pairs])
    tp, to = _pack([p[1] for p in pairs])
    g = torch.from_numpy(np.stack(guesses).astype(np.float32)).cuda()
    out = ops.icp(sp, so, tp, to, g, max(len(p[0]) for p in pairs), max(len(p[1]) for p in pairs), _lib.IcpParams(**kw))
    return {k: v.cpu().numpy() for k, v in out.items()}


def _f64_icp(src, tgt, guess, iters):
    """Independent float64 arm: scipy cKDTree NN + closed-form 2-D rigid fit, fixed iteration count."""
    src, tgt = src.astype(np.float64), tgt.astype(np.float64)
    tree = cKDTree(tgt)
    T = np.array(guess, np.float64)
    keep = None
    for _ in range(iters):
        p = src @ T[:2, :2].T + T[:2, 2]
        d, j = tree.query(p, distance_upper_bound=10.0)
        fin = np.isfinite(d)
        d2 = d ** 2
        lim = np.sort(d2[fin])[int(np.float32(fin.sum()) * np.float32(0.8))]
        keep = fin & (d2 <= 9.0) & (d2 <= lim)
        a, b = p[keep], tgt[j[keep]]
        ma, mb = a.mean(0), b.mean(0)
        M = (b - mb).T @ (a - ma)
        th = np.arctan2(M[1, 0] - M[0, 1], M[0, 0] + M[1, 1])
        c, s = np.cos(th), np.sin(th)
        dT = np.eye(3)
        dT[:2, :2] = [[c, -s], [s, c]]
        dT[:2, 2] = mb - dT[:2, :2] @ ma
        T = dT @ T
    return T, int(keep.sum())


def _hist(x):
    x = np.asarray(x, np.float64)
    edges = [0, 1e-6, 1e-5, 1e-4, 2e-4, 4e-4, 6e-4, 8e-4, 1e-3, 2e-3, np.inf]
    cnt, _ = np.histogram(x, edges)
    return {"edges": [str(e) for e in edges], "counts": cnt.tolist(), "p50": float(np.percentile(x, 50)),
            "p90": float(np.percentile(x, 90)), "p99": float(np.percentile(x, 99)), "max": float(x.max())}


def _sweep(name, pairs, guesses, kw, fixed_iters):
    okw = {k: v for k, v in kw.items()}
    want = [orc.icp(s, t, g.astype(np.float32), orc.IcpParams(**okw)) for (s, t), g in zip(pairs, guesses)]
    par = _gpu(pairs, guesses, **kw)              # default = parity mode (sequential float32 sums)
    f64 = _gpu(pairs, guesses, flags=2, **kw)     # float64 accumulation
    n = len(pairs)
    dev_t, dev_r, iter_diff = [], [], 0
    for i, w in enumerate(want):
        # ---- default mode: bit-identical to the oracle
        assert par["status"][i] == w["status"], (name, i)
        assert par["iterations"][i] == w["iterations"] and par["inliers"][i] == w["inliers"], (name, i)
        assert np.array_equal(par["T"][i].view(np.uint32), w["T"].view(np.uint32)), (name, i, par["T"][i], w["T"])
        # ---- float64-accumulation mode: same outcome class; deviations are recorded
        assert f64["status"][i] == w["status"], (name, i)
        if w["status"] != 0:
            continue
        if f64["iterations"][i] != w["iterations"]:
            iter_diff += 1        # a stop decision on the knife edge (checkers mode only)
            continue
        d = np.abs(_pose(f64["T"][i]) - _pose(w["T"]))
        dev_t.append(d[:2].max())
        dev_r.append(d[2])
    rep = {"problems": n, "default_mode_bit_identical_to_oracle": n, "float64_mode_vs_oracle_trans": _hist(dev_t),
           "float64_mode_vs_oracle_rot": _hist(dev_r), "float64_mode_iteration_count_differs": iter_diff}
    assert np.percentile(dev_t, 90) < 1e-3 and max(dev_t) < 1e-2 and max(dev_r) < 1e-3, (name, _hist(dev_t))
    if fixed_iters:
        assert iter_diff == 0
        g_t, o_t = [], []
        for i, ((s, t), g) in enumerate(zip(pairs, guesses)):
            if want[i]["status"] != 0:
                continue
            Tn, _ = _f64_icp(s, t, g, fixed_iters)
            g_t.append(np.abs(_pose(f64["T"][i]) - _pose(Tn)).max())
            o_t.append(np.abs(_pose(want[i]["T"]) - _pose(Tn)).max())
        rep["float64_mode_vs_float64_arm"] = _hist(g_t)
        rep["oracle_and_default_mode_vs_float64_arm"] = _hist(o_t)
        # the float64-accumulating mode is not farther from the float64 arm than the float32 chain is
        assert np.percentile(g_t, 90) <= np.percentile(o_t, 90) * 1.5 + 1e-5, (np.percentile(g_t, 90), np.percentile(o_t, 90))
        assert max(g_t) < 5e-3 and max(o_t) < 5e-3
    else:
        assert iter_diff <= max(4, n // 20), iter_diff
    print(name, json.dumps(rep))
    return rep


@pytest.fixture(scope="module")
def sweep_log():
    log = {}
    yield log
    if os.environ.get("SFE_ICP_SWEEP_REPORT"):
        with open(os.environ["SFE_ICP_SWEEP_REPORT"], "w") as f:
            json.dump(log, f, indent=1)


@pytest.mark.parametrize("mode", ["fixed20", "checkers"])
def test_config3_sweep(gpu_ctx, mode, sweep_log):
    kw = dict(smooth_length=0, max_iterations=20) if mode == "fixed20" else {}
    pairs = [synth.make_icp_pair(s)[:2] for s in range(N_SWEEP)]
    guesses = [np.eye(3)] * len(pairs)
    sweep_log["config3_" + mode] = _sweep("config3_" + mode, pairs, guesses, kw, 20 if mode == "fixed20" else 0)


@pytest.mark.parametrize("mode", ["fixed20", "checkers"])
def test_pipeline_sized_sweep(gpu_ctx, mode, sweep_log):
    kw = dict(smooth_length=0, max_iterations=20) if mode == "fixed20" else {}
    rng = np.random.default_rng(77)
    pairs, guesses = [], []
    for s in range(N_SWEEP):
        ns, nt = int(rng.integers(250, 640)), int(rng.integers(700, 1536))
        src, tgt, Tgt = synth.make_icp_pair(5000 + s, n_source=ns, n_target=nt)
        pairs.append((src, tgt))
        # odometry-like guess: the ground truth disturbed by the odometry noise of a step
        guesses.append(Tgt @ synth.se2(*rng.normal(0, [0.1, 0.1, 0.01])))
    sweep_log["pipeline_" + mode] = _sweep("pipeline_" + mode, pairs, guesses, kw, 20 if mode == "fixed20" else 0)
