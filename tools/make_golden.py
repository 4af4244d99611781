#!/usr/bin/env python
"""Generate the committed golden fixtures under tests/golden/ by RUNNING THE REFERENCE.

Runs only in the dev container (needs /root/reference).  The reference's Python is
imported unmodified from /root/reference/bruce_slam/src; what is missing in this
image is stubbed *around* it, never inside it:

  * ROS / gtsam / matplotlib / shapely imports  -> auto-generated stub modules
    (they are plumbing: subscribers, publishers, message types, plotting);
  * bruce_slam.cfar (pybind module built from cpp/cfar.cpp) -> a thin module over
    oracle/_ref/libcfar_ref.so, i.e. the UNMODIFIED cfar.cpp compiled against the
    storage-only Eigen shim (oracle/Makefile);
  * bruce_slam.pcl (libpointmatcher / PCL wrapper) -> identity stand-ins, so that
    the fixture captures the cloud BEFORE pcl.downsample / pcl.remove_outlier
    (those two are third-party arithmetic -- "parity unpinned", see DESIGN.md).

Fixtures written:
  tests/golden/cfar_tau.json        threshold factors from the reference's CFAR.py
                                    (CFAR.py:71-121) for several (Ntc,Ngc,Pfa,rank)
  tests/golden/cfar_masks.npz       packed CFAR masks (+ a threshold-image digest) of
                                    the config-1 frame from the reference cfar.cpp
  tests/golden/featx_config1.npz    FeatureExtraction.callback on the config-1 ping:
                                    map_x/map_y digests + samples, Cartesian (row,col)
                                    list and the metric points it publishes
  tests/golden/slam_host.npz        host-side numpy logic of SLAM.get_points (slam.py:229-292),
                                    SLAM.get_overlap (:389-424) and SLAM.compute_icp_with_cov
                                    (:325-387) run unmodified, with bruce_slam.pcl.{downsample,match}
                                    served by the CPU oracle and ICP.compute returning preset
                                    transforms (the natives themselves are covered elsewhere)
  tests/golden/globalinit.npz       SLAM.get_matching_cost_subroutine1 (slam.py:461-570) run
                                    unmodified on a synthetic source/target pair: the dilated
                                    target grid (packed) and the cost of 96 candidate poses.
                                    gtsam is absent: gtsam.Pose2 is replaced by the SE(2) class
                                    of oracle/globalinit_ref.py, everything else is the reference
  tests/golden/cfar_reference.npz   the unmodified cfar.cpp on the inputs of
                                    tests/test_oracle_cfar.py (masks, threshold digests + samples)
"""
import hashlib
import importlib
import importlib.abc
import importlib.machinery
import json
import os
import sys
import types
from unittest import mock

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SRC = "/root/reference/bruce_slam/src"
sys.path.insert(0, REPO)

STUB_ROOTS = {
    "rospy", "gtsam", "cv_bridge", "sensor_msgs", "geometry_msgs", "ros_numpy", "matplotlib",
    "shapely", "std_msgs", "visualization_msgs", "rti_dvl", "bar30_depth", "sonar_oculus", "tf",
    "message_filters", "nav_msgs", "rosbag", "kvh_gyro", "tf2_ros", "std_srvs", "bruce_msgs",
}


class _StubModule(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        m = mock.MagicMock(name=f"{self.__name__}.{name}")
        setattr(self, name, m)
        return m


class _StubFinder(importlib.abc.MetaPathFinder, importlib.abc.Loader):
    def find_spec(self, fullname, path, target=None):
        if fullname.split(".")[0] in STUB_ROOTS:
            return importlib.machinery.ModuleSpec(fullname, self, is_package=True)
        return None

    def create_module(self, spec):
        m = _StubModule(spec.name)
        m.__path__ = []
        return m

    def exec_module(self, module):
        pass


def _install_gtsam_stub():
    """gtsam with a working Pose2 (the cost function composes poses); the rest stays a mock."""
    from oracle import globalinit_ref

    g = _StubModule("gtsam")
    g.__path__ = []
    class Pose2(globalinit_ref.Pose2):  # + the accessor compute_icp_with_cov uses (slam.py:377)
        def rotation(self):
            R = self.matrix()[:2, :2]
            return types.SimpleNamespace(matrix=lambda: R)

        def compose(self, other):
            o = globalinit_ref.Pose2.compose(self, other)
            return Pose2(o.x(), o.y(), o.theta())

        def between(self, other):
            o = globalinit_ref.Pose2.between(self, other)
            return Pose2(o.x(), o.y(), o.theta())

    g.Pose2 = Pose2
    for name in ("Rot3", "Pose3"):  # conversions.g2n does isinstance() against these
        setattr(g, name, type(name, (), {}))
    g.Point2 = lambda *a: np.zeros(2)
    g.Point3 = lambda *a: np.zeros(3)
    sys.modules["gtsam"] = g


def _install_reference():
    from oracle import oracle as orc

    _install_gtsam_stub()
    sys.meta_path.insert(0, _StubFinder())
    sys.path.insert(0, REF_SRC)
    pkg = importlib.import_module("bruce_slam")

    cfar = types.ModuleType("bruce_slam.cfar")

    def _mk(alg, two):
        def f(img, train_hs, guard_hs, *rest):
            if alg == 3:
                k, tau = rest
            else:
                (tau,), k = rest, 0
            mask, thr = orc.cfar_reference(alg, np.asarray(img, np.float32), train_hs, guard_hs, int(k), float(tau), want_thr=two)
            return (mask, thr) if two else mask
        return f

    for i, nm in enumerate(["ca", "soca", "goca", "os"]):
        setattr(cfar, nm, _mk(i, False))
        setattr(cfar, nm + "2", _mk(i, True))
    sys.modules["bruce_slam.cfar"] = cfar
    pkg.cfar = cfar

    pcl = types.ModuleType("bruce_slam.pcl")
    pcl.downsample = lambda pts, *a: pts
    pcl.remove_outlier = lambda pts, *a: pts
    sys.modules["bruce_slam.pcl"] = pcl
    pkg.pcl = pcl
    return pkg


def _digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def main():
    from sonar_slam_b200 import synth

    out = os.path.join(REPO, "tests", "golden")
    os.makedirs(out, exist_ok=True)
    _install_reference()
    from bruce_slam.CFAR import CFAR  # the reference's own class

    # ---- threshold factors -------------------------------------------------------
    taus = []
    for (Ntc, Ngc, Pfa, rank) in [(40, 10, 0.1, 10), (40, 10, 1e-2, None), (24, 4, 0.05, 6),
                                   (16, 8, 1e-3, 15), (40, 10, 0.1, 0), (8, 2, 0.2, 3)]:
        try:
            c = CFAR(Ntc, Ngc, Pfa, rank)
        except ValueError as e:  # the reference itself gives up on some parameter sets
            taus.append(dict(Ntc=Ntc, Ngc=Ngc, Pfa=Pfa, rank=rank, raises=str(e)))
            continue
        taus.append(dict(Ntc=Ntc, Ngc=Ngc, Pfa=Pfa, rank=rank,
                         CA=float(c.threshold_factor_CA), SOCA=float(c.threshold_factor_SOCA),
                         GOCA=float(c.threshold_factor_GOCA), OS=float(c.threshold_factor_OS),
                         str=str(c)))
    with open(os.path.join(out, "cfar_tau.json"), "w") as f:
        json.dump(taus, f, indent=1)

    # ---- CFAR masks of the config-1 frame through the reference's CFAR class -----
    img = synth.make_frame(seed=1)
    det = CFAR(40, 10, 0.1, 10)
    masks = {}
    for alg in ["CA", "SOCA", "GOCA", "OS"]:
        m = det.detect(img, alg)
        m2, thr = det.detect2(img, alg)
        assert np.array_equal(m, m2)
        masks[alg] = np.packbits(np.ascontiguousarray(m))
        masks[alg + "_count"] = np.int64(m.sum())
        masks[alg + "_thr_sha256"] = np.array(_digest(np.ascontiguousarray(thr)))
        masks[alg + "_thr_sample"] = np.ascontiguousarray(thr)[::37, ::41].copy()
    np.savez_compressed(os.path.join(out, "cfar_masks.npz"), **masks)

    # ---- FeatureExtraction.callback on the config-1 ping --------------------------
    fe_mod = importlib.import_module("bruce_slam.feature_extraction")
    res = {}
    for tag, bearings in [("uniform", synth.bearings_uniform(512)), ("oculus", synth.bearings_oculus(512))]:
        fe = fe_mod.FeatureExtraction()
        fe.Ntc, fe.Ngc, fe.Pfa, fe.rank, fe.alg = 40, 10, 0.1, 10, "SOCA"
        fe.threshold, fe.resolution, fe.skip = 65, 0.5, 1
        fe.outlier_filter_radius, fe.outlier_filter_min_points = 1.0, 5
        fe.compressed_images = False
        fe.feature_img_pub = mock.MagicMock()
        fe.configure()
        captured = {}
        fe.publish_features = lambda ping, pts: captured.__setitem__("pts", np.array(pts))
        ping = synth.Ping(ping_id=0, image=img, range_resolution=30.0 / 512, num_ranges=512,
                          bearings=bearings)
        msg = types.SimpleNamespace(ping_id=0, ping=img, range_resolution=ping.range_resolution,
                                    num_ranges=512, bearings=list(bearings), header=mock.MagicMock())
        with mock.patch.object(fe_mod.ros_numpy.image, "image_to_numpy", lambda x: x):
            fe.callback(msg)
        pts = captured["pts"]
        # recover (row, col) exactly as the callback derived the points from them
        import cv2
        peaks = det.detect(img, "SOCA")
        peaks &= img > 65
        cart = cv2.remap(peaks, fe.map_x, fe.map_y, cv2.INTER_LINEAR)
        locs = np.c_[np.nonzero(cart)]
        res[tag + "_rows_cols"] = np.array([fe.rows, fe.cols], np.int64)
        res[tag + "_width_height_res"] = np.array([fe.width, fe.height, fe.res], np.float64)
        res[tag + "_map_x_sha256"] = np.array(_digest(fe.map_x))
        res[tag + "_map_y_sha256"] = np.array(_digest(fe.map_y))
        res[tag + "_map_x_sample"] = fe.map_x[::31, ::29].copy()
        res[tag + "_map_y_sample"] = fe.map_y[::31, ::29].copy()
        res[tag + "_locs"] = locs.astype(np.int32)
        res[tag + "_points"] = pts.astype(np.float64)
        assert len(locs) == len(pts)
        print(tag, "rows/cols", fe.rows, fe.cols, "polar det", int(peaks.sum()), "cart px", len(locs))
    np.savez_compressed(os.path.join(out, "featx_config1.npz"), **res)

    # ---- SLAM.get_matching_cost_subroutine1 on a synthetic pair -------------------
    slam_mod = importlib.import_module("bruce_slam.slam")
    gtsam = sys.modules["gtsam"]
    src, tgt, _ = synth.make_icp_pair(7, n_source=700, n_target=5000, extent=36.0, sensor_range=18.0)
    source_pose, target_pose = gtsam.Pose2(3.0, -1.5, 0.4), gtsam.Pose2(2.6, -1.1, 0.33)
    # the function is used unbound: it only reads self.point_noise (slam.py:73)
    fake_self = types.SimpleNamespace(point_noise=0.5)
    subroutine, pose_samples = slam_mod.SLAM.get_matching_cost_subroutine1(
        fake_self, src, source_pose, tgt, target_pose, np.diag([0.04, 0.04, 0.0004]))
    cells = {c.cell_contents.shape: c.cell_contents for c in subroutine.__closure__
             if isinstance(c.cell_contents, np.ndarray) and c.cell_contents.ndim == 2
             and c.cell_contents.dtype == np.uint8}
    (grid,) = cells.values()
    rng = np.random.default_rng(11)
    xs = np.concatenate([np.zeros((1, 3)), rng.uniform(-1, 1, (95, 3)) * np.array([1.0, 1.0, 0.1])])
    xs[1] = [0.4, -0.4, 0.07]
    costs = np.array([subroutine(x) for x in xs], np.int64)
    gi = dict(source=src, target=tgt, source_pose=np.array([3.0, -1.5, 0.4]), target_pose=np.array([2.6, -1.1, 0.33]),
              xs=xs, costs=costs, pose_samples=np.array(pose_samples), grid_shape=np.array(grid.shape, np.int64),
              grid_packed=np.packbits(grid > 0), grid_sha256=np.array(_digest(grid)))
    np.savez_compressed(os.path.join(out, "globalinit.npz"), **gi)
    # ---- host-side logic of get_points / get_overlap / compute_icp_with_cov ----------
    from oracle import oracle as orc
    pcl_stub = sys.modules["bruce_slam.pcl"]

    def _downsample(points, *rest):  # both pybind overloads (pcl.cpp:128,143), arithmetic = CPU oracle
        if len(rest) == 1:
            out, _ = orc.downsample(np.asarray(points, np.float32), rest[0])
            return out
        desc, res = rest
        out, idx = orc.downsample(np.asarray(points, np.float32), res)
        return out, np.asarray(desc)[idx]

    def _match(ref, pts, knn, max_dist):
        assert knn == 1
        return orc.match(np.asarray(ref, np.float32), np.asarray(pts, np.float32), max_dist)

    pcl_stub.downsample, pcl_stub.match = _downsample, _match
    rng = np.random.default_rng(5)
    kfs, kf_arrays = [], {}
    for k in range(4):
        c, _, _ = synth.make_icp_pair(30 + k, n_source=300 + 40 * k, n_target=400, extent=30.0, sensor_range=15.0)
        pose = gtsam.Pose2(0.4 * k, -0.2 * k, 0.05 * k)
        kf = types.SimpleNamespace(points=c, pose=pose, transf_points=slam_mod.Keyframe.transform_points(c, pose))
        kfs.append(kf)
        kf_arrays[f"kf{k}_points"] = c
        kf_arrays[f"kf{k}_pose"] = np.array([pose.x(), pose.y(), pose.theta()])
    fake = types.SimpleNamespace(current_key=4, keyframes=kfs, point_resolution=0.5, point_noise=0.5,
                                 icp_odom_sigmas=np.array([0.1, 0.1, 0.01]))
    S = slam_mod.SLAM
    sh = dict(kf_arrays)
    sh["points_all"] = S.get_points(fake)
    sh["points_ref_idx"] = S.get_points(fake, [0, 1, 2], 3)
    sh["points_ref_pose"] = S.get_points(fake, [1, 3], gtsam.Pose2(1.0, 0.5, -0.2))
    pk, kk = S.get_points(fake, [0, 2, 3], 1, True)
    sh["points_keys_pts"], sh["points_keys_keys"] = pk, kk
    n_ov, ind = S.get_overlap(fake, kfs[1].points, kfs[2].points, kfs[1].pose, kfs[2].pose, True)
    sh["overlap_count"], sh["overlap_indices"] = np.int64(n_ov), ind
    sh["overlap_plain"] = np.int64(S.get_overlap(fake, kfs[0].points, kfs[3].points))
    # compute_icp_with_cov: 14 guesses, ICP answers preset (3 failures); MinCovDet draws from numpy's global RNG
    Ts = []
    for i in range(14):
        th = 0.03 + rng.normal(0, 0.004)
        T = np.array([[np.cos(th), -np.sin(th), 0.5 + rng.normal(0, 0.02)],
                      [np.sin(th), np.cos(th), -0.3 + rng.normal(0, 0.02)], [0, 0, 1]], np.float32)
        if i == 4:
            T[0, 2] += 0.8  # an outlier the robust estimate should ignore
        Ts.append(("success" if i not in (2, 7, 11) else "ErrorMnimizer: no point to minimize", T))
    calls = iter(Ts)
    fake.icp = types.SimpleNamespace(compute=lambda s_, t_, g_: next(calls))
    guesses = [gtsam.Pose2(0.01 * i, 0.0, 0.0) for i in range(14)]
    np.random.seed(1234)
    msg, m, cov, samples = S.compute_icp_with_cov(fake, kfs[0].points, kfs[1].points, guesses)
    sh["cov_T"] = np.array([t for _, t in Ts])
    sh["cov_ok"] = np.array([m_ == "success" for m_, _ in Ts])
    sh["cov_msg"] = np.array(msg)
    sh["cov_mean"] = np.array([m.x(), m.y(), m.theta()])
    sh["cov_cov"], sh["cov_samples"] = cov, samples
    calls = iter(Ts[:5])  # four successes: below the five the reference asks for (slam.py:362-363)
    msg2 = S.compute_icp_with_cov(fake, kfs[0].points, kfs[1].points, guesses[:5])
    sh["cov_few_msg"] = np.array(msg2[0])
    np.savez_compressed(os.path.join(out, "slam_host.npz"), **sh)
    print("slam_host: all", sh["points_all"].shape, "keys", pk.shape, kk.shape, "overlap", int(n_ov), "cov msg", msg,
          "mean", sh["cov_mean"], "few:", msg2[0])
    print("globalinit: grid", grid.shape, "occupied", int((grid > 0).sum()), "costs", costs[:6], "min", costs.min())
    print("golden fixtures written to", out)


def fov_fixture():
    """tests/golden/fov_select.npz: the reference's own lines slam.py:876-899 (field-of-view pre-filter of the
    loop-closure targets), exec'ed verbatim on seeded inputs.  The lines sit inside a long method, so they are read
    from the reference file by number (and checked to be the expected statements) rather than called."""
    import textwrap
    from sonar_slam_b200 import synth
    _install_reference()
    slam_objects = importlib.import_module("bruce_slam.slam_objects")
    gtsam = sys.modules["gtsam"]
    with open(os.path.join(REF_SRC, "bruce_slam", "slam.py")) as f:
        lines = f.read().split("\n")
    block = lines[875:899]  # 1-based 876 .. 899
    assert block[0].strip().startswith("# Loop over the source frames") or "sel = np.zeros" in "".join(block[:4]), block[0]
    assert block[-1].strip() == "target_keys = target_keys[sel]", block[-1]
    code = textwrap.dedent("\n".join(block))
    rng = np.random.default_rng(21)
    _, tgt, _ = synth.make_icp_pair(3, n_source=100, n_target=6000, extent=80.0)
    target_points = (tgt + rng.normal(0, 0.01, tgt.shape)).astype(np.float32)
    target_keys = rng.integers(0, 40, (len(target_points), 1)).astype(np.float32)
    kfs = {}
    poses, covs = [], []
    for k in (17, 16, 15):
        pose = gtsam.Pose2(*(rng.uniform(-1, 1, 3) * [12.0, 12.0, 1.5]))
        A = rng.normal(0, 0.3, (3, 3))
        cov = A @ A.T * np.array([1.0, 1.0, 0.01])[:, None] * np.array([1.0, 1.0, 0.01])[None, :] + np.diag([0.05, 0.05, 1e-4])
        kfs[k] = types.SimpleNamespace(pose=pose, cov=cov)
        poses.append([pose.x(), pose.y(), pose.theta()])
        covs.append(cov)
    oculus = types.SimpleNamespace(max_range=30.0, horizontal_aperture=np.radians(130.0))
    ns = dict(np=np, Keyframe=slam_objects.Keyframe, source_frames=range(17, 14, -1),
              self=types.SimpleNamespace(keyframes=kfs, oculus=oculus),
              target_points=target_points.copy(), target_keys=target_keys.copy())
    exec(code, ns)  # noqa: S102 -- the reference's own statements
    out = os.path.join(REPO, "tests", "golden", "fov_select.npz")
    np.savez_compressed(out, target_points=target_points, target_keys=target_keys, poses=np.array(poses),
                        covs=np.array(covs), source_frames=np.array([17, 16, 15]), sel=ns["sel"],
                        kept_points=ns["target_points"], kept_keys=ns["target_keys"],
                        max_range=np.float64(30.0), horizontal_aperture=np.float64(np.radians(130.0)))
    print("fov_select:", len(target_points), "targets ->", int(ns["sel"].sum()), "kept; written to", out)


def cfar_reference_fixture():
    """tests/golden/cfar_reference.npz: the unmodified reference cfar.cpp (oracle/_ref/libcfar_ref.so) on the inputs
    of tests/test_oracle_cfar.py, every algorithm, two threshold factors.  Masks are stored packed; threshold images by
    the SHA-256 of their bytes (bit-exact) and a strided sample.  Needs the reference tree to build oracle/_ref."""
    from oracle import oracle as orc
    sys.path.insert(0, os.path.join(REPO, "tests"))
    from test_oracle_cfar import ALGS, TAU, _inputs
    orc.build()
    assert orc.have_reference(), "oracle/_ref/libcfar_ref.so was not built (reference tree absent)"
    g = {}
    for name, img, T, G, k in _inputs():
        g[name + "_input_sha256"] = np.array(_digest(img))
        for alg in ALGS:
            for i, tau in enumerate((TAU[alg], 0.37)):
                m, thr = orc.cfar_reference(alg, img, T, G, k, tau, want_thr=True)
                m_only, _ = orc.cfar_reference(alg, img, T, G, k, tau, want_thr=False)
                assert np.array_equal(m, m_only), (name, alg, i)
                thr = np.ascontiguousarray(thr)
                key = f"{name}_{alg}_{i}"
                g[key + "_mask"] = np.packbits(np.ascontiguousarray(m))
                g[key + "_thr_sha256"] = np.array(_digest(thr))
                g[key + "_thr_sample"] = thr[::7, ::5].copy()
    out = os.path.join(REPO, "tests", "golden", "cfar_reference.npz")
    np.savez_compressed(out, **g)
    print("cfar_reference:", len(g), "arrays written to", out)


if __name__ == "__main__":
    if "--only-fov" in sys.argv:
        fov_fixture()
    elif "--only-cfar-reference" in sys.argv:
        cfar_reference_fixture()
    else:
        main()
        fov_fixture()
        cfar_reference_fixture()
