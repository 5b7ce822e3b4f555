"""Pins the CPU restatement (oracle/) against the reference's OWN sources.

tests/golden/reference_pin.npz holds what the reference computed -- tools/mad_tree.cpp, odometry/mad_icp.cpp,
odometry/vel_estimator.cpp and odometry/pipeline.cpp compiled unmodified against oracle/eigen_standin
(oracle/_ref/libmadicp_ref.so) -- on the inputs below; tests/golden/make_reference_golden.py wrote it.  Everything the
reference decides -- split order, leaf selection, normal inheritance, NaN handling of 1-point nodes, gate, kernel,
accumulation order, keyframe promotion -- runs as written by its authors; the restatement must reproduce it bit for
bit.  What stays unpinned is the evaluation order INSIDE Eigen's operators, which the stand-in takes from the
restatement (see its header).  Large arrays are stored as digests of their values (tests/util.py, fingerprint).

CPU only.
"""
import ctypes as C
import os

import numpy as np
import pytest

from mad_icp_b200 import synth
from util import same

GOLD = os.path.join(os.path.dirname(__file__), "golden", "reference_pin.npz")
B_MAX_WALLS = (0.2, 1e-5)
REG_CASES = ((1, 1), (3, 2), (4, 4))
SWEEP = ((0.1, 0.05, 0.05, 0.01), (0.4, 0.2, 0.3, 0.05), (0.2, 0.1, 1e-3, 0.0))
LOOP_KEYS = ("X_hist", "H_hist", "b_hist", "X", "matched")


# ---- the inputs, shared with tests/golden/make_reference_golden.py
def walls(points_per_wall):
    np.random.seed(42)
    return synth.four_walls(points_per_wall=points_per_wall)


def degenerate_clouds():
    rs = np.random.RandomState(3)
    return (rs.rand(1, 3), rs.rand(2, 3), rs.rand(3, 3), np.repeat(rs.rand(1, 3), 50, axis=0),
            np.c_[rs.rand(200, 2), np.zeros(200)], np.c_[rs.rand(64), np.zeros((64, 2))])


def demo_guess():
    """apps/utils/tools/mad_registration.py: the four-walls cloud (seed 42) and the initial guess drawn after it."""
    cloud = walls(1000)
    T = np.eye(4)
    T[:3, :3] = synth.euler_xyz(0.1, 0.1, 0.1)
    T[:3, 3] = np.random.rand(3)
    return cloud, T


def sequence(n, beams=16, azimuths=512):
    scene = synth.StreetScene(seed=7)
    for i in range(n):
        base = synth.pose_xyyaw(0.8 * i, 1.0 + 0.02 * i, 0.004 * i)
        yield 0.1 * i, np.ascontiguousarray(synth.lidar_scan(scene, base, beams=beams, azimuths=azimuths, seed=100 + i))


DESKEW_POSES = (synth.pose_xyyaw(0.0, 1.0, 0.0), synth.pose_xyyaw(0.8, 1.05, 0.03))


# ---- the checks
@pytest.fixture(scope="module")
def ref():
    """The reference's results, by name."""
    with np.load(GOLD, allow_pickle=False) as z:
        return dict(z)


def _same_tree(t, ref, key):
    assert (t.num_nodes, t.num_leaves) == tuple(ref[f"{key}.size"]), key
    for k, v in t.export().items():  # eigenvectors of 1-point nodes are NaN in both (0/0 covariance)
        assert same(v, ref[f"{key}.{k}"]), (key, k)
    assert same(t.cloud(), ref[f"{key}.cloud"]), key  # the build reorders and writes into the caller's vector


def _same_loop(r, ref, key):
    for k in LOOP_KEYS:
        assert same(r[k], ref[f"{key}.{k}"]), (key, k)


@pytest.mark.parametrize("b_max", B_MAX_WALLS)
def test_tree_build_is_the_references(oracle, ref, b_max):
    cloud = walls(2000)
    assert same(cloud, ref[f"walls_{b_max}.input"])
    _same_tree(oracle.OracleTree(cloud, b_max=b_max), ref, f"walls_{b_max}")


def test_tree_build_lidar_scan_and_async_levels(oracle, ref):
    """max_parallel_level > 0 takes the reference's std::async branch (mad_tree.cpp:106-128): same tree."""
    case = synth.registration_case(K=1, beams=32, azimuths=1024)
    pts = case["scans"][0]
    assert same(pts, ref["lidar.input"])
    o = oracle.OracleTree(pts)
    _same_tree(o, ref, "lidar_level0")
    _same_tree(o, ref, "lidar_level3")
    o.apply_transform(case["kf_poses"][0])
    _same_tree(o, ref, "lidar_moved")
    q = case["query"][:5000]
    assert same(o.search(q), ref["lidar_moved.search"])


def test_degenerate_clouds(oracle, ref):
    for i, pts in enumerate(degenerate_clouds()):
        _same_tree(oracle.OracleTree(pts, b_max=0.05), ref, f"degenerate{i}")


@pytest.mark.parametrize("K,threads", REG_CASES)
def test_registration_loop_is_the_references(oracle, ref, K, threads):
    case = synth.registration_case(K=K, beams=16, azimuths=512)
    assert same(case["query"], ref[f"loop_{K}_{threads}.input"])
    kfo = []
    for s in range(K):
        a = oracle.OracleTree(case["scans"][s])
        a.apply_transform(case["kf_poses"][s])
        kfo.append(a)
    mo = oracle.OracleTree(case["query"])
    ro = oracle.icp_run(kfo, mo, case["T_guess"], iters=10, num_threads=threads)
    _same_loop(ro, ref, f"loop_{K}_{threads}")
    # the correspondences themselves: the reference's bestMatchingLeafFast on its own X_ * mean_, every round
    for it in range(10):
        assert same(np.asarray(ro["idx_hist"][it]), ref[f"loop_{K}_{threads}.idx{it}"]), it


def test_four_walls_demo_is_the_references(oracle, ref):
    """apps/utils/tools/mad_registration.py through both: same 15 poses, same H/b, converge to identity."""
    cloud, T = demo_guess()
    assert same(cloud, ref["demo.input"]) and same(T, ref["demo.T"])
    ro = oracle.icp_run([oracle.OracleTree(cloud)], oracle.OracleTree(cloud), T, iters=15, record_matches=False)
    _same_loop(ro, ref, "demo")
    assert np.abs(ref["demo.X"] - np.eye(4)[:3]).max() < 1e-6


@pytest.mark.parametrize("deskew", [False, True])
def test_pipeline_is_the_references(oracle, ref, deskew):
    """Streaming odometry: pose, smoothed velocity and keyframe decisions of every scan, bit for bit.
    (The keyframe weight det(H^-1) is computed by two independently written LU routines; only the
    decisions it drives are compared.)"""
    L = oracle.lib()
    L.orc_pipeline_create.restype = C.c_void_p
    L.orc_pipeline_create.argtypes = [C.c_double, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                      C.c_int, C.c_int, C.c_int]
    L.orc_pipeline_compute.argtypes = [C.c_void_p, C.c_double, oracle._dp, C.c_int]
    L.orc_pipeline_state.argtypes = [C.c_void_p, oracle._dp]
    L.orc_pipeline_free.argtypes = [C.c_void_p]
    po = C.c_void_p(L.orc_pipeline_create(10.0, int(deskew), 0.2, 0.1, 0.8, 0.1, 0.02, 4, 4, 0))
    states = ref[f"pipeline_{deskew}.states"]
    st = np.zeros(23)
    promoted = 0
    for i, (stamp, pts) in enumerate(sequence(16)):
        assert same(pts, ref[f"sequence.input{i}"]), i
        L.orc_pipeline_compute(po, stamp, oracle._d(pts), pts.shape[0])
        L.orc_pipeline_state(po, oracle._d(st))
        sr = states[i]
        assert np.array_equal(st[:12], sr[:12]), i          # frame_to_map_
        assert np.array_equal(st[12:16], sr[12:16]), i      # map updated, ids, number of keyframes
        assert np.array_equal(st[17:], sr[17:]), i          # VelEstimator state
        promoted += int(st[12])
    assert i == states.shape[0] - 1 and promoted >= 4
    L.orc_pipeline_free(po)


def test_deskew_is_the_references(oracle, ref):
    L = oracle.lib()
    L.orc_pipeline_create.restype = C.c_void_p
    L.orc_pipeline_create.argtypes = [C.c_double, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                      C.c_int, C.c_int, C.c_int]
    L.orc_pipeline_deskew.argtypes = [C.c_void_p, oracle._dp, C.c_int, oracle._dp, oracle._dp]
    L.orc_pipeline_free.argtypes = [C.c_void_p]
    po = C.c_void_p(L.orc_pipeline_create(10.0, 1, 0.2, 0.1, 0.8, 0.1, 0.02, 4, 1, 0))
    _, pts = next(sequence(1))
    Ta, Tb = DESKEW_POSES
    mine = pts.copy()
    L.orc_pipeline_deskew(po, oracle._d(mine), mine.shape[0], oracle._d(np.ascontiguousarray(Ta[:3])),
                          oracle._d(np.ascontiguousarray(Tb[:3])))
    assert same(mine, ref["deskew.output"])
    assert np.abs(mine - pts).max() > 1e-3  # it did something
    L.orc_pipeline_free(po)


@pytest.mark.parametrize("b_max,b_min,rho_ker,b_ratio", SWEEP)
def test_parameter_sweep_is_the_references(oracle, ref, b_max, b_min, rho_ker, b_ratio):
    """Other leaf sizes, kernel widths and gate ratios than the defaults: trees and every GN round."""
    case = synth.registration_case(K=2, beams=16, azimuths=512, seed=9)
    key = f"sweep_{b_max}_{b_min}_{rho_ker}_{b_ratio}"
    kfo = []
    for s, (scan, P) in enumerate(zip(case["scans"], case["kf_poses"])):
        a = oracle.OracleTree(scan, b_max=b_max, b_min=b_min)
        _same_tree(a, ref, f"{key}.kf{s}")
        a.apply_transform(P)
        kfo.append(a)
    mo = oracle.OracleTree(case["query"], b_max=b_max, b_min=b_min)
    ro = oracle.icp_run(kfo, mo, case["T_guess"], iters=6, min_ball=b_max, rho_ker=rho_ker, b_ratio=b_ratio, num_threads=2,
                        record_matches=False)
    _same_loop(ro, ref, key)
