"""GPU parity tests (run on the B200 box with `-m gpu`): the CUDA path, called through the C ABI,
against the CPU oracle on the same seeded inputs and against the committed golden vectors.

Bars (BASELINE.json north_star): correspondence indices bit-exact (teacher-forced with the oracle's
pose of every iteration), H/b relative 1e-12, final SE(3) pose within 1e-5 rad / 1e-4 m."""
import os

import numpy as np
import pytest

from mad_icp_b200 import FlatTree, MadIcpError, Registrar, synth
from util import HB_REL, POSE_M, POSE_RAD, bits_equal, pose_error, same

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _rel(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-300))


def _check_Hb(H, b, H_ref, b_ref, tol=HB_REL):
    """H: norm-wise relative error.  b = sum sJ*e cancels towards zero at the optimum, so its error is
    measured against the magnitude of the terms being summed (|e| < 1 => bounded by max|H|), not |b|."""
    scale = max(np.abs(H_ref).max(), np.abs(b_ref).max())
    eh = float(np.abs(H - H_ref).max() / scale)
    eb = float(np.abs(b - b_ref).max() / scale)
    assert eh <= tol and eb <= tol, (eh, eb)


def _setup(case, oracle, max_keyframes=None):
    K = len(case["scans"])
    reg = Registrar(device=0, max_keyframes=max_keyframes or max(K, 1))
    otrees = []
    for k, (scan, P) in enumerate(zip(case["scans"], case["kf_poses"])):
        ft = FlatTree(scan)
        ft.apply_transform(P)
        reg.put_keyframe(k, ft)
        ot = oracle.OracleTree(scan)
        ot.apply_transform(P)
        otrees.append(ot)
    fq, oq = FlatTree(case["query"]), oracle.OracleTree(case["query"])
    reg.set_moving(fq.leaf_means())
    return reg, otrees, oq


def _four_walls_case(g):
    np.random.seed(42)
    cloud = synth.four_walls(points_per_wall=1000)
    return dict(scans=[cloud], kf_poses=[np.eye(4)], query=cloud.copy(), T_guess=g["T_guess"])


@pytest.fixture(scope="module")
def lidar_small(oracle):
    g = np.load(os.path.join(GOLD, "lidar_small_registration.npz"))
    c = synth.registration_case(K=2, beams=16, azimuths=512, seed=3)
    return g, c, _setup(c, oracle)


@pytest.fixture(scope="module")
def walls(oracle):
    g = np.load(os.path.join(GOLD, "four_walls_registration.npz"))
    c = _four_walls_case(g)
    return g, c, _setup(c, oracle)


# ------------------------------------------------------------------ golden vectors (committed)
@pytest.mark.parametrize("which", ["walls", "lidar_small"])
def test_golden_indices_bit_exact_teacher_forced(which, request):
    g, c, (reg, _, _) = request.getfixturevalue(which)
    for it in range(g["X_hist"].shape[0]):
        idx = reg.search(g["X_hist"][it])
        assert idx.shape == g["idx_hist"][it].shape
        assert (idx == g["idx_hist"][it]).all(), f"iteration {it}: {(idx != g['idx_hist'][it]).sum()} indices differ"


@pytest.mark.parametrize("which", ["walls", "lidar_small"])
def test_golden_H_b_teacher_forced(which, request):
    g, c, (reg, _, _) = request.getfixturevalue(which)
    for it in range(g["X_hist"].shape[0]):
        H, b, _ = reg.linearize(g["X_hist"][it])
        _check_Hb(H, b, g["H_hist"][it], g["b_hist"][it])


@pytest.mark.parametrize("which,iters", [("walls", 15), ("lidar_small", 10)])
def test_golden_register_pose(which, iters, request):
    g, c, (reg, _, _) = request.getfixturevalue(which)
    out = reg.register(c["T_guess"], iters=iters)
    ang, dt = pose_error(out["X"], g["X"])
    assert ang < POSE_RAD and dt < POSE_M, (ang, dt)
    assert (out["matched"] == g["matched"]).all()
    assert out["n_matched"] == int(g["matched"].sum())
    # per-round trajectory follows the oracle's
    tr = reg.register_trace()
    assert tr.shape[0] == iters + 1 and bits_equal(tr[0], c["T_guess"][:3])
    for it in range(iters):
        ang, dt = pose_error(tr[it], g["X_hist"][it])
        assert ang < POSE_RAD and dt < POSE_M, (it, ang, dt)
    # H of the last round is what Pipeline reads (pipeline.cpp:223)
    assert _rel(out["H"], g["H_hist"][-1]) < 1e-6


def test_register_matches_step_api_and_is_deterministic(lidar_small):
    g, c, (reg, _, _) = lidar_small
    a = reg.register(c["T_guess"], iters=10)
    b = reg.register(c["T_guess"], iters=10)
    assert bits_equal(a["X"], b["X"]) and bits_equal(a["H"], b["H"]) and (a["matched"] == b["matched"]).all()
    # same loop driven from the host through the step API (K1+K2 kernels, K3 solve kernel)
    X = c["T_guess"][:3].copy()
    for _ in range(10):
        H, bb, m = reg.linearize(X)
        X = reg.solve_update(H, bb, X)
    ang, dt = pose_error(a["X"], X)
    assert ang < 1e-9 and dt < 1e-9
    assert (m == a["matched"]).all()


def test_linearize_matched_flags_and_oracle_linearize(lidar_small, oracle):
    g, c, (reg, otrees, oq) = lidar_small
    for X in (c["T_guess"], g["X"]):
        H, b, m = reg.linearize(X)
        Ho, bo, mo = oracle.icp_linearize(otrees, oq, X)
        assert (m == mo).all()
        _check_Hb(H, b, Ho, bo)


def test_solve_update_kernel(lidar_small, oracle):
    g, c, (reg, _, _) = lidar_small
    rs = np.random.RandomState(5)
    for it in range(g["H_hist"].shape[0]):
        Xn = reg.solve_update(g["H_hist"][it], g["b_hist"][it], g["X_hist"][it])
        _, Xo = oracle.solve_update(g["H_hist"][it], g["b_hist"][it], g["X_hist"][it])
        ang, dt = pose_error(Xn, Xo)
        assert ang < 1e-12 and dt < 1e-12
    # rank-deficient and zero systems stay finite (pseudo-inverse of D)
    X0 = np.eye(4)[:3]
    assert bits_equal(reg.solve_update(np.zeros((6, 6)), np.zeros(6), X0), X0)
    H = np.diag([1.0, 2.0, 0.0, 0.0, 3.0, 0.0])
    Xn = reg.solve_update(H, np.ones(6), X0)
    assert np.isfinite(Xn).all() and np.allclose(Xn[:, 3], [-1, -0.5, 0])


# ------------------------------------------------------------------ NN tool (pymadtree surface)
def test_kat_self_query_zero_error_on_gpu(oracle):
    """nn_search.py known answer: b_max=1e-5, querying the cloud against itself gives error == 0."""
    np.random.seed(42)
    cloud = synth.four_walls()  # 50 000 points
    ft = FlatTree(cloud, b_max=1e-5)
    reg = Registrar(device=0, max_keyframes=1)
    reg.put_keyframe(0, ft)
    out = reg.search_cloud(0, cloud)
    assert np.linalg.norm(out["points"] - cloud, axis=1).sum() == 0.0
    assert (out["dists"] == 0).all()
    ot = oracle.OracleTree(cloud, b_max=1e-5)
    assert (out["ordinals"] == ot.search(cloud)).all()
    means, normals, _, _ = ot.leaves()
    assert bits_equal(out["normals"], normals[out["ordinals"]])
    # off-tree queries: distances bit-equal to the host formula
    rs = np.random.RandomState(0)
    q = cloud[:5000] + rs.normal(0, 0.05, (5000, 3))
    out = reg.search_cloud(0, q)
    oi = ot.search(q)
    assert (out["ordinals"] == oi).all() and bits_equal(out["points"], means[oi])


# ------------------------------------------------------------------ full BASELINE sizes
@pytest.fixture(scope="module")
def full16(oracle):
    c = synth.registration_case(K=16)  # 16 keyframes x 131 072 points, 64 x 2048 query
    return c, _setup(c, oracle)


def test_full_size_cfg3_indices_and_pose(full16, oracle):
    c, (reg, otrees, oq) = full16
    ref = oracle.icp_run(otrees, oq, c["T_guess"], iters=10, num_threads=min(16, oracle.max_threads()))
    for it in (0, 1, 4, 9):
        idx = reg.search(ref["X_hist"][it])
        assert (idx == ref["idx_hist"][it]).all(), f"iteration {it}"
        H, b, _ = reg.linearize(ref["X_hist"][it])
        _check_Hb(H, b, ref["H_hist"][it], ref["b_hist"][it], tol=10 * HB_REL)  # 3e5 terms summed sequentially on the CPU
    out = reg.register(c["T_guess"], iters=10)
    ang, dt = pose_error(out["X"], ref["X"])
    assert ang < POSE_RAD and dt < POSE_M, (ang, dt)
    assert (out["matched"] == ref["matched"]).mean() > 0.9999
    # free-running index agreement (informational bar: the poses differ in the last bits)
    tr = reg.register_trace()
    agree = (reg.search(tr[9]) == ref["idx_hist"][9]).mean()
    assert agree > 0.999, agree
    # converges to the simulated truth within sensor noise
    ang, dt = pose_error(out["X"], c["T_true"])
    assert ang < 2e-3 and dt < 3e-2


def test_full_size_cfg3_against_the_compiled_reference(full16):
    """The same check against what the reference's OWN sources computed on the CPU (mad_tree.cpp and mad_icp.cpp
    compiled against oracle/eigen_standin, stored in golden/reference_full16.npz by golden/make_reference_golden.py;
    tests/test_reference_pin.py): GPU correspondences == the reference's own at every round / keyframe / leaf, H/b at
    its poses, final pose."""
    c, (reg, _, _) = full16
    with np.load(os.path.join(GOLD, "reference_full16.npz"), allow_pickle=False) as z:
        ref = dict(z)
    assert same(c["query"], ref["query.input"]) and all(same(s, ref[f"scan{k}.input"]) for k, s in enumerate(c["scans"]))
    # the reference's OWN correspondences (its bestMatchingLeafFast on its own X_ * mean_, mad_icp.cpp:78-79),
    # every round, every keyframe, every moving leaf: bit-exact, no sampling
    for it in range(10):
        idx = reg.search(ref["loop.X_hist"][it])
        assert idx.shape == (16, int(ref["num_leaves"]))
        assert same(idx, ref[f"loop.idx{it}"]), f"round {it}: correspondences differ from the reference's"
        H, b, _ = reg.linearize(ref["loop.X_hist"][it])
        _check_Hb(H, b, ref["loop.H_hist"][it], ref["loop.b_hist"][it], tol=10 * HB_REL)
    out = reg.register(c["T_guess"], iters=10)
    ang, dt = pose_error(out["X"], ref["loop.X"])
    assert ang < POSE_RAD and dt < POSE_M, (ang, dt)
    assert (out["matched"] == ref["loop.matched"]).mean() > 0.9999


def _moving_means(rtree):
    e = rtree.export()
    leaf = e["leaf_ordinal"] >= 0
    order = np.argsort(e["leaf_ordinal"][leaf])
    return e["mean"][leaf][order]


def test_full_size_cfg2_single_keyframe(full16, oracle):
    c, (reg16, otrees, oq) = full16
    reg = Registrar(device=0, max_keyframes=1)
    ft = FlatTree(c["scans"][15])
    ft.apply_transform(c["kf_poses"][15])
    reg.put_keyframe(0, ft)
    reg.set_moving(FlatTree(c["query"]).leaf_means())
    ref = oracle.icp_run([otrees[15]], oq, c["T_guess"], iters=10)
    assert (reg.search(ref["X_hist"][3])[0] == ref["idx_hist"][3][0]).all()
    out = reg.register(c["T_guess"], iters=10)
    ang, dt = pose_error(out["X"], ref["X"])
    assert ang < POSE_RAD and dt < POSE_M


def test_full_size_properties(full16):
    """Size-independent properties at BASELINE size: a permutation of the moving leaves permutes the
    correspondences; results do not depend on which slot a keyframe sits in; ordinals in range."""
    c, (reg, _, _) = full16
    means = FlatTree(c["query"]).leaf_means()
    X = c["T_guess"]
    base = reg.search(X)
    for k, s in enumerate(reg.active_slots()):
        assert base[k].min() >= 0 and base[k].max() < reg_leaves(reg, s)
    perm = np.random.RandomState(0).permutation(means.shape[0])
    reg.set_moving(means[perm])
    assert (reg.search(X) == base[:, perm]).all()
    Hp, bp, _ = reg.linearize(X)
    reg.set_moving(means)
    H, b, _ = reg.linearize(X)
    _check_Hb(Hp, bp, H, b, tol=1e-11)  # same terms, different summation order


def reg_leaves(reg, slot):
    from mad_icp_b200 import _capi
    return _capi.lib().madicp_keyframe_leaves(reg._h, slot)


# ------------------------------------------------------------------ edge cases
def test_single_moving_leaf_and_single_leaf_keyframe(oracle):
    reg = Registrar(device=0, max_keyframes=2)
    tiny = np.array([[1.0, 0.0, 0.0], [1.01, 0.0, 0.0], [1.0, 0.01, 0.0]])
    ft = FlatTree(tiny)
    assert ft.num_leaves == 1 and ft.num_nodes == 1
    reg.put_keyframe(1, ft)
    reg.set_moving(np.array([[1.0, 0.0, 0.05]]))
    assert reg.search(np.eye(4)).tolist() == [[0]]
    H, b, m = reg.linearize(np.eye(4))
    ot, oq = oracle.OracleTree(tiny), oracle.OracleTree(np.array([[1.0, 0.0, 0.05]]))
    Ho, bo, mo = oracle.icp_linearize([ot], oq, np.eye(4))
    assert (m == mo).all() and np.allclose(H, Ho, rtol=1e-13, atol=0) and np.allclose(b, bo, rtol=1e-13, atol=0)
    out = reg.register(np.eye(4), iters=3)
    assert np.isfinite(out["X"]).all()


def test_everything_gated_out_leaves_pose_unchanged(lidar_small):
    g, c, (reg, _, _) = lidar_small
    far = c["T_guess"] @ synth.pose_xyyaw(500.0, 300.0, 1.0)
    out = reg.register(far, iters=4)
    assert out["n_matched"] == 0 and not out["matched"].any()
    assert (out["H"] == 0).all() and (out["b"] == 0).all()
    assert bits_equal(out["X"], far[:3])  # H = 0 -> dx = 0 (pseudo-inverse), expmap(0) = I


def test_slot_reuse_drop_and_errors(lidar_small, oracle):
    g, c, _ = lidar_small
    reg = Registrar(device=0, max_keyframes=3)
    with pytest.raises(MadIcpError):
        reg.register(np.eye(4), iters=2)  # no moving leaves yet
    fts = []
    for scan, P in zip(c["scans"], c["kf_poses"]):
        ft = FlatTree(scan)
        ft.apply_transform(P)
        fts.append(ft)
    reg.set_moving(FlatTree(c["query"]).leaf_means())
    with pytest.raises(MadIcpError):
        reg.register(np.eye(4), iters=2)  # no keyframe yet
    reg.put_keyframe(2, fts[0])
    reg.put_keyframe(0, fts[1])
    assert reg.active_slots() == [0, 2]
    idx = reg.search(g["X_hist"][0])
    assert (idx[0] == g["idx_hist"][0][1]).all() and (idx[1] == g["idx_hist"][0][0]).all()
    reg.drop_keyframe(0)
    assert reg.num_keyframes == 1 and (reg.search(g["X_hist"][0])[0] == g["idx_hist"][0][0]).all()
    reg.put_keyframe(0, fts[0])  # overwrite with a different (larger/smaller) tree
    assert (reg.search(g["X_hist"][0])[0] == g["idx_hist"][0][0]).all()
    with pytest.raises(MadIcpError):
        reg.register(np.eye(4), iters=-1)
    with pytest.raises(MadIcpError):
        reg.register_async(np.eye(4), iters=65)  # one launch holds 64 rounds (register() chains launches beyond that)
    with pytest.raises(MadIcpError):
        reg.put_keyframe(3, fts[0])


def test_iters_one_clears_and_sets_matched(lidar_small, oracle):
    g, c, (reg, otrees, oq) = lidar_small
    out = reg.register(c["T_guess"], iters=1)
    ref = oracle.icp_run(otrees, oq, c["T_guess"], iters=1, num_threads=1)
    assert (out["matched"] == ref["matched"]).all()
    ang, dt = pose_error(out["X"], ref["X"])
    assert ang < 1e-9 and dt < 1e-9


def test_pool_growth_and_few_moving_leaves(oracle):
    """A keyframe larger than the initial pool slot (65 576 nodes) arrives after a small one: the pool is
    re-homed and both stay correct.  Also fewer moving leaves than CTAs (most CTAs own no work)."""
    rs = np.random.RandomState(3)
    small = synth.registration_case(K=1, beams=8, azimuths=256, seed=21)
    big_cloud = np.concatenate([synth.four_walls(points_per_wall=60000, rng=rs) * [10, 10, 3],
                                rs.uniform(-1, 41, (60000, 3)) * [1, 1, 0.1]])
    reg = Registrar(device=0, max_keyframes=3)
    f_small = FlatTree(small["scans"][0])
    f_small.apply_transform(small["kf_poses"][0])
    reg.put_keyframe(0, f_small)
    f_big = FlatTree(big_cloud, b_max=0.05)
    assert f_big.num_nodes > 70000
    reg.put_keyframe(2, f_big)                     # forces the pool (and the shadow arrays) to grow
    o_small = oracle.OracleTree(small["scans"][0])
    o_small.apply_transform(small["kf_poses"][0])
    o_big = oracle.OracleTree(big_cloud, b_max=0.05)
    q = FlatTree(small["query"])
    oq = oracle.OracleTree(small["query"])
    reg.set_moving(q.leaf_means())
    X = small["T_guess"]
    idx = reg.search(X)
    assert (idx[0] == o_small.search((X[:3, :3] @ q.leaf_means().T).T + X[:3, 3])).all()
    assert (idx[1] == o_big.search((X[:3, :3] @ q.leaf_means().T).T + X[:3, 3])).all()
    ref = oracle.icp_run([o_small, o_big], oq, X, iters=5, min_ball=0.2)
    out = reg.register(X, iters=5)
    ang, dt = pose_error(out["X"], ref["X"])
    assert ang < POSE_RAD and dt < POSE_M and (out["matched"] == ref["matched"]).all()
    # three moving leaves only
    few = q.leaf_means()[:3].copy()
    reg.set_moving(few)
    out = reg.register(X, iters=3)
    H, b, m = reg.linearize(X)
    assert np.isfinite(out["X"]).all() and out["matched"].shape == (3,) and m.shape == (3,)
    assert (reg.search(X)[:, :3] == idx[:, :3]).all()


def test_very_deep_tree():
    """A hand-made caterpillar tree 40 levels deep (every internal node: a leaf on the left, the rest on the
    right; split planes x = d + 0.5).  Far deeper than the implicit-heap experiments support; the default
    4-ary walk has no depth limit.  The answer is analytic: the leaf reached is min(floor(x + 0.5), D)."""
    from mad_icp_b200 import _capi
    D = 40
    recs = np.zeros(2 * D + 1, dtype=_capi.REC_DTYPE)
    for d in range(D):            # internal node of depth d at index 2d, children at 2d+1 (leaf), 2d+2
        recs[2 * d]["mean"] = [d + 0.5, 0, 0]
        recs[2 * d]["dir"] = [1, 0, 0]
        recs[2 * d]["link"] = 2 * d + 1
        recs[2 * d + 1]["mean"] = [d, 0, 0]
        recs[2 * d + 1]["dir"] = [0, 0, 1]
        recs[2 * d + 1]["link"] = -1 - d
    recs[2 * D]["mean"] = [D, 0, 0]
    recs[2 * D]["dir"] = [0, 0, 1]
    recs[2 * D]["link"] = -1 - D
    reg = Registrar(device=0, max_keyframes=1)
    reg.put_keyframe_records(0, recs, D + 1)
    x = np.random.RandomState(0).uniform(-2, D + 3, 5000)
    q = np.stack([x, np.zeros_like(x), np.zeros_like(x)], axis=1)
    out = reg.search_cloud(0, q)
    want = np.clip(np.floor(x + 0.5), 0, D).astype(np.int32)
    assert (out["ordinals"] == want).all()
    assert (out["points"][:, 0] == want).all()
    exact = np.arange(D + 1) + 0.5          # queries exactly ON the planes: s == 0 is "not < 0" -> right
    out = reg.search_cloud(0, np.stack([exact[:-1], np.zeros(D), np.zeros(D)], axis=1))
    assert (out["ordinals"] == np.arange(1, D + 1)).all()
