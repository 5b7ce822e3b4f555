"""Writes tests/golden/reference_pin.npz and tests/golden/reference_full16.npz: what the reference's OWN sources
compute (oracle/_ref/libmadicp_ref.so, built by `make -C oracle ref` from a checkout of the reference, see
oracle/Makefile) on the inputs of tests/test_reference_pin.py and of test_full_size_cfg3_against_the_compiled_reference
in tests/test_gpu_parity.py.  Only needed again when those inputs change; the tests read the files and need no
reference checkout.  Arrays larger than tests/util.GOLDEN_INLINE_BYTES are stored as digests of their values.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]
from mad_icp_b200 import synth  # noqa: E402
from oracle import reference as R  # noqa: E402
import test_reference_pin as T  # noqa: E402
from util import fingerprint  # noqa: E402

LOOP_KEYS = T.LOOP_KEYS


def tree(out, key, t):
    out[f"{key}.size"] = np.array([t.num_nodes, t.num_leaves])
    for k, v in t.export().items():
        out[f"{key}.{k}"] = fingerprint(v)
    out[f"{key}.cloud"] = fingerprint(t.cloud())


def loop(out, key, r):
    for k in LOOP_KEYS:
        out[f"{key}.{k}"] = fingerprint(r[k])
    if "idx_hist" in r:
        for it in range(r["idx_hist"].shape[0]):
            out[f"{key}.idx{it}"] = fingerprint(r["idx_hist"][it])


def reference_pin():
    out = {}
    cloud = T.walls(2000)
    for b_max in T.B_MAX_WALLS:
        out[f"walls_{b_max}.input"] = fingerprint(cloud)
        tree(out, f"walls_{b_max}", R.ReferenceTree(cloud, b_max=b_max))

    case = synth.registration_case(K=1, beams=32, azimuths=1024)
    pts = case["scans"][0]
    out["lidar.input"] = fingerprint(pts)
    tree(out, "lidar_level0", R.ReferenceTree(pts, max_parallel_level=0))
    tree(out, "lidar_level3", R.ReferenceTree(pts, max_parallel_level=3))
    r = R.ReferenceTree(pts)
    r.apply_transform(case["kf_poses"][0])
    tree(out, "lidar_moved", r)
    out["lidar_moved.search"] = fingerprint(r.search(case["query"][:5000]))

    for i, pts in enumerate(T.degenerate_clouds()):
        tree(out, f"degenerate{i}", R.ReferenceTree(pts, b_max=0.05))

    for K, threads in T.REG_CASES:
        case = synth.registration_case(K=K, beams=16, azimuths=512)
        out[f"loop_{K}_{threads}.input"] = fingerprint(case["query"])
        kfr = []
        for s in range(K):
            b = R.ReferenceTree(case["scans"][s])
            b.apply_transform(case["kf_poses"][s])
            kfr.append(b)
        mr = R.ReferenceTree(case["query"])
        loop(out, f"loop_{K}_{threads}", R.icp_run(kfr, mr, case["T_guess"], iters=10, num_threads=threads, record_idx=True))

    cloud, Tg = T.demo_guess()
    out["demo.input"], out["demo.T"] = fingerprint(cloud), fingerprint(Tg)
    loop(out, "demo", R.icp_run([R.ReferenceTree(cloud)], R.ReferenceTree(cloud), Tg, iters=15))

    for deskew in (False, True):
        pr = R.ReferencePipeline(deskew=deskew, num_keyframes=4, num_threads=4)
        states = []
        for i, (stamp, pts) in enumerate(T.sequence(16)):
            out[f"sequence.input{i}"] = fingerprint(pts)
            pr.compute(stamp, pts)
            states.append(pr.state())
        out[f"pipeline_{deskew}.states"] = np.array(states)

    pr = R.ReferencePipeline(deskew=True, num_threads=1)
    _, pts = next(T.sequence(1))
    out["deskew.output"] = fingerprint(pr.deskew(pts, *T.DESKEW_POSES))

    case = synth.registration_case(K=2, beams=16, azimuths=512, seed=9)
    for b_max, b_min, rho_ker, b_ratio in T.SWEEP:
        key = f"sweep_{b_max}_{b_min}_{rho_ker}_{b_ratio}"
        kfr = []
        for s, (scan, P) in enumerate(zip(case["scans"], case["kf_poses"])):
            b = R.ReferenceTree(scan, b_max=b_max, b_min=b_min)
            tree(out, f"{key}.kf{s}", b)
            b.apply_transform(P)
            kfr.append(b)
        mr = R.ReferenceTree(case["query"], b_max=b_max, b_min=b_min)
        loop(out, key, R.icp_run(kfr, mr, case["T_guess"], iters=6, min_ball=b_max, rho_ker=rho_ker, b_ratio=b_ratio,
                                 num_threads=2))
    return out


def reference_full16():
    """BASELINE size: 16 keyframes x 131 072 points, 64 x 2048 query, 10 GN rounds."""
    c = synth.registration_case(K=16)
    out = {"query.input": fingerprint(c["query"])}
    rtrees = []
    for s, (scan, P) in enumerate(zip(c["scans"], c["kf_poses"])):
        out[f"scan{s}.input"] = fingerprint(scan)
        t = R.ReferenceTree(scan, max_parallel_level=2)
        t.apply_transform(P)
        rtrees.append(t)
    rq = R.ReferenceTree(c["query"])
    out["num_leaves"] = np.array(rq.num_leaves)
    r = R.icp_run(rtrees, rq, c["T_guess"], iters=10, num_threads=min(16, R.max_threads()), record_idx=True)
    loop(out, "loop", r)
    out["loop.matched"] = r["matched"]  # whole: the GPU test bounds the share of flags that differ
    return out


def main():
    R.lib()
    for name, make in (("reference_pin", reference_pin), ("reference_full16", reference_full16)):
        out = make()
        path = os.path.join(HERE, f"{name}.npz")
        np.savez_compressed(path, **out)
        print(f"{path}: {len(out)} arrays, {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main()
