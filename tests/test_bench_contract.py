"""bench.py's contract: the reference arm prints one JSON line with the keys a reader of the line expects, without a
GPU the product arm fails loudly instead of falling back, and (`-m gpu`) --dump-outputs writes what the timed
registration returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=600):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=timeout, cwd=ROOT)


def test_reference_arm_line(built):
    p = _run("--impl", "reference", "--steps", "2", "--warmup", "1", "--beams", "8", "--azimuths", "256")
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "scans/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["n_gpus"] == 1 and line["gpu_launches"] == 0
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == line["value"]
    e = line["e2e"]
    assert e["value"] == line["value"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert "workload" in line["config"] and "model" not in line["config"]


def test_reference_arm_other_ranks_exit_quietly(built):
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--beams", "8", "--azimuths", "256"], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_product_arm_needs_a_gpu(built):
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("GPU present")
    p = _run("--steps", "1", "--warmup", "1", "--beams", "8", "--azimuths", "256", "--no-cpu-baseline")
    assert p.returncode != 0
    assert "CUDA" in (p.stderr + p.stdout)


def test_dump_outputs_is_for_the_product_arm(tmp_path):
    p = _run("--impl", "reference", "--steps", "1", "--dump-outputs", str(tmp_path / "out"))
    assert p.returncode == 2 and "--dump-outputs" in p.stderr
    assert not (tmp_path / "out").exists()


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_registration(built, tmp_path):
    """The last timed step's pose, H, b, matched flags and their count, as float64 / float32 .npy files; --steps sets
    the number of timed steps; a second run with the same arguments computes the same arrays bit for bit."""
    args = ("--steps", "3", "--warmup", "1", "--beams", "8", "--azimuths", "256", "--no-cpu-baseline", "--stream-scans", "0")
    dumps = []
    for run in ("a", "b"):
        p = _run(*args, "--dump-outputs", str(tmp_path / run))
        assert p.returncode == 0, p.stderr[-2000:]
        line = json.loads(p.stdout.strip().splitlines()[-1])
        assert line["steps"] == 3
        d = {n: np.load(tmp_path / run / f"{n}.npy") for n in ("X", "H", "b", "matched", "n_matched")}
        assert sorted(os.listdir(tmp_path / run)) == sorted(f"{n}.npy" for n in d)
        assert d["X"].shape == (3, 4) and d["H"].shape == (6, 6) and d["b"].shape == (6,)
        assert d["X"].dtype == d["H"].dtype == d["b"].dtype == np.float64 and d["matched"].dtype == np.float32
        assert d["matched"].shape == (line["config"]["moving_leaves"],) and set(np.unique(d["matched"])) <= {0.0, 1.0}
        assert d["n_matched"][0] == d["matched"].sum() == line["result"]["n_matched"]
        assert d["X"][:, 3].tolist() == line["result"]["pose_t"]
        dumps.append(d)
    for n in dumps[0]:
        assert np.array_equal(dumps[0][n], dumps[1][n]), n


def test_ranks_next_to_one_socket_get_whole_physical_cores():
    """bench.pin_to_gpu: four ranks next to a 32-core / 64-thread socket numbered [0..31 | 64..95] must not sit on each
    other's hyperthreads (the sorted CPU list cut into four runs did exactly that)."""
    sys.path.insert(0, ROOT)
    import bench
    cores = list(range(0, 32)) + list(range(64, 96))
    sets = [[c, c + 64] for c in range(32)]
    shares = [bench.share_of_cores(cores, k, 4, sibling_sets=sets) for k in range(4)]
    assert shares[0] == list(range(0, 8)) + list(range(64, 72))
    assert sorted(c for sh in shares for c in sh) == sorted(cores)
    phys = [{c % 64 for c in sh} for sh in shares]
    for a in range(4):
        assert len(shares[a]) == 16
        for b in range(a + 1, 4):
            assert not (phys[a] & phys[b])
    # no SMT / topology unreadable: every CPU is its own core; more ranks than cores: everybody keeps the whole set
    assert bench.share_of_cores([0, 1, 2, 3], 1, 2, sibling_sets=[[0], [1], [2], [3]]) == [2, 3]
    assert bench.share_of_cores([0, 1], 2, 4, sibling_sets=[[0], [1]]) == [0, 1]
    assert bench._sibling_sets(sorted(os.sched_getaffinity(0)))  # reads /sys without raising


def test_latency_model_is_a_pure_function_of_the_walk_counts():
    """bench.latency_model on the numbers of profiles/r03f_bench.json: the memory-only floor is the figure the earlier
    bench lines carried (0.0312 ms, frac 0.183); the full floor adds the dependent FP64 chain of every pass."""
    sys.path.insert(0, ROOT)
    import bench
    walked = [307232, 281829, 107440, 14523, 1799, 206, 9, 0, 0, 0]
    m = bench.latency_model(walked, 46436884, 10, 16, 19202, 0.1703627222031355e-3)
    assert m["passes_per_round"] == 3 and abs(m["mean_nodes_per_walk"] - 15.1146) < 1e-3
    assert abs(m["floor_memory_only_ms"] - 0.031205134883585593) < 1e-9
    assert abs(m["frac_memory_only"] - 0.18316879702343278) < 1e-9
    extra_cycles = 10 * 3 * (34 * 19.0 + 8 * 30.0)
    assert abs(m["floor_ms"] - (m["floor_memory_only_ms"] + extra_cycles / 1.92e9 * 1e3)) < 1e-12
    assert m["floor_memory_only_ms"] < m["floor_ms"] < m["measured_ms"] and 0 < m["frac"] < 1
    json.dumps(m)  # goes into the bench line as it is
