#!/usr/bin/env python
"""bench.py -- scans/sec of the MAD-ICP registration hot path on B200.

Workload (BASELINE.json configs[2] at N=1, configs[3] at N>1): one synthetic 64-beam x 2048-azimuth
scan (131 072 points -> ~19k moving leaves) registered against a 16-keyframe model with `--iters`
Gauss-Newton rounds (default 10, as BASELINE's configs[1]).  A *step* is one whole registration.

  value  : scans/s with the model and the moving leaves resident in HBM (CUDA events on the launch
           stream around the persistent GN kernel; L2 flushed between steps, outside the events).
  e2e    : the same through the public call with HOST buffers: pinned H2D of the moving leaves and the
           initial pose, the kernel, D2H of pose + H/b + matched flags, host synchronisation.
  N > 1  : `value` is the throughput deployment: every GPU holds the full 16-keyframe model and
           registers its own scan (independent units, no data-path collective, "scaling": "weak").
           `sharded` reports north_star's single-scan mode beside it: keyframe slot s on rank s % N
           (2 per GPU at N=8), the 48-value H/b tile all-reduced inside the persistent kernel every GN
           round through NVLink peer mailboxes (strong scaling of ONE scan's latency, which is bounded
           by the per-round barrier + solve, not by the tree walks; DESIGN.md section 7).
  --impl reference : the reference's CPU implementation of the path on the host cores: its own sources
           compiled against oracle/eigen_standin (oracle/_ref, shipped prebuilt) and the Eigen-free restatement
           (oracle/) are both timed and the faster one is the line's value (the stand-in is slower than Eigen).
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "scans/sec (130k-pt scan vs 16-keyframe model)"
K_MODEL = 16


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--stream-scans", type=int, default=-1,
                    help="cfg5 streaming block: scans of the synthetic sequence (default 1000 at N=1, 250 per rank at N>1; 0: off)")
    ap.add_argument("--stream-cpu-scans", type=int, default=200,
                    help="how many of them the CPU pipeline also runs (trajectory error and keyframe decisions)")
    ap.add_argument("--beams", type=int, default=64)
    ap.add_argument("--azimuths", type=int, default=2048)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed registration returned in its last step to DIR/<name>.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 arm")
    return a


def dump_outputs(path, res):
    """The arrays a caller of the timed registration receives (pose, last round's H and b, matched flags and their
    count), one float64 / float32 .npy each.  The inputs are seeded, so the same arguments give the same inputs and two
    builds can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    for name in ("X", "H", "b"):
        np.save(os.path.join(path, f"{name}.npy"), np.asarray(res[name], dtype=np.float64))
    np.save(os.path.join(path, "matched.npy"), np.asarray(res["matched"], dtype=np.float32))
    np.save(os.path.join(path, "n_matched.npy"), np.array([res["n_matched"]], dtype=np.float64))


def workload_name(a, n):
    shard = ("all keyframes on one GPU" if n == 1 else
             f"{n} replicas: every GPU holds the 16-keyframe model and registers its own scan (the keyframe-sharded "
             f"single-scan mode is reported under 'sharded')")
    return (f"{a.beams}x{a.azimuths}-ray synthetic scan ({a.beams * a.azimuths} pts) vs {K_MODEL}-keyframe model, "
            f"{a.iters} GN iters, {shard}")


# --------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """Polls NVML (SM clock + clock-event reasons) while the timed region runs.  (The polling period is not what costs
    the host-timed `e2e` its efficiency at N > 1: 2, 10 and 50 ms measured the same within the run-to-run spread at N=2,
    profiles/r03_sampler_period_2gpu.txt.)"""
    PERIOD_S = float(os.environ.get("MADICP_BENCH_SAMPLER_MS", "2")) * 1e-3
    BITS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
            0x80: "hw_power_brake_slowdown"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz, self.ok = None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def run(self):
        if not self.ok:
            return
        while not self.stop_flag:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                try:
                    r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.BITS.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(self.PERIOD_S)

    def summary(self):
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "note": "nvml unavailable"}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def _sibling_sets(cores):
    """Hardware threads of `cores` grouped by physical core (sorted by their lowest CPU number)."""
    seen, sets = set(), []
    for c in sorted(cores):
        if c in seen:
            continue
        sib = {c}
        try:
            with open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list") as f:
                for part in f.read().strip().split(","):
                    lo, _, hi = part.partition("-")
                    sib.update(range(int(lo), int(hi or lo) + 1))
        except (OSError, ValueError):
            pass
        sib &= set(cores)
        sib.add(c)
        seen |= sib
        sets.append(sorted(sib))
    return sets


def share_of_cores(cores, k, m, sibling_sets=None):
    """The k-th of m shares of `cores`, in WHOLE physical cores: ranks next to one socket should not end up on each
    other's hyperthreads.  (The sorted CPU list cut into m runs does that on a host numbered [0..31 | 64..95] per socket:
    rank 0 gets the CPUs 0-15 and rank 2 their siblings 64-79.  At N=2 the two cuts measure the same,
    profiles/r03_pinning_2gpu.txt; whether it is what the host-timed `e2e` loses at N=8 -- 0.76 of N x the single-GPU
    rate against 0.99 for the device-timed `value` -- could not be measured in round 2.)"""
    if os.environ.get("MADICP_BENCH_PIN_LEGACY"):  # the old cut, for A/B runs (profiles/r03_pinning_2gpu.txt)
        share = max(4, len(cores) // m)
        return sorted(cores)[k * share:(k + 1) * share] or sorted(cores)
    sets = sibling_sets if sibling_sets is not None else _sibling_sets(cores)
    per = max(1, len(sets) // m)
    mine = sets[k * per:(k + 1) * per] or sets
    return sorted(c for s0 in mine for c in s0)


def pin_to_gpu(dev, local_rank, world):
    """Keeps this process (and the pinned buffers it is about to allocate) on the CPU cores next to its GPU: with one
    process per GPU the host side of a step is a handful of latency-bound driver calls, and a remote NUMA node or a core
    shared with another rank's threads costs more than the kernel.  Returns a description for the JSON line."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(dev)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cores = [i for i in range(ncpu) if (words[i // 64] >> (i % 64)) & 1]
        if not cores:
            return None
        note = ""
        if world > 1:  # ranks whose GPUs share a node split its physical cores between them
            peers = []
            for d in range(world):
                w2 = pynvml.nvmlDeviceGetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(d), (ncpu + 63) // 64)
                if list(w2) == list(words):
                    peers.append(d)
            cores = share_of_cores(cores, peers.index(dev), len(peers))
            note = ", whole physical cores"
        os.sched_setaffinity(0, cores)
        return f"{len(cores)} hardware threads next to GPU {dev} ({cores[0]}-{cores[-1]}{note})"
    except Exception as e:  # noqa: BLE001  (no NVML / no permission: run unpinned)
        return f"unpinned ({type(e).__name__})"


def leaf_depths(recs):
    """Depth (internal nodes above) of every leaf ordinal, from the breadth-first records."""
    n = recs.shape[0]
    depth = np.zeros(n, np.int32)
    link = recs["link"]
    internal = np.nonzero(link >= 0)[0]
    for i in internal:  # BFS order => parents before children
        depth[link[i]] = depth[i] + 1
        depth[link[i] + 1] = depth[i] + 1
    leaf = link < 0
    out = np.zeros(int(leaf.sum()), np.int32)
    out[-1 - link[leaf]] = depth[leaf]
    return out


def algorithmic_bytes(reg, depth_tables, trace, iters, L):
    """SURVEY 8d, fused kernel: per round sum over (q,k) of 56*d (internal: mean 24 + split dir 24 +
    links 8) + 56 (leaf: mean 24 + normal 24 + bbox0 8) + 24 (moving mean), + L matched bytes in the
    last round + 27*8 per CTA partials (negligible, omitted).  d(q,k) is measured, not estimated: it is
    looked up from this run's own correspondences at every round's pose."""
    total, visits = 0, 0
    for it in range(iters):
        idx = reg.search(trace[it])
        for k in range(idx.shape[0]):
            d = depth_tables[k][idx[k]].astype(np.int64)
            total += int((56 * d + 56 + 24).sum())
            visits += int(d.sum()) + idx.shape[1]
    return total + L, visits


# --------------------------------------------------------------------------------------------
def latency_model(walked, visits, iters, K, L, measured_s, sm=148, warps_per_sm=24):
    """Latency floor of one k_gn_loop launch (what bounds the kernel, DESIGN.md 4.1): an SM runs its warp-items in passes
    of `warps_per_sm` resident warps, and a pass cannot be shorter than the chain of DEPENDENT operations of one item:
      * memory: a walk is one L2 round trip per two tree levels + the leaf record; a remembered item the memo word + the
        leaf record;
      * arithmetic (added in the second half of round 2; `floor_memory_only_ms` keeps the earlier definition): the FP64
        operations of one item that depend on each other -- pose applied (4), displacement, norm, square root and margin
        of the memo check (17), gate, error, Jacobian and scale (13), counted in kernels.cuh / device_kernels.cuh -- at the
        ~19 cycles a dependent FP64 operation takes on this part (scripts/fp64_probe.cu), and the 8 dependent DMMAs of the
        fold at ~30;
    and every round ends with the fold (one L2 round trip), the 6x6 solve + exponential map (~150 dependent FP64
    operations) and the pose hand-over (one L2 round trip).  Nothing here is a tuning constant of the kernel."""
    clk_ghz, l2_lat, fp64_lat, dmma_lat = 1.92, 250.0, 19.0, 30.0
    chain_ops = 4 + 17 + 13
    items_sm = K * L / sm / 32.0
    passes = int(np.ceil(items_sm / float(warps_per_sm)))
    dbar = visits / max(1, iters * K * L)  # mean nodes visited per walk (internal + leaf)
    mem_cycles = arith_cycles = 0.0
    for w in walked:
        frac_w = w / float(K * L)
        trips = frac_w * (dbar / 2.0 + 1.0) + (1.0 - frac_w) * 2.0
        mem_cycles += passes * trips * l2_lat + (2 * l2_lat + 150 * fp64_lat)
        arith_cycles += passes * (chain_ops * fp64_lat + 8 * dmma_lat)
    mem_s, floor_s = mem_cycles / (clk_ghz * 1e9), (mem_cycles + arith_cycles) / (clk_ghz * 1e9)
    return {"floor_ms": floor_s * 1e3, "floor_memory_only_ms": mem_s * 1e3, "measured_ms": measured_s * 1e3,
            "frac": floor_s / measured_s, "frac_memory_only": mem_s / measured_s, "passes_per_round": passes,
            "mean_nodes_per_walk": dbar, "walked_pairs_per_round": list(walked),
            "assumed": {"l2_hit_latency_cycles": l2_lat, "fp64_dependent_latency_cycles": fp64_lat,
                        "dmma_dependent_latency_cycles": dmma_lat, "dependent_fp64_ops_per_item": chain_ops,
                        "sm_ghz": clk_ghz, "resident_warps_per_sm": warps_per_sm},
            "note": "lower bound on the launch time if every dependent load were an L2 hit, every dependent FP64 operation "
                    "issued the cycle its operand arrived and nothing else cost time; frac = floor / measured (1.0 = at the "
                    "latency floor); frac_memory_only is the figure reported until the first half of round 2"}


def cpu_reference_leg(a, steps, warmup, budget_s=None):
    """Times the reference's OpenMP registration loop on the host cores.  Two CPU builds exist: the reference's
    own sources compiled against an Eigen stand-in (oracle/_ref, kind "reference") and the Eigen-free
    restatement (oracle/, kind "port"); they compute the same bits (tests/test_reference_pin.py) but the
    plain value-type stand-in costs the reference build some speed that real Eigen would not.  So that the
    baseline is not handicapped, both are timed (half the budget each) and the FASTER one is reported; the
    other one's figure stays in `sample`.  A step is one whole registration of the same workload, trees
    pre-built (SURVEY 8d)."""
    from mad_icp_b200 import synth
    from oracle import oracle as O
    from oracle import reference as R
    O.build()
    case = synth.registration_case(K=K_MODEL, beams=a.beams, azimuths=a.azimuths)
    threads = min(16, os.cpu_count() or 1)
    arms = [("port", O, O.OracleTree)]
    if R.available():
        try:
            R.lib()
            arms.insert(0, ("reference", R, R.ReferenceTree))
        except (OSError, RuntimeError):
            pass
    results = []
    for kind, M, Tree in arms:
        trees = [Tree(s) for s in case["scans"]]
        for t, P in zip(trees, case["kf_poses"]):
            t.apply_transform(P)
        q = Tree(case["query"])
        for _ in range(warmup):
            M.icp_run(trees, q, case["T_guess"], iters=a.iters, num_threads=threads, record=False)
        secs, t0 = [], time.perf_counter()
        for i in range(max(1, steps)):  # every CPU build runs the SAME number of steps (bounded by its budget share)
            last = M.icp_run(trees, q, case["T_guess"], iters=a.iters, num_threads=threads, record=False)
            secs.append(last["seconds"])
            if budget_s is not None and time.perf_counter() - t0 > budget_s / len(arms) and i >= 2:
                break
        total = float(sum(secs))
        results.append(dict(kind=kind, value=len(secs) / total, seconds=total, steps=len(secs), L=q.num_leaves,
                            X=np.asarray(last["X"], dtype=np.float64)[:3].copy(), n_matched=int(np.count_nonzero(last["matched"])),
                            matched=np.asarray(last["matched"]).astype(np.uint8).copy()))
        del trees, q
    best = max(results, key=lambda r: r["value"])
    names = {"reference": "reference sources (mad_tree.cpp, mad_icp.cpp) built against oracle/eigen_standin",
             "port": "Eigen-free restatement (oracle/)"}
    others = "; ".join(f"{names[r['kind']]}: {r['value']:.2f} scans/s over {r['steps']} registrations"
                       for r in results if r is not best)
    return dict(value=best["value"], seconds=best["seconds"], steps=best["steps"], cores=threads, kind=best["kind"],
                host_cores=os.cpu_count(), L=best["L"], X=best["X"], n_matched=best["n_matched"], matched=best["matched"],
                sample=f"{best['steps']} full registrations ({a.iters} GN iters, {K_MODEL} keyframes, {best['L']} moving "
                       f"leaves), trees pre-built, {threads} OpenMP threads over keyframes; {names[best['kind']]} "
                       f"(the faster of the CPU builds" + (f"; {others})" if others else ")"))


def pose_error(Xa, Xb):
    """(rotation angle [rad], translation distance [m]) between two 3x4 poses."""
    Xa, Xb = np.asarray(Xa)[:3], np.asarray(Xb)[:3]
    dR = Xa[:, :3] @ Xb[:, :3].T
    s = 0.5 * np.linalg.norm([dR[2, 1] - dR[1, 2], dR[0, 2] - dR[2, 0], dR[1, 0] - dR[0, 1]])
    return float(np.arctan2(s, (np.trace(dR) - 1.0) / 2.0)), float(np.linalg.norm(Xa[:, 3] - Xb[:, 3]))


def run_reference(a, rank):
    """--impl reference.  N = 1: one CPU registration loop (16 OpenMP threads over keyframes).  N > 1: the GPU arm
    runs N replicas (N scans in flight), so the CPU arm runs N replicas too -- N concurrent processes, each with its
    own 16 threads pinned to its own cores -- and reports their aggregate: like for like."""
    if rank != 0:
        return
    n = max(1, a.gpus)
    if n == 1:
        r = cpu_reference_leg(a, a.steps, max(a.warmup, 1), budget_s=150.0)
        value, steps, seconds, note = r["value"], r["steps"], r["seconds"], ""
    else:
        import subprocess
        threads = min(16, os.cpu_count() or 1)
        procs = []
        for i in range(n):
            env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_PORT",
                                                                     "MASTER_ADDR", "TORCHELASTIC_RUN_ID")}
            if (os.cpu_count() or 1) >= threads * n:
                env["OMP_PLACES"] = "{%d:%d}" % (threads * i, threads)
                env["OMP_PROC_BIND"] = "close"
            else:
                env["OMP_PROC_BIND"] = "false"
            procs.append(subprocess.Popen([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--gpus", "1",
                                           "--steps", str(a.steps), "--warmup", str(a.warmup), "--iters", str(a.iters),
                                           "--beams", str(a.beams), "--azimuths", str(a.azimuths)],
                                          env=env, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True))
        lines = []
        for p in procs:
            out, _ = p.communicate(timeout=1200)
            lines.append(json.loads([ln for ln in out.splitlines() if ln.startswith("{")][-1]))
        r = dict(lines[0]["cpu_baseline"], steps=lines[0]["steps"])
        r["sample"] = f"{n} concurrent CPU replicas, each: " + r["sample"]
        r["cores"] = threads * n
        value = float(sum(ln["value"] for ln in lines))  # replicas run concurrently: aggregate scans/s of the box
        steps = int(sum(ln["steps"] for ln in lines))
        seconds = max(ln["ms_per_step"] * ln["steps"] for ln in lines) * 1e-3
        r["value"] = value
        note = f"; {n} concurrent replicas x {threads} threads (the GPU arm at N={n} is {n} replicas too)"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "scans/s", "n_gpus": a.gpus,
            "steps": steps, "warmup": a.warmup, "ms_per_step": 1e3 * seconds / max(steps, 1) * (n if n > 1 else 1),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(a, n), "impl_note": "the reference's OpenMP registration loop on the "
                       "host cores; kind=reference: its own sources built against an Eigen stand-in (no Eigen in "
                       "the image), kind=port: the restatement" + note},
            "cpu_baseline": {"value": value, "unit": "scans/s", "cores": r["cores"], "kind": r["kind"],
                             "sample": r["sample"], "host_cores": r.get("host_cores", os.cpu_count())},
            "e2e": {"value": value, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
def stream_block(a, scans, rank, world, dev):
    """BASELINE.json configs[4]: streaming odometry over a synthetic KITTI-shape sequence, num_keyframes=16,
    p_th 0.8, no deskew, END TO END per scan through the reference-named Pipeline (pypeline): host float64 cloud in,
    H2D, float conversion / MAD-tree build / registration / keyframe promotion on the device, pose out.  The CPU
    pipeline (the reference's own Pipeline when oracle/_ref is shipped, else the restatement) runs the first
    --stream-cpu-scans scans: absolute trajectory error and keyframe decisions against it, and its scans/s."""
    os.environ.setdefault("MADICP_DEVICE", str(dev))
    from mad_icp_b200.pybind.pypeline import Pipeline
    threads = min(16, os.cpu_count() or 1)
    kw = dict(sensor_hz=10.0, deskew=False, b_max=0.2, rho_ker=0.1, p_th=0.8, b_min=0.1, b_ratio=0.02,
              num_keyframes=K_MODEL, num_threads=threads, realtime=False)
    import torch
    torch.cuda.set_device(dev)
    pipe = Pipeline(**kw)
    n = len(scans)
    # the scans wait in pinned host memory, as a driver's DMA buffers would (same rule as `e2e`: inputs start on the host)
    scans = [torch.from_numpy(np.ascontiguousarray(s0)).pin_memory().numpy() for s0 in scans]
    pipe.compute(0.0, scans[0])  # initialise: keyframe 0 (also first-touch allocations)
    traj, kf = [], []
    torch.cuda.synchronize(dev)
    depth = int(os.environ.get("MADICP_BENCH_LOOKAHEAD", "32"))  # scans handed over ahead of their turn: their trees are built in batches (0: none)
    t0 = time.perf_counter()
    for k in range(1, min(1 + depth, n)):  # the scans in flight ahead of the one being registered
        pipe.prefetch(scans[k])
    for i in range(1, n):
        pipe.compute(0.1 * i, scans[i])
        if depth > 0 and i + depth < n:  # a scan arrives: it goes up now, its tree is built with the next batch
            pipe.prefetch(scans[i + depth])
        traj.append(pipe.currentPose()[:3, 3].copy())
        kf.append((bool(pipe.isMapUpdated()), int(pipe.keyframeID())))
    t_gpu = time.perf_counter() - t0
    out = {"scans": n - 1, "points_per_scan": int(scans[0].shape[0]), "num_keyframes": K_MODEL, "p_th": 0.8,
           "value": (n - 1) / t_gpu, "unit": "scans/s", "ms_per_scan": 1e3 * t_gpu / (n - 1),
           "device_tree_build": bool(pipe.gpuBuild()), "lookahead_scans": depth, "keyframes_at_end": int(pipe.numKeyframes()),
           "path_length_m": float(np.linalg.norm(traj[-1] - traj[0])),
           "h2d_bytes_per_scan": int(scans[0].nbytes), "d2h_bytes_per_scan": 16 + 43 * 8 + 96,
           "note": "Pipeline.compute per scan, pinned host cloud in / pose out; tree build (batched look-ahead), registration and "
                   "keyframe promotion on the device"}
    m = min(a.stream_cpu_scans, n)
    if rank == 0 and m > 1:
        from oracle import oracle as O
        from oracle import reference as R
        kind = "port"
        cpu = None
        if R.available():
            try:
                R.lib()
                cpu, kind = R.ReferencePipeline(**kw), "reference"
            except (OSError, RuntimeError):
                cpu = None
        if cpu is None:
            O.build()
            cpu = O.OraclePipeline(**kw)
        cpu.compute(0.0, scans[0])
        ctraj, ckf = [], []
        t0 = time.perf_counter()
        for i in range(1, m):
            cpu.compute(0.1 * i, scans[i])
            st = cpu.state()
            ctraj.append(st[[3, 7, 11]].copy())
            ckf.append((bool(st[12]), int(st[14])))
        t_cpu = time.perf_counter() - t0
        g, c = np.array(traj[:m - 1]), np.array(ctraj)
        out.update({"cpu_scans": m - 1, "cpu_value": (m - 1) / t_cpu, "cpu_kind": kind, "cpu_threads": threads,
                    "ate_m": float(np.sqrt(((g - c) ** 2).sum(1).mean())), "ate_max_m": float(np.sqrt(((g - c) ** 2).sum(1)).max()),
                    "keyframe_decisions_equal": kf[:m - 1] == ckf})
    del pipe
    return out


# --------------------------------------------------------------------------------------------
def main():
    a = parse()
    if int(os.environ.get("WORLD_SIZE", "1")) == 1 or a.impl == "reference":
        os.environ.setdefault("OMP_PROC_BIND", "close")  # BASELINE.md section 3: the CPU arm's thread placement
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.impl == "reference":
        run_reference(a, rank)
        return

    from mad_icp_b200 import synth as _synth
    n_stream = a.stream_scans if a.stream_scans >= 0 else (1000 if world == 1 else 250)
    stream_scans = None
    if n_stream > 1:  # ray-cast the sequence in forked workers BEFORE CUDA is initialised in this process
        workers = max(1, min(32, (os.cpu_count() or 1) // max(world, 1)))
        stream_scans = _synth.sequence(n_stream + 1, a.beams, a.azimuths, workers=workers)["scans"]
    import torch
    import torch.distributed as dist
    from mad_icp_b200 import FlatTree, Registrar, synth
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n = world
    dev = local_rank if world > 1 else 0
    affinity = pin_to_gpu(dev, local_rank, world)
    torch.cuda.set_device(dev)

    # ---------------- inputs (synthetic, deterministic, identical on every rank)
    case = synth.registration_case(K=K_MODEL, beams=a.beams, azimuths=a.azimuths)
    stream = torch.cuda.Stream(device=dev)
    trees = []
    for s in range(K_MODEL):
        ft = FlatTree(case["scans"][s])
        ft.apply_transform(case["kf_poses"][s])
        trees.append(ft)
    # primary context: the FULL 16-keyframe model on this GPU.  N = 1: the whole job.  N > 1: one
    # replica per GPU, every rank registers its own scan (throughput mode, no exchange, weak scaling).
    reg = Registrar(device=dev, max_keyframes=K_MODEL)
    reg.set_stream(stream.cuda_stream)
    depth_tables, model_bytes = [], 0
    for s in range(K_MODEL):
        reg.put_keyframe(s, trees[s])
        depth_tables.append(leaf_depths(trees[s].records()))
        model_bytes += trees[s].num_nodes * (64 + 16 + 4)
    qtree = FlatTree(case["query"])
    means = qtree.leaf_means()
    L = means.shape[0]
    pinned = torch.from_numpy(means).pin_memory()
    X0 = case["T_guess"]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{dev}")  # > 126 MB L2

    def l2_flush():
        with torch.cuda.stream(stream):
            flush.fill_(1)

    def barrier():
        # Drain the GPU BEFORE the NCCL barrier: the sharded persistent kernel owns every SM and waits for
        # its peers' kernels; an NCCL kernel that slips in between two of them on one rank would wait for
        # the other rank's NCCL kernel, which is queued behind a persistent kernel that is waiting for
        # this rank -> deadlock.  Rule: no collective while cross-GPU registrations are in flight.
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed_resident(r):
        """K registrations with resident inputs: per-step event pairs (L2 flushed in between), summed,
        max over ranks.  Returns (total_ms, launches)."""
        for _ in range(max(a.warmup, 3)):
            l2_flush()
            r.register_async(X0, a.iters)
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
        l0 = r.kernel_launches
        barrier()
        for s0, s1 in ev:
            l2_flush()
            s0.record(stream)
            r.register_async(X0, a.iters)
            s1.record(stream)
        barrier()
        ms = float(sum(s0.elapsed_time(s1) for s0, s1 in ev))
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=f"cuda:{dev}")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, r.kernel_launches - l0

    # ---------------- resident-input throughput (`value`)
    reg.set_moving(pinned)
    sampler = ClockSampler(dev)
    sampler.start()
    total_ms, launches = timed_resident(reg)
    res = reg.register_fetch(want_matched=True)

    # ---------------- end to end through the public call with host buffers (`e2e`)
    for _ in range(3):
        l2_flush()
        reg.set_moving(pinned)
        reg.register(X0, a.iters)
    barrier()
    e2e_s = 0.0
    for _ in range(a.steps):
        l2_flush()
        barrier()  # sync - NCCL barrier - sync: the barrier's own kernel must be off the GPU before the clock starts
        t0 = time.perf_counter()
        reg.set_moving(pinned)                       # H2D: L x 24 B from pinned host memory
        out = reg.register(X0, a.iters)              # H2D pose, kernels, D2H pose/H/b/matched, sync
        e2e_s += time.perf_counter() - t0
    sampler.stop_flag = True
    sampler.join(timeout=1.0)
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=f"cuda:{dev}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    h2d = L * 24 + 96 + 16
    d2h = 16 + 42 * 8 + 96 + L

    # ---------------- N > 1: the SAME scan registered jointly (north_star's sharding): keyframe slot s on
    # rank s % N, the 48-value H/b tile all-reduced inside the persistent kernel every GN round (NVLink
    # peer mailboxes).  Strong scaling of one scan's latency; reported beside the replica throughput.
    sharded = None
    if world > 1:
        sh = Registrar(device=dev, max_keyframes=K_MODEL)
        sh.set_stream(stream.cuda_stream)
        for s in range(K_MODEL):
            if s % n == rank:
                sh.put_keyframe(s, trees[s])
        sh.set_moving(pinned)
        h = torch.tensor(list(sh.comm_export()), dtype=torch.uint8, device=f"cuda:{dev}")
        allh = [torch.empty_like(h) for _ in range(world)]
        dist.all_gather(allh, h)
        sh.comm_connect(rank, world, [bytes(t.cpu().tolist()) for t in allh])
        dist.barrier()
        sh_ms, _ = timed_resident(sh)
        sh_res = sh.register_fetch(want_matched=True)
        dpose = float(np.abs(sh_res["X"] - res["X"]).max())
        sharded = {"value": a.steps / (sh_ms * 1e-3), "unit": "scans/s", "ms_per_scan": sh_ms / a.steps,
                   "scaling": "strong", "max_abs_pose_diff_vs_single_gpu": dpose,
                   "n_matched_equal_vs_single_gpu": int(sh_res["n_matched"]) == int(res["n_matched"]),
                   "matched_flags_equal_vs_single_gpu": bool(np.array_equal(sh_res["matched"], res["matched"])),
                   "note": f"one scan, keyframe slot s on rank s%{n}, in-kernel NVLink all-reduce of H/b each GN round"}
        sh.close()

    # ---------------- cfg5: streaming odometry, end to end (every rank its own replica of the sequence at N > 1)
    stream = None
    if stream_scans is not None:
        barrier()
        stream = stream_block(a, stream_scans, rank, world, dev)
        if world > 1:
            t = torch.tensor([stream["ms_per_scan"]], dtype=torch.float64, device=f"cuda:{dev}")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            stream["ms_per_scan"] = float(t.item())
            stream["value"] = n * 1e3 / stream["ms_per_scan"]
            stream["note"] += f"; {n} independent replicas of the sequence, slowest rank's time"
        del stream_scans

    # ---------------- roofline of the dominant kernel (k_gn_loop) + parity guard
    trace = reg.register_trace()
    rf = None
    if world == 1:
        walked = reg.register_walked().astype(int).tolist()
        abytes, visits = algorithmic_bytes(reg, depth_tables, trace, a.iters, L)
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"
        avg_launch_s = (total_ms * 1e-3) / a.steps
        achieved = abytes / avg_launch_s / 1e9
        prof = {}
        tp = os.path.join(ROOT, "profiles", "gn_loop_traffic.json")
        if os.path.exists(tp):
            prof = json.load(open(tp))
        # L2 read bandwidth of THIS device, measured here: repeated reduction of a 48 MiB (L2-resident) buffer
        buf = torch.empty(48 << 20, dtype=torch.uint8, device=f"cuda:{dev}").view(torch.float32)
        for _ in range(3):
            buf.sum()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            buf.sum()
        e1.record()
        torch.cuda.synchronize(dev)
        l2_peak = 20 * buf.numel() * 4 / (e0.elapsed_time(e1) * 1e-3) / 1e9
        l2_bytes = prof.get("l2_to_l1_bytes_per_launch")
        l2 = {"bytes_per_launch": l2_bytes, "achieved": (l2_bytes / avg_launch_s / 1e9) if l2_bytes else None,
              "peak": l2_peak, "unit": "GB/s", "frac": (l2_bytes / avg_launch_s / 1e9 / l2_peak) if l2_bytes else None,
              "source": "lts__t_sectors_srcunit_tex_op_read.sum x 32 B of the committed ncu capture (profiles/); peak = "
                        "torch sum over a 48 MiB L2-resident buffer, measured in this run"}
        lat = latency_model(walked, visits, a.iters, K_MODEL, L, avg_launch_s)
        rf = {"kernel": "k_gn_loop (persistent: search + linearize + reduce + solve, all GN rounds)", "bound": "hbm",
              "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
              "traffic": prof.get("dram_bytes_per_launch"),
              "algorithmic_bytes_per_launch": abytes, "node_visits_per_launch": visits, "peak_source": peak_src,
              "avg_launch_ms": avg_launch_s * 1e3, "model_bytes": model_bytes, "l2": l2, "latency_model": lat,
              "note": "SURVEY 8d's algorithmic bytes are those of the reference's algorithm (every pair walked in every round); "
                      "the model is L2-resident and from round 1 on the kernel proves most walks unchanged and skips them "
                      "(walked_pairs_per_round), so DRAM traffic << algorithmic bytes and frac exceeds 1: HBM is not the bound. "
                      "The falsifiable figures are `l2` (bandwidth) and `latency_model` (dependent round trips)."}

    cpu, parity = None, None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        r = cpu_reference_leg(a, steps=1000, warmup=1, budget_s=a.cpu_seconds)
        cpu = {"value": r["value"], "unit": "scans/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"],
               "host_cores": r["host_cores"]}
        # in-run parity guard: the GPU result of the timed workload against the CPU leg's, same inputs
        ang, dt = pose_error(res["X"], r["X"])
        parity = {"against": r["kind"], "pose_rad": ang, "pose_m": dt, "tol_rad": 1e-5, "tol_m": 1e-4,
                  "n_matched_gpu": int(res["n_matched"]), "n_matched_cpu": int(r["n_matched"]),
                  "n_matched_equal": int(res["n_matched"]) == int(r["n_matched"]),
                  "matched_flags_equal": bool(res["matched"] is not None and np.array_equal(res["matched"] != 0, r["matched"] != 0)),
                  "ok": bool(ang < 1e-5 and dt < 1e-4 and int(res["n_matched"]) == int(r["n_matched"]))}
        if not parity["ok"]:
            print(f"bench.py: PARITY FAILURE against the CPU {r['kind']}: {parity}", file=sys.stderr, flush=True)

    if rank == 0:
        clocks = sampler.summary()
        line = {"metric": METRIC, "value": n * a.steps / (total_ms * 1e-3), "unit": "scans/s", "n_gpus": n,
                "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": total_ms / a.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic",
                "config": {"workload": workload_name(a, n), "moving_leaves": L, "keyframes": K_MODEL,
                           "gn_iters": a.iters, "l2": "flushed between steps (256 MiB fill, outside the per-step events)",
                           "timing": "per-step CUDA event pairs on the launch stream, summed; max over ranks",
                           "host_affinity": affinity},
                "e2e": {"value": n * a.steps / e2e_s, "unit": "scans/s", "h2d_bytes_per_step": h2d,
                        "d2h_bytes_per_step": d2h, "ms_per_step": 1e3 * e2e_s / a.steps,
                        "timing": "host wall clock around set_moving+register (pinned H2D, kernel, D2H, sync)"},
                "gpu_launches": int(launches), "clocks": clocks,
                "result": {"n_matched": int(res["n_matched"]), "pose_t": [float(v) for v in res["X"][:, 3]]}}
        if rf:
            line["roofline"] = rf
        if cpu:
            line["cpu_baseline"] = cpu
        if parity:
            line["parity"] = parity
        if sharded:
            line["sharded"] = sharded
        if stream:
            line["stream"] = stream
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, res)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
