#!/usr/bin/env python
"""bench.py -- the BASELINE.json metric: observations/s and LM iterations/s of bundle adjustment on the
10k-camera / 2M-point / 20M-observation synthetic scene (configs[2]), strong-scaled over N GPUs.

A "step" is one Levenberg-Marquardt iteration (linear solve by Schur-complement PCG, candidate evaluation,
re-linearisation).  `python bench.py --gpus N --steps K --warmup W` (under torchrun for N > 1, one rank per GPU):
  * every rank builds the same seeded scene and keeps its shard of points + their observations,
  * W untimed LM iterations (warm-up solve), parameters reset,
  * exactly K LM iterations timed on the device (CUDA events on the engine stream, per iteration; the
    initial evaluation is included), bracketed by barrier + synchronize, max over ranks,
  * `e2e`: the same K iterations through the drop-in C-ABI call tba_solve() with HOST buffers
    (pack + H2D + solve + D2H inside the timed region, wall clock, max over ranks),
  * `roofline`: the dominant kernel (implicit-Schur matvec) timed with CUDA events inside the timed solve,
  * `cpu_baseline` (N = 1, rank 0): the CPU oracle (port of the Theia+Ceres path; Ceres itself is not
    installable here) on a bounded sample.
`--impl reference` times that CPU restatement alone with all host threads.
`--dump-outputs DIR` (one process) writes what the timed solve computed as float64 arrays DIR/<name>.npy: the cameras,
the intrinsics, a fixed seeded sample of the points and the per-iteration costs.  When the solve reaches the fp64 floor
before K iterations, these are its results there, not those of the restarts that fill up K (which repeat its start).  The
scene is seeded, so the same arguments give the same inputs and two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from theiasfm_b200 import _abi, synthetic  # noqa: E402

METRIC = "observations/s = N_obs x LM iterations / solve time (10k-cam / 2M-pt / 20M-obs BA, ITERATIVE_SCHUR + SCHUR_JACOBI)"
SAMPLE_CONFIG = dict(n_cam=1_000, n_pt=100_000, obs_per_pt=10, model=_abi.MODEL_PINHOLE, shared_intrinsics=True, seed=20240612)


def solver_kwargs(max_iters):
    # tolerances at zero so that exactly `max_iters` LM iterations run (no early convergence inside the timed region)
    return dict(use_inner_iterations=0, linear_solver_type=_abi.ITERATIVE_SCHUR, preconditioner_type=_abi.PRECOND_SCHUR_JACOBI,
                max_num_iterations=max_iters, function_tolerance=0.0, gradient_tolerance=0.0, parameter_tolerance=0.0)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (profiling recipe's clocks line).
    Started before the warm-up (nvidia-smi takes ~1 s to come up); samples are filtered to the timed window."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self, t_begin, t_end):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.1)
        self.proc.terminate()
        ok = [r for t, r in self.rows if len(r) >= 10 and r[2].replace(".", "").isdigit()]
        inside = [r for t, r in self.rows if len(r) >= 10 and r[2].replace(".", "").isdigit() and t_begin - 0.02 <= t <= t_end + 0.05]
        rows = inside if inside else ok
        sm = [float(r[2]) for r in rows]
        mx = [float(r[3]) for r in rows]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in rows for n, v in zip(names, r[6:10]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "window": "timed region" if inside else "whole run (timed region shorter than the sampling period)",
                "power_w_max": max([float(r[4]) for r in rows if r[4].replace(".", "").isdigit()], default=None)}


def _microbench_call(symbol, n_out, device):
    code = ("import ctypes, json; L = ctypes.CDLL(%r); out = (ctypes.c_double * %d)(); rc = L.%s(%d, out); "
            "print(json.dumps({'rc': rc, 'v': list(out)}))"
            % (os.path.join(ROOT, "theiasfm_b200", "libtheia_microbench_b200.so"), n_out, symbol, device))
    try:
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
        d = json.loads(r.stdout.strip().splitlines()[-1])
        return d["v"] if d["rc"] == 0 else None
    except Exception:  # noqa: BLE001 -- the micro-benchmarks are optional evidence, never a reason to fail the bench
        return None


def run_microbench(device):
    """fp64 FMA peak, fp64 RED rate and 48-byte gather rate of this GPU (theiasfm_b200/csrc/tba_microbench.cu), measured
    in SEPARATE processes before the solve so that they cannot disturb the timed region; None if anything goes wrong.
    The second call (tba_microbench_ex) answers design questions for the next kernel generation and may fail on its own."""
    v = _microbench_call("tba_microbench", 3, device)
    if v is None:
        return None
    ex = _microbench_call("tba_microbench_ex", 6, device)
    gaps = _microbench_call("tba_microbench_gaps", 5, device)
    return {"fp64_fma_tflops": v[0], "fp64_red_gops": v[1], "gather48_grows": v[2],
            # launch gaps (us): small kernel alone; 220 KB-shared-memory kernel spinning ~20 us alone; the pair big + small; the pair with
            # the small kernel hinted to the maximum shared-memory carve-out; the pair with the small kernel launched with 220 KB itself
            "launch_gap_us": dict(zip(("small", "big_20us", "big_plus_small", "big_plus_small_carveout_hint", "big_plus_small_same_smem"), gaps)) if gaps else None,
            # design questions for the next kernel generation (NOTES.md section 3): REDs emitted element-major (6 lanes per
            # 48-byte row), shared-memory fp64 atomicAdd (CAS loop), global REDs confined to a 1200-camera window per CTA
            "fp64_red_rows_gops": ex[0] if ex else None, "fp64_smem_atomic_gops": ex[1] if ex else None,
            "fp64_red_window_gops": ex[2] if ex else None,
            # gather strategies for the 48-byte camera rows, G rows/s like gather48_grows (the shipped 3 x LDG.128 lane-per-row):
            # chunk-major loads transposed through shared memory, 64-byte padded rows with one 256-bit + one 128-bit load,
            # element-major 64-bit loads
            "gather48_coop_grows": ex[3] if ex else None, "gather64_ld256_grows": ex[4] if ex else None,
            "gather48_elem_grows": ex[5] if ex else None,
            "how": "tba_microbench: 8 DFMA chains/thread; RED.ADD.F64 and 3xLDG.128 gathers over a 60k-double vector, "
                   "32 distinct rows per warp; best of 5 after warm-up"}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def physical_cores():
    """Physical cores this process may run on (SMT siblings counted once): distinct (package, core) pairs of the allowed CPUs."""
    allowed = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))
    seen = set()
    for cpu in allowed:
        try:
            with open("/sys/devices/system/cpu/cpu%d/topology/physical_package_id" % cpu) as f:
                pkg = f.read().strip()
            with open("/sys/devices/system/cpu/cpu%d/topology/core_id" % cpu) as f:
                core = f.read().strip()
            seen.add((pkg, core))
        except OSError:
            seen.add(("?", cpu))
    return max(1, len(seen))


def pin_openmp():
    """Must run before libgomp is loaded (it reads these once): one thread per physical core, bound, no migration.  The round-1
    reference arm moved 17x between two boxes with unbound threads on all 128 logical CPUs."""
    os.environ["OMP_NUM_THREADS"] = str(physical_cores())
    os.environ["OMP_PROC_BIND"] = "close"
    os.environ["OMP_PLACES"] = "cores"
    os.environ["OMP_DYNAMIC"] = "false"
    os.environ.setdefault("OMP_WAIT_POLICY", "active")


def sample_workload_text(n_obs=None):
    c = SAMPLE_CONFIG
    return ("cpu_sample_1kcam: %d cameras / %d points / ~%d observations (same generator, same solver options as c3_10kcam: PINHOLE, one "
            "shared intrinsics group, TRIVIAL loss, default intrinsics mask, use_inner_iterations=false); the CPU restatement of the "
            "Theia+Ceres path is timed on this bounded sample, obs/s is size-normalised" %
            (c["n_cam"], c["n_pt"], n_obs if n_obs else c["n_pt"] * c["obs_per_pt"]))


def cpu_baseline(steps, warmup=0):
    """The CPU restatement (oracle/, kind 'port') on a bounded sample: a 1k-camera / 100k-point / 1M-observation scene.
    Call only in a process whose OpenMP runtime was configured by pin_openmp() (the reference arm / its child process)."""
    from oracle import oracle_py
    oracle_py.set_num_threads(int(os.environ.get("OMP_NUM_THREADS", "0")) or physical_cores())
    p = synthetic.make_scene(**SAMPLE_CONFIG)
    n_obs = p.n_obs
    if warmup:
        oracle_py.solve(p.copy(), oracle_py.default_options(**solver_kwargs(warmup)))
    s = oracle_py.solve(p, oracle_py.default_options(**solver_kwargs(steps)))
    iters = s.num_iterations - 1
    return {"value": n_obs * iters / s.solve_time_in_seconds, "unit": "obs/s", "cores": oracle_py.num_threads(), "kind": "port",
            "sample": "%d LM iterations of the same solver on a 1k-camera / 100k-point / %d-observation scene (same generator); "
                      "%.2f s solve, %.2f s problem setup; threads bound one per physical core (OMP_PROC_BIND=close, OMP_PLACES=cores)"
                      % (iters, n_obs, s.solve_time_in_seconds, s.setup_time_in_seconds),
            "lm_iters_per_s": iters / s.solve_time_in_seconds, "ms_per_step": 1e3 * s.solve_time_in_seconds / max(iters, 1),
            "linear_solver_iterations": s.num_linear_solver_iterations, "n_obs": n_obs, "logical_cpus": len(os.sched_getaffinity(0))}


def cpu_baseline_subprocess(steps, timeout=240):
    """cpu_baseline of the GPU arm: run the reference arm in its own process (fresh, pinned OpenMP runtime; torch's bundled
    libgomp in this process was initialised long ago) and keep its cpu_baseline object."""
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "OMP_NUM_THREADS")}
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(steps), "--warmup", "0"],
                           capture_output=True, text=True, timeout=timeout, env=env)
        return json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
    except Exception as e:  # noqa: BLE001 -- reported, never a reason to lose the GPU line
        return {"value": None, "unit": "obs/s", "cores": None, "kind": "port", "sample": "failed: %s: %s" % (type(e).__name__, e)}


SWITCHES = ("TBA_TRED", "TBA_LIN_OCC", "TBA_ABLATE", "TBA_MATVEC", "TBA_PCG")
# "default" = the shipped kernels (persistent streaming Schur kernels).  "tile_kernels" = the round-1 tile-per-CTA Schur kernels with
# the transposed RED emission; "r1_kernels" = the round-1 defaults.  The TBA_ABLATE variants switch parts of the matvec OFF (wrong
# results by construction, timing only): they say how much of the launch each part costs in situ.
VARIANTS = (("default", {}), ("split_pcg", {"TBA_PCG": "split"}), ("tile_kernels", {"TBA_MATVEC": "tile"}), ("r1_kernels", {"TBA_MATVEC": "tile", "TBA_TRED": "0", "TBA_LIN_OCC": "2"}),
            ("ablate_no_red", {"TBA_ABLATE": "1"}), ("ablate_no_gather", {"TBA_ABLATE": "2"}),
            ("ablate_no_segreduce", {"TBA_ABLATE": "8"}), ("ablate_all", {"TBA_ABLATE": "15"}))


def experiments_child(workload, K, device):
    """Runs in its OWN process (bench.py --experiments-child), after the measured solve of the parent is over: the same
    workload solved once per compiled-in experiment switch (NOTES.md section 3; all default off), one JSON line per variant
    with its per-stage device times and its per-iteration costs relative to the default kernels.  Diagnostics for the
    next round's kernel work -- never part of `value` / `e2e`; a variant that fails only loses its own line."""
    from theiasfm_b200 import engine
    full = synthetic.make_config(workload)
    init = full.copy()
    ref = None
    for name, env in VARIANTS:
        for k in SWITCHES:
            os.environ.pop(k, None)
        os.environ.update(env)
        line = {"variant": name}
        try:
            eng = engine.Engine(device=device)  # the switches are read when the context is created
            eng.upload(full, engine.default_options(**solver_kwargs(K)))
            eng.minimize()                      # warm-up
            eng.reset_parameters(init)
            eng.set_profiling(True)
            s = eng.minimize()
            st = eng.profile_stages()
            eng.set_profiling(False)
            eng.close()
            iters = max(s.num_iterations - 1, 1)
            costs = np.asarray(s.costs, dtype=np.float64)
            if ref is None and not name.startswith("ablate"):
                ref = costs
            n = min(len(ref), len(costs))
            line.update({"rc": int(s.rc), "ms_per_step": 1e3 * sum(it["iteration_time_in_seconds"] for it in s.iterations) / iters,
                         "steps_run": iters, "pcg_iterations": int(s.num_linear_solver_iterations), "final_cost": float(s.final_cost),
                         "max_rel_cost_diff_vs_default": None if name.startswith("ablate") else (float(np.max(np.abs(costs[:n] - ref[:n]) / ref[:n])) if n else None),
                         "stage_ms_per_step": {k: v["ms"] / iters for k, v in st.items()},
                         "matvec_ms_per_launch": st["matvec"]["ms"] / max(st["matvec"]["launches"], 1)})
        except Exception as e:  # noqa: BLE001
            line["error"] = "%s: %s" % (type(e).__name__, e)
        print(json.dumps(line), flush=True)
    # secondary path (BASELINE.json configs[4], SURVEY a16): the CUDA-core brute-force matcher on a sample of config 5's
    # image pairs (5k x 5k SIFT-128 each, ratio test + symmetric intersection); host buffers in, match lists out
    line = {"variant": "matcher_sample"}
    try:
        import ctypes as C
        from theiasfm_b200 import matcher
        rng = np.random.default_rng(0)
        n_img, n, dim = 4, int(os.environ.get("TBA_BENCH_MATCHER_N", "5000")), 128  # the variable only shrinks the CPU test of this code
        base = np.abs(rng.normal(size=(n, dim)))
        # every image sees the same features in its own order, with noise: the ratio test keeps most true matches
        desc = np.concatenate([base[rng.permutation(n)] + 0.05 * rng.normal(size=(n, dim)) for _ in range(n_img)]).astype(np.float32)
        desc /= np.linalg.norm(desc, axis=1, keepdims=True)
        off = (np.arange(n_img + 1) * n).astype(np.int64)
        pr = np.array([(i, j) for i in range(n_img) for j in range(i + 1, n_img)], np.int32)
        cap = len(pr) * n + 1
        out = (matcher.tbm_match * cap)()
        moff = np.zeros(len(pr) + 1, np.int64)
        ok = np.zeros(len(pr), np.uint8)
        opt = matcher.default_options()
        L = matcher.lib()

        def call():
            return L.tbm_match_all(device, desc.ctypes.data_as(C.POINTER(C.c_float)), off.ctypes.data_as(C.POINTER(C.c_int64)), n_img, dim,
                                   pr.ctypes.data_as(C.POINTER(C.c_int32)), len(pr), C.byref(opt), out, cap,
                                   moff.ctypes.data_as(C.POINTER(C.c_int64)), ok.ctypes.data_as(C.POINTER(C.c_uint8)))
        rc = call()  # warm-up
        t0 = time.perf_counter()
        reps = 3
        for _ in range(reps):
            rc = call()
        dt = (time.perf_counter() - t0) / reps
        line.update({"rc": int(rc), "images": n_img, "descriptors_per_image": n, "dim": dim, "pairs": int(len(pr)), "seconds_per_call": dt,
                     "pairs_per_s": len(pr) / dt, "matches": int(moff[-1]),
                     "distance_evaluations_per_s": len(pr) * float(n) * n / dt,
                     "note": "end to end through tbm_match_all with host buffers (H2D, top-2 kernel, D2H, host ratio test / intersection)"})
    except Exception as e:  # noqa: BLE001
        line["error"] = "%s: %s" % (type(e).__name__, e)
    print(json.dumps(line), flush=True)
    return 0


def run_experiments(workload, K, device, timeout=180):
    """Parent side: spawn the child, keep whatever lines it managed to print."""
    env = {k: v for k, v in os.environ.items() if k not in SWITCHES and k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    cmd = [sys.executable, os.path.abspath(__file__), "--experiments-child", "--workload", workload, "--steps", str(K), "--device", str(device)]
    out, note = "", None
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
        out = r.stdout
        if r.returncode != 0:
            note = "child exit code %d: %s" % (r.returncode, r.stderr.strip().splitlines()[-1] if r.stderr.strip() else "")
    except subprocess.TimeoutExpired as e:
        out = e.stdout.decode() if isinstance(e.stdout, bytes) else (e.stdout or "")
        note = "child killed after %d s" % timeout
    except Exception as e:  # noqa: BLE001 -- optional evidence, never a reason to fail the bench
        note = "%s: %s" % (type(e).__name__, e)
    res = {}
    for ln in out.splitlines():
        try:
            d = json.loads(ln)
            res[d.pop("variant")] = d
        except Exception:  # noqa: BLE001
            continue
    if note:
        res["note"] = note
    return res


# ---------------------------------------------------------------------------------------------------------------------------
# BASELINE.json configs[4] (SURVEY 8 row a16): BruteForceFeatureMatcher on 5k x 5k SIFT-128 image pairs.
MATCHER_METRIC = ("image pairs/s = matched image pairs / time (BruteForceFeatureMatcher::MatchImagePair semantics: 5000 x 5000 SIFT-128 "
                  "descriptors per pair, squared L2, Lowe ratio 0.8, symmetric, min 30 matches)")
MATCHER_N, MATCHER_DIM = 5000, 128


def matcher_scene(n_img, n=MATCHER_N, seed=20240613):
    """SIFT-like images: every image sees the same physical features (non-negative unit descriptors) in its own order with noise,
    plus 20 % unrelated descriptors: the ratio test keeps most true matches and rejects the rest."""
    rng = np.random.default_rng(seed)
    n_true = int(0.8 * n)
    base = np.abs(rng.normal(size=(n_true, MATCHER_DIM))).astype(np.float32)
    sets = []
    for _ in range(n_img):
        s = base[rng.permutation(n_true)] + 0.05 * np.abs(rng.normal(size=(n_true, MATCHER_DIM))).astype(np.float32)
        s = np.concatenate([s, np.abs(rng.normal(size=(n - n_true, MATCHER_DIM))).astype(np.float32)])
        s = s[rng.permutation(n)]
        sets.append(np.ascontiguousarray(s / np.linalg.norm(s, axis=1, keepdims=True), np.float32))
    return sets


def matcher_cpu_pairs_per_s(sets, n_pairs=2):
    """The CPU restatement of MatchImagePair (oracle/matcher_oracle.c, one thread: the reference runs one pair per pool thread)."""
    import ctypes as C
    from theiasfm_b200 import matcher
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "libmatcher_oracle.so"], stdout=subprocess.DEVNULL)
    M = C.CDLL(os.path.join(ROOT, "oracle", "libmatcher_oracle.so"))
    o = matcher.default_options()
    fp = C.POINTER(C.c_float)
    out = (matcher.tbm_match * len(sets[0]))()
    n = C.c_int()
    t0 = time.perf_counter()
    for p in range(n_pairs):
        a, b = sets[p % len(sets)], sets[(p + 1) % len(sets)]
        M.matcher_match_image_pair(a.ctypes.data_as(fp), len(a), b.ctypes.data_as(fp), len(b), MATCHER_DIM, C.byref(o), out, C.byref(n))
    dt = time.perf_counter() - t0
    return n_pairs / dt, dt


def matcher_main(args):
    """python bench.py --workload c5_matcher [--gpus N]: a "step" = this rank's share of all image pairs of a 48-image sample of
    config 5 (1128 pairs of 5000 x 5000 descriptors) through tbm_match_all; pairs are independent units, sharded round-robin over
    the ranks with no collective (descriptors replicated) -- strong scaling over a fixed pair list."""
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    K, W = args.steps, max(args.warmup, 0)
    n_img = int(os.environ.get("TBA_BENCH_MATCHER_IMAGES", "48"))
    n_desc = int(os.environ.get("TBA_BENCH_MATCHER_N", str(MATCHER_N)))
    config = {"workload": "c5_matcher: %d-image sample of config 5 (10k images x 5k SIFT-128): all %d image pairs, %d x %d descriptors per pair, "
                          "ratio 0.8, symmetric, min 30 matches" % (n_img, n_img * (n_img - 1) // 2, n_desc, n_desc),
              "parallelism": "image pairs sharded round-robin over %d GPU(s), descriptors replicated, no collective" % world,
              "l2_policy": "every step re-uploads the descriptors and streams %d candidate tiles per query block; the distance matrices are never stored; ratio test / symmetric filter on the device, only the kept matches are copied back" % ((n_desc + 127) // 128)}
    sets = matcher_scene(n_img, n_desc)
    if args.impl == "reference":
        if rank != 0:
            return 0
        v, dt = matcher_cpu_pairs_per_s(sets, 3)
        line = {"impl": "reference", "metric": MATCHER_METRIC, "value": v, "unit": "pairs/s", "n_gpus": args.gpus, "steps": K, "warmup": W,
                "ms_per_step": 1e3 * dt / 3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": config, "cpu_baseline": {"value": v, "unit": "pairs/s", "cores": 1, "kind": "port",
                                                    "sample": "3 image pairs of the same scene through oracle/matcher_oracle.c (one thread), %.2f s" % dt},
                "e2e": {"value": v, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
        print(json.dumps(line))
        return 0
    import torch
    import torch.distributed as dist
    from theiasfm_b200 import matcher
    if world > 1:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(local_rank)

    def allred(v, op):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64)
        dist.all_reduce(t, op=op)
        return float(t[0])
    all_pairs = [(i, j) for i in range(n_img) for j in range(i + 1, n_img)]
    mine = all_pairs[rank::world]
    opt = matcher.default_options()
    # the C-ABI call itself (host buffers in, match lists out): what a C++ caller times -- no Python list building around it
    import ctypes as C
    L = matcher.lib()
    off = np.zeros(n_img + 1, np.int64); off[1:] = np.cumsum([len(d) for d in sets])
    desc = np.ascontiguousarray(np.concatenate(sets, axis=0), np.float32)
    pr = np.ascontiguousarray(np.array(mine, np.int32).reshape(-1, 2))
    cap = int(len(mine)) * n_desc + 1
    out = (matcher.tbm_match * cap)()
    moff = np.zeros(len(pr) + 1, np.int64)
    okb = np.zeros(max(len(pr), 1), np.uint8)

    def call():
        rc = L.tbm_match_all(local_rank, desc.ctypes.data_as(C.POINTER(C.c_float)), off.ctypes.data_as(C.POINTER(C.c_int64)), n_img, MATCHER_DIM,
                             pr.ctypes.data_as(C.POINTER(C.c_int32)), len(pr), C.byref(opt), out, cap, moff.ctypes.data_as(C.POINTER(C.c_int64)),
                             okb.ctypes.data_as(C.POINTER(C.c_uint8)))
        assert rc == 0, rc
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(W):
        call()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    tw0 = time.time()
    t0 = time.perf_counter()
    gemm_ms = exact_ms = h2d_ms = 0.0
    n_matches = 0
    for _ in range(K):
        call()
        tm = matcher.last_timing()
        gemm_ms += tm["gemm_ms"]; exact_ms += tm["exact_ms"]; h2d_ms += tm["h2d_ms"]
        n_exh = tm["exhaustive_queries"]
        n_matches = int(moff[len(pr)])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    wall = allred(time.perf_counter() - t0, dist.ReduceOp.MAX if world > 1 else None)
    clocks = sampler.stop(tw0, time.time())
    dev_s = allred(1e-3 * (gemm_ms + exact_ms), dist.ReduceOp.MAX if world > 1 else None)
    gemm_s = allred(1e-3 * gemm_ms, dist.ReduceOp.MAX if world > 1 else None)
    pairs_total = len(all_pairs) * K
    n_matches = allred(float(n_matches), dist.ReduceOp.SUM if world > 1 else None)
    flops = 2.0 * n_desc * n_desc * MATCHER_DIM * 2 * len(all_pairs) * K  # both directions of every pair
    peak = 1414.5
    pk = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak_src = "fallback"
    if os.path.exists(pk):
        with open(pk) as f:
            peak = float(json.load(f)["bf16_tflops_sustained"]); peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    achieved = flops / gemm_s / 1e12 / world if gemm_s > 0 else 0.0   # per GPU
    cb = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, dt = matcher_cpu_pairs_per_s(sets, 2)
        cb = {"value": v, "unit": "pairs/s", "cores": 1, "kind": "port", "sample": "2 image pairs of the same scene through oracle/matcher_oracle.c (one thread), %.2f s" % dt}
    if rank == 0:
        line = {"metric": MATCHER_METRIC, "value": pairs_total / dev_s if dev_s > 0 else 0.0, "unit": "pairs/s", "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": 1e3 * dev_s / K, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 (TF32 tensor-core ranking, exact f32 decision)",
                "data": "synthetic", "config": config, "clocks": clocks,
                "e2e": {"value": pairs_total / wall, "unit": "pairs/s", "h2d_bytes_per_step": float(n_img * n_desc * MATCHER_DIM * 4) * world,
                        "d2h_bytes_per_step": float(n_matches * 12 + len(all_pairs) * 5), "seconds": wall},
                # per call: k_row_norms once; per chunk of <= 4M queries: k_expand_segments, k_nn_candidates, k_exact_top2, k_pair_decide, k_gather_matches
                "gpu_launches": int(K * (1 + 5 * max(1, (len(mine) * 2 * n_desc + (4 << 20) - 1) // (4 << 20)))) * world,
                "roofline": {"kernel": "k_nn_candidates (TF32 tcgen05.mma distance GEMM + fused top-8 epilogue from TMEM)", "bound": "tensor", "achieved": achieved,
                             "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                             "note": "algorithmic flops 2*n1*n2*128 per direction on the TF32 path (nominal dense TF32 = half the bf16 rate the peak is quoted for); per GPU",
                             "gemm_seconds": gemm_s, "exact_seconds": allred(1e-3 * exact_ms, dist.ReduceOp.MAX if world > 1 else None)},
                "cpu_baseline": cb, "matches_per_step": n_matches, "exhaustive_queries_per_step_rank0": n_exh, "queries_per_step": 2 * n_desc * len(all_pairs), "distance_evaluations_per_s": 2.0 * n_desc * n_desc * pairs_total / dev_s if dev_s > 0 else 0.0}
        print(json.dumps(line))
    elif world > 1:
        allred(1e-3 * exact_ms, dist.ReduceOp.MAX)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c3_10kcam", choices=list(synthetic.CONFIGS) + ["c5_matcher"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-experiments", action="store_true", help="skip the diagnostic pass over the compiled-in experiment switches")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed solve computed as DIR/<name>.npy (float64, "
                                                          "about 9 MB for c3_10kcam); bundle adjustment on one GPU")
    ap.add_argument("--experiments-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--device", type=int, default=0, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload == "c5_matcher" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs writes the bundle-adjustment result of one GPU (no --impl reference, c5_matcher or WORLD_SIZE > 1)")
    if args.experiments_child:
        return experiments_child(args.workload, args.steps, args.device)
    if args.workload == "c5_matcher":
        return matcher_main(args)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    K, W = args.steps, max(args.warmup, 0)
    cfg = synthetic.CONFIGS[args.workload]
    model_name = "PINHOLE" if cfg["model"] == _abi.MODEL_PINHOLE else "PINHOLE_RADIAL_TANGENTIAL"
    groups = "one shared intrinsics group" if cfg["shared_intrinsics"] else "one intrinsics group per camera"
    config = {"workload": "%s: %d cameras / %d points / ~%d observations, %s, %s, TRIVIAL loss, default intrinsics mask "
                          "(FOCAL_LENGTH|RADIAL_DISTORTION free), use_inner_iterations=false" %
                          (args.workload, cfg["n_cam"], cfg["n_pt"], cfg["n_pt"] * cfg["obs_per_pt"], model_name, groups),
              "parallelism": ("points+observations sharded over %d GPU(s), cameras replicated; per PCG iteration the matvec kernel itself exchanges the partial sums over NVLink peer memory "
                               "(TBA_P2P=0: NCCL all-reduce), three NCCL all-reduces per LM iteration" % world) if world > 1 else "one GPU",
              "l2_policy": ("inputs larger than L2: the stored linearisation streamed by every kernel is %.2f GB at N=1 "
                            "(L2 = 0.126 GB), no flush needed" if cfg["n_pt"] * cfg["obs_per_pt"] * 160 > 2 * 126e6 * world else
                            "WARNING: the stored linearisation (%.2f GB at N=1) is not larger than L2 per GPU at this N: "
                            "kernel times are L2-assisted") % (cfg["n_pt"] * cfg["obs_per_pt"] * 160 / 1e9)}

    if args.impl == "reference":
        # the reference arm: Theia+Ceres cannot be built in this image (Ceres/Eigen/glog absent), so the CPU
        # restatement of its path is timed on the host cores; rank 0 only.  It runs -- and NAMES -- a bounded sample
        # workload (the full 20 M-observation scene would take ~20 min per run on the host); obs/s is normalised by size.
        if rank != 0:
            return 0
        pin_openmp()
        cb = cpu_baseline(K, W)
        ref_config = dict(config)
        ref_config["workload"] = sample_workload_text(cb["n_obs"])
        ref_config["parallelism"] = "OpenMP over points, %d threads bound one per physical core" % cb["cores"]
        ref_config["l2_policy"] = "CPU run"
        ref_config["gpu_arm_workload"] = config["workload"]
        line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "obs/s", "n_gpus": args.gpus, "steps": K,
                "warmup": W, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "config": ref_config, "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "obs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "lm_iters_per_s": cb["lm_iters_per_s"]}
        print(json.dumps(line))
        return 0

    import torch
    import torch.distributed as dist
    from theiasfm_b200 import engine

    if world > 1:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.cuda.set_device(local_rank)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    def sum_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t[0])

    nccl_id = None
    if world > 1:
        obj = [engine.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(obj, src=0)
        nccl_id = obj[0]
    micro = run_microbench(local_rank) if rank == 0 else None
    eng = engine.Engine(device=local_rank, rank=rank, world_size=world, nccl_id=nccl_id)

    full = synthetic.make_config(args.workload)
    n_obs_total = full.n_obs
    if world > 1:
        shard, _, _ = full.shard(rank, world)
        del full
    else:
        shard = full
    init = shard.copy()

    sampler = ClockSampler(local_rank)
    sampler.start()
    # ---- warm-up: W LM iterations, then restore the initial estimate
    eng.upload(shard, engine.default_options(**solver_kwargs(max(W, 1))))
    if W > 0:
        eng.minimize()
    eng.reset_parameters(init)
    # ---- timed: exactly K LM iterations on device-resident inputs.  Tolerances are zero, so a solve only stops early when it
    # reaches the fp64 floor of this scene (cost change exactly 0 after ~16 iterations); the remaining iterations then come
    # from further solves restarted at the initial estimate (each pays its own initial evaluation inside the timed region).
    eng.upload(shard, engine.default_options(**solver_kwargs(K)))  # same packing, K iterations
    eng.reset_parameters(init)
    eng.set_profiling(os.environ.get("TBA_BENCH_NOPROF") is None)  # (TBA_BENCH_NOPROF=1: experiment -- what do the stage events cost? no roofline then)
    barrier()
    tw0 = time.time()
    t0 = time.perf_counter()
    iters, dev_s, launches_local, pcg_total, solves, s, result = 0, 0.0, 0.0, 0, 0, None, None
    while iters < K:
        if solves > 0:
            eng.reset_parameters(init)
        eng.set_max_iterations(K - iters)
        si = eng.minimize()
        solves += 1
        got = si.num_iterations - 1
        if s is None:
            s = si
        iters += got
        dev_s += sum(it["iteration_time_in_seconds"] for it in si.iterations)
        launches_local += float(si.num_kernel_launches)
        pcg_total += int(si.num_linear_solver_iterations)
        if got <= 0:
            raise RuntimeError("a solve from the initial estimate ran no LM iteration (%d of %d done): %s" % (iters, K, si.message))
        if args.dump_outputs and solves == 1 and iters < K:
            result = init.copy()  # the restarts overwrite the first solve's result on the device (the copy is not device-timed)
            eng.download(result)
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop(tw0, time.time())
    prof = eng.profile()
    stages = eng.profile_stages()
    eng.set_profiling(False)
    if args.dump_outputs:
        if result is None:
            result = init.copy()
            eng.download(result)
        write_outputs(args.dump_outputs, result, s.costs)
    t_max = max_over_ranks(dev_s if dev_s > 0 else wall)  # device time of the iterations; the wall clock only if the engine reported none
    launches = sum_over_ranks(launches_local)
    note = None if solves == 1 else ("%d LM iterations timed as %d solves restarted from the initial estimate (the first stopped after %d: %s)"
                                     % (iters, solves, s.num_iterations - 1, s.message))
    value = n_obs_total * iters / t_max
    # ---- roofline of the dominant kernel (implicit-Schur matvec; DESIGN.md section 5)
    peak, peak_src = load_peaks()
    nj = prof["doubles_per_obs"]
    alg_bytes = prof["observations"] * (8 + 8 * nj) + prof["points"] * (80 + 8) + full_cam_bytes(shard)
    mv_ms = prof["matvec_ms"] / max(prof["matvec_launches"], 1)
    achieved = alg_bytes / (mv_ms * 1e-3) / 1e9 if mv_ms > 0 else 0.0
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and args.workload == "c3_10kcam" and world == 1:  # the ncu capture is of this exact launch shape
        with open(tpath) as f:
            traffic = json.load(f).get("k_schur_matvec_dram_bytes_per_launch")
    lin_ms = prof["linearize_ms"] / max(prof["linearize_launches"], 1)
    lin_bytes = prof["observations"] * (8 + 16 + 8 * nj + 16) + prof["points"] * (32 + 112) + shard.n_cam * (48 + 160 + 96)
    roofline = {"kernel": "k_schur_stream<IMASK,0> (implicit Schur-complement matvec, persistent streaming kernel, one launch per PCG iteration)", "bound": "hbm",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "peak_source": peak_src, "algorithmic_bytes_per_launch": alg_bytes, "avg_launch_ms": mv_ms,
                "launches_timed": prof["matvec_launches"], "share_of_step": prof["matvec_ms"] * 1e-3 / dev_s if dev_s > 0 else None,
                # the matvec issues 6 fp64 REDs and 1 48-byte gather per observation: floors from the measured rates
                "atomic_floor_ms": (6.0 * prof["observations"] / (micro["fp64_red_gops"] * 1e9) * 1e3) if micro else None,
                "gather_floor_ms": (prof["observations"] / (micro["gather48_grows"] * 1e9) * 1e3) if micro else None,
                "hbm_floor_ms": alg_bytes / (peak * 1e9) * 1e3,
                "linearize": {"avg_launch_ms": lin_ms, "algorithmic_bytes_per_launch": lin_bytes,
                              "achieved": lin_bytes / (lin_ms * 1e-3) / 1e9 if lin_ms > 0 else 0.0,
                              "frac": (lin_bytes / (lin_ms * 1e-3) / 1e9 / peak) if lin_ms > 0 else 0.0,
                              "share_of_step": prof["linearize_ms"] * 1e-3 / dev_s if dev_s > 0 else None,
                              # SURVEY 8d: the linearisation is the fp64-heavy kernel (about 650 flop / observation: residual +
                              # analytic Jacobian 450, block outer products 200): report it against the measured DFMA peak too
                              "fp64_tflops_estimate": (650.0 * prof["observations"] / (lin_ms * 1e-3) * 1e-12) if lin_ms > 0 else None,
                              "frac_of_measured_fp64": (650.0 * prof["observations"] / (lin_ms * 1e-3) * 1e-12 / micro["fp64_fma_tflops"])
                              if (lin_ms > 0 and micro and micro.get("fp64_fma_tflops")) else None}}
    # ---- e2e: the drop-in call with host buffers (pack + H2D + solve + D2H inside the timed region)
    e2e = None
    if not args.no_e2e:
        host = init.copy()
        barrier()
        t0 = time.perf_counter()
        se = eng.solve(host, engine.default_options(**solver_kwargs(K)))
        barrier()
        t_e2e = max_over_ranks(time.perf_counter() - t0)
        assert se.rc == 0, se.message
        e_iters = max(se.num_iterations - 1, 1)
        e2e = {"value": n_obs_total * e_iters / t_e2e, "unit": "obs/s", "h2d_bytes_per_step": sum_over_ranks(se.h2d_bytes) / e_iters,
               "d2h_bytes_per_step": sum_over_ranks(se.d2h_bytes) / e_iters, "seconds": t_e2e, "steps_run": e_iters,
               "host_pack_and_upload_seconds": max_over_ranks(se.setup_time_in_seconds), "final_cost": se.final_cost}
    cb = None
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        cb = cpu_baseline_subprocess(3)
    eng.close()
    experiments = None
    if world == 1 and rank == 0 and not args.no_experiments and not any(k in os.environ for k in SWITCHES):
        experiments = run_experiments(args.workload, K, local_rank)
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "obs/s", "n_gpus": world, "steps": iters, "warmup": W,
                "ms_per_step": 1e3 * t_max / iters, "steps_requested": K, "solves_in_timed_region": solves, "note": note, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": config, "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches),
                "roofline": roofline, "microbench": micro, "cpu_baseline": cb, "lm_iters_per_s": iters / t_max,
                # SURVEY 8d: observation passes = linearisations + PCG matvecs + step evaluations, all ranks' shards together
                "obs_passes_per_s": n_obs_total * (prof["linearize_launches"] + prof["matvec_launches"] + iters) / t_max,
                "pcg_iterations": pcg_total, "initial_cost": s.initial_cost, "final_cost": s.final_cost,
                "wall_seconds_timed_region": wall, "n_obs": n_obs_total,
                # per-stage device time (CUDA events on the engine stream inside the timed region), ms per LM iteration
                "stage_ms_per_step": {k: v["ms"] / iters for k, v in stages.items()},
                "experiment_switches": {k: os.environ[k] for k in SWITCHES if k in os.environ}}
        line["experiments"] = experiments
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


DUMP_POINTS = 1 << 18  # points written by --dump-outputs: a seeded sample of this many rows when the scene has more (8 MB)


def write_outputs(out_dir, p, costs):
    """--dump-outputs: the adjusted parameters a caller of the timed path downloads (cameras [n_cam, 6], intrinsics [n_group, 10],
    points [n_pt, 4], sampled to DUMP_POINTS sorted rows by a fixed seed) and the per-iteration costs of the solve."""
    os.makedirs(out_dir, exist_ok=True)
    pt = p.pt
    if len(pt) > DUMP_POINTS:
        pt = pt[np.sort(np.random.default_rng(0).choice(len(pt), DUMP_POINTS, replace=False))]
    for name, a in (("cameras", p.ext), ("intrinsics", p.intr), ("points", pt), ("costs", costs)):
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, np.float64))


def full_cam_bytes(p):
    return p.n_cam * 96 + p.n_group * 160


if __name__ == "__main__":
    sys.exit(main())
