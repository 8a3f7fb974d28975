"""bench.py and __graft_entry__.smoke() need a GPU; their Python logic (argument handling, the JSON line and every derived field,
the oracle comparison of smoke) is exercised here on the CPU by running them in a subprocess against tests/mock_engine_py.py, a
stand-in for the engine answered by the oracle.  Says nothing about the CUDA engine or about performance."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

PRELUDE = """
import sys
sys.path.insert(0, %r); sys.path.insert(0, %r)
import mock_engine_py; mock_engine_py.install()
import torch
torch.cuda.set_device = lambda d: None
torch.cuda.synchronize = lambda *a, **k: None
""" % (os.path.join(ROOT, "tests"), ROOT)


def _run(code):
    return subprocess.run([sys.executable, "-c", PRELUDE + code], capture_output=True, text=True, timeout=600, cwd=ROOT)


def test_bench_line_has_every_contract_field():
    out = _run("""
import bench
bench.run_microbench = lambda d: {"fp64_fma_tflops": 37.0, "fp64_red_gops": 200.0, "gather48_grows": 50.0, "how": "mock"}
sys.argv = ["bench.py", "--workload", "c1_50cam", "--steps", "2", "--warmup", "1", "--no-cpu-baseline"]
bench.run_experiments = lambda w, k, d: {"default": {"rc": 0}}
bench.main()
""")
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["experiments"] == {"default": {"rc": 0}} and set(line["stage_ms_per_step"]) >= {"matvec", "linearize", "precond_ext", "rhs"}
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"):
        assert key in line, key
    assert line["unit"] == "obs/s" and line["dtype"] == "f64" and line["data"] == "synthetic" and "workload" in line["config"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(line["roofline"])
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(line["e2e"])
    assert line["steps"] == 2 and line["steps_requested"] == 2 and line["value"] > 0 and line["obs_passes_per_s"] >= line["value"]


def _bench_line(*argv):
    out = _run("""
import bench
bench.run_microbench = lambda d: None
sys.argv = ["bench.py", "--workload", "c1_50cam", "--warmup", "1", "--no-cpu-baseline", "--no-e2e", "--no-experiments"] + %r
bench.main()
""" % list(argv))
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_bench_runs_exactly_the_requested_steps():
    """Each solve of this scene stops at its fp64 floor after a few dozen LM iterations at most; the rest of the 400 come from
    solves restarted at the initial estimate, as many as it takes."""
    line = _bench_line("--steps", "400")
    assert line["steps"] == line["steps_requested"] == 400 and line["solves_in_timed_region"] > 8


def test_bench_dump_outputs(tmp_path):
    """--dump-outputs writes the timed solve's result; a second run with the same arguments starts from the same inputs."""
    dumps = []
    for run in ("a", "b"):
        assert _bench_line("--steps", "3", "--dump-outputs", str(tmp_path / run))["steps"] == 3
        dumps.append({f.stem: np.load(f) for f in (tmp_path / run).iterdir()})
    a, b = dumps
    assert {k: v.shape for k, v in a.items()} == {"cameras": (50, 6), "intrinsics": (1, 10), "points": (5000, 4), "costs": (4,)}
    for k in a:
        assert a[k].dtype == np.float64 and np.allclose(a[k], b[k], rtol=1e-12, atol=0), k
    assert a["costs"][3] < a["costs"][0]


def test_dump_outputs_of_the_largest_scene_stay_under_64_mb(tmp_path):
    """c3_10kcam: 2 M points (64 MB of float64 alone) are written as a fixed, sorted sample."""
    import bench

    class P:
        ext, intr, pt = np.zeros((10_000, 6)), np.zeros((1, 10)), np.arange(8.0 * 10 ** 6).reshape(-1, 4)
    bench.write_outputs(str(tmp_path / "a"), P, np.ones(21))
    bench.write_outputs(str(tmp_path / "b"), P, np.ones(21))
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64 << 20
    pts = np.load(tmp_path / "a" / "points.npy")
    assert pts.shape == (bench.DUMP_POINTS, 4) and np.all(np.diff(pts[:, 0]) > 0) and np.all(pts[:, 0] % 4 == 0)
    assert np.array_equal(pts, np.load(tmp_path / "b" / "points.npy"))


def test_smoke_logic():
    out = _run("import __graft_entry__ as g\ng.smoke()\n")
    assert out.returncode == 0, out.stderr[-2000:]
    assert "smoke ok" in out.stdout


def test_bench_experiments_child_logic():
    """The diagnostic pass over the experiment switches (bench.py --experiments-child): one JSON line per variant."""
    out = _run("""
import bench, os, subprocess
# the matcher sample runs through the SIMT-emulation build of the matcher library (tests/emu), shrunk to 48 descriptors per image
emu = os.path.join(%r, "tests", "emu")
subprocess.check_call(["make", "-C", emu, "libtheia_matcher_b200_emu.so"], stdout=subprocess.DEVNULL)
from theiasfm_b200 import matcher
matcher.LIB_PATH = os.path.join(emu, "libtheia_matcher_b200_emu.so")
os.environ["TBA_BENCH_MATCHER_N"] = "48"
bench.experiments_child("c1_50cam", 2, 0)
""" % ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [json.loads(ln) for ln in out.stdout.strip().splitlines() if ln.startswith("{")]
    assert [d["variant"] for d in lines] == [v[0] for v in __import__("bench").VARIANTS] + ["matcher_sample"]
    m = lines.pop()
    assert "error" not in m and m["rc"] == 0 and m["pairs"] == 6 and m["matches"] > 0, m
    for d in lines:
        assert "error" not in d, d
        assert d["rc"] == 0 and d["steps_run"] == 2
        assert d["variant"].startswith("ablate") or d["max_rel_cost_diff_vs_default"] <= 1e-12
        assert set(d["stage_ms_per_step"]) >= {"matvec", "linearize", "precond_ext", "precond_intr", "rhs", "backsub", "candidate_cost"}


def test_bench_experiments_parent_survives_a_failing_child(monkeypatch):
    """Without a GPU the real child cannot create an engine: every variant reports its error (or the child dies), the parent
    returns a dictionary either way and never raises.  The child inherits an empty CUDA_VISIBLE_DEVICES, so it sees no GPU on
    a machine that has one too."""
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    sys.path.insert(0, ROOT)
    import bench
    res = bench.run_experiments("c1_50cam", 1, 0, timeout=240)
    assert isinstance(res, dict) and res
    assert all(("error" in v or v.get("rc") != 0) for k, v in res.items() if k != "note") or "note" in res


def test_bench_main_and_experiments_child_against_the_emulated_engine(tmp_path):
    """The same two entry points through the REAL ctypes binding and the real engine code (tests/emu SIMT-emulation build) instead of the
    mock: catches attribute / signature drift between engine.py and what bench.py expects (it did: minimize()'s summary had no rc)."""
    emu = os.path.join(ROOT, "tests", "emu")
    subprocess.check_call(["make", "-C", emu], stdout=subprocess.DEVNULL)
    code = """
import sys, os, json
sys.path.insert(0, %r)
import torch
torch.cuda.set_device = lambda d: None
torch.cuda.synchronize = lambda *a, **k: None
from theiasfm_b200 import engine, matcher
engine.LIB_PATH = os.path.join(%r, "libtheia_ba_b200_emu.so"); engine._LIB = None
matcher.LIB_PATH = os.path.join(%r, "libtheia_matcher_b200_emu.so"); matcher._LIB = None
os.environ["TBA_BENCH_MATCHER_N"] = "32"
import bench
bench.run_microbench = lambda d: None
bench.run_experiments = lambda w, k, d: {"skipped": True}
sys.argv = ["bench.py", "--workload", "c1_50cam", "--steps", "1", "--warmup", "1", "--no-cpu-baseline", "--no-e2e", "--dump-outputs", %r]
bench.main()
bench.experiments_child("c1_50cam", 1, 0)
""" % (ROOT, emu, emu, str(tmp_path))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [json.loads(ln) for ln in out.stdout.strip().splitlines() if ln.startswith("{")]
    main, child = lines[0], lines[1:]
    assert np.load(tmp_path / "points.npy").shape == (5000, 4) and np.load(tmp_path / "costs.npy").shape == (2,)
    assert main["steps"] == 1 and main["gpu_launches"] > 0 and set(main["stage_ms_per_step"]) == set(__import__("bench").VARIANTS and
                                                                                                      ("matvec", "linearize", "precond_ext", "precond_intr", "rhs", "backsub", "candidate_cost", "prepare_fused"))
    assert [d["variant"] for d in child] == [v[0] for v in __import__("bench").VARIANTS] + ["matcher_sample"]
    for d in child:
        assert "error" not in d and d["rc"] == 0, d
    assert all(d["max_rel_cost_diff_vs_default"] <= 1e-9 for d in child[:-1] if not d["variant"].startswith("ablate"))


def test_smoke_against_the_emulated_engine():
    emu = os.path.join(ROOT, "tests", "emu")
    subprocess.check_call(["make", "-C", emu], stdout=subprocess.DEVNULL)
    code = """
import sys, os
sys.path.insert(0, %r)
from theiasfm_b200 import engine
engine.LIB_PATH = os.path.join(%r, "libtheia_ba_b200_emu.so"); engine._LIB = None
import __graft_entry__ as g
g.smoke()
""" % (ROOT, emu)
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0 and "smoke ok" in out.stdout, out.stderr[-2000:]
