"""The driver's bench contract, CPU side: `bench.py --impl reference` (the CPU oracle arm) prints ONE JSON line with the
keys the driver reads, on the smoke-sized workload; under torchrun every rank but 0 exits without work."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env=None, steps=2, extra_args=()):
    env = dict(os.environ)
    env.update(extra_env or {})
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "small", "--steps", str(steps), "--warmup", "0",
                        *extra_args], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return [l for l in r.stdout.splitlines() if l.strip()]


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "LM iterations/sec" and d["unit"] == "it/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 0 and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["config"]["workload"] == "small" and d["dtype"] == "f64" and d["data"] == "synthetic" and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_without_output():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []


def test_reference_arm_ignores_omp_num_threads_of_torchrun():
    # torch.distributed.run exports OMP_NUM_THREADS=1 to its workers: the CPU arm must still use every core it may run
    # on (round 1: the 30 M-observation reference run was single threaded under torchrun and timed out at N = 2, 4, 8)
    lines = _run({"OMP_NUM_THREADS": "1", "RANK": "0", "WORLD_SIZE": "2", "LOCAL_RANK": "0"})
    assert len(lines) == 1
    d = json.loads(lines[0])
    want = len(os.sched_getaffinity(0))
    assert d["cpu_baseline"]["cores"] == want
    assert d["cpu_baseline"]["final_cost"] > 0


def test_both_arms_print_the_same_config_keys():
    # the driver compares the two `config` objects: same keys (values are checked on the GPU box where both arms run)
    import bench
    ref = json.loads(_run()[0])["config"]
    job = bench.Job("small", 0, 1)
    ours = bench.config_of(job, "small", 1, 2, 300)
    assert sorted(ref) == sorted(ours)
    assert all(ref[k] == ours[k] for k in ref if k not in ("rcs_solver", "rcs_dim"))


def test_reference_arm_dumps_the_last_step_of_the_timed_solves(tmp_path, oracle):
    """--dump-outputs: 7 steps are one solve of 5 LM iterations and one of 2; the dump is the parameter vector and the rows of
    that last solve, the same as a 2-iteration oracle solve from the workload's start."""
    import numpy as np
    import bench
    out = tmp_path / "dump"
    d = json.loads(_run(steps=7, extra_args=("--dump-outputs", str(out)))[0])
    assert d["steps"] == 7
    arrays = {p.stem: np.load(p) for p in out.glob("*.npy")}
    assert sorted(arrays) == sorted(("parameters", "final_cost") + bench.DUMP_ROW_FIELDS)
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert sum(p.stat().st_size for p in out.glob("*.npy")) <= 64 << 20
    job = bench.Job("small", 0, 1)
    o = oracle.default_options()
    o.function_tolerance = 0.0; o.parameter_tolerance = 0.0; o.gradient_tolerance = 0.0; o.max_num_iterations = 2
    x, s, rows = job.oracle_solve(oracle, o, bench.host_threads())
    assert arrays["parameters"].shape == x.shape and np.abs(arrays["parameters"] - x).max() < 1e-9
    assert arrays["cost"].shape == (3,) and np.allclose(arrays["cost"], [r["cost"] for r in rows], rtol=1e-12, atol=0)
    assert np.isclose(arrays["final_cost"][0], s.final_cost, rtol=1e-12, atol=0)


def test_dump_of_a_large_parameter_vector_is_a_fixed_sample(tmp_path):
    import numpy as np
    import bench
    x = np.arange(bench.DUMP_MAX_FULL + 5, dtype=np.float64) * 0.5
    rows = [{k: float(i) for k in bench.DUMP_ROW_FIELDS} for i in range(3)]

    class Summary:
        final_cost = 2.0
    for sub in ("a", "b"):
        bench.dump_outputs(str(tmp_path / sub), x, Summary, rows)
    a, b = (np.load(tmp_path / sub / "parameters.npy") for sub in ("a", "b"))
    ia = np.load(tmp_path / "a" / "parameters_index.npy")
    assert a.dtype == ia.dtype == np.float64 and a.shape == ia.shape == (bench.DUMP_SAMPLE,)
    assert np.array_equal(a, b) and np.array_equal(a, 0.5 * ia) and np.all(np.diff(ia) > 0)
    assert sum(p.stat().st_size for p in (tmp_path / "a").glob("*.npy")) <= 64 << 20


def test_committed_traffic_numbers_belong_to_this_tree():
    """roofline.traffic comes from profiles/traffic.json; bench.py only uses an entry whose kernel_source_hash is the hash of
    the csrc/ files it runs.  The committed entries of the default workload must be the ones of the committed kernels."""
    import json
    import bench
    with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
        t = json.load(f)
    h = bench.kernel_source_hash()
    entries = t[bench.DEFAULT_WORKLOAD]
    assert entries and all(e.get("kernel_source_hash") == h for e in entries.values()), (h, entries)
