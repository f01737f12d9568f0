"""bench.py's reference arm runs here (CPU only): one JSON line with the contract's keys, the CPU path timed on a bounded
sample, nothing from the GPU arm touched.  (The GPU arm's line is checked on the B200 box by test_gpu_parity / the driver.)"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*extra):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-pairs", "1", *extra], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr
    lines = [l for l in p.stdout.strip().splitlines() if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def test_reference_arm_line_has_the_contract_keys():
    d = _run()
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "pairs/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["gpu_launches"] == 0 and d["dtype"] == "u8" and d["data"] == "synthetic"
    assert d["config"]["workload"] == "c2_1280x720_orb5000" and "model" not in d["config"]
    assert d["e2e"] == {"value": d["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    # same config as the GPU arm (the bounded sample is stated separately) and --warmup honoured as given
    assert d["config"]["pairs_per_gpu_per_step"] == 96 and cb["sample_pairs"] == 1 and d["warmup"] == 0 and d["steps"] == 1


def test_reference_arm_sharded_c5_workload_is_selectable():
    d = _run("--workload", "c5_1024_sharded")
    assert d["config"]["workload"] == "c5_1024_sharded" and d["config"]["global_pairs_per_step"] == 1024
    assert d["config"]["width"] == 1920 and d["config"]["n_features"] == 10000


def test_reference_arm_other_ranks_print_nothing():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_dump_outputs_is_bounded_padded_and_repeatable(tmp_path):
    """--dump-outputs: float files only, within the budget at the largest batch shape, rows past each count zeroed, the counts
    and the sampled pairs' lists equal to what the batch held, the same files from the same results."""
    import numpy as np
    import bench
    from front_end_b200 import KPOINT, MATCH
    P, cap = 96, 8192
    rng = np.random.default_rng(3)
    res = dict(kps=np.zeros((2 * P, cap), KPOINT), desc=rng.integers(0, 256, (2 * P, cap, 32), dtype=np.uint8),
               n_kps=rng.integers(0, cap + 100, 2 * P).astype(np.int32), matches_a=np.zeros((P, cap), MATCH),
               n_a=rng.integers(0, cap, P).astype(np.int32), matches_b=np.zeros((P, cap), MATCH), n_b=rng.integers(0, cap, P).astype(np.int32))
    for k in KPOINT.names:
        res["kps"][k] = rng.integers(-1, 2000, (2 * P, cap))
    for k in ("matches_a", "matches_b"):
        for f in MATCH.names:
            res[k][f] = rng.integers(0, cap, (P, cap))
    tracks = (np.zeros((P, cap), MATCH), rng.integers(0, cap, P).astype(np.int32))
    tracks[0]["trainIdx"] = rng.integers(0, cap, (P, cap))
    a = bench.dump_outputs(str(tmp_path / "a"), res, cap, tracks)
    b = bench.dump_outputs(str(tmp_path / "b"), res, cap, tracks)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(k + ".npy" for k in a) and sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64_000_000
    for f in files:
        x = np.load(tmp_path / "a" / f)
        assert x.dtype in (np.float32, np.float64) and np.array_equal(x, np.load(tmp_path / "b" / f)), f
    pairs = a["pairs"].astype(int)
    assert len(pairs) >= 8 and len(set(pairs)) == len(pairs) and pairs.max() < P - 1
    assert np.array_equal(a["n_kps"], res["n_kps"]) and np.array_equal(a["n_b"], res["n_b"])
    for s, p in enumerate(pairs):
        for e in range(2):
            m = min(int(res["n_kps"][2 * p + e]), cap)
            assert np.array_equal(a["desc"][s, e, :m], res["desc"][2 * p + e, :m]) and not a["desc"][s, e, m:].any()
            assert np.array_equal(a["kps"][s, e, :m, 5], res["kps"]["octave"][2 * p + e, :m]) and not a["kps"][s, e, m:].any()
        m = int(res["n_a"][p])
        assert np.array_equal(a["matches_a"][s, :m, 1], res["matches_a"]["trainIdx"][p, :m]) and not a["matches_a"][s, m:].any()
        m = int(tracks[1][p])
        assert np.array_equal(a["tracks"][s, :m, 1], tracks[0]["trainIdx"][p, :m]) and not a["tracks"][s, m:].any()


def test_dump_outputs_needs_the_gpu_arm():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", "x"],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert p.returncode == 2 and "--dump-outputs" in p.stderr


def test_reference_arm_surf_workload_is_bounded_and_says_what_it_scaled():
    """BASELINE config 3 on the CPU: the numpy SURF restatement is timed on a keypoint sample and scaled (a full pair would take
    ~25 s); the line says so."""
    d = _run("--workload", "c3_1280x720_surf128")
    cb = d["cpu_baseline"]
    assert d["config"]["workload"] == "c3_1280x720_surf128" and cb["extrapolated"] is True and "SCALED" in cb["sample"]
    assert 0 < d["value"] < 5 and cb["kind"] == "port"
