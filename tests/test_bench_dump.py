"""`bench.py --dump-outputs DIR`: what the last timed step returned, as float32 / float64 .npy files of at most 64 MB.
CPU: the writer (types, the seeded server sample) and the argument checks.  GPU: a short run of config 2 whose dumped
pair records, winners, decisions and per-type totals equal the oracle's."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def _case(S, A, seed=1):
    rng = np.random.default_rng(seed)
    per_server = {"key": rng.integers(-1, A, S).astype(np.int32), "cost": rng.uniform(0, 1e3, S).astype(np.float32)}
    per_pair = {"replicas": rng.integers(0, 1 << 40, S * A).astype(np.int64), "feasible": rng.integers(0, 2, S * A).astype(np.uint8),
                "rho": rng.uniform(0, 1, S * A).astype(np.float32)}
    per_type = {"type_count": rng.integers(0, 1000, 3).astype(np.int64), "type_cost": rng.uniform(0, 1e4, 3).astype(np.float32)}
    return per_server, per_pair, per_type


def test_dump_writes_every_array_exactly(tmp_path):
    per_server, per_pair, per_type = _case(50, 4)
    bench.dump_outputs(str(tmp_path), per_server, per_pair, per_type, 4)
    got = _load(str(tmp_path))
    want = {**per_server, **per_pair, **per_type}
    assert sorted(got) == sorted(want)
    for k, a in want.items():
        assert got[k].dtype == (np.float32 if a.dtype == np.float32 else np.float64), k
        assert np.array_equal(got[k], a), k


def test_dump_samples_servers_within_the_limit(tmp_path):
    S, A, limit = 20_000, 8, 400_000
    per_server, per_pair, per_type = _case(S, A)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), per_server, per_pair, per_type, A, limit=limit)
        assert sum(os.path.getsize(tmp_path / run / f) for f in os.listdir(tmp_path / run)) <= limit
    got, again = _load(str(tmp_path / "a")), _load(str(tmp_path / "b"))
    assert sorted(got) == sorted(again) and all(np.array_equal(got[k], again[k]) for k in got)
    srv = got["sampled_servers"].astype(np.int64)
    assert len(srv) > 1000 and np.all(np.diff(srv) > 0) and srv[-1] < S
    rows = (srv[:, None] * A + np.arange(A)).ravel()
    for k, a in per_server.items():
        assert np.array_equal(got[k], a[srv]), k
    for k, a in per_pair.items():
        assert np.array_equal(got[k], a[rows]), k
    for k, a in per_type.items():
        assert np.array_equal(got[k], a), k


@pytest.mark.parametrize("extra", [["--impl", "reference", "--dump-outputs", "x"], ["--steps", "0"]])
def test_bench_rejects_bad_arguments(extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert out.returncode == 2 and out.stdout.strip() == "", out.stderr[-2000:]


@pytest.mark.gpu
def test_dumped_outputs_equal_the_oracle(wva, oracle, tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "2", "--steps", "2", "--warmup", "3",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.strip()][-1])
    assert line["steps"] == 2 and line["e2e"]["steps"] == 2
    files = os.listdir(tmp_path)
    assert sum(os.path.getsize(tmp_path / f) for f in files) <= 64_000_000
    got = _load(str(tmp_path))
    assert "sampled_servers" not in got and all(a.dtype in (np.float32, np.float64) for a in got.values())
    abi = wva.abi
    img, c = wva.synth.baseline_config(2)

    def allocs(prefix):
        a = abi.AllocArrays(len(got[prefix + "acc"]))
        for n, dt in abi.ALLOC_FIELDS:
            getattr(a, n)[:] = got[prefix + n].astype(dt)
        return a

    o_pairs, o_feas, _ = oracle.analyze_pairs(img, threads=oracle.hardware_threads())
    assert np.array_equal(got["pairs_feasible"], o_feas)
    ok, field = allocs("pairs_").equal_bits(o_pairs)
    assert ok, field
    o_acc, o_chosen = oracle.solve(img, o_pairs, o_feas, unlimited=True)
    assert np.array_equal(got["chosen_key"], o_acc)
    ok, field = allocs("chosen_").equal_bits(o_chosen)
    assert ok, field
    o_count, o_cost = oracle.allocate_by_type(img, o_acc, o_chosen)
    assert np.array_equal(got["type_count"], o_count) and got["type_cost"].tobytes() == o_cost.tobytes()
    o_best, _, _, _ = oracle.analyze_grid(img, c["r_max"], c["b_max"], want_cube=False, threads=oracle.hardware_threads())
    best = np.zeros(img.S, dtype=abi.GRID_BEST_DTYPE)
    for n in best.dtype.names:
        best[n] = got["winner_" + n]
    assert best.tobytes() == o_best.tobytes()
