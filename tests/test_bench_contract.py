"""bench.py contract on the CPU: the reference arm (the only arm that runs without a GPU) prints exactly ONE JSON line
on stdout with the keys the driver reads; non-zero ranks of a torchrun launch stay silent; the B200 arm fails loudly
(no JSON, non-zero exit) when there is no CUDA device -- there is no CPU fallback to fall into."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, cwd=ROOT, env=e, timeout=600)


def test_reference_arm_prints_one_json_line():
    r = _run(["--impl", "reference", "--log-n", "10", "--steps", "2", "--warmup", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "GB/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["steps"] == 2 and d["gpu_launches"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def test_reference_arm_other_ranks_are_silent():
    r = _run(["--impl", "reference", "--gpus", "2", "--log-n", "10", "--steps", "1", "--warmup", "1"], env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_b200_arm_without_a_gpu_fails_loudly():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = _run(["--steps", "1", "--warmup", "1", "--no-cpu-baseline", "--no-e2e"], env={"CUDA_VISIBLE_DEVICES": ""})
    assert r.returncode != 0
    assert r.stdout.strip() == ""                      # nothing that could be mistaken for a measurement


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_dump_sample_is_fixed_and_bounded():
    """--dump-outputs writes the same parity blocks on every run of the same shape, at most 64 MiB of float64."""
    import numpy as np
    bench = _bench_module()
    assert np.array_equal(bench.dump_rows(64, 1024), np.arange(64))
    for log_n, S in ((19, 1024), (20, 1024), (16, 1 << 20)):
        rows = bench.dump_rows(1 << log_n, S)
        assert np.array_equal(rows, bench.dump_rows(1 << log_n, S))
        assert 1 <= len(rows) <= bench.DUMP_ROWS and len(rows) * S * 8 <= 64 << 20
        assert np.all(np.diff(rows) > 0) and rows[0] >= 0 and rows[-1] < 1 << log_n


@pytest.mark.gpu
def test_dump_outputs_is_the_parity_of_the_last_timed_step(tmp_path, oracle):
    """The timed path encodes its array in place: after 3 warm-up and 2 timed steps it holds fill A encoded five times."""
    import numpy as np
    import oracle_lib as ol
    r = _run(["--log-n", "11", "--steps", "2", "--warmup", "3", "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(tmp_path)])
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 2
    want = ol.fill_A(oracle, 1 << 11, 1024)
    for _ in range(5):
        want = ol.o_encode(oracle, want)
    got = np.load(tmp_path / "parity.npy")
    assert got.dtype == np.float64
    assert np.array_equal(got, want[_bench_module().dump_rows(1 << 11, 1024)])


def test_dump_outputs_is_refused_by_the_reference_arm(tmp_path):
    r = _run(["--impl", "reference", "--log-n", "10", "--steps", "1", "--warmup", "1", "--dump-outputs", str(tmp_path)])
    assert r.returncode != 0 and r.stdout.strip() == "" and "--dump-outputs" in r.stderr


def test_fill_a_rows_is_the_reference_fill_dealt_cyclically():
    """bench.py fills every rank's shard directly (global block l*G + rank = local row l of data0[i] = i % P, RS.cpp:28-29)."""
    import numpy as np
    import torch
    bench = _bench_module()
    N, S, G = 64, 12, 4
    full = (np.arange(N * S, dtype=np.uint64) % bench.P).astype(np.uint32).reshape(N, S)
    for r in range(G):
        got = bench.fill_a_rows(torch, "cpu", r, G, N // G, S).numpy().view(np.uint32)
        assert np.array_equal(got, full[r::G])
    assert bench.GOLDEN_PARITY_HASH_FILL_A[(19, 1024)] == 4272226309       # SURVEY 8c
    class A: log_n = 19; block_bytes = 4096
    assert bench.check_golden(A, 4272226309, "x")["golden_match"] is True
    try:
        bench.check_golden(A, 1, "x")
        assert False, "a wrong hash must abort the run"
    except SystemExit as e:
        assert "PARITY FAILURE" in str(e)
