"""bench.py is the driver's contract and cannot run its real path without a GPU: its CPU self-test mode
(GLLM_BENCH_CPU_SELFTEST=1: tiny random model, host clocks) executes the same control flow — argument handling,
per-pass prompt sets, warm-up, both timed regions, statistics, JSON line, orderly teardown — so a typo in the script
is caught here and not at round end."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra, env_extra=None, nproc=1, port=29951):
    env = dict(os.environ, GLLM_BENCH_CPU_SELFTEST="1", GLLM_B200_LOG="WARNING", PYTHONPATH=ROOT)
    env.update(env_extra or {})
    base = [os.path.join(ROOT, "bench.py"), "--gpus", str(nproc), "--steps", "2", "--warmup", "1", "--num-prompts", "6",
            "--maxp", "256", "--maxd", "16"] + extra
    if nproc == 1:
        cmd = [sys.executable] + base
    else:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
               "--master-addr", "127.0.0.1", "--master-port", str(port)] + base
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-1500:] + r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, r.stdout[-2000:]
    return json.loads(lines[0])


def test_bench_contract_single_process():
    d = _run([])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "latency"):
        assert key in d, key
    assert d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["value"] > 0 and d["e2e"]["value"] > 0
    assert d["config"]["num_prompts"] == 6 and d["config"]["output_tokens_per_step"] > 0
    assert d["e2e"]["h2d_bytes_per_step"] >= 0 and "SELF-TEST" in d["data"]
    kinds = d["config"]["device_ms_by_step_kind"]
    assert kinds == {} or all(len(v) == 3 for v in kinds.values())


def test_bench_dump_outputs_are_reproducible(tmp_path):
    """`--dump-outputs DIR`: the generated token ids of the last timed pass, as float .npy files, identical when the
    same arguments run again."""
    import numpy as np
    runs = []
    for name in ("a", "b"):
        d = _run(["--dump-outputs", str(tmp_path / name)])
        runs.append({k: np.load(tmp_path / name / f"{k}.npy")
                     for k in ("output_token_ids", "output_lens", "request_index")})
    a, b = runs
    for k in a:
        assert a[k].dtype == np.float64 and np.array_equal(a[k], b[k]), k
    assert a["request_index"].tolist() == list(range(6)) and a["output_lens"].sum() == a["output_token_ids"].size
    assert a["output_token_ids"].size == d["config"]["output_tokens_per_step"]


def test_bench_contract_two_ranks_and_named_config():
    d = _run(["--config", "mixtral-8x7b-ep"], nproc=2)
    assert d["n_gpus"] == 2 and d["config"]["parallelism"] == "tp2" and d["value"] > 0
    assert "Mixtral" in d["config"]["model"] and d["config"]["named_config"] == "mixtral-8x7b-ep"


def test_bench_reference_arm_reports_unavailable_without_a_gpu():
    env = dict(os.environ, PYTHONPATH=ROOT, GLLM_REF_TIMEOUT="300")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    assert r.returncode == 0
    line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1]
    d = json.loads(line)
    assert d["impl"] == "reference" and ("unavailable" in d or d.get("value", 0) > 0)


def test_bench_contract_pipeline_config():
    d = _run(["--config", "llama3-70b-pp4tp2"], nproc=2, port=29961)
    assert d["config"]["parallelism"] == "tp1pp2" and d["config"]["schedule_method"] == "token_throttling"
    assert d["value"] > 0
