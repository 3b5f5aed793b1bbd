#!/usr/bin/env python
"""Headline benchmark: offline serving throughput (output tokens/s) of Qwen3-8B bf16 with TP=N on N
B200s, on synthetic ShareGPT-shaped requests with random-init weights (BASELINE.json metric;
workload definition = the reference's benchmarks/benchmark_throughput.py: all requests submitted at
t=0, prompt <= 1024, prompt+output <= 2048, greedy, ignore_eos).

One *step* = one complete pass over the request set (`--num-prompts` requests, all prompt and output
tokens) through the engine's public API `LLM.generate(tokens=..., output_lens=...)`: continuous
batching, chunked prefill, paged KV, CUDA-graph decode, sampling, with the per-iteration H2D copy of
the batch arrays from pinned memory and the D2H read of the sampled tokens.

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 \
        --master-port 29500 bench.py --gpus 8 --steps 3 --warmup 3

Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


# BASELINE.json configurations: model preset, pipeline stages (tp = gpus / pp), schedule policy, metric label
CONFIGS = {
    "qwen3-8b-tp": dict(model="qwen3-8b", pp=1, method="chunked_prefill", label="Qwen3-8B TP"),
    "mixtral-8x7b-ep": dict(model="mixtral-8x7b", pp=1, method="chunked_prefill", label="Mixtral-8x7B EP"),
    "llama3-70b-pp4tp2": dict(model="llama-3-70b", pp=4, method="token_throttling",
                              label="Llama-3-70B PP4xTP2 token-throttled"),
    "deepseek-v3-fp8-ep": dict(model="deepseek-v3", pp=1, method="chunked_prefill",
                               label="DeepSeek-V3 fp8 block-scaled EP"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3, help="timed passes over the request set")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="preset:qwen3-8b")
    ap.add_argument("--num-prompts", type=int, default=1000,
                    help="the reference harness default (benchmarks/benchmark_throughput.py:359)")
    ap.add_argument("--maxp", type=int, default=4096)
    ap.add_argument("--maxd", type=int, default=1024)
    ap.add_argument("--max-cuda-graph-bs", type=int, default=512)
    ap.add_argument("--tp-mode", default="fused", choices=["fused", "nccl"])
    ap.add_argument("--schedule-method", default="chunked_prefill")
    ap.add_argument("--pp", type=int, default=1)
    ap.add_argument("--config", default="qwen3-8b-tp", choices=sorted(CONFIGS),
                    help="named BASELINE.json configuration (model + parallel layout + schedule policy)")
    ap.add_argument("--layers", type=int, default=0, help="override num_hidden_layers (0 = the model's own); a "
                    "reduced depth is reported in `config.model` and is NOT the named model")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--async-schedule", action=argparse.BooleanOptionalAction, default=True,
                    help="lookahead decode scheduling (engine default; --no-async-schedule for the synchronous loop)")
    ap.add_argument("--disable-cuda-graph", action="store_true", help="debugging: every step runs eagerly")
    ap.add_argument("--num-gpu-pages", type=int, default=None, help="debugging: fixed KV pool size (pages)")
    ap.add_argument("--fixed-prompts", action="store_true",
                    help="re-use the same token ids in every pass (with prefix caching the prompts of later passes "
                         "would then be served from the cache: NOT the benchmark; for debugging only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed passes, write what the last pass returned (generated token ids) as "
                         "DIR/*.npy, so that two builds can be compared output for output")
    return ap.parse_args()


def reference_arm(args):
    """Run the unmodified reference (baseline/install_reference.sh -> baseline/_ref) through its own public API in
    a subprocess (baseline/run_reference.py) and forward its JSON line. The reference pins vLLM 0.11 / torch 2.8 /
    transformers < 5, this image has vLLM 0.22 / torch 2.11 / transformers 5: if its native ops or imports do not
    line up on the box, the arm reports {"impl": "reference", "unavailable": <why>} and exits 0 (DESIGN.md)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return 0          # the reference spawns its own per-GPU workers: only one front-end process
    root = os.path.dirname(os.path.abspath(__file__))
    ref_root = os.path.join(root, "baseline", "_ref")

    def unavailable(why):
        print(json.dumps({"impl": "reference", "unavailable": " ".join(str(why).split())[:600]}), flush=True)
        return 0

    if not os.path.isfile(os.path.join(ref_root, "gllm", "llm_engine.py")):
        return unavailable("baseline/_ref is not populated (run baseline/install_reference.sh; the reference's "
                           "setup.py needs a vLLM wheel for its native kernels, see DESIGN.md)")
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "TORCHELASTIC_USE_AGENT_STORE",
              "GROUP_RANK", "ROLE_RANK", "LOCAL_WORLD_SIZE", "TORCHELASTIC_RUN_ID", "OMP_NUM_THREADS"):
        env.pop(k, None)  # the reference does its own rendezvous
    env["PYTHONPATH"] = os.pathsep.join([ref_root, os.path.join(root, "baseline", "shims"),
                                         env.get("PYTHONPATH", "")])
    try:
        import importlib.util
        vdir = os.path.dirname(importlib.util.find_spec("vllm").origin)
        stable = os.path.join(vdir, "_C_stable_libtorch.abi3.so")
        if os.path.exists(stable):
            env["GLLM_REF_PRELOAD_LIBS"] = stable
        env["GLLM_REF_ALIAS_VLLM"] = "1"
    except Exception:  # noqa: BLE001
        pass
    cmd = [sys.executable, os.path.join(root, "baseline", "run_reference.py"), "--gpus", str(args.gpus),
           "--steps", str(args.steps), "--warmup", str(args.warmup), "--num-prompts", str(args.num_prompts),
           "--maxp", str(args.maxp), "--maxd", str(args.maxd), "--max-cuda-graph-bs", str(args.max_cuda_graph_bs),
           "--seed", str(args.seed)]
    limit = int(os.environ.get("GLLM_REF_TIMEOUT", "1650"))
    env.setdefault("GLLM_REF_BUDGET_S", str(limit - 200))   # engine start-up (graph capture) ~80-120 s   # run_reference.py stops timing new passes after this
    try:
        # own process group: on a timeout the reference's spawned workers are taken down with the front-end
        proc = subprocess.Popen(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                                start_new_session=True)
        import signal
        timed_out = False
        try:
            out, err = proc.communicate(timeout=limit)
        except subprocess.TimeoutExpired:
            timed_out = True
        finally:
            try:       # always: worker processes the reference spawned must not keep GPU memory after the arm
                os.killpg(proc.pid, signal.SIGKILL)
            except (ProcessLookupError, PermissionError):
                pass
        if timed_out:
            proc.communicate()
            return unavailable(f"reference run exceeded {limit}s")
    except Exception as e:  # noqa: BLE001
        return unavailable(f"could not launch the reference: {e!r}")
    for line in reversed(out.splitlines()):
        if line.startswith("{") and '"impl": "reference"' in line:
            print(line)
            return 0
    # the reference's front-end only `sys.exit()`s when a worker died: the worker's traceback is further up
    lines = [ln for ln in (err + "\n" + out).replace("\r", "\n").splitlines() if ln.strip() and "it/s]" not in ln]
    sys.stderr.write("---- reference arm failed; last 60 lines of its output ----\n" + "\n".join(lines[-60:]) + "\n")
    errs = [ln for ln in lines if "Error" in ln or "error" in ln]
    tail = (errs or lines or ["no output"])[-1]
    return unavailable(f"reference failed on this image (vLLM 0.22 / torch 2.11 / transformers 5 instead of its "
                       f"pinned 0.11 / 2.8 / <5): {tail}")


def synth_requests(n, vocab, seed, pass_idx=0):
    """ShareGPT-shaped lengths: log-normal prompt/output lengths clipped by the reference's dataset
    filter (prompt >= 4, output >= 4, prompt <= 1024, prompt + output <= 2048). The LENGTHS depend on `seed` only
    (every pass is the same workload); the token ids also on `pass_idx`: both arms keep prefix caching on (the
    reference's default), and a pass that re-submitted the previous pass's prompts would find them in the cache
    and skip its prefill."""
    import numpy as np
    rng = np.random.default_rng(seed)
    lens, outs = [], []
    while len(lens) < n:
        p = int(rng.lognormal(5.0, 1.0))
        o = int(rng.lognormal(5.2, 0.9))
        if p < 4 or o < 4 or p > 1024 or p + o > 2048:
            continue
        lens.append(p)
        outs.append(o)
    trng = np.random.default_rng([seed, 7919, pass_idx])
    prompts = [trng.integers(10, vocab - 10, size=p).tolist() for p in lens]
    return prompts, outs


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, seqs, seed):
    """Write what `LLM.generate` returned to its caller in one pass: the generated token ids of every request,
    concatenated in request order (`output_token_ids.npy`), how many each request generated (`output_lens.npy`) and
    which requests these are (`request_index.npy`). float64 holds token ids exactly. When the whole set would exceed
    64 MB, a fixed sample of requests drawn with `seed` is written instead."""
    import numpy as np
    gen = [np.asarray(q.token_ids[q.prompt_len:], dtype=np.float64) for q in seqs]
    idx = np.arange(len(gen))
    if sum(g.nbytes + 16 for g in gen) > DUMP_LIMIT_BYTES:
        order = np.random.default_rng([seed, 4099]).permutation(len(gen))
        sizes = np.cumsum([gen[i].nbytes + 16 for i in order])
        idx = np.sort(order[:int(np.searchsorted(sizes, DUMP_LIMIT_BYTES, side="right"))])
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "output_token_ids.npy"),
            np.concatenate([gen[i] for i in idx]) if len(idx) else np.zeros(0, np.float64))
    np.save(os.path.join(out_dir, "output_lens.npy"), np.array([len(gen[i]) for i in idx], dtype=np.float64))
    np.save(os.path.join(out_dir, "request_index.npy"), idx.astype(np.float64))


class ClockSampler(threading.Thread):
    QUERY = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active," \
            "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index=0):
        super().__init__(daemon=True)
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu_index)], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:  # noqa: BLE001
            pass

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
                for nme, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:  # noqa: BLE001
                continue
        sm.sort()
        # median over samples under load (upper half of the distribution)
        load = sm[len(sm) // 2:] if sm else []
        med = load[len(load) // 2] if load else None
        return {"sm_mhz": med, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def main():
    args = parse()
    if args.impl == "reference":
        return reference_arm(args)
    import torch
    import torch.distributed as dist
    from gllm_b200 import LLM
    from gllm_b200.ops import sm100

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert world == args.gpus or (world == 1 and args.gpus == 1), \
        f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})"
    conf = CONFIGS[args.config]
    model_name = args.model.replace("preset:", "")
    model = args.model
    # Self-test of this script's control flow on a box without a GPU (tests/test_bench_cpu.py): a tiny random model
    # on the CPU, host clocks instead of CUDA events. Never a benchmark number (`"data"` says so).
    cpu_selftest = os.environ.get("GLLM_BENCH_CPU_SELFTEST") == "1" and not torch.cuda.is_available()
    if args.config != "qwen3-8b-tp":
        model_name = conf["model"]
        model = "preset:" + model_name
        if args.pp == 1:
            args.pp = min(conf["pp"], args.gpus)
        if args.schedule_method == "chunked_prefill":
            args.schedule_method = conf["method"]
    if args.layers > 0:
        from gllm_b200.models.presets import PRESETS
        model = dict(PRESETS[model_name], num_hidden_layers=args.layers)
        model_name = f"{model_name} REDUCED to {args.layers} layers"
    if cpu_selftest:
        from gllm_b200.models.presets import PRESETS, tiny
        arch = PRESETS.get(model_name.split(" ")[0], PRESETS["qwen3-8b"])["architectures"][0]
        if arch.startswith("Deepseek"):
            arch = "Qwen3ForCausalLM"
        over = dict(num_local_experts=4, num_experts_per_tok=2) if arch == "MixtralForCausalLM" else {}
        model = tiny(arch, num_hidden_layers=2 * args.pp, max_position_embeddings=4096, **over)
        model_name = f"tiny {arch} self-test model (CPU)"
    tp = args.gpus // args.pp
    llm = LLM(model, load_format="dummy", tp_size=tp, pp_size=args.pp, maxp=args.maxp, maxd=args.maxd,
              max_cuda_graph_bs=args.max_cuda_graph_bs, schedule_method=args.schedule_method,
              enable_prefix_caching=True, gpu_memory_util=0.9, model_max_length=2048 + 16,
              tp_mode=args.tp_mode, log_stats=False, launch_mode="inproc", seed=args.seed,
              async_schedule=args.async_schedule, disable_cuda_graph=args.disable_cuda_graph,
              num_gpu_pages=args.num_gpu_pages, **({"device": "cpu", "num_cpu_pages": 2048} if cpu_selftest else {}))
    vocab = llm.loader.config["vocab_size"]
    prompts, out_lens = synth_requests(args.num_prompts, vocab, args.seed)
    if cpu_selftest:      # the CPU oracle path is slow: a few tokens per request exercise the same control flow
        out_lens = [min(o, 6) for o in out_lens]
    total_out = sum(out_lens)
    total_in = sum(len(p) for p in prompts)
    runner = llm.worker.runner

    # token ids of every pass prepared up front (host work outside the timed region; the reference arm does the same)
    n_pass = args.warmup + args.steps
    pass_prompts = [prompts if (args.fixed_prompts or i == 0) else synth_requests(args.num_prompts, vocab, args.seed, i)[0]
                    for i in range(n_pass)]
    if cpu_selftest:
        pass_prompts = [[p[:40] for p in ps_] for ps_ in pass_prompts]
    pass_no = [0]

    def one_pass():
        toks = pass_prompts[min(pass_no[0], n_pass - 1)]
        pass_no[0] += 1
        return llm.generate(tokens=toks, output_lens=out_lens, ignore_eos=True, top_k=1, temperature=0.0)

    def barrier():
        if world > 1:
            dist.barrier()
        if not cpu_selftest:
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        one_pass()

    # ---- the K timed passes through the public API (LLM.generate: every iteration copies its batch arrays
    # host->device from pinned memory and reads the sampled tokens back), bracketed by barrier + sync. CUDA events on
    # the launching stream -> `value`; the host's wall clock around the same bracket -> `e2e`.
    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0"))) if rank == 0 else None
    if sampler:
        sampler.start()
    runner.time_steps = True
    runner.gpu_busy_ms()
    stats0 = dict(runner.stats)
    launches0 = sm100.launches()
    barrier()
    t0 = time.perf_counter()
    if not cpu_selftest:
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
    seqs = None
    for _ in range(args.steps):
        seqs = one_pass()
    if not cpu_selftest:
        ev1.record()
    barrier()
    wall_s = time.perf_counter() - t0
    dev_ms = wall_s * 1e3 if cpu_selftest else ev0.elapsed_time(ev1)
    busy_ms = runner.gpu_busy_ms()
    runner.time_steps = False
    stats1 = dict(runner.stats)
    launches = (sm100.launches() - launches0) + (stats1["graph_kernel_launches"] - stats0["graph_kernel_launches"])
    if sampler:
        sampler.stop()
    if world > 1:
        t = torch.tensor([dev_ms, wall_s * 1e3, busy_ms], device="cpu" if cpu_selftest else "cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dev_ms, wall_ms, busy_ms = t.tolist()
        wall_s = wall_ms / 1e3
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, seqs, args.seed)
    if rank == 0:
        value = args.steps * total_out / (dev_ms / 1e3)
        e2e = args.steps * total_out / wall_s
        base = None
        try:
            pub = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "BASELINE.json"))).get("published", {})
            base = pub.get("output_tokens_per_s")
        except Exception:  # noqa: BLE001
            pass
        eng_steps = stats1["steps"] - stats0["steps"]
        # request latencies of the last timed pass (all requests arrive together at t0: offline workload)
        lat = None
        try:
            ttft = sorted((q.first_token_time - q.arrival_time) * 1e3 for q in seqs if q.first_token_time)
            tpot = sorted((q.finish_time - q.first_token_time) * 1e3 / max(q.num_output_tokens - 1, 1)
                          for q in seqs if q.first_token_time and q.finish_time and q.num_output_tokens > 1)
            lat = {"p50_ttft_ms": round(ttft[len(ttft) // 2], 1), "p99_ttft_ms": round(ttft[int(len(ttft) * 0.99)], 1),
                   "p50_tpot_ms": round(tpot[len(tpot) // 2], 2), "p99_tpot_ms": round(tpot[int(len(tpot) * 0.99)], 2),
                   "arrival": "all requests at t0 (offline batch)", "source": "last timed pass"}
        except Exception:  # noqa: BLE001
            pass
        out = {
            "metric": "output tokens/sec, offline throughput (benchmark_throughput workload), " + conf["label"],
            "value": round(value, 1), "unit": "tokens/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(dev_ms / args.steps, 2), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": (value / base) if base else None, "dtype": "bf16",
            "data": "synthetic ShareGPT-shaped token ids (log-normal lengths, reference dataset filter); random-init weights"
                    + (" -- CPU SELF-TEST OF bench.py, NOT A MEASUREMENT" if cpu_selftest else ""),
            "impl": "ours",
            "config": {"model": model_name, "named_config": args.config, "num_prompts": args.num_prompts,
                       "global_batch": args.num_prompts, "seq_len": "prompt<=1024, prompt+output<=2048",
                       "input_tokens_per_step": total_in, "output_tokens_per_step": total_out,
                       "parallelism": f"tp{tp}" + (f"pp{args.pp}" if args.pp > 1 else ""), "tp_mode": args.tp_mode,
                       "schedule_method": args.schedule_method, "async_schedule": bool(args.async_schedule),
                       "enable_prefix_caching": True, "max_cuda_graph_bs": args.max_cuda_graph_bs,
                       "prompts": "same lengths every pass, fresh token ids per pass (no cross-pass prefix-cache hits)"
                       if not args.fixed_prompts else "IDENTICAL token ids every pass (prefill served from cache)",
                       "maxp": args.maxp, "maxd": args.maxd,
                       "l2": "inputs larger than L2 (16 GB of weights + multi-GB KV streamed every iteration)",
                       "engine_iterations_per_step": eng_steps // max(args.steps, 1),
                       "cuda_graph_iterations": (stats1["graph_steps"] - stats0["graph_steps"]) // max(args.steps, 1),
                       "gpu_busy_fraction": round(busy_ms / dev_ms, 3),
                       "device_ms_by_step_kind": {k: [v[0] // args.steps, round(v[1] / args.steps, 1), v[2] // args.steps]
                                                  for k, v in sorted(getattr(runner, "busy_by_kind", {}).items())},
                       "total_tokens_per_s": round(args.steps * (total_in + total_out) / (dev_ms / 1e3), 1)},
            "clocks": sampler.summary() if sampler else None,
            "e2e": {"value": round(e2e, 1), "unit": "tokens/s",
                    "h2d_bytes_per_step": (stats1["h2d_bytes"] - stats0["h2d_bytes"]) // max(args.steps, 1),
                    "d2h_bytes_per_step": (stats1["d2h_bytes"] - stats0["d2h_bytes"]) // max(args.steps, 1)},
            "gpu_launches": int(launches),
            "latency": lat,
        }
        print(json.dumps(out), flush=True)
    sys.stdout.flush()
    sys.stderr.flush()
    teardown(llm, world)
    return 0


def teardown(llm, world):
    """Orderly exit (no os._exit: exit-time hooks must run): quiesce the GPU, stop the engine, drop the symmetric
    memory handles while every peer is still alive, then destroy the process group. A watchdog bounds a teardown
    that stalls (it has not been seen to, but a hang here would hold the GPUs until the caller's timeout)."""
    import torch
    import torch.distributed as dist

    def _bail():
        sys.stderr.write("bench.py: teardown stalled for 120 s, forcing exit\n")
        sys.stderr.flush()
        os._exit(0)
    dog = threading.Timer(120.0, _bail)
    dog.daemon = True
    dog.start()
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    if world > 1 and dist.is_initialized():
        dist.barrier()
    try:
        llm.close()
    finally:
        if world > 1 and dist.is_initialized():
            dist.barrier()
            dist.destroy_process_group()
    dog.cancel()


if __name__ == "__main__":
    sys.exit(main())
