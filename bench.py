"""Headline benchmark: Qwen3-4B W4A16 decode / prefill tokens/s on B200 (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload decode|prefill|serve|serve8k] [--no-extra] [--no-cpu-baseline]
                    [--dump-outputs DIR]

Workloads (BASELINE.json `configs`; SURVEY.md section 8d):

  decode   (default; config 2, the one the metric is quoted on) Qwen3-4B-shaped random W4A16 weights,
           ONE request per GPU, 128-token prompt (chunk-prefilled through the paged path), greedy decode
           with paged-KV GQA attention + dequant matvec.  A "step" is one decode step (one token per GPU).
           The line also carries, under `extra`, the config-2 sweeps (context S in {128,1K,4K,8K} at B=1,
           batch B in {1..64} at S=128) and a short config-3 prefill measurement with its two rooflines.
  prefill  (config 3) a 4096-token prompt through Qwen3ModelWeek3.__call__ in one chunk (and in 512 /
           128-token chunks under `extra`); a "step" is one whole prefill.  roofline = the tcgen05 W4A16
           GEMM (tensor bound) + the tcgen05 paged FlashAttention under `extra.attention_roofline`.
  serve    (config 4) continuous batching, 64 decode slots, 128 requests per GPU, prompts U[128,1024],
           outputs U[32,128], prefill_step 128, page 128, seed 0 (protocol of the reference's
           benches/bench.py:351-572); a "step" is one scheduler iteration, the run is the whole queue.
  serve8k  (config 5) 8K-context requests sharded i mod N over the ranks, 64 decode slots per GPU;
           --requests defaults to 64 * N (every GPU carries config 5's per-GPU load: at N = 8 this is
           exactly the 512-request configuration), prefill_step 1024.

At N > 1 every rank serves its own requests (request i -> rank i mod N); weights are drawn on rank 0
and broadcast once over NCCL; there is no data-path collective.

Numbers on the JSON line (decode):
  value     decode tok/s, whole job, device-resident: K replays of the captured decode step with
            token feedback on the device (CUDA events, max over ranks)
  e2e       same metric through the public model call, per step: pinned-host token -> device copy,
            model(...), device -> host read of the sampled token
  roofline  the W4A16 weight-streaming kernel: the 145 projection launches of one token exactly as the
            decode graph issues them (2.137 GB of packed weights, > L2), replayed from a CUDA graph,
            CUDA-event timed; achieved = algorithmic bytes / time, traffic = ncu DRAM bytes of the same
            launches (read from the committed capture named in `traffic_source`, null if there is none)
  cpu_baseline  the reference's CPU path (oracle.model: dense bf16 weights, readable operators) on the
            host cores, bounded sample

--dump-outputs DIR (decode) writes what the last timed step handed its caller, rank 0: DIR/logits.npy
(float32 [1, vocab]) and DIR/next_tokens.npy (the greedy token, float64 [1]).  Weights and prompt are
seeded, so two builds run with the same arguments can be compared output for output.
"""

from __future__ import annotations

import argparse
import importlib.util
import json
import os
import random
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path[:0] = [str(ROOT), str(ROOT / "tiny-llm_b200")]

import torch  # noqa: E402

UNIT = "tok/s"
MODEL = "qwen3-4b"
PROMPT_LEN = 128
PAGE_SIZE = 128
METRICS = {
    "decode": "Qwen3-4B W4A16 decode tok/s",
    "prefill": "Qwen3-4B W4A16 prefill tok/s",
    "serve": "Qwen3-4B W4A16 continuous-batching output tok/s",
    "serve8k": "Qwen3-4B W4A16 data-parallel serving output tok/s (8K context)",
}


def measured_peaks() -> dict:
    path = ROOT / "MEASURED_PEAKS.json"
    if path.exists():
        data = json.loads(path.read_text())
        return {"hbm_gbs": float(data["hbm_gbs"]), "bf16_tflops": float(data.get("bf16_tflops", 1682.0)),
                "bf16_tflops_sustained": float(data.get("bf16_tflops_sustained", data.get("bf16_tflops", 1442.5))),
                "source": "MEASURED_PEAKS.json"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1680.0, "bf16_tflops_sustained": 1440.0, "source": "fallback (B200_PROFILING.md)"}


def committed_traffic(kernel: str):
    """(bytes per launch, file) from the committed ncu capture of this round, or (None, None)."""
    path = ROOT / "profiles" / "traffic.json"
    if not path.exists():
        return None, None
    try:
        entry = json.loads(path.read_text()).get(kernel)
        return (int(entry["dram_bytes_per_launch"]), f"profiles/{entry['source']}") if entry else (None, None)
    except (ValueError, KeyError, TypeError):
        return None, None


def synthetic_prompt(seed: int, length: int, vocab: int) -> list[int]:
    """Token ids as benches/bench.py:190-225 draws them: uniform in [256, V-1]."""
    rng = random.Random(seed)
    return [rng.randint(256, vocab - 1) for _ in range(length)]


class ClockSampler:
    """nvidia-smi clocks/throttle reasons sampled during the timed region."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines: list[str] = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, flag in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[3:7]):
                if flag.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cuda_time_ms(fn, stream=None) -> float:
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record(stream)
    fn()
    end.record(stream)
    end.synchronize()
    return start.elapsed_time(end)


def dump_outputs(out_dir: str, **arrays: torch.Tensor) -> None:
    """Each float32 / float64 tensor as ``out_dir/<name>.npy``."""
    import numpy as np

    path = Path(out_dir)
    path.mkdir(parents=True, exist_ok=True)
    for name, tensor in arrays.items():
        np.save(path / f"{name}.npy", tensor.cpu().numpy())


def base_line(args, world: int, workload: str) -> dict:
    return {
        "metric": METRICS[workload], "value": None, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16 activations, 4-bit weights (W4A16), fp32 accumulation",
        "data": "synthetic (random Qwen3-4B-shaped W4A16 weights, random prompts)",
    }


def setup(args):
    from extensions_b200 import tiny_llm_ext_b200 as ext
    from tiny_llm_b200 import Qwen3ModelWeek3
    from tiny_llm_b200.parallel import init_distributed, replicated_model

    rank, world, device = init_distributed("cuda")
    assert world == args.gpus or world == 1, f"launched with WORLD_SIZE={world} but --gpus {args.gpus}"
    pdl = os.environ.get("TL_PDL", "1") != "0"
    ext.set_pdl(pdl)
    t_load = time.perf_counter()
    model_ns, broadcast_bytes = replicated_model(MODEL, seed=0, rank=rank, device=device)
    model = Qwen3ModelWeek3(model_ns, page_size=PAGE_SIZE)
    info = {"weights_load_s": round(time.perf_counter() - t_load, 2), "broadcast_bytes": broadcast_bytes, "pdl": int(pdl)}
    return ext, model, model_ns, rank, world, device, info


# ------------------------------------------------------------------ workload: decode
def run_decode(args) -> None:
    from tiny_llm_b200.batch import greedy_tokens
    from tiny_llm_b200.parallel import barrier, max_over_ranks
    from tiny_llm_b200.synthetic import weight_stream_bytes

    ext, model, model_ns, rank, world, device, info = setup(args)
    margs = model_ns.args
    steps, warmup = args.steps, max(args.warmup, 3)
    max_seq = PROMPT_LEN + 2 * (steps + warmup) + 64
    model.decode_graph_max_seq_len = ((max_seq + PAGE_SIZE - 1) // PAGE_SIZE) * PAGE_SIZE
    engine = model.decode_engine(1)

    prompt = synthetic_prompt(1000 + rank, PROMPT_LEN, margs.vocab_size)
    cache = model.create_kv_cache()
    t0 = time.perf_counter()
    first = model(torch.tensor([prompt], dtype=torch.int32, device=device), 0, cache, logits_to_keep=1)
    token = int(greedy_tokens(first[:, -1, :])[0])
    torch.cuda.synchronize()
    info["prefill_128_s"] = round(time.perf_counter() - t0, 3)

    # ---- value: device-resident decode (graph replays, token feedback on device)
    offset = PROMPT_LEN
    engine.decode_on_device([token], [offset], cache, min(warmup, engine.log_capacity))
    torch.cuda.synchronize()
    offset += warmup
    token = int(engine.next_tokens[0])
    sampler = ClockSampler(device.index or 0)
    if rank == 0:
        sampler.start()
    launches0 = ext.launch_count()
    replays0 = engine.graph_replays
    barrier(device)
    torch.cuda.synchronize()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    done = 0
    while done < steps:  # one call unless --steps exceeds the engine's on-device token log (4096)
        take = min(steps - done, engine.log_capacity)
        out_tokens = engine.decode_on_device([token], [offset + done], cache, take)
        done += take
        if done < steps:
            token = int(out_tokens[-1, 0])
    end.record()
    torch.cuda.synchronize()
    barrier(device)
    ms = max_over_ranks(start.elapsed_time(end), device)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:  # before the e2e calls below replay the same engine and overwrite its buffers
        dump_outputs(args.dump_outputs, logits=engine.logits[:1].float(), next_tokens=out_tokens[-1].double())
    # graph replays do not pass through the C ABI; the launches recorded when the step was captured
    # are what each replay executes (plus whatever went through the ABI directly in the region)
    gpu_launches = engine.kernels_per_step * (engine.graph_replays - replays0) + (ext.launch_count() - launches0)
    offset += steps
    token = int(out_tokens[-1, 0])
    value = world * steps / (ms / 1e3)

    # ---- e2e: public API per step, pinned host token in, sampled token out
    e2e_steps = min(steps, 64)
    pinned_in = torch.empty(1, 1, dtype=torch.int32, pin_memory=True)
    pinned_out = torch.empty(1, dtype=torch.int32, pin_memory=True)
    for phase, count in (("warm", 3), ("timed", e2e_steps)):
        barrier(device)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(count):
            pinned_in[0, 0] = token
            tok_dev = pinned_in.to(device, non_blocking=True)
            logits = model(tok_dev, offset, cache, logits_to_keep=1)  # the call a user makes
            pinned_out.copy_(greedy_tokens(logits[:, -1, :]), non_blocking=True)
            torch.cuda.synchronize()
            token = int(pinned_out[0])
            offset += 1
        e2e_s = time.perf_counter() - t0
    e2e_s = max_over_ranks(e2e_s, device)
    e2e_value = world * e2e_steps / e2e_s
    meta_bytes = engine.upload_bytes_per_step()

    roofline = matvec_roofline(model, engine, ext, device) if rank == 0 else None
    for c in cache:
        c.release()

    extra = {}
    if rank == 0 and world == 1 and not args.no_extra:
        for name, fn in (("context_sweep", lambda: context_sweep(model, device, margs)),
                         ("batch_sweep", lambda: batch_sweep(model, device, margs)),
                         ("prefill", lambda: prefill_measure(model, ext, device, margs, tokens=4096, reps=3, chunked=False))):
            try:
                extra[name] = fn()
            except Exception as exc:  # an extra must never cost the headline line
                extra[name] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
            torch.cuda.empty_cache()

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = run_cpu_baseline(sample_steps=9, warmup_steps=3)

    if rank == 0:
        stream_bytes = weight_stream_bytes(margs)
        kv_bytes = 147456 * (PROMPT_LEN + warmup + steps // 2)
        peak = measured_peaks()
        line = base_line(args, world, "decode")
        line.update({
            "value": round(value, 2), "ms_per_step": round(ms / steps, 4),
            "config": {
                "workload": "Qwen3-4B W4A16 single-request decode, batch=1 per GPU, paged-KV GQA + dequant matvec",
                "prompt_len": PROMPT_LEN, "page_size": PAGE_SIZE, "requests_per_gpu": 1, "parallelism": f"dp{world}",
                "l2_policy": "inputs larger than L2: each step streams 2.14 GB of packed weights (L2 = 126 MB)",
                "decode_graph": "cuda-graph replay, fused=%s, pdl=%s" % (engine.fused, info["pdl"]),
            },
            "e2e": {"value": round(e2e_value, 2), "unit": UNIT, "h2d_bytes_per_step": 4 + meta_bytes, "d2h_bytes_per_step": 4, "steps": e2e_steps},
            "gpu_launches": int(gpu_launches), "kernels_per_step": int(engine.kernels_per_step), "clocks": clocks, "roofline": roofline,
            "token_roofline": {
                "bytes_per_token": stream_bytes + kv_bytes,
                "achieved_gbs": round((stream_bytes + kv_bytes) / (ms / steps / 1e3) / 1e9, 1),
                "frac": round((stream_bytes + kv_bytes) / (ms / steps / 1e3) / 1e9 / peak["hbm_gbs"], 4),
                "peak_gbs": peak["hbm_gbs"], "peak_source": peak["source"],
            },
            "cpu_baseline": cpu_baseline, "extra": extra, "setup": info,
        })
        print(json.dumps(line), flush=True)


def matvec_roofline(model, engine, ext, device) -> dict:
    """The projection launches of one decode token exactly as the engine issues them (per layer:
    rms_norm+q|k|v, o+residual, rms_norm+gate|up+swiglu, down+residual; then rms_norm+head), M = 1,
    from one captured graph: 2.137 GB of distinct packed weights per replay, so every launch
    streams from HBM (L2 = 126 MB)."""
    from tiny_llm_b200.synthetic import weight_stream_bytes

    H = model.hidden_size
    bf = torch.bfloat16
    x = torch.randn(1, H, device=device).to(bf)
    y = torch.randn(1, engine.Hq * engine.D, device=device).to(bf)
    res = torch.randn(1, H, device=device).to(bf)
    norm_w = torch.ones(H, device=device, dtype=bf)
    inter = model.layers_inner[0].mlp.hidden_dim
    act = torch.randn(1, inter, device=device).to(bf)
    head = model.w_lm_head if model.w_lm_head is not None else model.embedding.weight
    launches = 4 * len(model.layers_inner) + 1

    def body():
        for block, pk in zip(model.layers_inner, engine._packed):
            wo, wd = block.self_attn.wo, block.mlp.w_down
            ext.quantized_matmul_fused(pk.qkv.scales, pk.qkv.biases, pk.qkv.weight, x, norm_w, prologue=ext.PRO_RMSNORM, eps=1e-6)
            ext.quantized_matmul_fused(wo.scales, wo.biases, wo.weight, y, residual=res, epilogue=ext.EPI_RESIDUAL)
            ext.quantized_matmul_fused(pk.gate_up.scales, pk.gate_up.biases, pk.gate_up.weight, x, norm_w, prologue=ext.PRO_RMSNORM,
                                       eps=1e-6, epilogue=ext.EPI_SWIGLU_PAIRS)
            ext.quantized_matmul_fused(wd.scales, wd.biases, wd.weight, act, residual=res, epilogue=ext.EPI_RESIDUAL)
        ext.quantized_matmul_fused(head.scales, head.biases, head.weight, x, norm_w, prologue=ext.PRO_RMSNORM, eps=1e-6)

    stream = torch.cuda.Stream(device=device)
    with torch.cuda.stream(stream):
        body()
        stream.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            body()
        for _ in range(3):
            graph.replay()
        stream.synchronize()
        times = [cuda_time_ms(graph.replay, stream) for _ in range(10)]
    ms = statistics.median(times)
    # algorithmic bytes: every packed weight, scale and bias once (SURVEY 8d: 0.53125 B/weight) + activations in/out
    margs = model.mlx_model.args
    io = 2 * len(model.layers_inner) * (H + (engine.Hq + 2 * engine.Hkv) * engine.D + engine.Hq * engine.D + 2 * H + H + inter + inter + 2 * H)
    algorithmic = weight_stream_bytes(margs) + io + 2 * (H + margs.vocab_size)
    peak = measured_peaks()
    achieved = algorithmic / (ms / 1e3) / 1e9
    traffic, traffic_source = committed_traffic("w4a16_stream5_kernel")
    return {
        "kernel": "w4a16_stream5_kernel<bf16, M=1> (W4A16 dequant matvec with fused rms_norm / residual / SwiGLU epilogue)",
        "bound": "hbm", "achieved": round(achieved, 1), "peak": peak["hbm_gbs"], "peak_source": peak["source"], "unit": "GB/s",
        "frac": round(achieved / peak["hbm_gbs"], 4), "traffic": traffic, "traffic_source": traffic_source, "launches": launches,
        "avg_launch_us": round(ms * 1e3 / launches, 3), "algorithmic_bytes_per_launch": round(algorithmic / launches),
        "timing": f"cuda events on the launching stream around a graph replay of one token's {launches} projection launches, median of 10",
    }


def _prefill_request(model, device, prompt, chunk=2048):
    """One paged request cache holding `prompt` (chunked through the public call)."""
    cache = model.create_kv_cache()
    ids = torch.tensor([prompt], dtype=torch.int32, device=device)
    logits = None
    for off in range(0, len(prompt), chunk):
        logits = model(ids[:, off:off + chunk], off, cache, logits_to_keep=1)
    return cache, logits


def context_sweep(model, device, margs) -> list:
    """Config-2 context sweep (SURVEY 8d): B = 1, 64 device-resident decode steps after a real prefill of S tokens."""
    from tiny_llm_b200.batch import greedy_tokens
    from tiny_llm_b200.synthetic import weight_stream_bytes

    peak = measured_peaks()["hbm_gbs"]
    out, steps = [], 64
    model.decode_graph_max_seq_len = 8192 + 256
    engine = model.decode_engine(1)
    for S in (128, 1024, 4096, 8192):
        cache, logits = _prefill_request(model, device, synthetic_prompt(7 + S, S, margs.vocab_size))
        token = int(greedy_tokens(logits[:, -1, :])[0])
        engine.decode_on_device([token], [S], cache, 8)
        torch.cuda.synchronize()
        token = int(engine.next_tokens[0])
        ms = cuda_time_ms(lambda: engine.decode_on_device([token], [S + 8], cache, steps)) / steps
        for c in cache:
            c.release()
        nbytes = weight_stream_bytes(margs) + 147456 * (S + 8 + steps // 2) + 147456
        out.append({"context": S, "ms_per_token": round(ms, 4), "tok_s": round(1e3 / ms, 1), "bytes_per_token": nbytes,
                    "hbm_frac": round(nbytes / (ms / 1e3) / 1e9 / peak, 4)})
    return out


def batch_sweep(model, device, margs) -> list:
    """Config-2 batch sweep: B requests of 128 prompt tokens decoded together (weights counted once per step)."""
    from tiny_llm_b200.batch import greedy_tokens
    from tiny_llm_b200.kv_cache import BatchingKvCache
    from tiny_llm_b200.synthetic import weight_stream_bytes

    peak = measured_peaks()["hbm_gbs"]
    out, steps, S = [], 32, PROMPT_LEN
    model.decode_graph_max_seq_len = 512
    for B in (1, 2, 4, 8, 16, 32, 64):
        engine = model.decode_engine(B)
        tables = [BatchingKvCache(max_active_requests=B, max_seq_len=512) for _ in range(model.num_hidden_layers)]
        tokens = []
        for b in range(B):
            cache, logits = _prefill_request(model, device, synthetic_prompt(100 + b, S, margs.vocab_size))
            tokens.append(int(greedy_tokens(logits[:, -1, :])[0]))
            for layer_cache, table in zip(cache, tables):
                table.add_request(layer_cache, b)
        engine.decode_on_device(tokens, [S] * B, tables, 4)
        torch.cuda.synchronize()
        tokens = engine.next_tokens.tolist()
        ms = cuda_time_ms(lambda: engine.decode_on_device(tokens, [S + 4] * B, tables, steps)) / steps
        for table in tables:
            for b in range(B):
                table.remove_request(b)
        nbytes = weight_stream_bytes(margs) + B * (147456 * (S + 4 + steps // 2) + 147456)
        out.append({"batch": B, "ms_per_step": round(ms, 4), "tok_s": round(B * 1e3 / ms, 1), "bytes_per_step": nbytes,
                    "hbm_frac": round(nbytes / (ms / 1e3) / 1e9 / peak, 4)})
    return out


# ------------------------------------------------------------------ workload: prefill (config 3)
def prefill_flops(margs, tokens: int) -> dict:
    H, I = margs.hidden_size, margs.intermediate_size
    qw, kvw = margs.num_attention_heads * margs.head_dim, margs.num_key_value_heads * margs.head_dim
    proj = 2.0 * tokens * margs.num_hidden_layers * (H * (qw + 2 * kvw) + qw * H + 3 * H * I)
    attn = 4.0 * margs.num_attention_heads * margs.head_dim * (tokens * (tokens + 1) / 2) * margs.num_hidden_layers
    return {"projections": proj, "attention": attn, "head_last_row": 2.0 * H * margs.vocab_size}


def prefill_measure(model, ext, device, margs, tokens: int, reps: int, chunked: bool) -> dict:
    """Whole-model prefill of `tokens` prompt tokens (CUDA events around the public call, median of reps)
    + the two tensor-bound kernels timed the way the model issues them."""
    peaks = measured_peaks()
    prompt = torch.tensor([synthetic_prompt(31, tokens, margs.vocab_size)], dtype=torch.int32, device=device)

    def one(chunk):
        cache = model.create_kv_cache()
        torch.cuda.synchronize()
        ms = cuda_time_ms(lambda: [model(prompt[:, off:off + chunk], off, cache, logits_to_keep=1) for off in range(0, tokens, chunk)])
        for c in cache:
            c.release()
        return ms

    one(tokens)
    whole = statistics.median(one(tokens) for _ in range(reps))
    flops = prefill_flops(margs, tokens)
    total = flops["projections"] + flops["attention"] + flops["head_last_row"]
    out = {"tokens": tokens, "ms": round(whole, 3), "tok_s": round(tokens / (whole / 1e3), 1),
           "model_tflops": round(total / (whole / 1e3) / 1e12, 1), "model_frac_of_sustained_peak": round(total / (whole / 1e3) / 1e12 / peaks["bf16_tflops_sustained"], 4)}
    if chunked:
        out["chunked"] = []
        for chunk in (512, 128):
            one(chunk)
            ms = statistics.median(one(chunk) for _ in range(2))
            out["chunked"].append({"prefill_step": chunk, "ms": round(ms, 3), "tok_s": round(tokens / (ms / 1e3), 1)})
    out["gemm_roofline"] = gemm_roofline(model, ext, device, margs, tokens)
    out["attention_roofline"] = attention_roofline(ext, device, margs, tokens)
    return out


def gemm_roofline(model, ext, device, margs, tokens: int) -> dict:
    """The 4 x 36 projection GEMMs of one prefill chunk, back to back over the model's own (distinct) weights."""
    peaks = measured_peaks()
    H, I = margs.hidden_size, margs.intermediate_size
    qw = margs.num_attention_heads * margs.head_dim
    bf = torch.bfloat16
    x = torch.randn(tokens, H, device=device).to(bf)
    y = torch.randn(tokens, qw, device=device).to(bf)
    act = torch.randn(tokens, I, device=device).to(bf)

    def mm(w, a):
        return ext.quantized_matmul(w.scales, w.biases, w.group_size, w.bits, a, w.weight, True)

    def body():
        for block in model.layers_inner:
            at, mlp = block.self_attn, block.mlp
            mm(at.wq, x), mm(at.wk, x), mm(at.wv, x), mm(at.wo, y), mm(mlp.w_gate, x), mm(mlp.w_up, x), mm(mlp.w_down, act)

    body()
    torch.cuda.synchronize()
    ms = statistics.median(cuda_time_ms(body) for _ in range(3))
    flops = prefill_flops(margs, tokens)["projections"]
    launches = 7 * len(model.layers_inner)
    achieved = flops / (ms / 1e3) / 1e12
    return {"kernel": "w4a16_gemm_kernel / w4a16_gemm2_kernel (tcgen05.mma kind::f16, the pair form cta_group::2 for q|k|v and gate|up; TMEM accumulators, TMA activations, in-kernel W4 dequant)",
            "bound": "tensor", "achieved": round(achieved, 1), "peak": peaks["bf16_tflops_sustained"], "peak_source": peaks["source"] + " (sustained)",
            "unit": "TFLOP/s", "frac": round(achieved / peaks["bf16_tflops_sustained"], 4), "traffic": None, "launches": launches,
            "avg_launch_us": round(ms * 1e3 / launches, 2), "algorithmic_flops_per_launch": round(flops / launches),
            "timing": f"cuda events around the {launches} projection GEMMs of a {tokens}-token chunk issued back to back, median of 3"}


def attention_roofline(ext, device, margs, tokens: int) -> dict:
    peaks = measured_peaks()
    Hq, Hkv, D = margs.num_attention_heads, margs.num_key_value_heads, margs.head_dim
    pages = (tokens + PAGE_SIZE - 1) // PAGE_SIZE
    bf = torch.bfloat16
    kp = torch.randn(pages, Hkv, PAGE_SIZE, D, device=device).to(bf)
    vp = torch.randn(pages, Hkv, PAGE_SIZE, D, device=device).to(bf)
    q = torch.randn(Hq, tokens, D, device=device).to(bf)
    bt = torch.arange(pages, dtype=torch.int32, device=device).reshape(1, pages)
    cl = torch.tensor([tokens], dtype=torch.int32, device=device)

    def call():
        ext.paged_attention(q, kp, vp, bt, cl, D**-0.5, is_causal=True, num_kv_heads=Hkv, num_heads=Hq)

    for _ in range(3):
        call()
    torch.cuda.synchronize()
    ms = statistics.median(cuda_time_ms(call) for _ in range(5))
    flops = 4.0 * Hq * D * (tokens * (tokens + 1) / 2)
    achieved = flops / (ms / 1e3) / 1e12
    return {"kernel": "paged causal FlashAttention prefill (tl_paged_attention, L > 8, bf16, D = 128)", "bound": "tensor",
            "achieved": round(achieved, 1), "peak": peaks["bf16_tflops"], "peak_source": peaks["source"] + " (burst: kernel timed alone)",
            "unit": "TFLOP/s", "frac": round(achieved / peaks["bf16_tflops"], 4), "traffic": None, "launches": 1, "avg_launch_us": round(ms * 1e3, 1),
            "algorithmic_flops_per_launch": round(flops), "timing": f"cuda events, L = S = {tokens}, causal, median of 5 after 3 warm-up calls"}


def run_prefill(args) -> None:
    from tiny_llm_b200.batch import greedy_tokens
    from tiny_llm_b200.parallel import barrier, max_over_ranks

    ext, model, model_ns, rank, world, device, info = setup(args)
    margs = model_ns.args
    tokens = args.prompt_len or 4096
    steps, warmup = max(1, args.steps), max(args.warmup, 3)
    prompts = [torch.tensor([synthetic_prompt(2000 + rank + 17 * i, tokens, margs.vocab_size)], dtype=torch.int32, device=device) for i in range(2)]
    host_prompt = torch.tensor([synthetic_prompt(2000 + rank, tokens, margs.vocab_size)], dtype=torch.int32).pin_memory()

    def one(ids):
        cache = model.create_kv_cache()
        logits = model(ids, 0, cache, logits_to_keep=1)
        tok = greedy_tokens(logits[:, -1, :])
        for c in cache:
            c.release()
        return tok

    for _ in range(warmup):
        one(prompts[0])
    sampler = ClockSampler(device.index or 0)
    if rank == 0:
        sampler.start()
    launches0 = ext.launch_count()
    barrier(device)
    torch.cuda.synchronize()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(steps):
        one(prompts[i % 2])
    end.record()
    torch.cuda.synchronize()
    barrier(device)
    ms = max_over_ranks(start.elapsed_time(end), device)
    clocks = sampler.stop() if rank == 0 else None
    gpu_launches = ext.launch_count() - launches0
    value = world * steps * tokens / (ms / 1e3)
    # e2e: prompt ids from pinned host memory, first token read back
    pinned_out = torch.empty(1, dtype=torch.int32, pin_memory=True)
    barrier(device)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        pinned_out.copy_(one(host_prompt.to(device, non_blocking=True)), non_blocking=True)
        torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0, device)
    extra = {}
    roofline = None
    if rank == 0:
        try:
            extra = prefill_measure(model, ext, device, margs, tokens, reps=3, chunked=not args.no_extra)
            roofline = extra.pop("gemm_roofline")
        except Exception as exc:
            extra = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    cpu_baseline = run_cpu_baseline(sample_steps=2, mode="prefill") if (rank == 0 and world == 1 and not args.no_cpu_baseline) else None
    if rank == 0:
        line = base_line(args, world, "prefill")
        line.update({
            "value": round(value, 1), "ms_per_step": round(ms / steps, 3),
            "config": {"workload": "Qwen3-4B W4A16 4K-context prefill, tiled FlashAttention + tensor-core GEMM, one request per GPU",
                       "prompt_len": tokens, "prefill_step": tokens, "page_size": PAGE_SIZE, "parallelism": f"dp{world}", "logits_to_keep": 1,
                       "l2_policy": "inputs larger than L2: 2.14 GB of packed weights + 0.6 GB of K/V pages per prefill; two prompts alternate"},
            "e2e": {"value": round(world * steps * tokens / e2e_s, 1), "unit": UNIT, "h2d_bytes_per_step": tokens * 4, "d2h_bytes_per_step": 4, "steps": steps},
            "gpu_launches": int(gpu_launches), "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline, "extra": extra, "setup": info,
        })
        print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ workloads: serve / serve8k (configs 4, 5)
def build_requests(seed: int, count: int, vocab: int, min_in: int, max_in: int, min_out: int, max_out: int):
    """benches/bench.py:201-225: prompt length, output budget, then the prompt ids from one seeded stream."""
    rng = random.Random(seed)
    reqs = []
    for _ in range(count):
        n_in, n_out = rng.randint(min_in, max_in), rng.randint(min_out, max_out)
        reqs.append(([rng.randint(256, vocab - 1) for _ in range(n_in)], n_out))
    return reqs


def run_serve(args, long_context: bool) -> None:
    from tiny_llm_b200.batch import ContinuousBatcher
    from tiny_llm_b200.parallel import barrier, max_over_ranks, shard, sum_over_ranks
    from tiny_llm_b200.synthetic import weight_stream_bytes

    ext, model, model_ns, rank, world, device, info = setup(args)
    margs = model_ns.args
    slots = args.slots
    if long_context:
        total = args.requests or 64 * world
        out_len = 128
        all_reqs = build_requests(0, total, margs.vocab_size, 8192 - out_len, 8192 - out_len, out_len, out_len)
        prefill_step, max_seq = args.prefill_step or 1024, 8192 + PAGE_SIZE
        workload = (f"Qwen3-4B data-parallel serving, {total} requests at 8K context (prompt {8192 - out_len} + {out_len} output tokens) "
                    f"sharded i mod {world}, {slots} decode slots per GPU")
    else:
        total = args.requests or 128 * world
        all_reqs = build_requests(0, total, margs.vocab_size, 128, 1024, 32, 128)
        prefill_step, max_seq = args.prefill_step or 128, 1024 + 128 + PAGE_SIZE
        workload = f"Qwen3-4B continuous batching, {slots} concurrent requests per GPU, {total} requests, chunked prefill + paged KV"
    mine = shard(all_reqs, rank, world)
    model.decode_graph_max_seq_len = ((max_seq + PAGE_SIZE - 1) // PAGE_SIZE) * PAGE_SIZE
    model.prefill_graph_len = int(os.environ.get("TL_PREFILL_GRAPH", str(prefill_step)))  # captured chunk graph (0: operator path)

    def serve(reqs, timing=True, step=None):
        step = step or prefill_step
        model.prefill_graph_len = int(os.environ.get("TL_PREFILL_GRAPH", str(step)))
        batcher = ContinuousBatcher(model, None, [p for p, _ in reqs], max_seq_len=max_seq, batch_size=slots, prefill_step=step,
                                    verbose=False, device=device, max_new_tokens=[n for _, n in reqs])
        batcher.record_timing = timing
        t0 = time.perf_counter()
        batcher.run()
        torch.cuda.synchronize()
        return batcher, time.perf_counter() - t0

    # warm-up: a short queue through the same scheduler (captures the B-slot decode graph, sizes the pools)
    warm = [(p[: min(len(p), 2 * prefill_step)], 4) for p, _ in mine[: min(len(mine), slots + 2)]]
    # ... plus one prompt with a ONE-token tail chunk: that tail is a B = 1 decode step, whose engine (private packed
    # weight copies + graph capture, 30-900 ms depending on the host) otherwise gets built inside the timed region by the
    # first such prompt of the queue
    long_enough = [p for p, _ in mine if len(p) > prefill_step + 1]
    if long_enough:
        warm.append((long_enough[0][: prefill_step + 1], 2))
    serve(warm, timing=False)
    sampler = ClockSampler(device.index or 0)
    if rank == 0:
        sampler.start()
    launches0 = ext.launch_count()
    engine = model.decode_engine(slots)
    replays0 = engine.graph_replays
    barrier(device)
    torch.cuda.synchronize()
    batcher, wall = serve(mine)
    barrier(device)
    wall_max = max_over_ranks(wall, device)
    clocks = sampler.stop() if rank == 0 else None
    generated = sum(batcher.generated.values())
    total_generated = sum_over_ranks(generated, device)
    total_prefill = sum_over_ranks(batcher.prefill_tokens, device)
    gpu_ms = batcher.gpu_phase_ms()  # device time per phase (CUDA events); the wall-time lists include queueing behind the other phase
    decode_ms = sum(gpu_ms["decode"]) or sum(batcher.decode_step_ms)
    prefill_ms = sum(gpu_ms["prefill"]) or sum(batcher.prefill_chunk_ms)
    gpu_launches = engine.kernels_per_step * (engine.graph_replays - replays0) + (ext.launch_count() - launches0)
    steps_sorted = sorted(gpu_ms["decode"] or batcher.decode_step_ms)
    pct = lambda q: steps_sorted[min(len(steps_sorted) - 1, int(q * len(steps_sorted)))] if steps_sorted else None
    mine_stats = {
        "requests": len(mine), "wall_s": round(wall, 3), "generated_tokens": generated, "prefill_tokens": batcher.prefill_tokens,
        "decode_steps": batcher.decode_steps, "decode_tokens": batcher.decode_tokens,
        "output_tok_s": round(generated / wall, 1), "prefill_tok_s": round(batcher.prefill_tokens / (prefill_ms / 1e3), 1) if prefill_ms else None,
        "decode_tok_s": round(batcher.decode_tokens / (decode_ms / 1e3), 1) if decode_ms else None,
        "decode_step_ms_p50": round(pct(0.5), 3) if steps_sorted else None, "decode_step_ms_p95": round(pct(0.95), 3) if steps_sorted else None,
        "time_in_decode_s": round(decode_ms / 1e3, 3), "time_in_prefill_s": round(prefill_ms / 1e3, 3),
        "timing": "per-phase device time from CUDA events on the scheduler's stream; wall_s is host wall-clock of the whole run",
        "prefill_chunk_ms_p50": round(sorted(gpu_ms["prefill"])[len(gpu_ms["prefill"]) // 2], 3) if gpu_ms["prefill"] else None,
        "prefill_chunk_ms_max": round(max(gpu_ms["prefill"]), 3) if gpu_ms["prefill"] else None,
        "prefill_chunks": len(gpu_ms["prefill"]), "prefill_chunks_over_2x_p50": (sum(1 for v in gpu_ms["prefill"] if v > 2 * sorted(gpu_ms["prefill"])[len(gpu_ms["prefill"]) // 2]) if gpu_ms["prefill"] else None),
        "row_variant_replays": {str(k): v for k, v in getattr(engine, "variant_replays", {}).items()},
        "graph_captures": {"decode": getattr(engine, "captures", None), "prefill": sum(getattr(e, "captures", 0) for e in getattr(model, "_prefill_engines", {}).values())},
        "peak_active_requests": batcher.peak_active_requests, "peak_live_pages": batcher.peak_live_pages,
        "peak_live_kv_gb": round(batcher.peak_live_pages * 2 * margs.num_key_value_heads * PAGE_SIZE * margs.head_dim * 2 / 1e9, 2),
    }
    # config 4 only: the same queue with larger prefill chunks (the chunk size is the scheduler's knob; 128 is the
    # reference protocol's default and stays the headline)
    sweep = []
    if not long_context and world == 1 and not args.no_extra and not args.prefill_step:
        for step in (256, 512):
            serve([(p[: min(len(p), 2 * step)], 4) for p, _ in mine[: min(len(mine), slots + 2)]], timing=False, step=step)
            b2, w2 = serve(mine, step=step)
            ms2 = b2.gpu_phase_ms()
            sweep.append({"prefill_step": step, "output_tok_s": round(sum(b2.generated.values()) / w2, 1), "wall_s": round(w2, 3),
                          "time_in_prefill_s": round(sum(ms2["prefill"]) / 1e3, 3), "time_in_decode_s": round(sum(ms2["decode"]) / 1e3, 3)})
    if rank == 0:
        peak = measured_peaks()
        # decode-step roofline: weights once + every live request's K/V once per step (median step)
        line = base_line(args, world, "serve8k" if long_context else "serve")
        iters = batcher.tick
        line.update({
            "value": round(total_generated / wall_max, 1), "steps": iters, "warmup": len(warm), "ms_per_step": round(1e3 * wall_max / max(iters, 1), 3),
            "scaling": "weak" if not args.requests else "strong",
            "config": {"workload": workload, "slots": slots, "prefill_step": prefill_step, "page_size": PAGE_SIZE, "seed": 0,
                       "requests_total": total, "parallelism": f"dp{world}", "max_seq_len": max_seq,
                       "protocol": "benches/bench.py:351-572 (run_batch_requests_serving): token-id requests, no tokenizer, greedy",
                       "l2_policy": "inputs larger than L2: every decode step streams 2.14 GB of weights + the live K/V"},
            "e2e": {"value": round(total_generated / wall_max, 1), "unit": UNIT,
                    "h2d_bytes_per_step": slots * 4 + engine.upload_bytes_per_step(), "d2h_bytes_per_step": slots * 4,
                    "note": "the serving loop IS the public API: tokens go host -> device and sampled ids device -> host every step"},
            "gpu_launches": int(gpu_launches), "clocks": clocks,
            "serving": mine_stats, "prefill_tok_s_all_ranks": round(total_prefill / wall_max, 1),
            "extra": {"prefill_step_sweep": sweep} if sweep else {},
            "roofline": {"bound": "hbm", "unit": "GB/s", "peak": peak["hbm_gbs"], "peak_source": peak["source"], "traffic": None,
                         "kernel": "whole decode step at the median live context (weights + live K/V once)",
                         "achieved": None, "frac": None},
            "setup": info,
        })
        if steps_sorted and batcher.decode_steps:
            avg_ctx_tokens = batcher.peak_live_pages / max(model.num_hidden_layers, 1) * PAGE_SIZE  # upper bound: pages at the peak
            step_bytes = weight_stream_bytes(margs) + 147456 * avg_ctx_tokens
            achieved = step_bytes / (pct(0.5) / 1e3) / 1e9
            line["roofline"].update({"achieved": round(achieved, 1), "frac": round(achieved / peak["hbm_gbs"], 4),
                                     "bytes_per_step_at_peak": int(step_bytes)})
        print(json.dumps(line), flush=True)


# ------------------------------------------------------------- CPU reference arm
CPU_SAMPLE_LAYERS = 8


def _load_standalone(name: str, path: Path):
    """Import one source file without its package (the reference arm must not pull in the product
    package: importing tiny_llm_b200 loads libtiny_llm_b200.so)."""
    spec = importlib.util.spec_from_file_location(name, path)
    module = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(module)
    return module


def run_cpu_baseline(sample_steps: int, warmup_steps: int = 1, mode: str = "decode") -> dict:
    """tiny_llm_ref's CPU-capable path (oracle.model) on the host cores, bounded: the same synthetic
    Qwen3-4B shapes with CPU_SAMPLE_LAYERS of the 36 transformer blocks (+ embedding and tied head), an
    8-token prompt and a few decode steps; the per-token time is scaled to the full depth by weight
    bytes (a decode step on the CPU is one pass over every dense weight).  Threads are pinned to
    min(32, cores): the bf16 GEMV of torch scales poorly past that and oversubscribed runs made the
    round-1 number swing by 80x."""
    from oracle.model import ReferenceCpuModel, greedy_decode

    synthetic = _load_standalone("_bench_synthetic", ROOT / "tiny-llm_b200" / "tiny_llm_b200" / "synthetic.py")
    cores = os.cpu_count() or 1
    threads = min(32, cores)
    # Pin the process to `threads` cores BEFORE the first parallel CPU op creates torch's worker pool (the workers
    # inherit the mask): on a 128-thread host the unpinned run swung 3x between two launches on the same box (22 vs
    # 69 ms per step: workers migrating across NUMA nodes away from the first-touched weights).
    allowed = None
    try:
        allowed = sorted(os.sched_getaffinity(0))
        os.sched_setaffinity(0, set(allowed[:threads]))
    except (AttributeError, OSError):
        allowed = None
    torch.set_num_threads(threads)
    try:
        return _cpu_baseline_pinned(sample_steps, warmup_steps, mode, synthetic, cores, threads)
    finally:
        if allowed is not None:
            os.sched_setaffinity(0, set(allowed))  # the calling thread only; the CPU workers keep their cores


def _cpu_baseline_pinned(sample_steps, warmup_steps, mode, synthetic, cores, threads) -> dict:
    from oracle.model import ReferenceCpuModel, greedy_decode

    full = synthetic.CONFIGS[MODEL]
    ns = synthetic.synthetic_qwen3(MODEL, seed=0, device="cpu", num_hidden_layers=CPU_SAMPLE_LAYERS)
    model = ReferenceCpuModel(ns)
    del ns
    H, inter = full["hidden_size"], full["intermediate_size"]
    q_w, kv_w = full["num_attention_heads"] * full["head_dim"], full["num_key_value_heads"] * full["head_dim"]
    layer_w = H * (q_w + 2 * kv_w) + q_w * H + 3 * H * inter
    head_w = full["vocab_size"] * H
    if mode == "prefill":
        tokens = 128
        prompt = synthetic_prompt(1000, tokens, model.args.vocab_size)
        samples = []
        for _ in range(1 + sample_steps):
            timings: dict = {}
            greedy_decode(model, prompt, 1, timings=timings)
            samples.append(timings["prefill_s"])
        sample_s = statistics.median(samples[1:])
        scale = (full["num_hidden_layers"] * layer_w) / (CPU_SAMPLE_LAYERS * layer_w)  # the head sees one row only
        value = tokens / (sample_s * scale)
        return {"value": round(value, 3), "unit": UNIT, "cores": threads, "host_cores": cores, "kind": "port",
                "sample": (f"oracle.model prefill of a {tokens}-token prompt, {CPU_SAMPLE_LAYERS} of {full['num_hidden_layers']} blocks, "
                           f"median of {sample_steps} ({1e3 * sample_s:.0f} ms), scaled x{scale:.2f} to the full depth"),
                "ms_per_step": round(1e3 * sample_s * scale, 1)}
    prompt = synthetic_prompt(1000, 8, model.args.vocab_size)
    timings = {}
    greedy_decode(model, prompt, 1 + warmup_steps + sample_steps, timings=timings)
    per_step = sorted(timings["decode_s"][warmup_steps:])
    scale = (full["num_hidden_layers"] * layer_w + head_w) / (CPU_SAMPLE_LAYERS * layer_w + head_w)
    # Best of N: the GPU boxes' hosts are shared and a CPU decode step (a 2.4 GB GEMV sweep) swings 2-3x from step to
    # step inside one run (median 20-25 ms, interquartile range > 2x the median on two consecutive runs); the fastest
    # step is the reproducible one, and it is the most favourable figure for the CPU path.
    median_s = statistics.median(per_step)
    sample_s = per_step[0]
    q1, q3 = per_step[len(per_step) // 4], per_step[(3 * len(per_step)) // 4]
    spread = (q3 - q1) / median_s if median_s else 0.0  # interquartile range over the median
    value = 1.0 / (sample_s * scale)
    return {"value": round(value, 4), "unit": UNIT, "cores": threads, "host_cores": cores, "kind": "port",
            "sample": (f"oracle.model (reference CPU path: dense bf16 weights, readable ops), {CPU_SAMPLE_LAYERS} of "
                       f"{full['num_hidden_layers']} Qwen3-4B blocks + tied head, 8-token prompt, best of {len(per_step)} decode steps "
                       f"({1e3 * sample_s:.1f} ms; median {1e3 * median_s:.0f} ms, interquartile spread {100 * spread:.0f} %: shared host), {threads} pinned threads, scaled x{scale:.2f} by weight bytes to the full depth"),
            "ms_per_step": round(1e3 * sample_s * scale, 1), "spread": round(spread, 3)}


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps
    workload = args.workload
    mode = "prefill" if workload == "prefill" else "decode"
    sample = min(max(steps, 9), 16) if mode == "decode" else 2  # a CPU decode step is 20-70 ms: 9-16 samples stay well under a second
    base = run_cpu_baseline(sample_steps=sample, warmup_steps=3, mode=mode)
    line = {
        "impl": "reference",
        "metric": METRICS[workload],
        "value": base["value"],
        "unit": UNIT,
        "n_gpus": args.gpus,
        "steps": sample,
        "warmup": 3,
        "ms_per_step": base["ms_per_step"],
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "bf16 weights/activations (dequantised W4), fp32 attention",
        "data": "synthetic (same random Qwen3-4B-shaped weights as the GPU arm)",
        "config": {"workload": f"Qwen3-4B single-request {mode}, batch=1, reference CPU path on host cores", "prompt_len": 8 if mode == "decode" else 128,
                   "note": "MLX cannot be installed here and the reference's native ops are GPU-only; this is the oracle port of tiny_llm_ref's CPU-capable path"},
        "cpu_baseline": {"kind": base["kind"], "cores": base["cores"], "sample": base["sample"], "value": base["value"], "unit": UNIT},
        "e2e": {"value": base["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(METRICS), default="decode")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the sweeps / secondary measurements under `extra`")
    ap.add_argument("--requests", type=int, default=0, help="serve/serve8k: total requests over all ranks")
    ap.add_argument("--slots", type=int, default=64, help="serve/serve8k: decode slots per GPU")
    ap.add_argument("--prefill-step", type=int, default=0)
    ap.add_argument("--prompt-len", type=int, default=0, help="prefill: prompt tokens (default 4096)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="decode: write the last timed step's logits and token as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = {"decode": 128, "prefill": 8}.get(args.workload, 0)
    if args.workload in ("decode", "prefill") and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "decode"):
        ap.error("--dump-outputs is implemented for --impl ours --workload decode")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "decode":
        run_decode(args)
    elif args.workload == "prefill":
        run_prefill(args)
    else:
        run_serve(args, long_context=args.workload == "serve8k")


if __name__ == "__main__":
    main()
