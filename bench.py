#!/usr/bin/env python
"""bench.py — decode tokens/s, Llama-2-7B-shaped Q4_K_M GGUF, batch 1 (BASELINE.json metric, configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one single-token decode pass of the whole hot path: ONE launch of the persistent step kernel (csrc/stream.cuh) whose
phases are the 129 mat-vecs over 225 weight tensors, 32 attention blocks at a context of 256..511 tokens, the embedding row and the greedy pick.  Workload: synthetic 7B-shaped model (random valid quant blocks in the reference's Q4_K_M tensor mix,
3.8 GB of weights ≫ the 126 MB L2, so every step streams its inputs from HBM — no L2 flush needed), 256-token prompt
prefilled untimed, then W warm-up + K timed decode steps (the context grows past 512 when K needs it).

  value     device-timed: K steps replayed as CUDA graphs with the token fed back on the device (the pick phase), CUDA events on the
            launching stream, max over ranks; tokens/s summed over ranks (replicas: one sequence per GPU, weak scaling).  The
            logits stay on the device (no D2H inside this number; e2e below includes the step's result read-back)
  e2e       the same K steps through the public API (llm.eval([tok]) + llm.sample(top_k=1)): token H2D, the greedy pick made on
            the device and its 8-byte read-back inside the timed region
  roofline  dominant kernel k_step, mat-vec phases (HBM-bound): the GGUF bytes of the weights the 129 mat-vec phases of a step read
            (4005.4 MB) ÷ the duration of a launch that holds exactly those phases (no attention / embedding / pick), measured live
            as a CUDA graph between CUDA events on the engine's stream; peak = MEASURED_PEAKS.json hbm_gbs; traffic = ncu dram
            bytes (profiles/k_step_traffic.json).  roofline.step = the same for the whole step (weights + KV + logits bytes ÷
            device-timed step)
  cpu_baseline / --impl reference: the UNMODIFIED reference (oracle/_ref/libctransformers_ref.so) on the host cores, same
            model file, same prompt, bounded sample, thread count swept (ggml's spin-wait pool collapses when oversubscribed).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

CTX = 512
PROMPT = 256
MODEL_DIR = Path(os.environ.get("CTB_MODEL_DIR", "/tmp/ctb_models"))
REF_SO = ROOT / "oracle" / "_ref" / "libctransformers_ref.so"


# --workload: the default is the BASELINE.json headline (configs[1]); "falcon7b" is configs[3] (not a driver bench line)
WORKLOADS = {
    "llama2-7b": dict(file="llama2-7b-shaped.Q4_K_M.synthetic.gguf", arch="llama", shape="LLAMA2_7B", ftype="Q4_K_M", lo=259,
                      metric="decode tokens/s Llama-2-7B Q4_K_M b=1", dtype="int8 (q4_K/q6_K weights x q8_K activations, mma.sync u8 x s8 -> exact int32), fp32 combine in the reference's order",
                      name="Llama-2-7B-shaped Q4_K_M GGUF"),
    "falcon7b": dict(file="falcon-7b-shaped.Q5_K_M.synthetic.gguf", arch="falcon", shape="FALCON_7B_SHAPED", ftype="Q5_K_M", lo=0,
                     metric="decode tokens/s Falcon-7B Q5_K_M b=1", dtype="int8 (q5_K/q6_K weights x q8_K activations, mma.sync u8 x s8 -> exact int32), fp32 combine in the reference's order",
                     name="Falcon-7B-shaped (n_embd 4608, multi-query) Q5_K_M GGUF"),
}
# configs[2]: prompt ingestion of the same model (the batched kernel of csrc/prefill.cuh); a separate bench line, not the driver's
WORKLOADS["prefill2048"] = dict(WORKLOADS["llama2-7b"], metric="prefill tokens/s Llama-2-7B Q4_K_M 2048-token prompt",
                                dtype="int8 mma.sync (u8 scale digits x s8 Q8_K activations, exact int32), fp32 combine in the reference's order")
# configs[4]: the 13B shape, tensor-sharded over the ranks (--mode tp); also runs on one GPU (world 1 = the plain engine)
WORKLOADS["llama2-13b"] = dict(file="llama2-13b-shaped.Q4_K_M.synthetic.gguf", arch="llama", shape="LLAMA2_13B", ftype="Q4_K_M", lo=259,
                               metric="decode tokens/s Llama-2-13B Q4_K_M b=1 tensor-sharded", dtype=WORKLOADS["llama2-7b"]["dtype"],
                               name="Llama-2-13B-shaped Q4_K_M GGUF")
WL = WORKLOADS["llama2-7b"]


def model_path():
    return MODEL_DIR / WL["file"]


def ensure_model(rank, world, barrier):
    from ctransformers_b200 import synth
    p = model_path()
    if rank == 0 and not p.exists():
        MODEL_DIR.mkdir(parents=True, exist_ok=True)
        tmp = p.with_suffix(".tmp")
        (synth.write_llama if WL["arch"] == "llama" else synth.write_falcon)(tmp, getattr(synth, WL["shape"]), WL["ftype"], seed=0)
        tmp.rename(p)
    barrier()
    return p


def prompt_ids():
    import numpy as np
    from ctransformers_b200 import synth
    ids = np.random.default_rng(1).integers(WL["lo"], getattr(synth, WL["shape"]).n_vocab, PROMPT).tolist()
    if WL["arch"] == "llama":
        ids[0] = 1
    return ids


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.proc = index, [], threading.Event(), None

    def run(self):
        # one long-running nvidia-smi in loop mode (a sample every 20 ms) instead of one process per sample
        cmd = ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "20"]
        try:
            self.proc = subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if line.strip():
                    self.rows.append([c.strip() for c in line.split(",")])
                if self.stop_flag.is_set():
                    break
        except Exception:
            pass
        finally:
            try:
                self.proc.kill()
            except Exception:
                pass

    def summary(self):
        self.stop_flag.set()
        try:
            self.proc.kill()
        except Exception:
            pass
        self.join(timeout=6)
        if not self.rows:   # loop mode unavailable: one direct query as a last resort
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(self.rows)}


def hbm_peak():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def context_for(n_tokens):
    """CTX, or longer when the prompt, warm-up and timed steps do not fit in it (so --steps is never cut short)."""
    return max(CTX, n_tokens + 1)


def dump_outputs(out_dir, llm, tokens):
    """--dump-outputs: what a caller of the timed path holds after its last step, for comparing two builds output for output
    (same arguments, same inputs): the greedy tokens of the timed steps, that step's logits and hidden state."""
    import numpy as np
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    np.save(d / "tokens.npy", np.array(tokens, np.float64))
    np.save(d / "logits.npy", np.array(llm.logits, np.float32))
    np.save(d / "embeddings.npy", np.array(llm.embeddings, np.float32))


def kv_bytes_per_step(n_layer, n_embd_gqa, t_avg):
    return 2 * n_layer * n_embd_gqa * t_avg * 2 + 2 * n_layer * n_embd_gqa * 2


def pick_threads(llm, tok, cores):
    """ggml's spinning thread pool degrades badly when oversubscribed; sweep like BASELINE.md's plan and keep the fastest."""
    forced = os.environ.get("CTB_REF_THREADS")
    if forced:
        return max(1, min(cores, int(forced))), {}
    cands = sorted({c for c in (4, 8, 16, 24, 32, 48, 64, cores // 2, cores) if 1 <= c <= cores})
    timing = {}
    for c in cands:
        t0 = time.perf_counter()
        for _ in range(2):
            llm.eval([tok], threads=c)
        timing[c] = (time.perf_counter() - t0) / 2
        if timing[c] > 4 * min(timing.values()):
            break                      # far past the optimum, more threads only get slower
    return min(timing, key=timing.get), {str(k): round(v, 4) for k, v in timing.items()}


def run_reference(args, rank, world, barrier):
    """The reference's own CPU implementation on the host cores (rank 0 only)."""
    if rank != 0:
        return
    if not REF_SO.exists():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libctransformers_ref.so was not built (needs /root/reference at build time)"}))
        return
    from ctransformers_b200 import AutoModelForCausalLM
    cores = os.cpu_count() or 1
    p = ensure_model(0, 1, lambda: None)
    steps = max(1, args.steps)
    ctx = context_for(PROMPT + 2 * 9 + args.warmup + steps)        # 9: the most thread counts pick_threads tries, 2 evals each
    llm = AutoModelForCausalLM.from_pretrained(str(p), lib=str(REF_SO), context_length=ctx, threads=min(cores, 16))
    ids = prompt_ids()
    llm.eval(ids, batch_size=256, threads=min(cores, 32))           # untimed prefill, one chunk
    tok = llm.sample(top_k=1, repetition_penalty=1.0, seed=0)
    threads, sweep = pick_threads(llm, tok, cores)
    for _ in range(args.warmup):
        llm.eval([tok], threads=threads); tok = llm.sample(top_k=1, repetition_penalty=1.0, seed=0)
    t0 = time.perf_counter()
    tokens = []
    for _ in range(steps):
        llm.eval([tok], threads=threads); tok = llm.sample(top_k=1, repetition_penalty=1.0, seed=0)
        tokens.append(tok)
    dt = time.perf_counter() - t0
    v = steps / dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, llm, tokens)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "tokens/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE,
        "data": "synthetic", "config": workload_config(1, ctx),
        "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": threads, "kind": "reference", "host_cores": cores, "thread_sweep_s_per_token": sweep,
                         "sample": f"{steps} decode steps at context {PROMPT}+ after a {PROMPT}-token prompt, llm.eval+llm.sample, unmodified reference CPU build (AVX2), {threads} threads (best of the sweep)"},
        "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


METRIC = WL["metric"]
DTYPE = WL["dtype"]


def run_prefill(args, path, rank, world, local, barrier, max_over_ranks, group):
    """configs[2]: a 2048-token prompt through llm.eval(tokens, batch_size=512) — 4 reference-sized chunks, 64 batched launches of
    32 tokens each (csrc/prefill.cuh) + the head mat-vec of the last token.  One "step" = one whole prompt."""
    import numpy as np
    from ctransformers_b200 import AutoModelForCausalLM, synth
    n_prompt, ctx = 2048, 2304
    llm = AutoModelForCausalLM.from_pretrained(str(path), context_length=ctx)
    shape = getattr(synth, WL["shape"])
    ids = np.random.default_rng(1).integers(WL["lo"], shape.n_vocab, n_prompt).tolist()
    ids[0] = 1
    steps, W = max(1, args.steps), 1

    def once():
        llm._context = []
        llm.eval(ids, batch_size=512)
        return llm.ctb_llm_last_eval_ms()
    for _ in range(W):
        once()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    t0 = time.perf_counter()
    dev_ms = [once() for _ in range(steps)]
    barrier()
    wall = max_over_ranks(time.perf_counter() - t0)
    clocks = sampler.summary()
    ms = max_over_ranks(sum(dev_ms))
    tok = llm.sample(top_k=1, repetition_penalty=1.0, seed=0)
    mk = 0   # Σ M·K over the mat-muls of a token
    for (m, k, cnt) in ((shape.n_embd, shape.n_embd, 2), (shape.n_embd // shape.n_head * shape.n_head_kv, shape.n_embd, 2), (shape.n_ff, shape.n_embd, 2), (shape.n_embd, shape.n_ff, 1)):
        mk += m * k * cnt * shape.n_layer
    flops = 2.0 * n_prompt * mk
    peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()) if (ROOT / "MEASURED_PEAKS.json").exists() else {}
    tf_peak = float(peaks.get("bf16_tflops", 1590.0))
    achieved = flops / (ms / steps / 1e3) / 1e12
    result = {
        "metric": METRIC, "value": world * n_prompt * steps / (ms / 1e3), "unit": "tokens/s", "n_gpus": world, "steps": steps, "warmup": W,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
        "config": {"workload": WL["name"] + " (synthetic random quant blocks), one 2048-token prompt per step, llm.eval(tokens, batch_size=512), ctx 2304",
                   "global_batch": world, "prompt": n_prompt, "batch_size": 512, "parallelism": f"replicas x{world}",
                   "l2": "each batched launch streams the 3.8 GB of layer weights once: inputs exceed the 126 MB L2"},
        "clocks": clocks,
        "e2e": {"value": world * n_prompt * steps / wall, "unit": "tokens/s", "h2d_bytes_per_step": 64 * 33 * 16, "d2h_bytes_per_step": 4,
                "how": "llm.eval(prompt, batch_size=512) wall clock per prompt: 64 state uploads of 33 x 16 B, the look-ahead pick read back"},
        "gpu_launches": steps * (n_prompt // 32 + 1),
        "roofline": {"bound": "tensor", "kernel": "k_pstep", "achieved": achieved, "peak": tf_peak, "unit": "TFLOP/s", "frac": achieved / tf_peak, "traffic": None,
                     "peak_source": "MEASURED_PEAKS.json bf16_tflops (no int8 figure is measured on this pool; the kernel's dense int8 mma.sync does 2 digit products per useful MAC)",
                     "algorithmic_flops_per_step": flops, "how": "2 * N * sum(M*K) of the layer mat-muls / device-timed prompt"},
        "first_token_after_prompt": int(tok),
    }
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, llm, [tok])
        print(json.dumps(result))
    group.close()


def run_tp(args, path, rank, world, local, barrier, max_over_ranks, group):
    """configs[4]: ONE sequence decoded by all ranks together (strong scaling): every rank holds its heads / n_ff slice of the
    layer weights, two NCCL all-reduces of n_embd floats per layer inside the step's CUDA graph (csrc/engine.cu build_ops)."""
    import torch
    import torch.distributed as dist
    from ctransformers_b200 import LLM, Config, synth
    from ctransformers_b200.tp import tensor_parallel_ticket
    shape = getattr(synth, WL["shape"])
    if world > 1:
        ticket = tensor_parallel_ticket()
    else:
        ticket = None
    steps = max(1, args.steps)
    W = max(args.warmup, 3)
    ctx = context_for(PROMPT + W + steps)
    llm = LLM(str(path), config=Config(context_length=ctx), tp=ticket)
    ids = prompt_ids()
    llm.eval(ids, batch_size=256)
    tok = llm.sample(top_k=1, repetition_penalty=1.0, seed=0)
    for _ in range(W):
        llm.eval([tok]); tok = llm.sample(top_k=1, repetition_penalty=1.0, seed=0)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    t0 = time.perf_counter()
    e2e_tokens = []
    for _ in range(steps):
        llm.eval([tok]); tok = llm.sample(top_k=1, repetition_penalty=1.0, seed=0)
        e2e_tokens.append(tok)
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    # device-timed: K steps with the token fed back on the device (every rank picks from the same all-reduced logits)
    llm._context = []
    llm.eval(ids, batch_size=256)
    first = llm.sample(top_k=1, repetition_penalty=1.0, seed=0)
    out = (C.c_int * (W + steps))()
    assert llm.ctb_llm_decode_greedy(first, PROMPT, W, out) >= 0
    barrier()
    ms = llm.ctb_llm_decode_greedy(int(out[W - 1]), PROMPT + W, steps, out)
    barrier()
    clocks = sampler.summary()
    assert ms > 0
    ms = max_over_ranks(ms)
    tokens_dev = list(out[:steps])
    ranks_agree = all(t == tokens_dev for t in group.gather_ints(tokens_dev))
    peak, peak_src = hbm_peak()
    wbytes = int(llm.ctb_llm_weight_bytes_per_token())           # this rank's share
    wb_max = max_over_ranks(float(wbytes))
    achieved = wb_max / (ms / 1e3 / steps) / 1e9
    launches = int(llm.ctb_llm_launches_per_token())
    result = {
        "metric": METRIC, "value": steps / (ms / 1e3), "unit": "tokens/s", "n_gpus": world, "steps": steps, "warmup": W, "ms_per_step": ms / steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
        "config": {"workload": WL["name"] + f" (synthetic random quant blocks), batch=1 decode, ctx={ctx}, 256-token prompt then decode", "global_batch": 1,
                   "ctx": ctx, "prompt": PROMPT, "parallelism": f"tp{world} (column-parallel q/k/v/gate/up, row-parallel wo/down, {2 * shape.n_layer} all-reduces of {shape.n_embd} floats per token over NCCL)",
                   "l2": "each rank streams its GBs of weights per step: inputs exceed the 126 MB L2"},
        "clocks": clocks,
        "e2e": {"value": steps / e2e_s, "unit": "tokens/s", "h2d_bytes_per_step": 16, "d2h_bytes_per_step": 8,
                "how": "llm.eval([tok]) + llm.sample(top_k=1) per step on every rank (same calls, same seed), wall clock, max over ranks"},
        "gpu_launches": launches * steps, "launches_per_token": launches, "comm_nranks": world,
        "roofline": {"bound": "hbm", "kernel": "k_step (all phases of a rank's step, exchanges included)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": None, "peak_source": peak_src, "weight_bytes_per_rank_per_step": wb_max,
                     "how": "largest rank's weight bytes per step / device-timed step (so the NCCL exchanges and launch boundaries count against it)"},
        "greedy_tokens_match_e2e": tokens_dev[:steps] == e2e_tokens[:steps], "ranks_agree": ranks_agree,
    }
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, llm, tokens_dev)
        print(json.dumps(result))
    del llm
    group.close()


def workload_config(n, ctx):
    return {"workload": WL["name"] + f" (synthetic random quant blocks), batch=1 decode, ctx={ctx}, 256-token prompt then decode",
            "global_batch": n, "ctx": ctx, "prompt": PROMPT, "parallelism": f"replicas x{n} (one sequence per GPU, no collective)",
            "l2": "inputs (GBs of weights per step) exceed the 126 MB L2; no flush needed"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=192)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="llama2-7b", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default="replicas", choices=["replicas", "tp"],
                    help="tp: ONE sequence, layer weights tensor-sharded over the ranks (BASELINE configs[4]; implies --workload llama2-13b unless one is given)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as DIR/<name>.npy (tokens, logits, embeddings)")
    args = ap.parse_args()
    global WL, METRIC, DTYPE
    if args.mode == "tp" and args.workload == "llama2-7b" and "--workload" not in sys.argv:
        args.workload = "llama2-13b"
    WL = WORKLOADS[args.workload]
    METRIC, DTYPE = WL["metric"], WL["dtype"]

    from ctransformers_b200 import replicas
    who = replicas.Rank.from_env()
    rank, world, local = who.rank, who.world, who.local
    if args.impl == "reference":
        if not replicas.reference_rank_runs(who):
            return                       # under torchrun only rank 0 times the CPU reference
        return run_reference(args, rank, world, lambda: None)

    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    group = replicas.Group(who, backend="nccl", device=f"cuda:{local}")

    def barrier():
        group.barrier(torch.cuda.synchronize)

    max_over_ranks = group.max

    from ctransformers_b200 import AutoModelForCausalLM, synth
    path = ensure_model(rank, world, barrier)
    if args.mode == "tp":
        return run_tp(args, path, rank, world, local, barrier, max_over_ranks, group)
    if args.workload == "prefill2048":
        return run_prefill(args, path, rank, world, local, barrier, max_over_ranks, group)
    steps = max(1, args.steps)
    W = max(args.warmup, 3)
    ctx = context_for(PROMPT + W + steps)
    llm = AutoModelForCausalLM.from_pretrained(str(path), context_length=ctx)
    shape = getattr(synth, WL["shape"])
    ids = prompt_ids()

    def prefill():
        llm._context = []
        llm.eval(ids, batch_size=256)
        return llm.sample(top_k=1, repetition_penalty=1.0, seed=0)

    # ------------------------------------------------------------------ end to end through the public API ("e2e")
    # (first: the engine's look-ahead only runs while decoding appends to the cache, see Engine::after_eval)
    tok = prefill()
    for _ in range(W):
        llm.eval([tok]); tok = llm.sample(top_k=1, repetition_penalty=1.0, seed=0)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    t0 = time.perf_counter()
    e2e_tokens = []
    for _ in range(steps):
        llm.eval([tok])                                   # H2D {token, n_past}; stream sync
        tok = llm.sample(top_k=1, repetition_penalty=1.0, seed=0)   # device penalty + top-k, candidates D2H, host draw
        e2e_tokens.append(tok)
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e = replicas.aggregate_tokens_per_s(world, steps, e2e_s * 1e3)
    device_samples = int(llm.ctb_llm_device_samples())

    # ------------------------------------------------------------------ device-timed ("value")
    first = prefill()
    out = (C.c_int * (W + steps))()
    assert llm.ctb_llm_decode_greedy(first, PROMPT, W, out) >= 0                      # warm-up steps at n_past = 256..
    barrier()
    ms = llm.ctb_llm_decode_greedy(int(out[W - 1]), PROMPT + W, steps, out)           # K timed steps, CUDA events inside
    barrier()
    clocks = sampler.summary()                                                        # covers the e2e AND the device-timed region
    assert ms > 0
    ms = max_over_ranks(ms)
    tokens_dev = list(out[:steps])
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, llm, tokens_dev)                              # before the profiling passes below overwrite them
    replicas_agree = all(t == tokens_dev for t in group.gather_ints(tokens_dev))   # every replica decodes the same sequence
    value = replicas.aggregate_tokens_per_s(world, steps, ms)

    # ------------------------------------------------------------------ roofline
    peak, peak_src = hbm_peak()
    wbytes = int(llm.ctb_llm_weight_bytes_per_token())
    t_avg = PROMPT + W + steps / 2
    gqa = shape.n_embd // shape.n_head * shape.n_head_kv
    step_bytes = wbytes + kv_bytes_per_step(shape.n_layer, gqa, t_avg) + shape.n_vocab * 4
    achieved = step_bytes / (ms / 1e3 / steps) / 1e9
    ms_kind = (C.c_double * 4)()
    cnt_kind = (C.c_int * 4)()
    prof_steps = 4
    for i in range(prof_steps):
        llm.ctb_llm_profile_step(tokens_dev[i], PROMPT + W + steps // 2 + i - prof_steps, ms_kind, cnt_kind)
    # dominant kernel = k_step's mat-vec phases: a launch holding exactly those, replayed as a CUDA graph between two CUDA events
    # on the engine's stream (after everything else, so the KV cache it leaves behind does not matter)
    n_mv = C.c_long(0)
    mv_ms = llm.ctb_llm_time_matvec_only(32, C.byref(n_mv))
    mv_ms = max_over_ranks(mv_ms)
    n_mv = max(1, n_mv.value)
    mv_achieved = wbytes / (mv_ms / 1e3) / 1e9
    traffic = None
    tf = ROOT / "profiles" / "k_step_traffic.json"
    if tf.exists() and args.workload == "llama2-7b":
        traffic = json.loads(tf.read_text()).get("dram_bytes_per_matvec_phase_avg")
    roofline = {
        "bound": "hbm", "kernel": "k_step (mat-vec phases)", "achieved": mv_achieved, "peak": peak, "unit": "GB/s", "frac": mv_achieved / peak, "traffic": traffic,
        "peak_source": peak_src, "matvec_phases_per_step": n_mv, "algorithmic_bytes_per_phase": wbytes / n_mv, "avg_phase_us": 1e3 * mv_ms / n_mv,
        "how": "weight bytes of the step's mat-vec phases / the duration of a k_step launch holding exactly those phases (no attention, embedding, pick), replayed as a CUDA graph, CUDA events on the launching stream, 32 replays; traffic = ncu dram bytes per phase",
        "step": {"achieved": achieved, "frac": achieved / peak, "bytes_per_step": step_bytes, "weight_bytes_per_step": wbytes,
                 "frac_vs_3.9GB_weights_only": (3.9e9 / (ms / 1e3 / steps) / 1e9) / peak,
                 "how": "weights + KV + logits bytes of a whole decode step / device-timed step (all kernels)"},
        "eager_ms_per_step_by_kind": {"matvec": ms_kind[0] / prof_steps, "attention": ms_kind[1] / prof_steps, "other": ms_kind[3] / prof_steps,
                                      "how": f"un-fused eager pass (one kernel per op), CUDA event after every kernel, {prof_steps} steps (share of the step by op class)"},
    }

    result = {
        "metric": METRIC, "value": value, "unit": "tokens/s", "n_gpus": world, "steps": steps, "warmup": W,
        "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": DTYPE, "data": "synthetic", "config": workload_config(world, ctx),
        "clocks": clocks,
        "e2e": {"value": e2e, "unit": "tokens/s", "h2d_bytes_per_step": 16, "d2h_bytes_per_step": 8,
                "how": "llm.eval([tok]) + llm.sample(top_k=1, repetition_penalty=1.0) per step, wall clock between device syncs; per step: H2D {token, position, step, n_total} (16 B), D2H {arg-max of the logits, number of logits equal to it} (8 B) — a greedy sample() is answered by the pick the engine made on the device (a sampled one would add the 64-token window up and a 2 KB candidate block down); the logits stay on the device until llm.logits is asked for",
                "lookahead_hits": int(llm.ctb_llm_speculative_hits()), "device_samples": device_samples},
        "value_excludes": "logits D2H (kept on the device; e2e includes the step's result read-back)",
        "gpu_launches": int(llm.ctb_llm_launches_per_token()) * steps,
        "roofline": roofline,
        "greedy_tokens_match_e2e": tokens_dev[:steps] == e2e_tokens[:steps], "replicas_agree": replicas_agree,
    }

    if rank == 0 and world == 1 and not args.no_cpu_baseline and REF_SO.exists():
        del llm
        cores = os.cpu_count() or 1
        ref = AutoModelForCausalLM.from_pretrained(str(path), lib=str(REF_SO), context_length=CTX, threads=min(cores, 16))
        n_prompt, n_dec = PROMPT, 12
        ref.eval(ids[:n_prompt], batch_size=256, threads=min(cores, 32))
        t = ref.sample(top_k=1, repetition_penalty=1.0, seed=0)
        threads, sweep = pick_threads(ref, t, cores)
        t0 = time.perf_counter()
        for _ in range(n_dec):
            t = ref.sample(top_k=1, repetition_penalty=1.0, seed=0)
            ref.eval([t], threads=threads)
        dt = time.perf_counter() - t0
        result["cpu_baseline"] = {"value": n_dec / dt, "unit": "tokens/s", "cores": threads, "kind": "reference", "host_cores": cores, "thread_sweep_s_per_token": sweep,
                                  "sample": f"{n_dec} decode steps after a {n_prompt}-token prompt (context ≈{n_prompt + 2 * len(sweep) + n_dec}), same model file, unmodified reference CPU build (AVX2), {threads} threads (best of the sweep)"}
    if rank == 0:
        print(json.dumps(result))
    group.close()


if __name__ == "__main__":
    main()
