"""Regenerates tests/golden/*.npz from the UNMODIFIED reference (oracle/_ref/libctransformers_ref.so, built from the
reference's sources by oracle/Makefile):  python tests/golden/make_golden.py [kat | pool | runs | <model case> ...]

Contents
  kat_quant.npz    seeded activations → the reference's Q8_K / Q8_0 block bytes; seeded weights quantized by the
                   reference → its vec_dot result per type (known-answer vectors for oracle and CUDA kernels)
  model_<case>.npz prompt, last-token logits / embeddings after the prompt, 24 greedy tokens, final logits, top-2 gaps
                   for each synthetic model in tests/modelcases.py (weights come from seeded random blocks, so the GGUF
                   is reproducible without the reference)
  host_logic.npz   tokenizer ids for a set of strings, detokenized pieces, and sampler picks for seeded logits
  ref_quant_pool.npz  blocks of every weight type made by the reference's quantizer from seeded rows (refs.pool_matrix)
  reference_runs.npz  what the tests that compare with the reference expect, for the inputs they build themselves:
                   SHA-256 digests of its outputs (they must match bit for bit), greedy tokens and dot products
"""
import ctypes as C
import json
import sys
import tempfile
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parent))
sys.path.insert(0, str(HERE.parent.parent))
import modelcases  # noqa: E402
import refs  # noqa: E402
from refs import Q4_0, Q4_K, Q5_0, Q5_K, Q6_K, Q8_0, Q8_K, ptr  # noqa: E402

TEXTS = ["AI is going to", "  hello  world ", "héllo ☃ the", "", "theof and123", "a\nb\tc", "The people of the water were very little.",
         "that's what they'll've said", "12345 67", "\x00\x01"]


def kat_quant():
    rng = np.random.default_rng(2024)
    out = {}
    for k in (256, 1024):
        x = (rng.standard_normal(k) * 3).astype(np.float32)
        out[f"x_{k}"] = x
        out[f"q8k_{k}"] = refs.ref_quantize_act(Q8_K, x)
        out[f"q80_{k}"] = refs.ref_quantize_act(Q8_0, x)
    k, m = 1024, 6
    w = (rng.standard_normal((m, k)) * 0.05).astype(np.float32)
    x = out["x_1024"]
    out["w_f32"] = w
    for t, at in ((Q4_0, Q8_0), (Q8_0, Q8_0), (Q4_K, Q8_K), (Q5_K, Q8_K), (Q6_K, Q8_K), (Q5_0, Q8_0)):   # (appended: earlier vectors keep their bytes)
        wq = refs.ref_quantize(t, w).reshape(m, -1)
        act = refs.ref_quantize_act(at, x)
        out[f"wq_{t}"] = wq
        out[f"dot_{t}"] = np.array([refs.ref_vec_dot(t, k, wq[i], act) for i in range(m)], np.float32)
        deq = np.zeros((m, k), np.float32)
        refs.ref_traits(t)["to_float"](ptr(wq), ptr(deq), m * k)
        out[f"deq_{t}"] = deq
    np.savez_compressed(HERE / "kat_quant.npz", **out)


def quant_pool():
    out = {}
    for t in (Q4_0, Q5_0, Q8_0, Q4_K, Q5_K, Q6_K):
        w = (np.random.default_rng(100 + t).standard_normal((16, 1024)) * 0.05 + 0.01).astype(np.float32)
        out[f"pool_{t}"] = refs.ref_quantize(t, w).reshape(-1, refs.BLOCK[t][1])
    np.savez_compressed(HERE / "ref_quant_pool.npz", **out)


def reference_runs(tmp):
    """The inputs are built exactly as the tests build them (tests/test_oracle.py, tests/test_model_gpu.py)."""
    from ctransformers_b200 import synth
    out = {}
    rng = np.random.default_rng(7)                                  # test_oracle: quantizers
    d8k, d80 = [], []
    for trial in range(60):
        x = (rng.standard_normal(2048) * rng.choice([1e-3, 1, 50])).astype(np.float32)
        if trial % 7 == 0:
            x[256:512] = 0
        d8k.append(refs.digest(refs.ref_quantize_act(Q8_K, x)))
        d80.append(refs.digest(refs.ref_quantize_act(Q8_0, x)))
    out["quant_q8k"], out["quant_q80"] = np.array(d8k), np.array(d80)
    for t, at in ((Q4_0, Q8_0), (Q5_0, Q8_0), (Q8_0, Q8_0), (Q4_K, Q8_K), (Q5_K, Q8_K), (Q6_K, Q8_K)):   # test_oracle: vec_dot
        rng = np.random.default_rng(t)
        k = 4096
        wq = refs.pool_matrix(t, 16, k, rng).reshape(16, -1)
        x = rng.standard_normal(k).astype(np.float32)
        act = refs.ref_quantize_act(at, x)
        out[f"vecdot_act_{t}"] = np.array(refs.digest(act))
        out[f"vecdot_{t}"] = np.array([refs.ref_vec_dot(t, k, wq[i], act) for i in range(16)], np.float32)
        blocks = np.ascontiguousarray(synth.random_blocks(t, 1024, 8, 0.02, np.random.default_rng(t)))   # random blocks
        deq = np.zeros(8 * 1024, np.float32)
        refs.ref_traits(t)["to_float"](ptr(blocks), ptr(deq), deq.size)
        out[f"randblk_deq_{t}"] = np.array(refs.digest(deq))
    for name in ("llama_tiny_q4km", "falcon_tiny_q5km"):            # test_oracle: whole model, three chunkings
        path, ctx = modelcases.build(name, tmp)
        arch, shape, _, _ = modelcases.CASES[name]
        ids = np.random.default_rng(9).integers(259 if arch == "llama" else 0, shape.n_vocab, 70).tolist()
        for bs in (8, 64, 33):
            llm = ref_llm(path, ctx)
            llm.eval(ids, batch_size=bs)
            ds = []
            for _ in range(3):
                a = np.array(llm.logits, dtype=np.float32)
                ds.append(refs.digest(a))
                llm.eval([int(np.argmax(a))])
            out[f"chunk_{name}_{bs}"] = np.array(ds)

    def store(key, run):
        out[key + "_digests"] = np.array(refs.run_digests(run))
        out[key + "_tokens"] = np.array(run[2])
    for name in ("llama_tiny_q4km", "llama_gqa_q5km", "falcon_tiny_q5km"):   # test_model_gpu: chunkings of the fixture prompt
        path, ctx = modelcases.build(name, tmp)
        for bs in (8, 64, 5):
            store(f"live_{name}_{bs}", modelcases.run_greedy(ref_llm(path, ctx), modelcases.prompt_for(name), modelcases.N_NEW, batch_size=bs))
    path = Path(tmp) / "realq.gguf"                                 # test_model_gpu: weights from the reference's quantizer
    shape = synth.LlamaShape(n_vocab=1024, n_embd=512, n_head=4, n_head_kv=4, n_ff=1536, n_layer=2, n_ctx_train=128)
    synth.write_llama(path, shape, "Q4_K_M", seed=3, quantizer=refs.pool_quantizer, sigma=0.05)
    prompt = [1] + np.random.default_rng(0).integers(259, 1024, 30).tolist()
    store("realq", modelcases.run_greedy(ref_llm(path, 64), prompt, 8))
    for name, bs in (("llama_wide_q4km", 512), ("llama_wide_q4km", 64), ("llama_gqa_q5km", 5), ("falcon_tiny_q5km", 512)):   # prefill
        path, _ = modelcases.build(name, tmp)
        arch, shape, _, _ = modelcases.CASES[name]
        prompt = np.random.default_rng(9).integers(259 if arch == "llama" else 0, shape.n_vocab, 70).tolist()
        if arch == "llama":
            prompt[0] = 1
        store(f"prefill_{name}_{bs}", modelcases.run_greedy(ref_llm(path, 96), prompt, 6, batch_size=bs))
    import bench                                                    # test_model_gpu: the 7B-shaped bench models
    for workload in ("llama2-7b", "falcon7b"):
        bench.WL = bench.WORKLOADS[workload]
        path = bench.ensure_model(0, 1, lambda: None)
        store(f"bench_{workload}", modelcases.run_greedy(ref_llm(path, 128), bench.prompt_ids()[:32], 8))
        print(workload, "done")
    np.savez_compressed(HERE / "reference_runs.npz", **out)


def ref_llm(path, ctx):
    from ctransformers_b200 import AutoModelForCausalLM
    return AutoModelForCausalLM.from_pretrained(str(path), lib=str(refs.REF_SO), context_length=ctx, threads=4)


def models(tmp, only=None):
    for name in modelcases.CASES:
        if only and name not in only:
            continue
        path, ctx = modelcases.build(name, tmp)
        llm = ref_llm(path, ctx)
        prompt = modelcases.prompt_for(name)
        first_logits, first_embd, toks, last_logits, gaps = modelcases.run_greedy(llm, prompt, modelcases.N_NEW)
        np.savez_compressed(HERE / f"model_{name}.npz", prompt=np.array(prompt), first_logits=first_logits, first_embd=first_embd,
                            tokens=np.array(toks), last_logits=last_logits, gaps=np.array(gaps))
        print(name, "tokens", toks[:8], "min top-2 gap", min(gaps))


def host_logic(tmp):
    out = {}
    for name in ("llama_tiny_q4km", "falcon_tiny_q5km"):
        path, ctx = modelcases.build(name, tmp)
        llm = ref_llm(path, ctx)
        for i, text in enumerate(TEXTS):
            if name.startswith("falcon") and not text.isascii():
                continue   # the synthetic BPE vocabulary only holds printable ASCII bytes
            if name.startswith("falcon") and any(ord(c) < 33 and c not in " " for c in text):
                continue
            ids = llm.tokenize(text)
            out[f"{name}_tok_{i}"] = np.array(ids, np.int32)
        pieces = [llm.detokenize([t], decode=False) for t in range(llm.vocab_size)]
        out[f"{name}_pieces"] = np.array([p.hex() for p in pieces])
        # sampler: seeded logits written through the mutable logits view, then sampled with several settings
        llm.eval([5, 6, 7])
        rng = np.random.default_rng(3)
        picks = []
        settings = [(40, 0.95, 0.8, 1.1, 1), (1, 1.0, 1.0, 1.0, 0), (5, 0.5, 1.3, 1.3, 7), (0, 0.9, 0.7, 1.0, 123), (1000, 1.0, 0.01, 1.2, 9)]
        lg_all = []
        for rep in range(4):
            lg = (rng.standard_normal(llm.vocab_size) * 3).astype(np.float32)
            lg_all.append(lg)
            view = llm.logits
            for j, v in enumerate(lg):
                view[j] = float(v)
            for (k, p, temp, pen, seed) in settings:
                picks.append(llm.sample(top_k=k, top_p=p, temperature=temp, repetition_penalty=pen, last_n_tokens=64, seed=seed))
        out[f"{name}_sample_logits"] = np.array(lg_all)
        out[f"{name}_sample_picks"] = np.array(picks, np.int32)
        out[f"{name}_sample_settings"] = np.array(settings, np.float64)
    out["texts"] = np.array(TEXTS)
    np.savez_compressed(HERE / "host_logic.npz", **out)


if __name__ == "__main__":
    assert refs.have_ref(), "build oracle/_ref first: make -C oracle ref"
    import sys
    only = sys.argv[1:]          # python make_golden.py [model case ...]: regenerate only those model fixtures
    with tempfile.TemporaryDirectory() as tmp:
        if only:                 # "kat" regenerates kat_quant.npz (its vectors are appended per type, earlier ones keep their bytes)
            if "kat" in only:
                kat_quant()
            if "pool" in only:
                quant_pool()
            if "runs" in only:   # reads ref_quant_pool.npz
                reference_runs(tmp)
            cases = [o for o in only if o not in ("kat", "pool", "runs")]
            if cases:
                models(tmp, cases)
        else:
            kat_quant()
            models(tmp)
            host_logic(tmp)
            quant_pool()
            reference_runs(tmp)
    print("golden vectors written to", HERE)
