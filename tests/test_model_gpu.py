"""GPU parity tests, whole path: synthetic GGUF models through the public Python API / the 17-function C ABI on the
B200 library, against (1) the committed golden fixtures the reference produced (tests/golden/model_*.npz) and (2) what
the unmodified reference produced on the same files for further chunkings, prompts and models (tests/golden/reference_runs.npz:
digests of its logits and hidden states, which must match bit for bit, and its greedy tokens).

Bar: the north star asks for logits within 1e-3 relative and identical greedy tokens; the kernels reproduce the
reference's accumulation order, so these tests demand the stronger thing — logits, embeddings and tokens IDENTICAL to the
reference's, bit for bit (LOGIT_TOL documents the contractual tolerance and is asserted first for a readable failure)."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

import modelcases
import refs

pytestmark = pytest.mark.gpu
GOLD = Path(__file__).resolve().parent / "golden"
LOGIT_TOL = 1e-3


def rel_err(a, b):
    return float(np.abs(a - b).max() / np.abs(b).max())


def same_as_reference(ours, key):
    """A modelcases.run_greedy result against the reference's stored one: same tokens, bit-identical logits and hidden state."""
    gold = refs.golden("reference_runs")
    assert ours[2] == gold[key + "_tokens"].tolist()
    assert refs.run_digests(ours) == gold[key + "_digests"].tolist(), "first logits / first embeddings / last logits differ from the reference's"


def same_bits(a, b):
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    assert rel_err(a, b) <= LOGIT_TOL, f"outside the contractual tolerance: {rel_err(a, b):.3e}"
    bad = a.view(np.uint32) != b.view(np.uint32)
    assert not bad.any(), f"{int(bad.sum())} of {bad.size} values differ from the reference (max rel {rel_err(a, b):.3e})"


@pytest.fixture(scope="module")
def model_dir(tmp_path_factory):
    return tmp_path_factory.mktemp("gpu_models")


def load(path, ctx, **kw):
    from ctransformers_b200 import AutoModelForCausalLM
    return AutoModelForCausalLM.from_pretrained(str(path), context_length=ctx, **kw)


@pytest.mark.parametrize("name", list(modelcases.CASES))
def test_against_golden_fixture(name, model_dir):
    gold = np.load(GOLD / f"model_{name}.npz")
    path, ctx = modelcases.build(name, model_dir)
    llm = load(path, ctx)
    first_logits, first_embd, toks, last_logits, _ = modelcases.run_greedy(llm, gold["prompt"].tolist(), modelcases.N_NEW)
    same_bits(first_logits, gold["first_logits"])
    same_bits(first_embd, gold["first_embd"])
    assert toks == gold["tokens"].tolist()
    same_bits(last_logits, gold["last_logits"])


@pytest.mark.parametrize("name", ["llama_tiny_q4km", "llama_gqa_q5km", "falcon_tiny_q5km"])
def test_against_live_reference(name, model_dir):
    path, ctx = modelcases.build(name, model_dir)
    prompt = modelcases.prompt_for(name)
    for bs in (8, 64, 5):   # the chunking is part of the contract: it fixes the row length of the attention mat-muls
        same_as_reference(modelcases.run_greedy(load(path, ctx), prompt, modelcases.N_NEW, batch_size=bs), f"live_{name}_{bs}")


def test_real_quantized_weights_against_live_reference(model_dir):
    """Weights made by the reference's own quantizer (blocks of tests/golden/ref_quant_pool.npz), not random blocks."""
    from ctransformers_b200 import synth
    path = model_dir / "realq.gguf"
    shape = synth.LlamaShape(n_vocab=1024, n_embd=512, n_head=4, n_head_kv=4, n_ff=1536, n_layer=2, n_ctx_train=128)
    synth.write_llama(path, shape, "Q4_K_M", seed=3, quantizer=refs.pool_quantizer, sigma=0.05)
    prompt = [1] + np.random.default_rng(0).integers(259, 1024, 30).tolist()
    same_as_reference(modelcases.run_greedy(load(path, 64), prompt, 8), "realq")


def test_logits_are_a_mutable_view_and_sampling_sees_edits(model_dir):
    """reference tests/test_model.py:10-16 — writes through llm.logits must be visible to the next sample()."""
    path, ctx = modelcases.build("llama_tiny_q4km", model_dir)
    llm = load(path, ctx)
    llm.eval([1, 300, 301])
    assert len(llm.logits) == llm.vocab_size == 1024
    best = int(np.argmax(np.array(llm.logits)))
    assert llm.sample(top_k=1, repetition_penalty=1.0) == best
    llm.logits[best] -= 1000.0
    assert abs(llm.logits[best] - (np.array(llm.logits)[best])) == 0
    assert llm.sample(top_k=1, repetition_penalty=1.0) != best
    assert len(llm.embeddings) == 256
    assert llm.context_length == ctx and llm.model_type == "llama" and llm.bos_token_id == 1 and llm.eos_token_id == 2


def test_prefix_reuse_and_kv_overwrite(model_dir):
    """Re-evaluating at a smaller n_past overwrites the cache (llama.cpp:2323-2335): same logits as a fresh run."""
    path, ctx = modelcases.build("llama_tiny_q4km", model_dir)
    a = load(path, ctx)
    a.eval([1, 400, 401, 402, 403])
    toks = [1, 400, 401, 500, 501]
    todo = a.prepare_inputs_for_generation(toks)
    assert todo == [500, 501]
    a.eval(todo)
    b = load(path, ctx)
    b.eval(toks)
    assert np.array_equal(np.array(a.logits), np.array(b.logits))


def test_every_chunking_matches_the_oracle(model_dir):
    """Like the reference, results depend (in the last bits) on how a prompt is chunked, because a chunk's n_past + N is the
    row length of its attention mat-muls.  Every chunking must equal the whole-model oracle run with the same chunking."""
    name = "llama_gqa_q5km"
    path, ctx = modelcases.build(name, model_dir)
    prompt = np.random.default_rng(4).integers(259, 2048, 70).tolist()
    for bs in (1, 8, 33, 64):
        llm = load(path, ctx)
        llm.eval(prompt, batch_size=bs)
        m = refs.OracleModel(path, ctx)
        want = m.eval(prompt, batch_size=bs)
        same_bits(np.array(llm.logits, dtype=np.float32), want)


def test_fused_greedy_decode_matches_stepwise(model_dir, lib):
    import ctypes as C
    path, ctx = modelcases.build("llama_tiny_q4km", model_dir)
    prompt = modelcases.prompt_for("llama_tiny_q4km")
    a = load(path, ctx)
    _, _, toks, last_logits, _ = modelcases.run_greedy(a, prompt, 16)
    b = load(path, ctx)
    b.eval(prompt)
    first = b.sample(top_k=1, repetition_penalty=1.0)
    out = (C.c_int * 16)()
    ms = b.ctb_llm_decode_greedy(first, len(prompt), 16, out)
    assert ms > 0
    # decode_greedy returns the token picked AFTER each step; the stepwise loop's tokens are the ones fed in
    assert [first] + list(out[:15]) == toks
    assert b.ctb_llm_launches_per_token() > 0 and b.ctb_llm_weight_bytes_per_token() > 0


def test_context_overflow_is_clamped_not_fatal(model_dir):
    path, _ = modelcases.build("llama_tiny_q4_0", model_dir)
    llm = load(path, 16)
    llm.eval(list(range(300, 316)))
    llm.eval([5])   # n_past is clamped to n_ctx - n like LLM::EvalInternal (llm.h:124-126); must not crash
    assert np.isfinite(np.array(llm.logits)).all()


def test_create_failure_modes(tmp_path):
    from ctransformers_b200 import AutoModelForCausalLM
    bad = tmp_path / "truncated.gguf"
    bad.write_bytes(b"GGUF" + b"\x02\0\0\0" + b"\xff" * 8)
    with pytest.raises(RuntimeError):
        AutoModelForCausalLM.from_pretrained(str(bad))
    with pytest.raises(ValueError):
        AutoModelForCausalLM.from_pretrained(str(tmp_path / "nope.gguf"))


def test_greedy_lookahead_hits_and_misses_match_the_oracle(model_dir, lib):
    """The engine starts the step for the greedy next token while the host samples (engine.cu: after_eval).  A run of greedy
    tokens (look-ahead hits), then off-greedy tokens (misses that must overwrite the guessed step), then greedy again:
    every logits vector must be the oracle's for the same token sequence."""
    name = "llama_tiny_q4km"
    path, ctx = modelcases.build(name, model_dir)
    llm = load(path, ctx)
    orc = refs.OracleModel(path, ctx)
    seq = modelcases.prompt_for(name)[:9]
    llm.eval(seq, batch_size=8)
    want = orc.eval(seq, batch_size=8).copy()
    hits0 = llm.ctb_llm_speculative_hits()
    for step in range(16):
        got = np.array(llm.logits, dtype=np.float32)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), f"step {step}"
        greedy = int(np.argmax(got))
        tok = greedy if step not in (6, 7, 12) else (greedy + 17) % llm.vocab_size
        llm.eval([tok])
        want = orc.eval([tok]).copy()
    assert llm.ctb_llm_speculative_hits() - hits0 >= 4


# ---- BASELINE-size models (configs[1] and configs[3]) against the reference: the same files bench.py times
@pytest.mark.parametrize("workload", ["llama2-7b", "falcon7b"])
def test_bench_model_against_live_reference(workload):
    """32-token prompt (reference default chunking, batch_size 8) + 8 greedy steps on the 7B-shaped bench model: logits after
    the prompt, the greedy tokens and the last logits must be the reference's, bit for bit."""
    import sys
    sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
    import bench
    bench.WL = bench.WORKLOADS[workload]
    path = bench.ensure_model(0, 1, lambda: None)          # bench.MODEL_DIR, shared with bench.py on the same machine
    prompt = bench.prompt_ids()[:32]
    same_as_reference(modelcases.run_greedy(load(path, 128), prompt, 8), f"bench_{workload}")


# ---- batched prefill (csrc/prefill.cuh): prompts longer than a few tokens go through the dense int8 tensor-core kernel
@pytest.mark.parametrize("name,bs", [("llama_wide_q4km", 512), ("llama_wide_q4km", 64), ("llama_gqa_q5km", 5), ("falcon_tiny_q5km", 512)])
def test_prefill_against_live_reference(name, bs, model_dir):
    """A prompt of 70 tokens (3 batched launches: 32 + 32 + 6) at batch_size 5 / 64 / 512: logits and hidden state after the
    prompt and the greedy continuation must be the reference's, bit for bit."""
    path, _ = modelcases.build(name, model_dir)
    arch, shape, _, _ = modelcases.CASES[name]
    rng = np.random.default_rng(9)
    prompt = rng.integers(259 if arch == "llama" else 0, shape.n_vocab, 70).tolist()
    if arch == "llama":
        prompt[0] = 1
    same_as_reference(modelcases.run_greedy(load(path, 96), prompt, 6, batch_size=bs), f"prefill_{name}_{bs}")


def test_prefill_equals_single_token_path(model_dir, monkeypatch):
    """The batched kernel and the single-token kernel are two implementations of the same arithmetic: identical bits."""
    path, _ = modelcases.build("llama_wide_q4km", model_dir)
    prompt = modelcases.prompt_for("llama_wide_q4km")
    a = modelcases.run_greedy(load(path, 96), prompt, 4, batch_size=16)
    monkeypatch.setenv("CTB_NO_PREFILL", "1")
    b = modelcases.run_greedy(load(path, 96), prompt, 4, batch_size=16)
    same_bits(a[0], b[0])
    same_bits(a[1], b[1])
    assert a[2] == b[2]


def test_device_sampler_draws_the_reference_tokens(model_dir):
    """sample() before anybody has asked for llm.logits runs repetition penalty + top-k on the device (csrc/sample_gpu.cuh) and
    the rest on the host; after llm.logits has been read the whole chain runs on the host logits like the reference's.  Same
    seeds, same tokens — and the host chain is the one pinned against the reference in test_host_logic.py."""
    path, ctx = modelcases.build("llama_tiny_q4km", model_dir)
    llm = load(path, ctx)
    prompt = modelcases.prompt_for("llama_tiny_q4km")
    llm.eval(prompt)
    last = prompt[-20:] + [7, 7, 300]
    cases = [(40, 0.95, 0.8, 1.1, s) for s in range(6)] + [(1, 1.0, 1.0, 1.0, 0), (5, 0.5, 1.3, 1.3, 3), (100, 0.9, 0.7, 1.0, 4), (64, 1.0, 2.0, 1.5, 5)]

    def draw(k, p, t, rp, seed):
        arr = (C.c_int * len(last))(*last)
        return llm.ctransformers_llm_sample(arr, len(last), k, p, t, rp, seed)

    before = llm.ctb_llm_device_samples()
    dev = [draw(*c) for c in cases]
    assert llm.ctb_llm_device_samples() - before >= len(cases) - 1       # (equal logits may send a case to the host path)
    _ = llm.logits[0]                                                      # a host view exists from here on
    mid = llm.ctb_llm_device_samples()
    host = [draw(*c) for c in cases]
    assert llm.ctb_llm_device_samples() == mid
    assert dev == host
    # and the lazily fetched logits are the eval's logits: a fresh engine that copies eagerly agrees
    llm2 = load(path, ctx)
    _ = llm2.logits
    llm2.eval(prompt)
    same_bits(np.array(llm.logits, np.float32), np.array(llm2.logits, np.float32))
    same_bits(np.array(llm.embeddings, np.float32), np.array(llm2.embeddings, np.float32))


def test_lazy_sampling_modes_match_the_eager_engine(model_dir):
    """A decode loop that never reads llm.logits: greedy calls are answered by the engine's own pick (no kernel), sampled calls by
    the device sampler with the look-ahead step launched behind it, and switching between the two keeps every token equal to an
    engine that copies its logits to the host after every eval and samples there (the reference's flow)."""
    path, ctx = modelcases.build("llama_tiny_q4km", model_dir)
    a, b = load(path, ctx), load(path, ctx)
    _ = b.logits                                               # b: eager host views from the start
    prompt = modelcases.prompt_for("llama_tiny_q4km")
    a.eval(prompt); b.eval(prompt)
    greedy = dict(top_k=1, repetition_penalty=1.0)
    sampled = dict(top_k=40, top_p=0.95, temperature=0.8, repetition_penalty=1.1)
    plan = [greedy] * 6 + [sampled] * 6 + [greedy] * 4 + [sampled] * 2 + [greedy] * 3 + [dict(top_k=1, repetition_penalty=1.3)] * 3
    before = a.ctb_llm_device_samples()
    for i, kw in enumerate(plan):
        ta, tb = a.sample(seed=i, **kw), b.sample(seed=i, **kw)
        assert ta == tb, (i, kw)
        a.eval([ta]); b.eval([tb])
    assert a.ctb_llm_device_samples() - before >= len(plan) - 2
    assert a.ctb_llm_speculative_hits() >= 6                   # the greedy stretches ride the look-ahead
    same_bits(np.array(a.logits, np.float32), np.array(b.logits, np.float32))
