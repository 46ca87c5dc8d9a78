"""BASELINE.json configs[0]: GPT-2 Q4_0 in the old GGML container, ctx 128, 32 new tokens, on the reference's CPU build.

There is no GPU kernel for this format (DESIGN.md §8); what the configuration checks is the plumbing every other measurement
stands on: model synthesis, the Python surface of this repository driving a library given through `lib=` (here the unmodified
reference), greedy determinism — and that this repository's own library declines the file the way the reference ABI
prescribes (NULL from create → RuntimeError)."""
import numpy as np
import pytest

import refs
from ctransformers_b200 import AutoModelForCausalLM, synth



@pytest.fixture(scope="module")
def gpt2_file(tmp_path_factory):
    shape = synth.GPT2Shape(n_vocab=640, n_ctx=128, n_embd=128, n_head=4, n_layer=2)
    return synth.write_gpt2_ggml(tmp_path_factory.mktemp("gpt2") / "gpt2-tiny.q4_0.bin", shape, "Q4_0", seed=3), shape


def run(path, n_new=32):
    llm = AutoModelForCausalLM.from_pretrained(str(path), model_type="gpt2", lib=str(refs.REF_SO), context_length=512, threads=2)
    ids = np.random.default_rng(1).integers(0, llm.vocab_size, 96).tolist()      # prompt + new tokens = the whole 128 context
    llm.eval(ids, batch_size=8)
    first = np.array(llm.logits, dtype=np.float32)
    toks = []
    for _ in range(n_new):
        t = llm.sample(top_k=1, repetition_penalty=1.0, seed=0)
        toks.append(int(t))
        llm.eval([t])
    return llm, first, toks


@pytest.mark.skipif(not refs.have_ref(), reason="needs oracle/_ref, the reference compiled from its sources (make -C oracle ref)")
def test_reference_runs_the_gpt2_file_through_this_python_surface(gpt2_file):
    path, shape = gpt2_file
    llm, first, toks = run(path)
    assert llm.vocab_size == shape.n_vocab
    assert llm.context_length == shape.n_ctx          # the file's own n_ctx wins over the requested context_length (gpt2.cc:85)
    assert first.shape == (shape.n_vocab,) and np.isfinite(first).all() and float(np.abs(first).max()) > 0
    assert len(toks) == 32 and all(0 <= t < shape.n_vocab for t in toks)
    _, first2, toks2 = run(path)
    assert np.array_equal(first.view(np.uint32), first2.view(np.uint32)) and toks == toks2   # greedy decoding is deterministic


def test_b200_library_declines_the_old_container(gpt2_file):
    path, _ = gpt2_file
    with pytest.raises(RuntimeError):
        AutoModelForCausalLM.from_pretrained(str(path), model_type="gpt2")
