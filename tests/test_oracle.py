"""CPU tests that pin the oracle: the plain-C restatement (oracle/ggml_oracle.c) against (1) the committed golden
vectors that the unmodified reference produced (tests/golden/make_golden.py), (2) what the compiled reference produced
for the inputs the tests below build (tests/golden/reference_runs.npz), (3) the known-answer thresholds of upstream test-quantize-fns.cpp
(models/submodules/llama.cpp/tests/test-quantize-fns.cpp:16-31, 76-113)."""
from pathlib import Path

import numpy as np
import pytest

import refs
from refs import Q4_0, Q4_K, Q5_0, Q5_K, Q6_K, Q8_0, Q8_K, ptr, row_bytes

GOLD = Path(__file__).resolve().parent / "golden"
TYPES = [(Q4_0, Q8_0), (Q5_0, Q8_0), (Q8_0, Q8_0), (Q4_K, Q8_K), (Q5_K, Q8_K), (Q6_K, Q8_K)]


@pytest.fixture(scope="module")
def kat():
    return np.load(GOLD / "kat_quant.npz")


def _oracle_quant(t, x):
    o = refs.oracle()
    out = np.zeros(row_bytes(t, x.size), np.uint8)
    (o.orc_quantize_row_q8_K if t == Q8_K else o.orc_quantize_row_q8_0)(ptr(np.ascontiguousarray(x)), ptr(out), x.size)
    return out


@pytest.mark.parametrize("k", [256, 1024])
def test_activation_quantizers_match_golden(kat, k):
    x = kat[f"x_{k}"]
    assert np.array_equal(_oracle_quant(Q8_K, x), kat[f"q8k_{k}"])
    assert np.array_equal(_oracle_quant(Q8_0, x), kat[f"q80_{k}"])


@pytest.mark.parametrize("t,at", TYPES)
def test_vec_dot_and_dequant_match_golden(kat, t, at):
    o = refs.oracle()
    wq, x = kat[f"wq_{t}"], kat["x_1024"]
    act = _oracle_quant(at, x)
    fn = getattr(o, f"orc_vec_dot_{refs.TYPE_NAME[t]}_{'q8_K' if at == Q8_K else 'q8_0'}")
    got = np.array([fn(1024, ptr(np.ascontiguousarray(wq[i])), ptr(act)) for i in range(wq.shape[0])], np.float32)
    want = kat[f"dot_{t}"]
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), "oracle dot must equal the reference bit for bit"
    deq = np.zeros_like(kat[f"deq_{t}"])
    getattr(o, "orc_dequantize_row_" + refs.TYPE_NAME[t])(ptr(np.ascontiguousarray(wq)), ptr(deq), deq.size)
    assert np.array_equal(deq.view(np.uint32), kat[f"deq_{t}"].view(np.uint32))


@pytest.mark.parametrize("t,at", TYPES)
def test_upstream_quantize_fns_thresholds(kat, t, at):
    """test-quantize-fns.cpp: dot(q(x), q8(y)) error / n < 0.02 on 0.1 + 2cos(i + offset), n = 4096·32 there, 4096 here;
    round-trip array_rmse (sqrt(sum sq)/n, test-quantize-fns.cpp:34-41) < 0.002.  Weights quantized by the reference (golden file) are not available for this vector, so the
    round trip uses the activation types we quantize ourselves, and the dot uses golden weights vs the float dot."""
    o = refs.oracle()
    wq, x, w = kat[f"wq_{t}"], kat["x_1024"], kat["w_f32"]
    act = _oracle_quant(at, x)
    fn = getattr(o, f"orc_vec_dot_{refs.TYPE_NAME[t]}_{'q8_K' if at == Q8_K else 'q8_0'}")
    for i in range(wq.shape[0]):
        got = fn(1024, ptr(np.ascontiguousarray(wq[i])), ptr(act))
        assert abs(got - float(w[i] @ x)) / 1024 < 0.02
    # Q8_0 / Q8_K round trip of the synthetic test vector
    n = 4096
    v = (0.1 + 2 * np.cos(np.arange(n) + 1.0)).astype(np.float32)
    q = _oracle_quant(Q8_0, v).reshape(-1, 34)
    d = q[:, :2].copy().view(np.float16).astype(np.float32)
    back = (q[:, 2:].view(np.int8).astype(np.float32) * d).reshape(-1)
    assert np.sqrt(np.sum((back - v) ** 2)) / n < 0.002   # upstream array_rmse = sqrt(sum of squares) / n


def test_fp16_conversions_exhaustive():
    o = refs.oracle()
    bits = np.arange(65536, dtype=np.uint16)
    f = bits.view(np.float16).astype(np.float32)
    mine = np.array([o.orc_fp16_to_fp32(int(b)) for b in bits], np.float32)
    ok = ~np.isnan(f)
    assert np.array_equal(mine.view(np.uint32)[ok], f.view(np.uint32)[ok])
    back = np.array([o.orc_fp32_to_fp16(float(v)) for v in f[ok]], np.uint16)
    assert np.array_equal(back, bits[ok])
    rng = np.random.default_rng(0)
    x = (rng.standard_normal(20000) * rng.choice([1e-8, 1e-5, 1e-3, 1, 100, 7e4], 20000)).astype(np.float32)
    assert np.array_equal(np.array([o.orc_fp32_to_fp16(float(v)) for v in x], np.uint16), x.astype(np.float16).view(np.uint16))


class TestAgainstCompiledReference:
    """Against what the compiled reference produced for the same seeded inputs (tests/golden/reference_runs.npz)."""

    def test_quantizers_bit_exact(self):
        gold = refs.golden("reference_runs")
        rng = np.random.default_rng(7)
        for trial in range(60):
            x = (rng.standard_normal(2048) * rng.choice([1e-3, 1, 50])).astype(np.float32)
            if trial % 7 == 0:
                x[256:512] = 0
            assert refs.digest(_oracle_quant(Q8_K, x)) == gold["quant_q8k"][trial], trial
            assert refs.digest(_oracle_quant(Q8_0, x)) == gold["quant_q80"][trial], trial

    @pytest.mark.parametrize("t,at", TYPES)
    def test_vec_dot(self, t, at):
        """Weights from the reference's quantizer, activations quantized by the oracle (identical to the reference's)."""
        gold = refs.golden("reference_runs")
        o = refs.oracle()
        rng = np.random.default_rng(t)
        k = 4096
        wq = refs.pool_matrix(t, 16, k, rng).reshape(16, -1)
        x = rng.standard_normal(k).astype(np.float32)
        act = _oracle_quant(at, x)
        assert refs.digest(act) == gold[f"vecdot_act_{t}"]
        fn = getattr(o, f"orc_vec_dot_{refs.TYPE_NAME[t]}_{'q8_K' if at == Q8_K else 'q8_0'}")
        got = np.array([fn(k, ptr(np.ascontiguousarray(wq[i])), ptr(act)) for i in range(16)], np.float32)
        assert np.array_equal(got.view(np.uint32), gold[f"vecdot_{t}"].view(np.uint32))

    def test_random_block_generator_is_valid_for_the_reference(self):
        """synth.random_blocks must produce blocks the reference dequantizes to finite, sensibly scaled weights (the oracle's
        dequantization of them is checked to be the reference's, bit for bit)."""
        from ctransformers_b200 import synth
        gold = refs.golden("reference_runs")
        o = refs.oracle()
        for t in (Q4_0, Q5_0, Q8_0, Q4_K, Q5_K, Q6_K):
            blocks = np.ascontiguousarray(synth.random_blocks(t, 1024, 8, 0.02, np.random.default_rng(t)))
            out = np.zeros(8 * 1024, np.float32)
            getattr(o, "orc_dequantize_row_" + refs.TYPE_NAME[t])(ptr(blocks), ptr(out), out.size)
            assert refs.digest(out) == gold[f"randblk_deq_{t}"], t
            assert np.isfinite(out).all()
            assert 0.01 < out.std() < 0.04, (t, out.std())
            assert abs(out.mean()) < 0.004


# ---- the whole-model restatement (oracle/llama_oracle.c) is pinned by the logits the reference produced
import modelcases  # noqa: E402


@pytest.mark.parametrize("name", list(modelcases.CASES))
def test_full_eval_matches_reference_golden(name, tmp_path_factory):
    gold = np.load(GOLD / f"model_{name}.npz")
    path, ctx = modelcases.build(name, tmp_path_factory.mktemp("orc"))
    m = refs.OracleModel(path, ctx)
    logits = m.eval(gold["prompt"].tolist()).copy()
    # bit-exact: the oracle reproduces the reference's fp32 accumulation order and FMA placement
    assert np.array_equal(logits.view(np.uint32), gold["first_logits"].view(np.uint32)), np.abs(logits - gold["first_logits"]).max()
    assert np.array_equal(m.embd.view(np.uint32), gold["first_embd"].view(np.uint32))
    toks = []
    for want in gold["tokens"][:6]:
        t = int(np.argmax(m.logits))
        toks.append(t)
        m.eval([t])
    assert toks == gold["tokens"][:6].tolist()


@pytest.mark.parametrize("name", ["llama_tiny_q4km", "falcon_tiny_q5km"])
def test_full_eval_matches_live_reference_for_any_chunking(name, tmp_path_factory):
    """70-token prompt (so the V·P f16 dot uses both its SIMD part and its scalar tail), three chunkings, then 3 decode steps:
    every logits vector is the reference's for the same chunking (tests/golden/reference_runs.npz)."""
    gold = refs.golden("reference_runs")
    path, ctx = modelcases.build(name, tmp_path_factory.mktemp("orc_live"))
    arch, shape, _, _ = modelcases.CASES[name]
    ids = np.random.default_rng(9).integers(259 if arch == "llama" else 0, shape.n_vocab, 70).tolist()
    for bs in (8, 64, 33):
        m = refs.OracleModel(path, ctx)
        m.eval(ids, batch_size=bs)
        for step in range(3):
            assert refs.digest(m.logits) == gold[f"chunk_{name}_{bs}"][step], (bs, step)
            m.eval([int(np.argmax(m.logits))])
