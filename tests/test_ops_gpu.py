"""GPU parity tests, op level: every CUDA stage of the hot path, called through the C ABI with host buffers, against
the plain-C oracle (oracle/ggml_oracle.c) on the same seeded inputs.

Bar: BIT-EXACT everywhere.  The oracle reproduces the reference's AVX2 accumulation order and FMA placement (it is pinned
bit for bit against the compiled reference in tests/test_oracle.py), and the CUDA kernels reproduce the same order, so
quantizers, norms, RoPE, embedding rows, every quantized dot product and the attention block must match to the last bit."""
import ctypes as C

import numpy as np
import pytest

import refs
from conftest import ptr
from refs import F16, F32, Q4_0, Q4_K, Q5_0, Q5_K, Q6_K, Q8_0, Q8_K, row_bytes

pytestmark = pytest.mark.gpu



def _rand_weights(t, k, m, seed, sigma=0.02):
    from ctransformers_b200 import synth
    return np.ascontiguousarray(synth.random_blocks(t, k, m, sigma, np.random.default_rng(seed))).view(np.uint8)


def _act(rng, k, scale=1.0):
    x = rng.standard_normal(k).astype(np.float32) * scale
    x[rng.integers(0, k, 8)] *= 17.0
    return x


@pytest.mark.parametrize("k", [256, 4096, 11008])
def test_quantize_q8_K_bit_exact(lib, k):
    o = refs.oracle()
    rng = np.random.default_rng(k)
    for trial in range(6):
        x = _act(rng, k, [1e-4, 1.0, 300.0][trial % 3])
        if trial == 3:
            x[:256] = 0.0                      # all-zero block → d = 0
        if trial == 4:
            x[5], x[9] = -3.5, 3.5             # |max| tie: the FIRST one fixes the sign
            x[:256] = np.clip(x[:256], -3.5, 3.5)
        a = np.zeros(row_bytes(Q8_K, k), np.uint8)
        b = np.zeros_like(a)
        o.orc_quantize_row_q8_K(ptr(x), ptr(a), k)
        assert lib.ctb_quantize_row_q8_K(ptr(x), ptr(b), k) == 0
        assert np.array_equal(a, b), f"trial {trial}: {(a != b).sum()} differing bytes"


@pytest.mark.parametrize("k", [32, 4096, 4544])
def test_quantize_q8_0_bit_exact(lib, k):
    o = refs.oracle()
    rng = np.random.default_rng(k + 1)
    for trial in range(4):
        x = _act(rng, k, [1e-3, 1.0, 50.0, 1.0][trial])
        if trial == 3:
            x[:32] = 0.0
        a = np.zeros(row_bytes(Q8_0, k), np.uint8)
        b = np.zeros_like(a)
        o.orc_quantize_row_q8_0(ptr(x), ptr(a), k)
        assert lib.ctb_quantize_row_q8_0(ptr(x), ptr(b), k) == 0
        assert np.array_equal(a, b)


def _same_bits(got, want):
    got, want = np.ascontiguousarray(got, np.float32), np.ascontiguousarray(want, np.float32)
    bad = got.view(np.uint32) != want.view(np.uint32)
    assert not bad.any(), f"{int(bad.sum())} of {bad.size} values differ; max |diff| {np.abs(got - want).max():.3e}"


@pytest.mark.parametrize("t", [Q4_K, Q5_K, Q6_K, Q4_0, Q5_0, Q8_0])
@pytest.mark.parametrize("k,m", [(256, 3), (4096, 64), (11008, 33)])
def test_mul_mat_vs_oracle(lib, t, k, m):
    o = refs.oracle()
    rng = np.random.default_rng(t * 1000 + k)
    w = _rand_weights(t, k, m, seed=t + k)
    n = 2
    x = np.stack([_act(rng, k), _act(rng, k, 0.05)])
    want = np.zeros((n, m), np.float32)
    got = np.zeros((n, m), np.float32)
    assert o.orc_mul_mat(t, ptr(w), ptr(x), ptr(want), k, m, n) == 0
    assert lib.ctb_mul_mat(t, ptr(w), ptr(x), ptr(got), k, m, n) == 0
    _same_bits(got, want)


@pytest.mark.parametrize("t", [Q4_K, Q5_K, Q6_K])
@pytest.mark.parametrize("k,m", [(4096, 4096 + 37), (4096, 22016), (11008, 4096), (2048, 1184 + 8), (256, 9000)])
def test_mul_mat_full_size_partitions(lib, t, k, m):
    """Bench-sized shapes: many row tiles per CTA, warp ranges that start and end in the middle of a row (fold state handed from
    warp to warp, parked terms), ranges longer and shorter than a row, a ragged last tile — all bit-exact with the oracle."""
    o = refs.oracle()
    rng = np.random.default_rng(t * 77 + k + m)
    w = _rand_weights(t, k, m, seed=t + k + m)
    x = _act(rng, k)[None, :]
    want = np.zeros((1, m), np.float32)
    got = np.zeros((1, m), np.float32)
    assert o.orc_mul_mat(t, ptr(w), ptr(x), ptr(want), k, m, 1) == 0
    assert lib.ctb_mul_mat(t, ptr(w), ptr(x), ptr(got), k, m, 1) == 0
    _same_bits(got, want)


@pytest.mark.parametrize("k", [512, 1000])
def test_mul_mat_f16_weights(lib, k):
    """F16 weights take ggml_vec_dot_f16 with the activation row rounded to f16 (ggml.c:1665-1675, 2392-2426)."""
    o = refs.oracle()
    o.orc_vec_dot_f16.restype = C.c_float
    m = 24
    rng = np.random.default_rng(k)
    w = (rng.standard_normal((m, k)) * 0.05).astype(np.float16)
    x = _act(rng, k)[None]
    got = np.zeros((1, m), np.float32)
    assert lib.ctb_mul_mat(F16, ptr(w), ptr(x), ptr(got), k, m, 1) == 0
    x16 = x[0].astype(np.float16)
    want = np.array([o.orc_vec_dot_f16(k, ptr(np.ascontiguousarray(w[i])), ptr(x16)) for i in range(m)], np.float32)
    _same_bits(got[0], want)


def test_mul_mat_f32_weights(lib):
    k, m = 512, 16
    rng = np.random.default_rng(3)
    w = (rng.standard_normal((m, k)) * 0.05).astype(np.float32)
    x = _act(rng, k)[None]
    got = np.zeros((1, m), np.float32)
    assert lib.ctb_mul_mat(F32, ptr(w), ptr(x), ptr(got), k, m, 1) == 0
    assert np.allclose(got[0], w @ x[0], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("mode", [1, 2])
def test_norm_bit_exact(lib, mode):
    o = refs.oracle()
    n = 4096
    rng = np.random.default_rng(mode)
    x, w, b = _act(rng, n, 3.0), (1 + 0.1 * rng.standard_normal(n)).astype(np.float32), (0.1 * rng.standard_normal(n)).astype(np.float32)
    want, got = np.zeros(n, np.float32), np.zeros(n, np.float32)
    if mode == 1:
        o.orc_rms_norm_mul(ptr(x), ptr(w), ptr(want), n, 1e-5)
        assert lib.ctb_norm(1, ptr(x), ptr(w), None, ptr(got), n, 1e-5) == 0
    else:
        o.orc_layer_norm_mul_add(ptr(x), ptr(w), ptr(b), ptr(want), n, 1e-5)
        assert lib.ctb_norm(2, ptr(x), ptr(w), ptr(b), ptr(got), n, 1e-5) == 0
    assert np.array_equal(want.view(np.uint32), got.view(np.uint32)), f"{(want != got).sum()} of {n} differ, max {np.abs(want - got).max()}"


@pytest.mark.parametrize("mode,hd", [(0, 128), (2, 64), (0, 64)])
def test_rope_bit_exact(lib, mode, hd):
    o = refs.oracle()
    rng = np.random.default_rng(hd + mode)
    for pos in (0, 1, 37, 511):
        x = rng.standard_normal((8, hd)).astype(np.float32)
        want, got = x.copy(), x.copy()
        o.orc_rope(ptr(want), 8, hd, pos, mode, 10000.0, 1.0)
        assert lib.ctb_rope(ptr(got), 8, hd, pos, mode, 10000.0, 1.0) == 0
        assert np.array_equal(want.view(np.uint32), got.view(np.uint32)), f"pos {pos}: max diff {np.abs(want - got).max()}"


@pytest.mark.parametrize("n_head,n_kv,hd,T,n_total", [(4, 4, 128, 1, 1), (4, 4, 128, 300, 300), (8, 1, 64, 77, 77), (8, 2, 128, 512, 512),
                                                      (4, 4, 64, 21, 24), (4, 2, 128, 40, 64), (2, 2, 128, 33, 33), (2, 1, 64, 257, 300),
                                                      (4, 4, 128, 1500, 1500), (4, 1, 64, 2047, 2048), (2, 2, 128, 1027, 1027)])
def test_attention_bit_exact(lib, n_head, n_kv, hd, T, n_total):
    """n_total = row length of the reference's V·P mat-mul (n_past + N of the eval call): it fixes where the f16 dot switches
    from its 32 SIMD lanes to the scalar double tail, so it is part of the contract."""
    o = refs.oracle()
    rng = np.random.default_rng(T + hd)
    q = rng.standard_normal((n_head, hd)).astype(np.float32)
    kc = (rng.standard_normal((T, n_kv, hd)) * 0.7).astype(np.float16)          # [T][n_kv*hd]
    vt = rng.standard_normal((n_kv * hd, T)).astype(np.float16)                  # transposed, like the reference cache
    scale = np.float32(1.0 / np.sqrt(np.float32(hd)))
    got = np.zeros((n_head, hd), np.float32)
    assert lib.ctb_attention(ptr(q), ptr(kc), ptr(vt), ptr(got), n_head, n_kv, hd, T, n_total, float(scale)) == 0
    want = np.zeros((n_head, hd), np.float32)
    # the oracle's V·P dot runs over n_total entries: pad the transposed cache with zeros probabilities beyond T
    vpad = np.zeros((n_kv * hd, n_total), np.float16)
    vpad[:, :T] = vt
    o.orc_attn_head_n.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]
    for h in range(n_head):
        kvh = h // (n_head // n_kv)
        kslice = np.ascontiguousarray(kc[:, kvh, :])
        vslice = np.ascontiguousarray(vpad[kvh * hd:(kvh + 1) * hd])
        o.orc_attn_head_n(ptr(q[h]), ptr(kslice), hd, ptr(vslice), n_total, hd, T, n_total, float(scale), ptr(want[h]))
    _same_bits(got, want)


@pytest.mark.parametrize("t", [Q4_K, Q5_K, Q4_0, Q5_0])
def test_ffn_gate_vs_oracle(lib, t):
    o = refs.oracle()
    k, m = 4096, 96
    rng = np.random.default_rng(t)
    w1, w3 = _rand_weights(t, k, m, 1), _rand_weights(t, k, m, 2)
    x = _act(rng, k)
    g, u = np.zeros(m, np.float32), np.zeros(m, np.float32)
    o.orc_mul_mat(t, ptr(w1), ptr(x), ptr(g), k, m, 1)
    o.orc_mul_mat(t, ptr(w3), ptr(x), ptr(u), k, m, 1)
    s = np.zeros(m, np.float32)
    o.orc_silu(ptr(g), ptr(s), m)
    want = s * u
    got = np.zeros(m, np.float32)
    assert lib.ctb_ffn_gate(t, ptr(w1), ptr(w3), ptr(x), ptr(got), k, m) == 0
    _same_bits(got, want)


@pytest.mark.parametrize("t", [Q4_K, Q5_K, Q6_K, Q4_0, Q5_0, Q8_0, F16, F32])
def test_get_row_bit_exact(lib, t):
    o = refs.oracle()
    k, rows = 512, 9
    if t == F32:
        tab = np.random.default_rng(1).standard_normal((rows, k)).astype(np.float32)
        want = tab
    elif t == F16:
        tab = np.random.default_rng(1).standard_normal((rows, k)).astype(np.float16)
        want = tab.astype(np.float32)
    else:
        tab = _rand_weights(t, k, rows, 5, sigma=1.0)
        want = np.zeros((rows, k), np.float32)
        getattr(o, "orc_dequantize_row_" + refs.TYPE_NAME[t])(ptr(tab), ptr(want), rows * k)
    for r in (0, 4, rows - 1):
        got = np.zeros(k, np.float32)
        assert lib.ctb_get_row(t, ptr(tab), k, rows, r, ptr(got)) == 0
        assert np.array_equal(got.view(np.uint32), np.ascontiguousarray(want[r]).view(np.uint32))


@pytest.mark.parametrize("t", [Q4_K, Q5_K, Q6_K, Q4_0, Q5_0, Q8_0])
@pytest.mark.parametrize("k", [512, 1024, 2816])
def test_mul_mat_real_quantized_weights(lib, t, k):
    """Weights made of blocks the reference's quantizer produced (all scale/min bit patterns occur, unlike the random-block
    generator): tests/golden/ref_quant_pool.npz."""
    o = refs.oracle()
    rng = np.random.default_rng(k + t)
    m = 48
    w = refs.pool_matrix(t, m, k, rng)
    x = _act(rng, k)[None]
    want, got = np.zeros((1, m), np.float32), np.zeros((1, m), np.float32)
    assert o.orc_mul_mat(t, ptr(w), ptr(x), ptr(want), k, m, 1) == 0
    assert lib.ctb_mul_mat(t, ptr(w), ptr(x), ptr(got), k, m, 1) == 0
    _same_bits(got, want)
