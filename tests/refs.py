"""ctypes loaders for the two CHECKERS (test infrastructure, never the product):

  * ``oracle()``  — oracle/_build/liboracle.so, our plain-C restatement (oracle/ggml_oracle.c)
  * ``ref()``     — oracle/_ref/libctransformers_ref.so, the unmodified reference compiled from its
                    sources by oracle/Makefile (only where those sources are present); the tests
                    compare with what it produced through tests/golden/, tests/golden/make_golden.py
                    regenerates that data from it
"""
import ctypes as C
import hashlib
import os
import subprocess
import zlib
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
ORACLE_SO = ROOT / "oracle" / "_build" / "liboracle.so"
REF_SO = ROOT / "oracle" / "_ref" / "libctransformers_ref.so"
GOLD = ROOT / "tests" / "golden"

# ggml type ids (ggml.h enum ggml_type)
F32, F16, Q4_0, Q5_0, Q8_0, Q4_K, Q5_K, Q6_K, Q8_K = 0, 1, 2, 6, 8, 12, 13, 14, 15
BLOCK = {Q4_0: (32, 18), Q5_0: (32, 22), Q8_0: (32, 34), Q4_K: (256, 144), Q5_K: (256, 176), Q6_K: (256, 210), Q8_K: (256, 292),
         F32: (1, 4), F16: (1, 2)}
TYPE_NAME = {Q4_0: "q4_0", Q5_0: "q5_0", Q8_0: "q8_0", Q4_K: "q4_K", Q5_K: "q5_K", Q6_K: "q6_K"}


def row_bytes(t, k):
    bs, sz = BLOCK[t]
    assert k % bs == 0
    return k // bs * sz


_oracle = None
_ref = None


def oracle():
    global _oracle
    if _oracle is None:
        if not ORACLE_SO.exists():
            subprocess.check_call(["make", "-C", str(ROOT / "oracle"), "oracle"])
        o = C.CDLL(str(ORACLE_SO))
        fp, vp, i = C.POINTER(C.c_float), C.c_void_p, C.c_int
        o.orc_fp16_to_fp32.restype = C.c_float
        o.orc_fp16_to_fp32.argtypes = [C.c_uint16]
        o.orc_fp32_to_fp16.restype = C.c_uint16
        o.orc_fp32_to_fp16.argtypes = [C.c_float]
        for n in ("orc_vec_dot_q4_0_q8_0", "orc_vec_dot_q5_0_q8_0", "orc_vec_dot_q8_0_q8_0", "orc_vec_dot_q4_K_q8_K", "orc_vec_dot_q5_K_q8_K",
                  "orc_vec_dot_q6_K_q8_K"):
            getattr(o, n).restype = C.c_float
            getattr(o, n).argtypes = [i, vp, vp]
        o.orc_mul_mat.restype = i
        o.orc_mul_mat.argtypes = [i, vp, vp, vp, i, i, i]
        o.orc_rms_norm_mul.argtypes = [vp, vp, vp, i, C.c_float]
        o.orc_layer_norm_mul_add.argtypes = [vp, vp, vp, vp, i, C.c_float]
        o.orc_rope.argtypes = [vp, i, i, i, i, C.c_float, C.c_float]
        o.orc_rope_table.argtypes = [vp, i, i, C.c_float, C.c_float]
        o.orc_attn_head.argtypes = [vp, vp, C.c_size_t, vp, C.c_size_t, i, i, C.c_float, vp]
        _oracle = o
    return _oracle


class _Traits(C.Structure):
    _fields_ = [("type_name", C.c_char_p), ("blck_size", C.c_int), ("type_size", C.c_size_t), ("is_quantized", C.c_bool),
                ("to_float", C.c_void_p), ("from_float", C.c_void_p), ("from_float_reference", C.c_void_p),
                ("vec_dot", C.c_void_p), ("vec_dot_type", C.c_int)]


def have_ref():
    return REF_SO.exists()


def ref():
    """The compiled reference (AVX2 build).  Also initialises ggml's fp16 tables once."""
    global _ref
    if _ref is None:
        r = C.CDLL(str(REF_SO))
        r.ggml_internal_get_type_traits.restype = _Traits
        r.ggml_internal_get_type_traits.argtypes = [C.c_int]

        class _IP(C.Structure):
            _fields_ = [("mem_size", C.c_size_t), ("mem_buffer", C.c_void_p), ("no_alloc", C.c_bool)]
        r.ggml_init.restype = C.c_void_p
        r.ggml_init.argtypes = [_IP]
        r.ggml_free.argtypes = [C.c_void_p]
        r.ggml_free(r.ggml_init(_IP(1 << 20, None, False)))  # builds table_silu_f16 & co (ggml.c:4319-4333)
        r.ggml_quantize_chunk.restype = C.c_size_t
        r.ggml_quantize_chunk.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        _ref = r
    return _ref


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def ref_traits(t):
    tr = ref().ggml_internal_get_type_traits(t)
    to_float = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p, C.c_int)(tr.to_float) if tr.to_float else None
    from_float = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p, C.c_int)(tr.from_float) if tr.from_float else None
    vec_dot = C.CFUNCTYPE(None, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p)(tr.vec_dot) if tr.vec_dot else None
    return dict(to_float=to_float, from_float=from_float, vec_dot=vec_dot, vec_dot_type=tr.vec_dot_type)


def ref_quantize(t, x):
    """Quantize f32 rows [M,K] with the reference's own quantizer (ggml.c:19319 ggml_quantize_chunk)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    m, k = x.shape
    out = np.zeros(m * row_bytes(t, k), dtype=np.uint8)
    hist = np.zeros(16, dtype=np.int64)
    n = ref().ggml_quantize_chunk(t, ptr(x), ptr(out), 0, m * k, ptr(hist))
    assert n == out.size, (n, out.size)
    return out


def ref_quantize_act(t, x):
    """Quantize an activation row with the reference's from_float for type t (Q8_K / Q8_0)."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    out = np.zeros(row_bytes(t, x.size), dtype=np.uint8)
    ref_traits(t)["from_float"](ptr(x), ptr(out), x.size)
    return out


def ref_vec_dot(t, k, wrow, act):
    s = np.zeros(1, dtype=np.float32)
    ref_traits(t)["vec_dot"](k, ptr(s), ptr(wrow), ptr(act))
    return float(s[0])


# --------------------------------------------------------------------------------------------------------------
# Stored reference results (tests/golden/make_golden.py writes them from the compiled reference)
def digest(a):
    """SHA-256 of an array's bytes: equal digests <=> bit-identical results (float32 for float arrays)."""
    a = np.ascontiguousarray(a, np.float32 if np.asarray(a).dtype.kind == "f" else None)
    return hashlib.sha256(a.tobytes()).hexdigest()


def run_digests(run):
    """modelcases.run_greedy's result as stored: digests of the first logits, first embeddings, last logits."""
    return [digest(run[0]), digest(run[1]), digest(run[3])]


_golden = {}


def golden(name):
    if name not in _golden:
        _golden[name] = dict(np.load(GOLD / f"{name}.npz"))
    return _golden[name]


def pool_matrix(t, m, k, rng):
    """[m, k] weights of type t made of blocks the reference's quantizer produced (tests/golden/ref_quant_pool.npz, from
    seeded N(0.01, 0.05²) rows): every scale / min bit pattern the real quantizer emits, drawn block by block with rng."""
    pool = golden("ref_quant_pool")[f"pool_{t}"]
    bs, _ = BLOCK[t]
    assert k % bs == 0
    return np.ascontiguousarray(pool[rng.integers(0, len(pool), m * (k // bs))]).reshape(-1)


def pool_quantizer(t, w):
    """synth.write_* quantizer that stands in for the reference's: blocks from the stored pool, drawn with a rng seeded
    from the f32 tensor the writer passes (so each tensor gets its own, reproducible draw)."""
    w = np.ascontiguousarray(w, np.float32)
    rng = np.random.default_rng(zlib.crc32(w[:4].tobytes()))
    return pool_matrix(t, w.shape[0], w.shape[1], rng)


# --------------------------------------------------------------------------------------------------------------
# Whole-model oracle (oracle/llama_oracle.c) driven from a GGUF file
def read_gguf(path):
    """Tiny GGUF v2/v3 reader: returns (kv dict, {name: (type, shape, np.uint8 view of the data)})."""
    import struct
    buf = np.memmap(path, dtype=np.uint8, mode="r")
    pos = [0]

    def rd(fmt):
        v = struct.unpack_from("<" + fmt, buf, pos[0])
        pos[0] += struct.calcsize("<" + fmt)
        return v[0] if len(v) == 1 else v

    def rstr():
        n = rd("Q")
        s = bytes(buf[pos[0]:pos[0] + n])
        pos[0] += n
        return s

    scalar = {0: "B", 1: "b", 2: "H", 3: "h", 4: "I", 5: "i", 6: "f", 7: "?", 10: "Q", 11: "q", 12: "d"}
    magic, version, n_tensors, n_kv = rd("I"), rd("I"), rd("Q"), rd("Q")
    assert magic == 0x46554747 and version >= 2
    kv = {}
    for _ in range(n_kv):
        key = rstr().decode()
        t = rd("I")
        if t == 8:
            kv[key] = rstr()
        elif t == 9:
            et, n = rd("I"), rd("Q")
            if et == 8:
                kv[key] = [rstr() for _ in range(n)]
            else:
                sz = struct.calcsize(scalar[et])
                kv[key] = np.frombuffer(buf, dtype=np.dtype("<" + scalar[et]), count=n, offset=pos[0]).copy()
                pos[0] += sz * n
        else:
            kv[key] = rd(scalar[t])
    infos = []
    for _ in range(n_tensors):
        name = rstr().decode()
        nd = rd("I")
        shape = [rd("Q") for _ in range(nd)]
        t, off = rd("I"), rd("Q")
        infos.append((name, t, shape, off))
    align = kv.get("general.alignment", 32)
    start = (pos[0] + align - 1) // align * align
    tensors = {}
    for name, t, shape, off in infos:
        rows = int(np.prod(shape[1:])) if len(shape) > 1 else 1
        nbytes = row_bytes(t, shape[0]) * rows
        tensors[name] = (t, shape, buf[start + off:start + off + nbytes])
    return kv, tensors


class OracleModel:
    """oracle/llama_oracle.c bound to one GGUF file (keeps the arrays alive)."""

    def __init__(self, path, n_ctx):
        o = oracle()
        kv, tensors = read_gguf(path)
        arch = kv["general.architecture"].decode()
        g = lambda k, d=None: kv.get(f"{arch}.{k}", d)
        self.falcon = arch == "falcon"
        self.n_vocab = len(kv["tokenizer.ggml.tokens"])
        self.n_embd, self.n_ff, self.n_head, self.n_layer = g("embedding_length"), g("feed_forward_length"), g("attention.head_count"), g("block_count")
        self.n_head_kv = g("attention.head_count_kv", self.n_head)
        eps = g("attention.layer_norm_epsilon") if self.falcon else g("attention.layer_norm_rms_epsilon")
        rope_base = g("rope.freq_base", 10000.0)
        lin = g("rope.scale_linear", 1.0)
        o.orc_model_new.restype = C.c_void_p
        o.orc_model_new.argtypes = [C.c_int] * 8 + [C.c_float] * 3
        o.orc_model_set_mat.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        o.orc_model_set_vec.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p]
        o.orc_model_set_trace.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        o.orc_model_free.argtypes = [C.c_void_p]
        o.orc_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        self.o, self.keep = o, []
        self.m = o.orc_model_new(int(self.falcon), self.n_vocab, self.n_embd, self.n_ff, self.n_head, self.n_head_kv, self.n_layer, n_ctx,
                                 eps, rope_base, 1.0 / lin if lin != 1.0 else 1.0)

        def mat(layer, slot, name):
            t, shape, data = tensors[name]
            a = np.ascontiguousarray(data)
            self.keep.append(a)
            o.orc_model_set_mat(self.m, layer, slot, t, shape[0], int(np.prod(shape[1:])), ptr(a))

        def vec(layer, slot, name):
            if name not in tensors:
                return
            a = np.ascontiguousarray(tensors[name][2]).view(np.float32)
            self.keep.append(a)
            o.orc_model_set_vec(self.m, layer, slot, ptr(a))

        mat(-1, 0, "token_embd.weight")
        mat(-1, 1, "output.weight")
        vec(-1, 0, "output_norm.weight")
        vec(-1, 1, "output_norm.bias")
        for il in range(self.n_layer):
            b = f"blk.{il}."
            vec(il, 0, b + "attn_norm.weight"); vec(il, 1, b + "attn_norm.bias")
            vec(il, 2, b + "attn_norm_2.weight"); vec(il, 3, b + "attn_norm_2.bias"); vec(il, 4, b + "ffn_norm.weight")
            names = ({3: "attn_qkv", 4: "attn_output", 6: "ffn_down", 7: "ffn_up"} if self.falcon else
                     {0: "attn_q", 1: "attn_k", 2: "attn_v", 4: "attn_output", 5: "ffn_gate", 6: "ffn_down", 7: "ffn_up"})
            for slot, nm in names.items():
                mat(il, slot, b + nm + ".weight")
        self.logits = np.zeros(self.n_vocab, np.float32)
        self.embd = np.zeros(self.n_embd, np.float32)
        self.trace_layers = np.zeros((self.n_layer, self.n_embd), np.float32)
        self.trace_attn = np.zeros((self.n_layer, self.n_embd), np.float32)
        o.orc_model_set_trace(self.m, ptr(self.trace_layers), ptr(self.trace_attn))
        self.n_past = 0

    def set_tp(self, world):
        """Switch the restatement to the sharded engine's summation order (oracle/llama_oracle.c: tp_world)."""
        from ctransformers_b200 import tp_plan
        sh = tp_plan.plan(self.n_embd, self.n_head, self.n_head_kv, self.n_ff, self.n_vocab, world)
        wo = (C.c_int * (world + 1))(*([s.attn_k[0] for s in sh] + [sh[-1].attn_k[1]]))
        w2 = (C.c_int * (world + 1))(*([s.ff[0] for s in sh] + [sh[-1].ff[1]]))
        self.o.orc_model_set_tp.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        assert self.o.orc_model_set_tp(self.m, world, wo, w2) == 0

    def eval(self, tokens, batch_size=8):
        """Same chunking as the reference's LLM::BatchEval (llm.h:40-54): the chunk an attention row belongs to fixes its length."""
        toks = np.asarray(tokens, dtype=np.int32)
        for start in range(0, len(toks), batch_size):
            t = np.ascontiguousarray(toks[start:start + batch_size])
            rc = self.o.orc_eval(self.m, ptr(t), len(t), self.n_past, ptr(self.logits), ptr(self.embd))
            assert rc == 0, rc
            self.n_past += len(t)
        return self.logits

    def __del__(self):
        if getattr(self, "m", None):
            self.o.orc_model_free(self.m)
            self.m = None
