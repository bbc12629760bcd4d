"""ctypes bindings for the CPU oracle (libtce_oracle.so) and the in-place reference builds (oracle/_ref).

TEST INFRASTRUCTURE ONLY -- see oracle/__init__.py.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
REF_DIR = HERE / "_ref"

_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(np.uint8, flags="C_CONTIGUOUS")
_i8p = np.ctypeslib.ndpointer(np.int8, flags="C_CONTIGUOUS")
_u16p = np.ctypeslib.ndpointer(np.uint16, flags="C_CONTIGUOUS")
_u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")


def build(ref: bool = True) -> None:
    """(Re)build the oracle .so and, with ref, oracle/_ref.  oracle/Makefile builds and rebuilds oracle/_ref from the reference tree
    (its REF, or TCE_REFERENCE_DIR when set) wherever that tree is readable, and leaves it alone elsewhere."""
    tree = os.environ.get("TCE_REFERENCE_DIR")
    targets = ["oracle"] + (["ref"] + ([f"REF={tree}"] if tree else []) if ref else [])
    subprocess.run(["make", "-s", "-C", str(HERE)] + targets, check=True)


_ORACLE = None


def lib() -> C.CDLL:
    global _ORACLE
    if _ORACLE is None:
        so = HERE / "libtce_oracle.so"
        if not so.exists():
            build(ref=False)
        _ORACLE = C.CDLL(str(so))
        L = _ORACLE
        L.orc_calculate_zeros_width.restype = C.c_int
        L.orc_w4a16_gemv.restype = C.c_int
        L.orc_w4a16_gemv.argtypes = [_u16p, _u32p, _u32p, _u16p, _f32p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_naive_mat_mul_int4.argtypes = [_f32p, _u8p, _f32p, C.c_float, _f32p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_naive_mat_mul_int4_with_offset.argtypes = [_f32p, _u8p, _f32p, _f32p, C.c_float, _f32p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_int4_fast_ref.argtypes = [_f32p, _u8p, _f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int]
        L.orc_naive_mat_mul_fp16_int4.argtypes = [_u16p, _i32p, _u16p, _u16p, C.c_int, C.c_int, C.c_int, C.c_int]
        L.orc_mat_mul_transposed.argtypes = [_f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int]
        L.orc_int8_matmul.argtypes = [_i8p, _i8p, _i8p, _i8p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int]
        L.orc_int8_matmul_nobias.argtypes = [_i8p, _i8p, _i8p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_int, C.c_int]
        L.orc_int8_matmul_nobias_batch.argtypes = L.orc_int8_matmul_nobias.argtypes
        L.orc_int8_matmul_bfp32_ofp32.argtypes = [_i8p, _i8p, _f32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_float]
        L.orc_int8_matmul_nobias_ofp32.argtypes = [_i8p, _i8p, _f32p, C.c_int, C.c_int, C.c_int, C.c_float]
        L.orc_int8_matmul_nobias_ofp32_batch.argtypes = L.orc_int8_matmul_nobias_ofp32.argtypes
        L.orc_naive_mat_mul_int8.argtypes = [_i8p, _i8p, _i8p, C.c_int, C.c_int, C.c_int, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_float, C.c_int, C.c_int]
        L.orc_rmsnorm.argtypes = [_f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_float]
        L.orc_layernorm_q.argtypes = [_f32p, _f32p, _f32p, _i8p, C.c_int, C.c_int]
        L.orc_rope.argtypes = [_f32p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, _f32p, _f32p, C.c_int]
        L.orc_llama_attention_core.restype = C.c_int
        L.orc_llama_attention_core.argtypes = [_f32p, _f32p, _f32p, C.c_void_p, C.c_void_p, _f32p, _f32p, _f32p, C.c_float,
                                               C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _f32p, _f32p, _f32p]
        L.orc_opt_int8_attention_core.restype = C.c_int
        L.orc_opt_int8_attention_core.argtypes = [_i8p, _i8p, _i8p, C.c_void_p, C.c_void_p, _f32p, C.c_float, C.c_float,
                                                  C.c_int, C.c_int, C.c_int, C.c_int, _i8p, _i8p, _i8p]
    return _ORACLE


# ----------------------------------------------------------------------------------------------
# numpy-level wrappers (the oracle's public face for tests)
# ----------------------------------------------------------------------------------------------

def zeros_width(ic: int, group: int = 128) -> int:
    return int(lib().orc_calculate_zeros_width(ic, group))


def w4a16_gemv(x_half: np.ndarray, w: np.ndarray, zeros: np.ndarray, scales_half: np.ndarray, group: int = 128):
    """x fp16 [M,IC]; w uint32 [OC,IC/8]; zeros uint32 [OC,zw]; scales fp16 [OC,zw*8] -> fp32 [M,OC]."""
    x_half = np.ascontiguousarray(x_half, dtype=np.float16)
    M, IC = x_half.shape
    OC = w.shape[0]
    y = np.zeros((M, OC), np.float32)
    rc = lib().orc_w4a16_gemv(x_half.view(np.uint16), np.ascontiguousarray(w, np.uint32), np.ascontiguousarray(zeros, np.uint32),
                              np.ascontiguousarray(scales_half, np.float16).view(np.uint16), y, None, M, IC, OC, group)
    assert rc == 0
    return y


def naive_mat_mul_int4(A, B, scales, zero_point=8.0, block_size=128):
    A = np.ascontiguousarray(A, np.float32)
    M, IC = A.shape
    OC = B.shape[0]
    out = np.zeros((M, OC), np.float32)
    lib().orc_naive_mat_mul_int4(A, np.ascontiguousarray(B, np.uint8), np.ascontiguousarray(scales, np.float32).ravel(), zero_point, out, M, IC, OC, block_size)
    return out


def int8_matmul(variant: int, A, B, bias8=None, biasf=None, alpha=1.0, beta=1.0, q_min=-128, q_max=127):
    """variant numbering = oracle/ref_shim.cc ref_int8_matmul.  B is [N,K] (or [M,N,K] for batch variants)."""
    A = np.ascontiguousarray(A, np.int8)
    B = np.ascontiguousarray(B, np.int8)
    M, K = A.shape
    N = B.shape[-2]
    L = lib()
    if variant in (0, 1):
        out = np.zeros((M, N), np.int8)
        L.orc_int8_matmul(A, B, np.ascontiguousarray(bias8, np.int8), out, M, N, K, alpha, beta, q_min, q_max)
    elif variant == 2:
        out = np.zeros((M, N), np.int8)
        L.orc_int8_matmul_nobias(A, B, out, M, N, K, alpha, q_min, q_max)
    elif variant == 3:
        out = np.zeros((M, N), np.int8)
        L.orc_int8_matmul_nobias_batch(A, B, out, M, N, K, alpha, q_min, q_max)
    elif variant in (4, 5):
        out = np.zeros((M, N), np.float32)
        L.orc_int8_matmul_bfp32_ofp32(A, B, np.ascontiguousarray(biasf, np.float32), out, M, N, K, alpha)
    elif variant == 6:
        out = np.zeros((M, N), np.float32)
        L.orc_int8_matmul_nobias_ofp32(A, B, out, M, N, K, alpha)
    elif variant == 7:
        out = np.zeros((M, N), np.float32)
        L.orc_int8_matmul_nobias_ofp32_batch(A, B, out, M, N, K, alpha)
    else:
        raise ValueError(variant)
    return out


def rmsnorm(x, weight, eps):
    x = np.ascontiguousarray(x, np.float32)
    out = np.zeros_like(x)
    lib().orc_rmsnorm(x, np.ascontiguousarray(weight, np.float32), out, x.shape[0], x.shape[1], eps)
    return out


def rope_tables(max_len: int, head_dim: int, theta: float = 10000.0):
    """cos/sin tables [max_len, head_dim] in the HF rotate-half convention the reference loads from
    ``rotary_emb/{cos,sin}_cached.bin`` (llm/src/ops/RotaryPosEmb.cc indexes cos(0, pos, j), j<head_dim)."""
    inv = 1.0 / (theta ** (np.arange(0, head_dim, 2, dtype=np.float64) / head_dim))
    t = np.arange(max_len, dtype=np.float64)
    fr = np.outer(t, inv)
    emb = np.concatenate([fr, fr], axis=1)
    return np.cos(emb).astype(np.float32), np.sin(emb).astype(np.float32)


def llama_attention_core(q, k, v, past_k, past_v, mask, cosb, sinb, alpha, H, KVH, hd):
    """fp32 GQA attention between the projections (see tce_oracle.c).  q [s,H*hd], k/v [s,KVH*hd],
    past_* [KVH,past,hd] or None.  Returns (attn_out [s,H*hd], final_k [KVH,tgz,hd], final_v)."""
    q = np.ascontiguousarray(q, np.float32)
    k = np.ascontiguousarray(k, np.float32)
    v = np.ascontiguousarray(v, np.float32)
    s = q.shape[0]
    past = 0 if past_k is None else past_k.shape[1]
    tgz = s + past
    out = np.zeros((s, H * hd), np.float32)
    fk = np.zeros((KVH, tgz, hd), np.float32)
    fv = np.zeros((KVH, tgz, hd), np.float32)
    pk = None if past_k is None else np.ascontiguousarray(past_k, np.float32)
    pv = None if past_v is None else np.ascontiguousarray(past_v, np.float32)
    rc = lib().orc_llama_attention_core(q, k, v, None if pk is None else pk.ctypes.data, None if pv is None else pv.ctypes.data,
                                        np.ascontiguousarray(mask, np.float32), np.ascontiguousarray(cosb, np.float32),
                                        np.ascontiguousarray(sinb, np.float32), alpha, s, past, H, KVH, hd, out, fk, fv)
    assert rc == 0
    return out, fk, fv


def opt_int8_attention_core(q8, k8, v8, past_k, past_v, mask, qk_alpha, pv_alpha, H, hd):
    q8 = np.ascontiguousarray(q8, np.int8)
    s = q8.shape[0]
    past = 0 if past_k is None else past_k.shape[1]
    tgz = s + past
    out = np.zeros((s, H * hd), np.int8)
    fk = np.zeros((H, tgz, hd), np.int8)
    fv = np.zeros((H, tgz, hd), np.int8)
    pk = None if past_k is None else np.ascontiguousarray(past_k, np.int8)
    pv = None if past_v is None else np.ascontiguousarray(past_v, np.int8)
    rc = lib().orc_opt_int8_attention_core(q8, np.ascontiguousarray(k8, np.int8), np.ascontiguousarray(v8, np.int8),
                                           None if pk is None else pk.ctypes.data, None if pv is None else pv.ctypes.data,
                                           np.ascontiguousarray(mask, np.float32), qk_alpha, pv_alpha, s, past, H, hd, out, fk, fv)
    assert rc == 0
    return out, fk, fv


def causal_mask(sqlen: int, past: int, neg: float = -3.402823466e38):
    """prepare_decoder_attention_mask semantics (llm/src/nn_modules/non_cuda/Int4llamaDecoder.cc): 0 on/below
    the diagonal (shifted by `past`), lowest-float above."""
    tgz = sqlen + past
    m = np.zeros((sqlen, tgz), np.float32)
    for i in range(sqlen):
        m[i, past + i + 1:] = neg
    return m


# ----------------------------------------------------------------------------------------------
# reference builds (oracle/_ref): only present when built in a container that has /root/reference
# ----------------------------------------------------------------------------------------------
_REF = {}


def ref_available(kind: str = "generic") -> bool:
    return (REF_DIR / f"libtce_ref_{kind}.so").exists()


def ref(kind: str = "generic") -> C.CDLL:
    if kind not in _REF:
        so = REF_DIR / f"libtce_ref_{kind}.so"
        if not so.exists():
            raise FileNotFoundError(f"{so} not built (needs /root/reference; run `make -C oracle ref`)")
        L = C.CDLL(str(so))
        L.ref_naive_mat_mul_int4.argtypes = [_f32p, _u8p, _f32p, _f32p, C.c_void_p, _f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        L.ref_int8_matmul.argtypes = [C.c_int, _i8p, _i8p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                      C.c_float, C.c_float, C.c_int, C.c_int, C.c_int]
        L.ref_naive_mat_mul_int8.argtypes = [_i8p, _i8p, _i8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int, C.c_int]
        L.ref_mat_mul_transposed.argtypes = [_f32p, _f32p, _f32p, C.c_int, C.c_int, C.c_int]
        if kind == "generic":
            L.ref_naive_mat_mul_fp16_int4.argtypes = [_u16p, _i32p, _u16p, _u16p, C.c_int, C.c_int, C.c_int, C.c_int]
        if kind == "avx":
            L.ref_w4a8_avx.argtypes = [C.c_void_p] * 6 + [C.c_int] * 4
        _REF[kind] = L
    return _REF[kind]


_REF_CUDA = None


def ref_cuda():
    """oracle/_ref/libtce_ref_cuda.so: the reference's own kernels/cuda/gemv_cuda.cu compiled for sm_100a (GPU-side baseline and
    second oracle).  Takes raw DEVICE pointers; launches on the legacy default stream like the reference."""
    global _REF_CUDA
    if _REF_CUDA is None:
        so = REF_DIR / "libtce_ref_cuda.so"
        if not so.exists():
            raise FileNotFoundError(f"{so} not built (needs /root/reference and nvcc; run `make -C oracle ref`)")
        L = C.CDLL(str(so))
        L.ref_cuda_gemv.restype = C.c_int
        L.ref_cuda_gemv.argtypes = [C.c_void_p] * 5 + [C.c_int] * 3
        _REF_CUDA = L
    return _REF_CUDA


_REF_GEN = None


def ref_sample_candidates(logits, window=(), top_k=40, top_p=0.95, temp=0.8, repeat_penalty=1.1, frequency_penalty=0.0, presence_penalty=0.0):
    """The reference's own sampling chain (llm/src/Generate.cc compiled in place, oracle/_ref/libtce_ref_generate.so) in the order of
    LLaMAGenerate.cu:112-166, without the final draw: -> (ids, probs) of the surviving candidates."""
    global _REF_GEN
    if _REF_GEN is None:
        import os

        so = REF_DIR / "libtce_ref_generate.so"
        if not so.exists():
            raise FileNotFoundError(f"{so} not built (needs /root/reference; run `make -C oracle ref`)")
        L = C.CDLL(str(so), mode=os.RTLD_LAZY)  # Generate.h drags in model classes the sampling functions never call
        L.ref_sample_candidates.restype = C.c_int
        L.ref_sample_candidates.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int] + [C.c_float] * 5 + [C.c_void_p, C.c_void_p]
        _REF_GEN = L
    lg = np.ascontiguousarray(logits, dtype=np.float32)
    win = np.ascontiguousarray(np.asarray(list(window), dtype=np.int32))
    ids = np.zeros(lg.size, dtype=np.int32)
    probs = np.zeros(lg.size, dtype=np.float32)
    n = _REF_GEN.ref_sample_candidates(lg.ctypes.data, lg.size, win.ctypes.data if win.size else None, int(win.size), int(top_k), float(top_p), float(temp),
                                       float(repeat_penalty), float(frequency_penalty), float(presence_penalty), ids.ctypes.data, probs.ctypes.data)
    return ids[:n].copy(), probs[:n].copy()


def ref_naive_mat_mul_int4(A, B, scales, zero_point=8.0, block_size=128, kind="generic"):
    A = np.ascontiguousarray(A, np.float32)
    M, IC = A.shape
    OC = B.shape[0]
    out = np.zeros((M, OC), np.float32)
    zp = np.array([zero_point], np.float32)
    ref(kind).ref_naive_mat_mul_int4(A, np.ascontiguousarray(B, np.uint8), np.ascontiguousarray(scales, np.float32).ravel(), zp, None, out,
                                     M, IC, OC, block_size, 0)
    return out


def ref_int8_matmul(variant: int, A, B, bias8=None, biasf=None, alpha=1.0, beta=1.0, q_min=-128, q_max=127, kind="generic", num_thread=1):
    A = np.ascontiguousarray(A, np.int8)
    B = np.ascontiguousarray(B, np.int8)
    M, K = A.shape
    N = B.shape[-2]
    c8 = np.zeros((M, N), np.int8)
    cf = np.zeros((M, N), np.float32)
    b8 = None if bias8 is None else np.ascontiguousarray(bias8, np.int8)
    bf = None if biasf is None else np.ascontiguousarray(biasf, np.float32)
    ref(kind).ref_int8_matmul(variant, A, B, None if b8 is None else b8.ctypes.data, None if bf is None else bf.ctypes.data,
                              c8.ctypes.data, cf.ctypes.data, M, N, K, alpha, beta, q_min, q_max, num_thread)
    return c8 if variant in (0, 1, 2, 3) else cf


def aligned_empty(shape, dtype, align: int = 64) -> np.ndarray:
    """32-byte alignment is mandatory for the reference AVX kernels (SURVEY.md 8b Ownership)."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    raw = np.empty(n + align, np.uint8)
    off = (-raw.ctypes.data) % align
    return raw[off:off + n].view(dtype).reshape(shape)


# ----------------------------------------------------------------------------------------------
# reference MODULE build (oracle/_ref/libtce_ref_modules.so: llm/src/nn_modules/Int8OPTAttention.cc + its ops, unmodified)
# ----------------------------------------------------------------------------------------------
def write_opt_attention_params(root, W, B, bo, a_qkv, b_qkv, qk_alpha, pv_alpha, a_out):
    """The parameter tree Int8OPTAttention's constructor loads (load_W8A8B8O8Linear_params etc., llm/src/ops/*.cc:6-13).
    W: dict q,k,v,o -> int8 [E][E]; B: dict q,k,v -> int8 [E]; bo: float32 [E]."""
    import os

    f32 = lambda v: np.array([v], np.float32)
    for k in "qkv":
        d = os.path.join(root, f"{k}_proj")
        os.makedirs(d, exist_ok=True)
        np.ascontiguousarray(W[k], np.int8).tofile(os.path.join(d, "weight.bin"))
        np.ascontiguousarray(B[k], np.int8).tofile(os.path.join(d, "bias_int8.bin"))
        f32(a_qkv).tofile(os.path.join(d, "alpha.bin"))
        f32(b_qkv).tofile(os.path.join(d, "beta.bin"))
    d = os.path.join(root, "out_proj")
    os.makedirs(d, exist_ok=True)
    np.ascontiguousarray(W["o"], np.int8).tofile(os.path.join(d, "weight.bin"))
    np.ascontiguousarray(bo, np.float32).tofile(os.path.join(d, "bias.bin"))
    f32(a_out).tofile(os.path.join(d, "alpha.bin"))
    for name, v in (("qk_bmm", qk_alpha), ("pv_bmm", pv_alpha)):
        d = os.path.join(root, name)
        os.makedirs(d, exist_ok=True)
        f32(v).tofile(os.path.join(d, "alpha.bin"))


def ref_int8_opt_attention(param_root, hidden, E, H, prefill, decode_steps, max_sqlen=256):
    """Runs the REFERENCE Int8OPTAttention::forward (prefill rows, then single-token steps).  Returns (out fp32 [T][E], K, V int8 [H][T][hd])."""
    so = REF_DIR / "libtce_ref_modules.so"
    if not so.exists():
        raise FileNotFoundError(f"{so} not built (needs /root/reference; run `make -C oracle ref`)")
    L = C.CDLL(str(so))
    L.ref_int8_opt_attention.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    hidden = np.ascontiguousarray(hidden, np.int8)
    T, hd = prefill + decode_steps, E // H
    out = np.zeros((T, E), np.float32)
    fk = np.zeros((H, T, hd), np.int8)
    fv = np.zeros((H, T, hd), np.int8)
    n = L.ref_int8_opt_attention(str(param_root).encode(), E, H, max_sqlen, hidden.ctypes.data, prefill, decode_steps, out.ctypes.data, fk.ctypes.data,
                                 fv.ctypes.data)
    assert n == T
    return out, fk, fv


def write_opt_decoder_layer_params(root, W, B, bo, ln, fc, scales):
    """Parameter tree of Int8OPTDecoderLayer's constructor (llm/src/nn_modules/Int8OPTDecoderLayer.cc:60-90): self_attn/... (as above),
    self_attn_layer_norm|final_layer_norm/{weight,bias}.bin, fc1/{weight,bias_int8,alpha,beta}.bin, fc2/{weight,bias,alpha}.bin.
    ln: dict ln1w, ln1b, ln2w, ln2b (float32 [E]); fc: dict w1 int8 [F][E], b1 int8 [F], w2 int8 [E][F], b2 float32 [E];
    scales: dict a_qkv, b_qkv, qk_alpha, pv_alpha, a_out, a1, b1, a2."""
    import os

    f32 = lambda v: np.array([v], np.float32)
    write_opt_attention_params(os.path.join(root, "self_attn"), W, B, bo, scales["a_qkv"], scales["b_qkv"], scales["qk_alpha"], scales["pv_alpha"], scales["a_out"])
    for name, w, b in (("self_attn_layer_norm", ln["ln1w"], ln["ln1b"]), ("final_layer_norm", ln["ln2w"], ln["ln2b"])):
        d = os.path.join(root, name)
        os.makedirs(d, exist_ok=True)
        np.ascontiguousarray(w, np.float32).tofile(os.path.join(d, "weight.bin"))
        np.ascontiguousarray(b, np.float32).tofile(os.path.join(d, "bias.bin"))
    d = os.path.join(root, "fc1")
    os.makedirs(d, exist_ok=True)
    np.ascontiguousarray(fc["w1"], np.int8).tofile(os.path.join(d, "weight.bin"))
    np.ascontiguousarray(fc["b1"], np.int8).tofile(os.path.join(d, "bias_int8.bin"))
    f32(scales["a1"]).tofile(os.path.join(d, "alpha.bin"))
    f32(scales["b1"]).tofile(os.path.join(d, "beta.bin"))
    d = os.path.join(root, "fc2")
    os.makedirs(d, exist_ok=True)
    np.ascontiguousarray(fc["w2"], np.int8).tofile(os.path.join(d, "weight.bin"))
    np.ascontiguousarray(fc["b2"], np.float32).tofile(os.path.join(d, "bias.bin"))
    f32(scales["a2"]).tofile(os.path.join(d, "alpha.bin"))


_MODLIBS = {}


def modules_lib(kind: str = "ref_modules"):
    """kind = "ref_modules": the reference's modules on the reference's own kernels/ref bodies (CPU).
    kind = "callsites_cuda": the SAME reference call sites compiled unchanged with -DQM_CUDA on this repo's library (the drop-in proof)."""
    if kind not in _MODLIBS:
        so = REF_DIR / f"libtce_{kind}.so"
        if not so.exists():
            raise FileNotFoundError(f"{so} not built (run `make -C oracle ref` where /root/reference exists)")
        L = C.CDLL(str(so))
        L.ref_int8_opt_attention.restype = C.c_int
        L.ref_int8_opt_attention.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, _i8p, C.c_int, C.c_int, _f32p, _i8p, _i8p]
        L.ref_int8_opt_decoder_layer.restype = C.c_int
        L.ref_int8_opt_decoder_layer.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, _f32p, C.c_int, C.c_int, _f32p, _i8p, _i8p]
        if kind == "callsites_cuda":
            L.ref_linear_half_int4.restype = C.c_int
            L.ref_linear_half_int4.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, _u16p, _u16p]
        _MODLIBS[kind] = L
    return _MODLIBS[kind]


def run_opt_decoder_layer(kind, param_root, hidden_f32, E, H, F, prefill, decode_steps, max_sqlen=256):
    hidden = np.ascontiguousarray(hidden_f32, np.float32)
    total = prefill + decode_steps
    out = np.zeros((total, E), np.float32)
    hd = E // H
    fk = np.zeros((H, total, hd), np.int8)
    fv = np.zeros((H, total, hd), np.int8)
    n = modules_lib(kind).ref_int8_opt_decoder_layer(str(param_root).encode(), E, H, F, max_sqlen, hidden, prefill, decode_steps, out, fk, fv)
    assert n == total
    return out, fk, fv


def run_opt_attention(kind, param_root, hidden_i8, E, H, prefill, decode_steps, max_sqlen=256):
    hidden = np.ascontiguousarray(hidden_i8, np.int8)
    total = prefill + decode_steps
    out = np.zeros((total, E), np.float32)
    hd = E // H
    fk = np.zeros((H, total, hd), np.int8)
    fv = np.zeros((H, total, hd), np.int8)
    n = modules_lib(kind).ref_int8_opt_attention(str(param_root).encode(), E, H, max_sqlen, hidden, prefill, decode_steps, out, fk, fv)
    assert n == total
    return out, fk, fv


def oracle_int8_opt_attention(hidden, W, B, bo, a_qkv, b_qkv, qk_alpha, pv_alpha, a_out, H, prefill, decode_steps):
    """The same module flow composed from the oracle: projections (orc_int8_matmul), core, out_proj."""
    E = hidden.shape[1]
    hd = E // H
    pk = pv = None
    past = row = 0
    outs = []
    for call in range(1 + decode_steps):
        s = prefill if call == 0 else 1
        x = hidden[row:row + s]
        q, k, v = (int8_matmul(0, x, W[n], B[n], None, a_qkv, b_qkv) for n in "qkv")
        core, pk, pv = opt_int8_attention_core(q, k, v, pk, pv, causal_mask(s, past), qk_alpha, pv_alpha, H, hd)
        outs.append(int8_matmul(4, core, W["o"], biasf=bo, alpha=a_out))
        past += s
        row += s
    return np.concatenate(outs), pk, pv


# ----------------------------------------------------------------------------------------------
# reference Int4llamaAttention MODULE (CPU, the reference's own x86 flags): oracle/_ref/libtce_ref_llama.so
# ----------------------------------------------------------------------------------------------
def selection_matrix(rows: int, cols: int, rng):
    """0/1 matrix picking `rows` distinct input channels: survives INT4 quantisation exactly, so the module's linears
    become exact channel selections and the attention core can be compared at fp32 round-off."""
    sel = rng.permutation(cols)[:rows]
    W = np.zeros((rows, cols), np.float32)
    W[np.arange(rows), sel] = 1.0
    return W, sel


def exact_w4a8_activations(shape, rng, unit=2.0 ** -6):
    """fp32 activations that the reference's per-32 int8 activation quantiser (matmul_avx_int8_int4.cc:259-316) reproduces
    exactly: integers in [-127, 127] times a power of two, every 32-block holding a +-127."""
    xi = rng.integers(-127, 128, shape).astype(np.float32)
    blocks = xi.reshape(shape[0], shape[1] // 32, 32)
    blocks[:, :, 0] = 127 * np.sign(rng.standard_normal(blocks.shape[:2]))
    return (xi * np.float32(unit)).astype(np.float32)


def w4a8_activation_roundtrip(x):
    """What an identity / selection Linear_FP_int4 returns on the x86 build: x quantised per 32-block to int8 and rescaled
    (d = amax/127, id = 127/amax, round to nearest even) -- restates matmul_avx_int8_int4.cc:259-316 for the test harness."""
    xb = np.ascontiguousarray(x, np.float32).reshape(-1, 32)
    amax = np.abs(xb).max(1, keepdims=True)
    d = (amax / np.float32(127)).astype(np.float32)
    inv = np.where(amax != 0, np.float32(127) / np.where(amax != 0, amax, 1), 0).astype(np.float32)
    q = np.rint((xb * inv).astype(np.float32))
    return (q * d).astype(np.float32).reshape(np.shape(x))


def write_llama_attention_params(root, W, cosb, sinb, alpha):
    """Parameter tree of the CPU Int4llamaAttention (QM_x86): W dict q_proj/k_proj/v_proj/o_proj -> fp32 matrices."""
    import os

    from . import quant

    for name, w in W.items():
        d = os.path.join(root, name)
        os.makedirs(d, exist_ok=True)
        qs, sc = quant.quantize_q4_3(w)
        qs.tofile(os.path.join(d, "weight_int4.bin"))
        sc.astype(np.float32).tofile(os.path.join(d, "scaling_factor_int4.bin"))
        np.array([8.0], np.float32).tofile(os.path.join(d, "zero_point_int4.bin"))
    d = os.path.join(root, "rotary_emb")
    os.makedirs(d, exist_ok=True)
    np.ascontiguousarray(cosb, np.float32).tofile(os.path.join(d, "cos_cached.bin"))
    np.ascontiguousarray(sinb, np.float32).tofile(os.path.join(d, "sin_cached.bin"))
    d = os.path.join(root, "qk_bmm")
    os.makedirs(d, exist_ok=True)
    np.array([alpha], np.float32).tofile(os.path.join(d, "alpha.bin"))


def ref_int4_llama_attention(param_root, hidden, E, H, KVH, prefill, decode_steps, max_sqlen, num_thread=None, timing=False):
    """Runs the REFERENCE Int4llamaAttention::forward (CPU).  Returns (out fp32 [T][E], K, V fp32 [KVH][T][hd]); with timing=True also the wall
    seconds of the decode steps alone.  num_thread: the reference's NUM_THREAD global (its worker pool is sized by the first call of the process)."""
    so = REF_DIR / "libtce_ref_llama.so"
    if not so.exists():
        raise FileNotFoundError(f"{so} not built (needs /root/reference; run `make -C oracle ref`)")
    L = C.CDLL(str(so))
    if num_thread is not None:
        C.c_int.in_dll(L, "NUM_THREAD").value = int(num_thread)
    L.ref_int4_llama_attention_timed.argtypes = [C.c_char_p] + [C.c_int] * 4 + [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    hidden = np.ascontiguousarray(hidden, np.float32)
    T, hd = prefill + decode_steps, E // H
    out = np.zeros((T, E), np.float32)
    fk = np.zeros((KVH, T, hd), np.float32)
    fv = np.zeros((KVH, T, hd), np.float32)
    secs = C.c_double(0.0)
    n = L.ref_int4_llama_attention_timed(str(param_root).encode(), E, H, KVH, max_sqlen, hidden.ctypes.data, prefill, decode_steps, out.ctypes.data,
                                         fk.ctypes.data, fv.ctypes.data, C.addressof(secs))
    assert n == T
    return (out, fk, fv, secs.value) if timing else (out, fk, fv)


def oracle_llama_attention_module(hidden, sel, cosb, sinb, alpha, H, KVH, prefill, decode_steps):
    """Same flow from the oracle: selection projections (exact), orc_llama_attention_core, o_proj = selection of the
    int8-round-tripped core output.  sel: dict q,k,v,o -> channel index arrays.  Returns (out, K, V, core)."""
    E = hidden.shape[1]
    hd = E // H
    pk = pv = None
    past = row = 0
    outs, cores = [], []
    for call in range(1 + decode_steps):
        s = prefill if call == 0 else 1
        x = hidden[row:row + s]
        core, pk, pv = llama_attention_core(x[:, sel["q"]], x[:, sel["k"]], x[:, sel["v"]], pk, pv, causal_mask(s, past), cosb, sinb, alpha, H, KVH, hd)
        cores.append(core)
        outs.append(w4a8_activation_roundtrip(core)[:, sel["o"]])
        past += s
        row += s
    return np.concatenate(outs), pk, pv, np.concatenate(cores)
