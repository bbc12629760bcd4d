#!/usr/bin/env python
"""Generate tests/golden/* from the REFERENCE ITSELF.

Sources (all need a TinyChatEngine source tree, named by the environment variable TCE_REFERENCE_DIR):

1. the reference's Python quantizer ``llm/tools/quantize_methods.py`` imported as-is -> packed INT4 formats
   (``quant_*.npz``): pins oracle/quant.py and tinychatengine_b200/formats.py byte-for-byte;
2. the reference's C++ kernels compiled in place (``make -C oracle ref`` -> oracle/_ref/*.so, entered through
   oracle/ref_shim.cc) -> outputs of naive_mat_mul_int4 / int8_ref_matmul* / naive_mat_mul_int8 /
   naive_mat_mul_fp16_int4 / the AVX W4A8 fast path (``kernels_*.npz``): pins oracle/tce_oracle.c;
3. the same builds on the seeded cases of tests/test_oracle_golden.py (``*_cases.npz``, ``int4_config1.npz``, ``norms.npz``) and
   the layout of the reference's kernels/matmul.h (``matmul_h_layout.txt``);
4. on a GPU, the reference's CUDA GEMV (oracle/_ref/libtce_ref_cuda.so, built beforehand) on the cases of
   tests/test_gpu_w4a16.py::test_reference_cuda_kernel_on_this_gpu (``reference_cuda_gemv.npz``).

Inputs are stored next to outputs, or regenerated from a seed by the test and fingerprinted, so the fixtures are self-contained.  Usage:

    TCE_REFERENCE_DIR=<tree> python tests/golden/make_golden.py              # 1-3
    TCE_REFERENCE_DIR=<tree> python tests/golden/make_golden.py recorded     # 3 only
    python tests/golden/make_golden.py cuda OUT_DIR                          # 4, on a GPU: OUT_DIR/reference_cuda_gemv.npz
"""
import os
import sys
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
OUT = Path(__file__).resolve().parent
TESTS = ROOT / "tests"


def ref_tree() -> Path:
    """The reference tree: its Python quantizer and headers are read directly, and capi.build() forwards it to oracle/Makefile as REF so
    that oracle/_ref is built from the same tree."""
    tree = os.environ.get("TCE_REFERENCE_DIR")
    if not tree:
        raise SystemExit("make_golden.py: set TCE_REFERENCE_DIR to a TinyChatEngine source tree")
    return Path(tree)


def ref_python_quantizer(w: np.ndarray, method: str):
    sys.path.insert(0, str(ref_tree() / "llm" / "tools"))
    import quantize_methods as qm  # the reference module, unmodified

    oc, ic = w.shape
    with tempfile.NamedTemporaryFile(suffix=".bin", delete=False) as f:
        f.write(np.ascontiguousarray(w, np.float32).tobytes())
        path = f.name
    try:
        qs, d, m, zp = getattr(qm, method)(path, oc * ic, "fp32", ic, oc)
    finally:
        os.unlink(path)
    return np.asarray(qs), np.asarray(d), np.asarray(zp)


def main():
    from oracle import capi

    capi.build(ref=True)
    rng = np.random.default_rng(20260922)

    # ---------------- 1. quantizer formats ----------------
    for name, (oc, ic) in {"a": (16, 256), "b": (8, 1408), "c": (8, 2048)}.items():
        w = (rng.standard_normal((oc, ic)) * 0.02).astype(np.float32)
        w[0, :128] = 0.0  # an all-zero block exercises the d == 0 branch
        out = {"w": w}
        qs, d, zp = ref_python_quantizer(w, "quantize_row_q4_6")
        # files are written int32 / fp16 / int32 for CUDA (model_quantizer.py:38-46)
        out["q4_6_qs"] = qs.astype(np.int32).view(np.uint32)
        out["q4_6_d"] = d.astype(np.float16)
        out["q4_6_zp"] = zp.astype(np.int32).view(np.uint32)
        if ic % 64 == 0:
            qs, d, zp = ref_python_quantizer(w, "quantize_row_q4_3")
            out["q4_3_qs"] = qs.astype(np.uint8).reshape(oc, ic // 2)
            out["q4_3_d"] = d.astype(np.float32).reshape(oc, ic // 32)
        qs, d, zp = ref_python_quantizer(w, "quantize_row_q4_5")
        out["q4_5_qs"] = qs.astype(np.int32)
        out["q4_5_d"] = d.astype(np.float16)
        np.savez_compressed(OUT / f"quant_{name}.npz", **out)

    # ---------------- 2. compiled reference kernels ----------------
    from oracle import quant

    G = capi.ref("generic")
    out = {}
    # naive_mat_mul_int4, generic branch, block 128 and 32 (kernels/matmul_int4.cc:106-127)
    for tag, (M, IC, OC, blk) in {"g128": (2, 512, 24, 128), "g32": (3, 256, 16, 32)}.items():
        w = (rng.standard_normal((OC, IC)) * 0.02).astype(np.float32)
        B, s = quant.quantize_q4_0_sequential(w, blk)
        A = rng.standard_normal((M, IC)).astype(np.float32)
        out[f"int4_{tag}_A"], out[f"int4_{tag}_B"], out[f"int4_{tag}_s"] = A, B, s
        out[f"int4_{tag}_C"] = capi.ref_naive_mat_mul_int4(A, B, s, 8.0, blk)
    # int8 family (kernels/ref/matmul_ref_int8.cc), alpha/beta from the reference's own op tests
    # (llm/tests/non_cuda/test_ops.cc:179: alpha=0.00050354, beta=0.0213013)
    M, N, K = 5, 24, 96
    A = rng.integers(-127, 128, (M, K), dtype=np.int8)
    B = rng.integers(-127, 128, (N, K), dtype=np.int8)
    Bb = rng.integers(-127, 128, (M, N, K), dtype=np.int8)
    b8 = rng.integers(-127, 128, (N,), dtype=np.int8)
    bf = rng.standard_normal(N).astype(np.float32)
    alpha, beta = np.float32(0.00050354), np.float32(0.0213013)
    out.update(i8_A=A, i8_B=B, i8_Bb=Bb, i8_b8=b8, i8_bf=bf, i8_alpha=alpha, i8_beta=beta)
    for v in range(8):
        Bv = Bb if v in (3, 7) else B
        qmin = 0 if v == 1 else -128  # variant 1 doubles as the ReLU flavour (W8A8B8O8LinearReLU: q_min = 0)
        out[f"i8_C{v}"] = capi.ref_int8_matmul(v, A, Bv, b8, bf, float(alpha), float(beta), qmin, 127)
    # a large-alpha case that saturates / hits the clamp
    out["i8_Csat"] = capi.ref_int8_matmul(0, A, B, b8, bf, 0.05, 1.0, -128, 127)
    # naive_mat_mul_int8 (kernels/matmul_int8.cc:8-30), B is [K][N]
    Bkn = np.ascontiguousarray(B.T)
    Cn = np.zeros((M, N), np.int8)
    G.ref_naive_mat_mul_int8(A, Bkn, Cn, M, N, K, 3, -2, 0.02, 0.01, 0.35, -128, 127)
    out["i8_naive_C"] = Cn
    # host fp16 reference, AWQ-GEMM layout (kernels/cuda/matmul_int4.cu:8-48)
    M, IC, OC = 2, 256, 16
    w = (rng.standard_normal((OC, IC)) * 0.02).astype(np.float32)
    qs5, d5 = quant.quantize_q4_5(w, 128)
    A16 = rng.standard_normal((M, IC)).astype(np.float16)
    C16 = np.zeros((M, OC), np.uint16)
    G.ref_naive_mat_mul_fp16_int4(A16.view(np.uint16), qs5, d5.view(np.uint16), C16, M, IC, OC, 128)
    out.update(f16_A=A16, f16_qs=qs5, f16_d=d5, f16_C=C16)
    # mat_mul_transposed
    A = rng.standard_normal((3, 40)).astype(np.float32)
    Bt = rng.standard_normal((7, 40)).astype(np.float32)
    Ct = np.zeros((3, 7), np.float32)
    G.ref_mat_mul_transposed(A, Bt, Ct, 3, 7, 40)
    out.update(t_A=A, t_B=Bt, t_C=Ct)
    np.savez_compressed(OUT / "kernels_generic.npz", **out)

    # the reference's AVX fast path (W4A8, g32): the timed CPU baseline; stored so the oracle/bench plumbing
    # can be sanity-checked without the reference tree
    X = capi.ref("avx")
    M, IC, OC = 1, 512, 64
    w = (rng.standard_normal((OC, IC)) * 0.02).astype(np.float32)
    qs3, d3 = quant.quantize_q4_3(w)
    A = capi.aligned_empty((M, IC), np.float32)
    A[:] = rng.standard_normal((M, IC)).astype(np.float32)
    Bq = capi.aligned_empty(qs3.shape, np.uint8)
    Bq[:] = qs3
    S = capi.aligned_empty(d3.shape, np.float32)
    S[:] = d3
    Cx = capi.aligned_empty((M, OC), np.float32)
    xi8 = capi.aligned_empty((M * IC,), np.int8)
    xs = capi.aligned_empty((M * IC // 32,), np.float32)
    X.ref_w4a8_avx(A.ctypes.data, Bq.ctypes.data, S.ctypes.data, Cx.ctypes.data, xi8.ctypes.data, xs.ctypes.data, M, IC, OC, 2)
    np.savez_compressed(OUT / "kernels_avx.npz", A=np.array(A), w=w, qs=qs3, d=d3, C=np.array(Cx))
    # the reference MODULE Int8OPTAttention (compiled in place, oracle/ref_modules_shim.cc): prefill of 9 tokens + 3 decode steps
    E, H, prefill, steps = 256, 4, 9, 3
    par = dict(a_qkv=np.float32(0.0009), b_qkv=np.float32(0.9), qk_alpha=np.float32(0.0007), pv_alpha=np.float32(0.011), a_out=np.float32(0.0008))
    W = {k: rng.integers(-127, 128, (E, E), dtype=np.int8) for k in "qkvo"}
    Bq8 = {k: rng.integers(-127, 128, (E,), dtype=np.int8) for k in "qkv"}
    bo = rng.standard_normal(E).astype(np.float32)
    hidden = rng.integers(-127, 128, (prefill + steps, E), dtype=np.int8)
    with tempfile.TemporaryDirectory() as d:
        capi.write_opt_attention_params(d, W, Bq8, bo, **par)
        out, fk, fv = capi.ref_int8_opt_attention(d, hidden, E, H, prefill, steps)
    np.savez_compressed(OUT / "opt_attention_module.npz", hidden=hidden, wq=W["q"], wk=W["k"], wv=W["v"], wo=W["o"], bq=Bq8["q"], bk=Bq8["k"], bv=Bq8["v"],
                        bo=bo, out=out, final_k=fk, final_v=fv, H=H, prefill=prefill, steps=steps, **par)
    # the reference MODULE Int4llamaAttention (CPU build, GQA 4:2, head_dim 128): prefill of 7 tokens + 3 decode steps.  The four
    # linears are 0/1 channel selections and the activations are exactly int8-representable, so the module output isolates the
    # attention core (RoPE, KV concat, GQA repeat, mask, in-place softmax, PV) at fp32 round-off.
    E, H, KVH, prefill, steps, max_sq = 512, 4, 2, 7, 3, 64
    hd = E // H
    Wsel, sel = {}, {}
    for name, rows in (("q", E), ("k", KVH * hd), ("v", KVH * hd), ("o", E)):
        Wsel[name + "_proj"], sel[name] = capi.selection_matrix(rows, E, rng)
    cosb, sinb = capi.rope_tables(max_sq, hd, 10000.0)
    alpha = np.float32(1.0 / np.sqrt(hd))
    hidden = capi.exact_w4a8_activations((prefill + steps, E), rng)
    with tempfile.TemporaryDirectory() as d:
        capi.write_llama_attention_params(d, Wsel, cosb, sinb, alpha)
        out, fk, fv = capi.ref_int4_llama_attention(d, hidden, E, H, KVH, prefill, steps, max_sq)
    np.savez_compressed(OUT / "llama_attention_module.npz", hidden=hidden, sel_q=sel["q"], sel_k=sel["k"], sel_v=sel["v"], sel_o=sel["o"], out=out,
                        final_k=fk, final_v=fv, H=H, KVH=KVH, prefill=prefill, steps=steps, max_sq=max_sq, alpha=alpha, theta=np.float32(10000.0))
    # the reference's sampling chain (llm/src/Generate.cc via oracle/_ref/libtce_ref_generate.so): candidate sets + probabilities for a few
    # configurations over one logits vector with distinct values (the order among equal logits is unspecified in the reference)
    V = 4096
    logits = (rng.standard_normal(V) * 3.0).astype(np.float32)
    window = rng.integers(0, V, 64).astype(np.int32)
    window[5] = window[9] = int(np.argmax(logits))  # the favourite is penalised, twice in the window
    cases = [dict(top_k=40, top_p=0.95, temp=0.8, repeat_penalty=1.1, frequency_penalty=0.0, presence_penalty=0.0),
             dict(top_k=40, top_p=0.5, temp=1.3, repeat_penalty=1.3, frequency_penalty=0.2, presence_penalty=0.1),
             dict(top_k=200, top_p=1.0, temp=0.7, repeat_penalty=1.0, frequency_penalty=0.0, presence_penalty=0.0),
             dict(top_k=1, top_p=0.95, temp=0.8, repeat_penalty=1.1, frequency_penalty=0.0, presence_penalty=0.0),
             dict(top_k=40, top_p=0.95, temp=0.0, repeat_penalty=1.5, frequency_penalty=0.0, presence_penalty=0.0)]
    samp = {"logits": logits, "window": window, "n_cases": len(cases)}
    for i, c in enumerate(cases):
        ids, probs = capi.ref_sample_candidates(logits, window, **c)
        samp[f"ids{i}"], samp[f"probs{i}"] = ids, probs
        samp[f"cfg{i}"] = np.array([c["top_k"], c["top_p"], c["temp"], c["repeat_penalty"], c["frequency_penalty"], c["presence_penalty"]], dtype=np.float64)
    np.savez_compressed(OUT / "sampling.npz", **samp)
    make_llama_model()
    make_recorded_cases()
    print("golden fixtures written to", OUT)


def make_llama_model():
    """The reference's WHOLE CPU model -- Int4LlamaForCausalLM -> Int4llamaDecoder -> Int4llamaDecoderLayer -> Int4llamaAttention, compiled in place
    (oracle/_ref/libtce_ref_llama_model.so) -- on a synthetic two-layer GQA model: logits of a 6-token prompt pass and 3 decode steps.  Only the
    seed travels (the weights are regenerated from it; `weights_crc` guards the generator), so the fixture stays a few KB.  Pins the composition
    oracle/llama_ref.py::llama_forward, which tests/helpers.py::oracle_decode_step runs for the GPU parity tests."""
    import zlib

    from oracle import capi, llama_ref

    E, H, KVH, L, F, V, prefill, steps, max_sq, seed, theta, eps = 256, 4, 2, 2, 512, 320, 6, 3, 640, 20260926, 500000.0, 1e-5
    rng = np.random.default_rng(seed)
    model = llama_ref.random_model(rng, E, H, KVH, L, F, V)
    tokens = rng.integers(0, V, prefill + steps).astype(np.int32)
    hd = E // H
    cosb, sinb = capi.rope_tables(max_sq, hd, theta)
    with tempfile.TemporaryDirectory() as d:
        handles = llama_ref.write_llama_model_params(d, model, cosb, sinb, np.float32(1.0 / np.sqrt(hd)))
        logits = llama_ref.ref_int4_llama_causal_lm(d, tokens, E, H, KVH, L, F, V, prefill, steps, max_sq, eps)
    crc = zlib.crc32(handles["lm_head"][0].tobytes()) ^ zlib.crc32(handles["layers"][0]["down"][0].tobytes())
    np.savez_compressed(OUT / "llama_model.npz", dims=np.array([E, H, KVH, L, F, V, prefill, steps, max_sq, seed], np.int64), theta=np.float64(theta),
                        eps=np.float64(eps), tokens=tokens, logits=logits, weights_crc=np.uint32(crc))


def _record(store, key, crc, **outputs):
    store[f"{key}__crc"] = np.uint32(crc)
    for name, a in outputs.items():
        store[f"{key}__{name}"] = a


def make_recorded_cases():
    """The reference's outputs on the seeded cases of tests/test_oracle_golden.py (the test's own builders make the inputs) and the struct
    layout of its kernels/matmul.h as printed by tests/test_host_header_abi.py's probe."""
    import ctypes as C
    import hashlib

    from oracle import capi, llama_ref

    sys.path.insert(0, str(TESTS))
    import test_host_header_abi as ABI
    import test_oracle_golden as T

    capi.build(ref=True)
    ref = ref_tree()
    layout = ABI.probe(str(ref / "kernels" / "matmul.h"), ["-DQM_CUDA", "-I" + str(ref / "llm" / "half-2.2.0" / "include")])
    (OUT / "matmul_h_layout.txt").write_text(layout + "\n")

    rec = {}
    for M in T.CONFIG1_M:
        _, x, _, _, _, B, sc, crc = T.config1_case(M)
        want = capi.ref_naive_mat_mul_int4(x.astype(np.float32), B, sc, 8.0, 128)
        _record(rec, f"M{M}", crc, sha256=np.array(hashlib.sha256(want.tobytes()).hexdigest()), sample=want.ravel()[::T.CONFIG1_SAMPLE_STRIDE].copy())
    np.savez_compressed(OUT / "int4_config1.npz", **rec)

    rec = {}
    for case in T.OPT_CASES:
        E, H_, prefill, steps, _ = case
        W, B, bo, hidden, par, crc = T.opt_attention_case(*case)
        with tempfile.TemporaryDirectory() as d:
            capi.write_opt_attention_params(d, W, B, bo, *par)
            out, k, v = capi.ref_int8_opt_attention(d, hidden, E, H_, prefill, steps)
        _record(rec, T.case_key(*case), crc, out=out, k=k, v=v)
    np.savez_compressed(OUT / "opt_attention_cases.npz", **rec)

    rec = {}
    for case in T.LLAMA_ATTENTION_CASES:
        E, H_, KVH, prefill, steps, _ = case
        W, _, cosb, sinb, alpha, hidden, max_sq, crc = T.llama_attention_case(*case)
        with tempfile.TemporaryDirectory() as d:
            capi.write_llama_attention_params(d, W, cosb, sinb, alpha)
            out, k, v = capi.ref_int4_llama_attention(d, hidden, E, H_, KVH, prefill, steps, max_sq)
        _record(rec, T.case_key(*case), crc, out=out, k=k, v=v)
    np.savez_compressed(OUT / "llama_attention_cases.npz", **rec)

    rec = {}
    X = capi.ref("avx")
    for case in T.W4A8_CASES:
        M, IC, OC, _ = case
        A0, qs, d, crc = T.w4a8_case(*case)
        A, Bq, S = (capi.aligned_empty(a.shape, a.dtype) for a in (A0, qs, d))  # the AVX kernels need aligned buffers
        A[:], Bq[:], S[:] = A0, qs, d
        Cx = capi.aligned_empty((M, OC), np.float32)
        xi8 = capi.aligned_empty((M * IC,), np.int8)
        xs = capi.aligned_empty((M * IC // 32,), np.float32)
        X.ref_w4a8_avx(A.ctypes.data, Bq.ctypes.data, S.ctypes.data, Cx.ctypes.data, xi8.ctypes.data, xs.ctypes.data, M, IC, OC, 2)
        _record(rec, T.case_key(*case), crc, C=np.array(Cx))
    np.savez_compressed(OUT / "w4a8_avx_cases.npz", **rec)

    rec = {}
    for case in T.LLAMA_MODEL_CASES:
        E, H_, KVH, L, F, V, prefill, steps, _ = case
        model, tokens, cosb, sinb, crc = T.llama_model_case(*case)
        with tempfile.TemporaryDirectory() as d:
            llama_ref.write_llama_model_params(d, model, cosb, sinb, np.float32(1.0 / np.sqrt(E // H_)))
            logits = llama_ref.ref_int4_llama_causal_lm(d, tokens, E, H_, KVH, L, F, V, prefill, steps, 640, 1e-6)
        _record(rec, T.case_key(*case), crc, logits=logits)
    np.savez_compressed(OUT / "llama_model_cases.npz", **rec)

    rec = {}
    Lm = C.CDLL(str(capi.REF_DIR / "libtce_ref_modules.so"))
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    for rows, dim, x, w, b, crc in T.norm_cases():
        rms = np.zeros_like(x)
        Lm.ref_llama_rmsnorm(vp(x), vp(w), vp(rms), rows, dim, C.c_float(1e-5))
        x8 = (x * 20).astype(np.float32)
        ln8 = np.zeros((rows, dim), np.int8)
        Lm.ref_layernorm_q(vp(x8), vp(w), vp(b), vp(ln8), rows, dim)
        _record(rec, T.case_key(rows, dim), crc, rmsnorm=rms, layernorm_q=ln8)
    np.savez_compressed(OUT / "norms.npz", **rec)

    rec = {}
    for trial, logits, window, cfg, crc in T.sampling_trials():
        ids, probs = capi.ref_sample_candidates(logits, window, **cfg)
        _record(rec, f"trial{trial}", crc, ids=ids, probs=probs)
    np.savez_compressed(OUT / "sampling_cases.npz", **rec)


def make_reference_cuda_gemv(out_dir):
    """On a GPU: the reference's gemv_kernel_g128 (oracle/_ref/libtce_ref_cuda.so) on the cases of test_reference_cuda_kernel_on_this_gpu."""
    import torch

    from oracle import capi

    sys.path.insert(0, str(TESTS))
    import test_gpu_w4a16 as T

    rec = {}
    for oc, ic in T.REFERENCE_CUDA_SHAPES:
        x, w, z, s, crc = T.reference_cuda_case(oc, ic)
        yr = torch.empty((1, oc), dtype=torch.float16, device=x.device)
        torch.cuda.synchronize()
        assert capi.ref_cuda().ref_cuda_gemv(x.data_ptr(), w.data_ptr(), z.data_ptr(), s.data_ptr(), yr.data_ptr(), 1, ic, oc) == 0
        torch.cuda.synchronize()
        _record(rec, f"{oc}x{ic}", crc, y=yr.cpu().numpy())
    np.savez_compressed(Path(out_dir) / "reference_cuda_gemv.npz", **rec)


if __name__ == "__main__":
    if sys.argv[1:] == ["recorded"]:
        make_recorded_cases()
    elif sys.argv[1:2] == ["cuda"] and len(sys.argv) == 3:
        make_reference_cuda_gemv(sys.argv[2])
    elif len(sys.argv) == 1:
        main()
    else:
        raise SystemExit(__doc__)
