"""The oracle (oracle/tce_oracle.c, oracle/quant.py) against fixtures produced by the reference itself
(tests/golden/make_golden.py: reference Python quantizer + reference C++ kernels compiled in place).

The seeded cases below (the *_CASES lists and the *_case builders) regenerate their inputs from a seed; the reference's outputs for
them are stored under tests/golden/ by make_golden.py, which calls the same builders."""
import zlib

import numpy as np
import pytest

from oracle import capi, quant


def inputs_crc(*arrays) -> int:
    """Fingerprint of a seeded case's inputs, stored beside the recorded outputs."""
    c = 0
    for a in arrays:
        c = zlib.crc32(np.ascontiguousarray(a).tobytes(), c)
    return c


def case_key(*params) -> str:
    return "_".join(str(p) for p in params)


def recorded(golden_dir, name, key, crc) -> dict:
    """The reference outputs recorded for case `key` in tests/golden/<name>.npz, after checking that this host regenerated the same inputs."""
    g = np.load(golden_dir / f"{name}.npz")
    assert int(g[f"{key}__crc"]) == crc, f"inputs of case {key} differ from the recorded ones: regenerate tests/golden/{name}.npz (make_golden.py)"
    return {k.split("__", 1)[1]: g[k] for k in g.files if k.startswith(key + "__")}


@pytest.mark.parametrize("name", ["a", "b", "c"])
def test_quantizer_formats_match_reference_python(golden_dir, name):
    g = np.load(golden_dir / f"quant_{name}.npz")
    w = g["w"]
    qs, d, zp = quant.quantize_q4_6(w)
    assert np.array_equal(qs, g["q4_6_qs"])
    assert np.array_equal(d.view(np.uint16), g["q4_6_d"].view(np.uint16))
    assert np.array_equal(zp, g["q4_6_zp"])
    assert zp.shape[1] == quant.calculate_zeros_width(w.shape[1]) == capi.zeros_width(w.shape[1])
    if "q4_3_qs" in g:
        qs3, d3 = quant.quantize_q4_3(w)
        assert np.array_equal(qs3, g["q4_3_qs"])
        assert np.array_equal(d3, g["q4_3_d"])
    qs5, d5 = quant.quantize_q4_5(w)
    assert np.array_equal(qs5, g["q4_5_qs"])
    assert np.array_equal(d5.view(np.uint16), g["q4_5_d"].view(np.uint16))


def test_naive_mat_mul_int4_bit_exact(golden_dir):
    g = np.load(golden_dir / "kernels_generic.npz")
    for tag, blk in (("g128", 128), ("g32", 32)):
        C = capi.naive_mat_mul_int4(g[f"int4_{tag}_A"], g[f"int4_{tag}_B"], g[f"int4_{tag}_s"], 8.0, blk)
        assert np.array_equal(C.view(np.uint32), g[f"int4_{tag}_C"].view(np.uint32)), tag


CONFIG1_M = [1, 16]
CONFIG1_SAMPLE_STRIDE = 97


def config1_case(M):
    """BASELINE.json configs[0] at its full size: IC 4096 x OC 11008, group 128.  -> (rng, x, qs, d, zp, B, sc, crc)"""
    rng = np.random.default_rng(1234)
    IC, OC = 4096, 11008
    w = (rng.standard_normal((OC, IC)) * 0.02).astype(np.float32)
    qs, d, zp = quant.quantize_q4_6(w)
    x = rng.standard_normal((M, IC)).astype(np.float16)
    B = quant.qmcuda_to_sequential_bytes(qs)
    sc = d[:, : IC // 128].astype(np.float32)
    return rng, x, qs, d, zp, B, sc, inputs_crc(x, B, sc)


@pytest.mark.parametrize("M", CONFIG1_M)
def test_naive_mat_mul_int4_full_size_config1_live(golden_dir, M):
    """BASELINE.json configs[0] at its full size (IC 4096 x OC 11008, group 128, M in {1, 16}, SURVEY.md 8(d) config 1): the oracle
    restatement vs the reference's own naive_mat_mul_int4 (kernels/matmul_int4.cc:106-127) compiled in place -- bit for bit -- and
    the QM_CUDA-layout oracle the GPU tests compare with vs both.  The reference's output is recorded as its SHA-256 and a strided
    sample (tests/golden/int4_config1.npz): the full product does not fit a small fixture."""
    import hashlib

    rng, x, qs, d, zp, B, sc, crc = config1_case(M)
    rec = recorded(golden_dir, "int4_config1", f"M{M}", crc)
    got = capi.naive_mat_mul_int4(x.astype(np.float32), B, sc, 8.0, 128)
    assert np.array_equal(got.ravel()[::CONFIG1_SAMPLE_STRIDE].view(np.uint32), rec["sample"].view(np.uint32))
    assert hashlib.sha256(got.tobytes()).hexdigest() == str(rec["sha256"])
    y = capi.w4a16_gemv(x, qs, zp, d)
    assert np.array_equal(y.view(np.uint32), got.view(np.uint32))
    # second weight set of config 1: random per-group zero points (the zero path), against float64
    zp2 = rng.integers(0, 2**32, zp.shape, dtype=np.uint32)
    y2 = capi.w4a16_gemv(x, qs, zp2, d)
    ref = x.astype(np.float64) @ quant.dequant_qmcuda(qs, d, zp2).astype(np.float64).T
    assert np.max(np.abs(y2 - ref)) <= 1e-5 * np.max(np.abs(ref))


def test_w4a16_gemv_oracle_consistent_with_naive(golden_dir):
    """The QM_CUDA-layout oracle (per-group zeros, fp16 scales) equals naive_mat_mul_int4 when zeros == 8 and the
    scales/activations are exactly representable in fp16."""
    rng = np.random.default_rng(5)
    OC, IC, M = 24, 1408, 2  # 11 groups -> zeros_w 2, scales padded to 16 (the IC=11008 padding quirk in small)
    w = (rng.standard_normal((OC, IC)) * 0.02).astype(np.float32)
    qs, d, zp = quant.quantize_q4_6(w)
    x = rng.standard_normal((M, IC)).astype(np.float16)
    y = capi.w4a16_gemv(x, qs, zp, d)
    y2 = capi.naive_mat_mul_int4(x.astype(np.float32), quant.qmcuda_to_sequential_bytes(qs), d[:, : IC // 128].astype(np.float32), 8.0, 128)
    # same products; (q-z)*s vs s*(q-z) commute exactly, accumulation order identical
    assert np.array_equal(y.view(np.uint32), y2.view(np.uint32))
    # and a dynamic-zero case against a float64 evaluation
    zp2 = rng.integers(0, 2**32, zp.shape, dtype=np.uint32)
    y3 = capi.w4a16_gemv(x, qs, zp2, d)
    ref = x.astype(np.float64) @ quant.dequant_qmcuda(qs, d, zp2).astype(np.float64).T
    assert np.max(np.abs(y3 - ref)) <= 1e-4 * max(1.0, np.max(np.abs(ref)))


def test_int8_family_bit_exact(golden_dir):
    g = np.load(golden_dir / "kernels_generic.npz")
    A, B, Bb, b8, bf = g["i8_A"], g["i8_B"], g["i8_Bb"], g["i8_b8"], g["i8_bf"]
    alpha, beta = float(g["i8_alpha"]), float(g["i8_beta"])
    for v in range(8):
        Bv = Bb if v in (3, 7) else B
        qmin = 0 if v == 1 else -128
        C = capi.int8_matmul(v, A, Bv, b8, bf, alpha, beta, qmin, 127)
        want = g[f"i8_C{v}"]
        if C.dtype == np.int8:
            assert np.array_equal(C, want), v
        else:
            assert np.array_equal(C.view(np.uint32), want.view(np.uint32)), v
    assert np.array_equal(capi.int8_matmul(0, A, B, b8, bf, 0.05, 1.0, -128, 127), g["i8_Csat"])
    assert np.abs(g["i8_Csat"].astype(np.int32)).max() == 128 or g["i8_Csat"].max() == 127


def test_naive_mat_mul_int8(golden_dir):
    g = np.load(golden_dir / "kernels_generic.npz")
    A, B = g["i8_A"], g["i8_B"]
    M, K = A.shape
    N = B.shape[0]
    C = np.zeros((M, N), np.int8)
    capi.lib().orc_naive_mat_mul_int8(A, np.ascontiguousarray(B.T), C, M, N, K, 3, -2, 0.02, 0.01, 0.35, -128, 127)
    assert np.array_equal(C, g["i8_naive_C"])


def test_fp16_int4_host_reference(golden_dir):
    g = np.load(golden_dir / "kernels_generic.npz")
    A, qs, d = g["f16_A"], g["f16_qs"], g["f16_d"]
    M, IC = A.shape
    OC = d.shape[1]
    C = np.zeros((M, OC), np.uint16)
    capi.lib().orc_naive_mat_mul_fp16_int4(A.view(np.uint16), qs, d.view(np.uint16), C, M, IC, OC, 128)
    assert np.array_equal(C, g["f16_C"])


def test_mat_mul_transposed(golden_dir):
    g = np.load(golden_dir / "kernels_generic.npz")
    C = np.zeros_like(g["t_C"])
    capi.lib().orc_mat_mul_transposed(g["t_A"], g["t_B"], C, 3, 7, 40)
    assert np.array_equal(C, g["t_C"])


def test_half_conversions_match_numpy():
    L = capi.lib()
    L.orc_half_to_float.restype = __import__("ctypes").c_float
    L.orc_float_to_half.restype = __import__("ctypes").c_uint16
    L.orc_float_to_half.argtypes = [__import__("ctypes").c_float]
    allh = np.arange(65536, dtype=np.uint16)
    f = allh.view(np.float16).astype(np.float32)
    for h in list(range(0, 65536, 97)) + [0x0001, 0x03ff, 0x0400, 0x7bff, 0x7c00, 0xfc00, 0x8000]:
        got = L.orc_half_to_float(int(h))
        if np.isnan(f[h]):
            assert np.isnan(got)
        else:
            assert got == f[h]
    rng = np.random.default_rng(0)
    xs = np.concatenate([rng.standard_normal(2000) * 10 ** rng.uniform(-9, 5, 2000), [65504, 65519.9, 65520, 1e-8, 2.0**-25, 2.0**-24, 0.0, -0.0]]).astype(np.float32)
    for x in xs:
        with np.errstate(over="ignore"):
            want = np.float32(x).astype(np.float16).view(np.uint16)
        assert L.orc_float_to_half(float(x)) == int(want), x


def _opt_fixture(golden_dir):
    g = np.load(golden_dir / "opt_attention_module.npz")
    W = {"q": g["wq"], "k": g["wk"], "v": g["wv"], "o": g["wo"]}
    B = {"q": g["bq"], "k": g["bk"], "v": g["bv"]}
    par = {k: float(g[k]) for k in ("a_qkv", "b_qkv", "qk_alpha", "pv_alpha", "a_out")}
    return g, W, B, par


def test_opt_attention_module_golden(golden_dir):
    """Oracle composition of Int8OPTAttention::forward == the compiled reference MODULE's recorded outputs (prefill 9 + 3 decode
    steps), bit for bit.  This fixture is what pinned the in-place softmax seed (softmax.cc:13 read after row 0 was overwritten)."""
    g, W, B, par = _opt_fixture(golden_dir)
    out, fk, fv = capi.oracle_int8_opt_attention(g["hidden"], W, B, g["bo"], par["a_qkv"], par["b_qkv"], par["qk_alpha"], par["pv_alpha"], par["a_out"],
                                                 int(g["H"]), int(g["prefill"]), int(g["steps"]))
    assert np.array_equal(fk, g["final_k"]) and np.array_equal(fv, g["final_v"])
    assert np.array_equal(out.view(np.uint32), g["out"].view(np.uint32))


OPT_CASES = [(128, 2, 5, 2, 1), (384, 6, 17, 4, 2), (256, 4, 1, 6, 3)]


def opt_attention_case(E, H, prefill, steps, seed):
    """-> (W, B, bo, hidden, par, crc)"""
    rng = np.random.default_rng(seed)
    W = {k: rng.integers(-127, 128, (E, E), dtype=np.int8) for k in "qkvo"}
    B = {k: rng.integers(-127, 128, (E,), dtype=np.int8) for k in "qkv"}
    bo = rng.standard_normal(E).astype(np.float32)
    hidden = rng.integers(-127, 128, (prefill + steps, E), dtype=np.int8)
    par = (np.float32(0.0011), np.float32(0.7), np.float32(0.0009), np.float32(0.013), np.float32(0.0006))
    return W, B, bo, hidden, par, inputs_crc(hidden, *W.values(), *B.values(), bo)


@pytest.mark.parametrize("E,H,prefill,steps,seed", OPT_CASES)
def test_opt_attention_module_live(golden_dir, E, H, prefill, steps, seed):
    """Same comparison on fresh random parameters per case, against the reference module's outputs recorded for them
    (tests/golden/opt_attention_cases.npz)."""
    W, B, bo, hidden, par, crc = opt_attention_case(E, H, prefill, steps, seed)
    rec = recorded(golden_dir, "opt_attention_cases", case_key(E, H, prefill, steps, seed), crc)
    got, gk, gv = capi.oracle_int8_opt_attention(hidden, W, B, bo, *par, H, prefill, steps)
    assert np.array_equal(gk, rec["k"]) and np.array_equal(gv, rec["v"])
    assert np.array_equal(got.view(np.uint32), rec["out"].view(np.uint32))


def test_llama_attention_module_golden(golden_dir):
    """orc_llama_attention_core == the compiled reference Int4llamaAttention MODULE (CPU build, GQA 4:2, head_dim 128, prefill 7 +
    3 decode steps) at fp32 round-off: K cache <= 1e-6, outputs <= 1e-5 of the maximum (the reference build uses -Ofast)."""
    g = np.load(golden_dir / "llama_attention_module.npz")
    H, KVH, max_sq = int(g["H"]), int(g["KVH"]), int(g["max_sq"])
    hd = g["hidden"].shape[1] // H
    cosb, sinb = capi.rope_tables(max_sq, hd, float(g["theta"]))
    sel = {k: g["sel_" + k] for k in "qkvo"}
    out, fk, fv, _ = capi.oracle_llama_attention_module(g["hidden"], sel, cosb, sinb, float(g["alpha"]), H, KVH, int(g["prefill"]), int(g["steps"]))
    assert np.abs(fk - g["final_k"]).max() <= 1e-6 * np.abs(g["final_k"]).max()
    assert np.array_equal(fv, g["final_v"])
    assert np.abs(out - g["out"]).max() <= 1e-5 * np.abs(g["out"]).max()


LLAMA_ATTENTION_CASES = [(256, 4, 4, 5, 2, 1), (256, 8, 2, 12, 3, 2), (512, 4, 1, 1, 5, 3)]


def llama_attention_case(E, H, KVH, prefill, steps, seed):
    """-> (W, sel, cosb, sinb, alpha, hidden, max_sq, crc)"""
    rng = np.random.default_rng(seed)
    hd, max_sq = E // H, 64
    W, sel = {}, {}
    for name, rows in (("q", E), ("k", KVH * hd), ("v", KVH * hd), ("o", E)):
        W[name + "_proj"], sel[name] = capi.selection_matrix(rows, E, rng)
    cosb, sinb = capi.rope_tables(max_sq, hd, 500000.0)
    alpha = np.float32(1.0 / np.sqrt(hd))
    hidden = capi.exact_w4a8_activations((prefill + steps, E), rng)
    return W, sel, cosb, sinb, alpha, hidden, max_sq, inputs_crc(hidden, *sel.values(), cosb, sinb)


@pytest.mark.parametrize("E,H,KVH,prefill,steps,seed", LLAMA_ATTENTION_CASES)
def test_llama_attention_module_live(golden_dir, E, H, KVH, prefill, steps, seed):
    """orc_llama_attention_core on fresh selection projections per case vs the reference module's outputs recorded for them
    (tests/golden/llama_attention_cases.npz)."""
    W, sel, cosb, sinb, alpha, hidden, max_sq, crc = llama_attention_case(E, H, KVH, prefill, steps, seed)
    rec = recorded(golden_dir, "llama_attention_cases", case_key(E, H, KVH, prefill, steps, seed), crc)
    want, wk, wv = rec["out"], rec["k"], rec["v"]
    got, gk, gv, _ = capi.oracle_llama_attention_module(hidden, sel, cosb, sinb, alpha, H, KVH, prefill, steps)
    assert np.abs(gk - wk).max() <= 1e-6 * np.abs(wk).max() and np.array_equal(gv, wv)
    # a score within round-off of an int8 rounding boundary may flip one quantisation step of the o_proj input: allow isolated steps
    diff = np.abs(got - want)
    assert (diff > 1e-5 * np.abs(want).max()).mean() <= 2e-3
    assert diff.max() <= np.abs(want).max() / 100


def test_w4a8_linear_restatement_matches_avx_fixture(golden_dir):
    """oracle/llama_ref.py::w4a8_linear (the projection arithmetic of the reference's CPU build: int8 activations per 32-block x int4 weights,
    kernels/avx/matmul_avx_int8_int4.cc) against the output of the compiled AVX kernel stored in kernels_avx.npz."""
    from oracle import llama_ref

    g = np.load(golden_dir / "kernels_avx.npz")
    got = llama_ref.w4a8_linear(g["A"], (llama_ref.unpack_q4_3(g["qs"]), g["d"].astype(np.float32)))
    assert got.shape == g["C"].shape
    assert np.abs(got - g["C"]).max() <= 2e-6 * np.abs(g["C"]).max()


W4A8_CASES = [(1, 4096, 256, 1), (3, 1024, 64, 2), (8, 512, 128, 3)]


def w4a8_case(M, IC, OC, seed):
    """-> (A, qs, d, crc)"""
    rng = np.random.default_rng(seed)
    w = (rng.standard_normal((OC, IC)) * 0.02).astype(np.float32)
    qs, d = quant.quantize_q4_3(w)
    A = rng.standard_normal((M, IC)).astype(np.float32)
    return A, qs, d, inputs_crc(A, qs, d)


@pytest.mark.parametrize("M,IC,OC,seed", W4A8_CASES)
def test_w4a8_linear_restatement_matches_avx_live(golden_dir, M, IC, OC, seed):
    """Same on fresh weights per case, against the compiled AVX kernel's outputs recorded for them (tests/golden/w4a8_avx_cases.npz)."""
    from oracle import llama_ref

    A, qs, d, crc = w4a8_case(M, IC, OC, seed)
    Cx = recorded(golden_dir, "w4a8_avx_cases", case_key(M, IC, OC, seed), crc)["C"]
    got = llama_ref.w4a8_linear(A, (llama_ref.unpack_q4_3(qs), d.astype(np.float32)))
    assert np.abs(got - Cx).max() <= 2e-6 * np.abs(Cx).max()


def test_llama_model_composition_golden(golden_dir):
    """oracle/llama_ref.py::llama_forward -- the composition of a Llama step that tests/helpers.py::oracle_decode_step runs for the GPU parity tests
    -- fed with the reference CPU build's arithmetic (fp32, W4A8 projections) reproduces the logits of the reference's WHOLE model
    (Int4LlamaForCausalLM::forward compiled in place: prompt pass of 6 tokens + 3 decode steps, 2 layers, GQA 4:2) to fp32 round-off."""
    import zlib

    from oracle import llama_ref

    g = np.load(golden_dir / "llama_model.npz")
    E, H, KVH, L, F, V, prefill, steps, max_sq, seed = (int(v) for v in g["dims"])
    rng = np.random.default_rng(seed)
    model = llama_ref.random_model(rng, E, H, KVH, L, F, V)
    tokens = rng.integers(0, V, prefill + steps).astype(np.int32)
    assert np.array_equal(tokens, g["tokens"]), "numpy's generator stream changed: regenerate tests/golden/llama_model.npz"
    handles = llama_ref.quantized_handles(model)
    crc = zlib.crc32(handles["lm_head"][0].tobytes()) ^ zlib.crc32(handles["layers"][0]["down"][0].tobytes())
    assert crc == int(g["weights_crc"]), "synthetic weights differ from the fixture's: regenerate tests/golden/llama_model.npz"
    cosb, sinb = capi.rope_tables(max_sq, E // H, float(g["theta"]))
    got = llama_ref.oracle_int4_llama_causal_lm(model, handles, tokens, cosb, sinb, H, KVH, prefill, steps, float(g["eps"]))
    want = g["logits"]
    assert got.shape == want.shape == (prefill + steps, V)
    _check_model_logits(got, want)


def _check_model_logits(got, want):
    """fp32 round-off (measured 2-6e-7 of the maximum) -- unless an activation that sits within round-off of an int8 rounding boundary of the W4A8
    activation quantiser (kernels/avx/matmul_avx_int8_int4.cc:259-316, the one discontinuity of the CPU path) rounds the other way on this host:
    seen on 5 of 40 seeds, echo <= 8e-3 of the maximum.  A wrong composition (order of norm / residual / activation) is an O(1) error."""
    import warnings

    rel = float(np.abs(got - want).max() / np.abs(want).max())
    assert rel <= 3e-2, rel
    if rel > 5e-6:
        warnings.warn(f"int8 activation-rounding flip against the reference build: logits differ by {rel:.1e} of the maximum instead of ~3e-7")


LLAMA_MODEL_CASES = [(256, 2, 2, 1, 256, 128, 1, 4, 2), (512, 4, 1, 2, 1024, 256, 9, 2, 3), (256, 4, 4, 3, 512, 192, 4, 1, 4)]


def llama_model_case(E, H, KVH, L, F, V, prefill, steps, seed):
    """-> (model, tokens, cosb, sinb, crc); the reference runs it with max_sqlen 640 and eps 1e-6"""
    from oracle import llama_ref

    rng = np.random.default_rng(seed)
    model = llama_ref.random_model(rng, E, H, KVH, L, F, V)
    tokens = rng.integers(0, V, prefill + steps).astype(np.int32)
    cosb, sinb = capi.rope_tables(640, E // H, 10000.0)
    weights = [model["embed"], model["final_norm"], model["lm_head"]] + [lt[k] for lt in model["layers"] for k in sorted(lt)]
    return model, tokens, cosb, sinb, inputs_crc(tokens, cosb, sinb, *weights)


@pytest.mark.parametrize("E,H,KVH,L,F,V,prefill,steps,seed", LLAMA_MODEL_CASES)
def test_llama_model_composition_live(golden_dir, E, H, KVH, L, F, V, prefill, steps, seed):
    """Same pin on fresh models per case (MHA, GQA and MQA, one to three layers, prompt-only / decode-only heavy call patterns), against the
    reference build's logits recorded for them (tests/golden/llama_model_cases.npz)."""
    from oracle import llama_ref

    model, tokens, cosb, sinb, crc = llama_model_case(E, H, KVH, L, F, V, prefill, steps, seed)
    want = recorded(golden_dir, "llama_model_cases", case_key(E, H, KVH, L, F, V, prefill, steps, seed), crc)["logits"]
    got = llama_ref.oracle_int4_llama_causal_lm(model, llama_ref.quantized_handles(model), tokens, cosb, sinb, H, KVH, prefill, steps, 1e-6)
    _check_model_logits(got, want)


def test_oracle_decode_step_is_the_pinned_composition():
    """tests/helpers.py::oracle_decode_step (the checker of the GPU decode step) goes through llama_forward -- no second statement of the layer
    order exists in the test tree."""
    import inspect

    import helpers

    src = inspect.getsource(helpers.oracle_decode_step)
    assert "llama_ref.llama_forward(" in src and "rmsnorm" not in src and "llama_attention_core" not in src


def norm_cases():
    """-> (rows, dim, x, w, b, crc) per case; LayerNormQ takes x * 20"""
    rng = np.random.default_rng(8)
    for rows, dim in ((1, 4096), (5, 768), (3, 130)):
        x = (rng.standard_normal((rows, dim)) * 3).astype(np.float32)
        w = (1 + 0.1 * rng.standard_normal(dim)).astype(np.float32)
        b = rng.standard_normal(dim).astype(np.float32)
        yield rows, dim, x, w, b, inputs_crc(x, w, b)


def test_norms_match_the_compiled_reference_ops(golden_dir):
    """orc_rmsnorm / orc_layernorm_q vs the reference's LlamaRMSNorm::forward / LayerNormQ::forward (compiled in place, strict IEEE
    flags; outputs recorded in tests/golden/norms.npz): RMSNorm bit-for-bit (it is the fused prologue of the decode GEMVs), LayerNormQ
    int8 outputs bit-for-bit."""
    for rows, dim, x, w, b, crc in norm_cases():
        rec = recorded(golden_dir, "norms", case_key(rows, dim), crc)
        got = capi.rmsnorm(x, w, 1e-5)
        assert np.array_equal(got.view(np.uint32), rec["rmsnorm"].view(np.uint32))
        x8 = (x * 20).astype(np.float32)
        got8 = np.zeros((rows, dim), np.int8)
        capi.lib().orc_layernorm_q(x8, w, b, got8, rows, dim)
        assert np.array_equal(got8, rec["layernorm_q"])


# ---- token sampling (SURVEY.md 8(f)3): oracle/sampling.py against the reference's Generate.cc -------------------------------------
def _sampling_cases(golden_dir):
    g = np.load(golden_dir / "sampling.npz")
    for i in range(int(g["n_cases"])):
        c = g[f"cfg{i}"]
        cfg = dict(top_k=int(c[0]), top_p=float(c[1]), temp=float(c[2]), repeat_penalty=float(c[3]), frequency_penalty=float(c[4]), presence_penalty=float(c[5]))
        yield g["logits"], g["window"], cfg, g[f"ids{i}"], g[f"probs{i}"]


def test_sampling_oracle_matches_reference_fixture(golden_dir):
    """tests/golden/sampling.npz was produced by the reference's own sample_* functions (make_golden.py)."""
    from oracle import sampling

    for logits, window, cfg, ids, probs in _sampling_cases(golden_dir):
        oi, op = sampling.candidates(logits, window, **cfg)
        assert np.array_equal(oi, ids), cfg
        np.testing.assert_allclose(op, probs, rtol=0, atol=1e-6)


def sampling_trials():
    """-> (trial, logits, window, cfg, crc) for six seeded draws of vocabulary size, window and configuration"""
    rng = np.random.default_rng(7)
    for trial in range(6):
        V = int(rng.integers(50, 3000))
        logits = (rng.standard_normal(V) * rng.uniform(0.5, 6)).astype(np.float32)
        window = rng.integers(0, V, int(rng.integers(0, 100))).astype(np.int32)
        cfg = dict(top_k=int(rng.integers(1, 80)), top_p=float(rng.uniform(0.3, 1.0)), temp=float(rng.uniform(0.2, 1.5)),
                   repeat_penalty=float(rng.uniform(1.0, 1.5)), frequency_penalty=float(rng.uniform(0, 0.3)), presence_penalty=float(rng.uniform(0, 0.3)))
        yield trial, logits, window, cfg, inputs_crc(logits, window, np.array(list(cfg.values()), np.float64))


def test_sampling_oracle_matches_reference_live(golden_dir):
    """Same, on fresh inputs per trial, against the candidates the compiled reference returned for them (tests/golden/sampling_cases.npz)."""
    from oracle import sampling

    for trial, logits, window, cfg, crc in sampling_trials():
        rec = recorded(golden_dir, "sampling_cases", f"trial{trial}", crc)
        oi, op = sampling.candidates(logits, window, **cfg)
        assert np.array_equal(oi, rec["ids"]), (trial, cfg)
        np.testing.assert_allclose(op, rec["probs"], rtol=0, atol=1e-6)
    # the draw: inverse CDF over the candidate probabilities
    ids, probs = sampling.candidates(logits, window, **cfg)
    assert sampling.draw(ids, probs, 0.0) == int(ids[0]) and sampling.draw(ids, probs, 0.999999) == int(ids[-1])
    assert 0.0 <= sampling.uniform01(1234, 5) < 1.0
