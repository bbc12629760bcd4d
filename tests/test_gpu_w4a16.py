"""W4A16 GEMV parity on the GPU: tce_w4a16_gemv (C ABI) vs the CPU oracle on the same packed bytes."""
import numpy as np
import pytest
import torch

from helpers import assert_w4_close, rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    from tinychatengine_b200.runtime import Context

    c = Context(0)
    yield c
    c.close()


def make_case(oc, ic, m, seed, random_zeros):
    from tinychatengine_b200.runtime import random_w4

    dev = torch.device("cuda", 0)
    w, z, s = random_w4(oc, ic, dev, seed, random_zeros=random_zeros)
    g = torch.Generator(device=dev)
    g.manual_seed(seed + 7)
    x = torch.randn((m, ic), device=dev, generator=g).to(torch.float16)
    return x, w, z, s


def oracle(x, w, z, s):
    from oracle import capi

    return capi.w4a16_gemv(x.cpu().numpy(), w.cpu().numpy().view(np.uint32), z.cpu().numpy().view(np.uint32), s.cpu().numpy())


# (OC, IC): config 1 of BASELINE.json (4096x11008 matmul, both orientations: IC=11008 has the padded 88-scale /
# 11-zero-word rows), Llama-3 down_proj depth, tiny and ragged row counts
SHAPES = [(11008, 4096), (4096, 11008), (1024, 14336), (16, 14336), (48, 128), (40, 256), (4, 1024)]


@pytest.mark.parametrize("impl", [1, 0])
@pytest.mark.parametrize("oc,ic", SHAPES)
def test_gemv_m1_matches_oracle(ctx, impl, oc, ic):
    ctx.set_option("gemv_impl", impl)
    for rz in (False, True):
        x, w, z, s = make_case(oc, ic, 1, 11 + oc + ic, rz)
        y = ctx.w4a16_gemv(x, w, z, s)
        torch.cuda.synchronize()
        assert_w4_close(y.float().cpu().numpy(), oracle(x, w, z, s), f"impl={impl} {oc}x{ic} rz={rz}")
    ctx.set_option("gemv_impl", 1)


@pytest.mark.parametrize("m", [2, 5, 8, 9, 17])
def test_gemv_small_batch(ctx, m):
    for oc, ic in ((256, 4096), (1024, 1152), (64, 11008)):
        x, w, z, s = make_case(oc, ic, m, 100 + m, True)
        y = ctx.w4a16_gemv(x, w, z, s)
        torch.cuda.synchronize()
        assert_w4_close(y.float().cpu().numpy(), oracle(x, w, z, s), f"M={m} {oc}x{ic}")


def _per_element_err(y, ref):
    """SURVEY.md 8(d) config 1, second criterion: relative error per element wherever |ref| > 1e-3 * max|ref|."""
    y, ref = np.asarray(y, np.float64), np.asarray(ref, np.float64)
    m = np.abs(ref) > 1e-3 * np.abs(ref).max()
    return float(np.max(np.abs(y - ref)[m] / np.abs(ref)[m]))


@pytest.mark.parametrize("m", [1, 3])
@pytest.mark.parametrize("factor", [100.0, 1000.0])
@pytest.mark.parametrize("kill", [False, True])
def test_gemv_massive_activation_channels(ctx, m, factor, kill):
    """AWQ exists because of massive-activation channels: one x`factor` outlier per 128-group.  The reference converts fp16
    activations to fp32 exactly (gemv_cuda.cu:181-184); this kernel re-quantises each group to block fixed point, so the outlier
    must not swamp the other 127 elements.  `kill`: the outlier channel's weights equal the zero point (it contributes nothing, the
    result is made of the small elements only) -- the worst case for a block format.  Checked on the max-norm AND per element."""
    oc, ic = 512, 4096
    x, w, z, s = make_case(oc, ic, m, 4242, True)
    gen = torch.Generator(device="cpu")
    gen.manual_seed(7)
    x = (x.float() * 0.05)
    ch = torch.randint(0, 128, (ic // 128,), generator=gen) + torch.arange(ic // 128) * 128  # one outlier channel per group
    x[:, ch] *= factor
    x = x.to(torch.float16)
    assert torch.isfinite(x).all()
    if kill:
        # nibble of channel c := zero point of its group, for every output row
        wn = w.cpu().numpy().view(np.uint32).copy()
        zn = z.cpu().numpy().view(np.uint32)
        for g_, c in enumerate(ch.tolist()):
            zg = (zn[:, g_ // 8] >> (4 * (g_ % 8))) & 0xF
            word, sh = c // 8, 4 * (c % 8)
            wn[:, word] = (wn[:, word] & ~np.uint32(0xF << sh)) | (zg.astype(np.uint32) << sh)
        w = torch.from_numpy(wn.view(np.int32)).to(x.device)
    y = ctx.w4a16_gemv(x, w, z, s)
    torch.cuda.synchronize()
    ref = oracle(x, w, z, s)
    got = y.float().cpu().numpy()
    assert_w4_close(got, ref, f"outliers x{factor} kill={kill}")
    e = _per_element_err(got, ref)
    assert e <= 1e-2, f"per-element rel err {e:.3e} (outliers x{factor}, kill={kill}, M={m})"


def test_gemv_tiny_and_mixed_magnitudes(ctx):
    """groups whose elements span the whole fp16 range, all-zero groups, and a denormal-only group"""
    oc, ic = 64, 1024
    x, w, z, s = make_case(oc, ic, 1, 99, True)
    xf = x.float()
    xf[:, 0:128] = 0.0
    xf[:, 128:256] *= 6e-6          # fp16 subnormals
    xf[:, 256:384] *= torch.logspace(-3, 3, 128, device=x.device)
    x = xf.to(torch.float16)
    y = ctx.w4a16_gemv(x, w, z, s)
    torch.cuda.synchronize()
    ref = oracle(x, w, z, s)
    assert_w4_close(y.float().cpu().numpy(), ref, "mixed magnitudes")
    assert _per_element_err(y.float().cpu().numpy(), ref) <= 1e-2


REFERENCE_CUDA_SHAPES = [(4096, 4096), (1024, 14336), (11008, 4096)]


def reference_cuda_case(oc, ic):
    """-> (x, w, z, s, crc of their bytes)"""
    import zlib

    x, w, z, s = make_case(oc, ic, 1, 5 + oc, True)
    crc = 0
    for t in (x, w, z, s):
        crc = zlib.crc32(t.cpu().numpy().tobytes(), crc)
    return x, w, z, s, crc


@pytest.mark.parametrize("oc,ic", REFERENCE_CUDA_SHAPES)
def test_reference_cuda_kernel_on_this_gpu(ctx, golden_dir, oc, ic):
    """The reference's own gemv_kernel_g128 (kernels/cuda/gemv_cuda.cu:140-194), compiled unchanged for sm_100a, run on a B200 on these
    inputs: a second, independent oracle.  Its arithmetic is fp32 FMA of exactly converted fp16 inputs; its outputs are recorded in
    tests/golden/reference_cuda_gemv.npz (make_golden.py cuda)."""
    x, w, z, s, crc = reference_cuda_case(oc, ic)
    g = np.load(golden_dir / "reference_cuda_gemv.npz")
    assert int(g[f"{oc}x{ic}__crc"]) == crc, "inputs differ from the recorded ones: regenerate tests/golden/reference_cuda_gemv.npz"
    yr = g[f"{oc}x{ic}__y"].astype(np.float32)
    y = ctx.w4a16_gemv(x, w, z, s)
    torch.cuda.synchronize()
    want = oracle(x, w, z, s)
    assert_w4_close(yr, want, "reference CUDA kernel vs oracle")
    assert_w4_close(y.float().cpu().numpy(), yr, "this kernel vs reference CUDA kernel")


@pytest.mark.parametrize("oc,ic,m", [(64, 1024, 1), (48, 4096, 2), (256, 192, 1)])
def test_group_64_path(ctx, oc, ic, m):
    """gemv_kernel_g64 (kernels/cuda/gemv_cuda.cu:68-123): one scale / zero per 64 channels, zeros_width(IC, 64) padded rows."""
    from oracle import capi
    from tinychatengine_b200.runtime import random_w4

    dev = torch.device("cuda", 0)
    w, z, s = random_w4(oc, ic, dev, 9 + oc, random_zeros=True, group=64)
    x = torch.randn((m, ic), device=dev).to(torch.float16)
    y = ctx.w4a16_gemv(x, w, z, s, group=64)
    torch.cuda.synchronize()
    ref = capi.w4a16_gemv(x.cpu().numpy(), w.cpu().numpy().view(np.uint32), z.cpu().numpy().view(np.uint32), s.cpu().numpy(), group=64)
    assert_w4_close(y.float().cpu().numpy(), ref, f"g64 {oc}x{ic}")


def test_gemm_entry_point_same_contract(ctx):
    x, w, z, s = make_case(128, 1024, 24, 5, False)
    y = ctx.w4a16_gemv(x, w, z, s, gemm=True)
    torch.cuda.synchronize()
    assert_w4_close(y.float().cpu().numpy(), oracle(x, w, z, s), "gemm slot")


def test_repeated_calls_are_deterministic_and_counters_rearm(ctx):
    """stream-K fix-up leaves its arrival counters at zero: many back-to-back launches give identical bits."""
    x, w, z, s = make_case(16 * 37, 2048, 1, 77, True)
    ref = None
    for _ in range(20):
        y = ctx.w4a16_gemv(x, w, z, s).clone()
        if ref is None:
            ref = y
        assert torch.equal(ref, y)
    for cw, cps in ((16, 1), (8, 1), (8, 2), (8, 3)):
        ctx.set_option("gemv_consumer_warps", cw)
        ctx.set_option("gemv_ctas_per_sm", cps)
        y = ctx.w4a16_gemv(x, w, z, s)
        assert rel_err(y.float().cpu().numpy(), ref.float().cpu().numpy()) < 1e-3
    ctx.set_option("gemv_consumer_warps", 16)
    ctx.set_option("gemv_ctas_per_sm", 1)


def test_full_size_properties_llama3_lm_head(ctx):
    """BASELINE.json full size (128256 x 4096 lm_head): too slow for the scalar oracle in full, so (a) a random
    row sample against the oracle, (b) the independent simple kernel on all rows, (c) linearity in x."""
    oc, ic = 128256, 4096
    x, w, z, s = make_case(oc, ic, 1, 2024, False)
    y = ctx.w4a16_gemv(x, w, z, s)
    rows = torch.randint(0, oc, (64,), device=x.device)
    ys = oracle(x, w[rows], z[rows], s[rows])
    assert_w4_close(y[:, rows].float().cpu().numpy(), ys, "lm_head sample")
    ctx.set_option("gemv_impl", 0)
    y0 = ctx.w4a16_gemv(x, w, z, s)
    ctx.set_option("gemv_impl", 1)
    assert rel_err(y.float().cpu().numpy(), y0.float().cpu().numpy()) < 2e-3
    y_again = ctx.w4a16_gemv(x, w, z, s)
    assert torch.equal(y, y_again), "same inputs must give the same bits (fixed-order stream-K fix-up)"
    y2 = ctx.w4a16_gemv((x * 2).to(torch.float16), w, z, s)  # linearity in x
    assert rel_err(y2.float().cpu().numpy(), 2 * y.float().cpu().numpy()) < 1e-3


def test_error_behaviour(ctx):
    from tinychatengine_b200 import _lib

    x, w, z, s = make_case(16, 256, 1, 1, False)
    with pytest.raises(_lib.TceError):  # reference: printf + exit(1) on a group size other than 64 / 128 (gemv_cuda.cu:253-257)
        ctx.w4a16_gemv(x, w, z, s, group=32)
    y = torch.empty((1, 16), dtype=torch.float16, device=x.device)
    rc = ctx.L.tce_w4a16_gemv(ctx.h, None, None, None, None, None, 1, 256, 16, 128)
    assert rc == -1
