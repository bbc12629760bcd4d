// capi.cu -- extern "C" surface of libtce_b200.so (include/tce_b200.h): argument checking, context and
// workspace management, dispatch to the sm_100a kernels.  No CPU fallback anywhere in this file.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/tce_b200.h"
#include "kernels.h"
#include "kernels_attn.h"
#include "kernels_w8a8.h"
#include "llama_decoder.h"

using namespace tce;

struct tce_ctx {
    Ctx c;
    int attn_chunk = 128;
};

static thread_local std::string g_err;

static int fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
int tce_fail_cuda(cudaError_t e, const char *what) {
    return fail(TCE_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}
#define CK(call, what)                                   \
    do {                                                 \
        cudaError_t e__ = (call);                        \
        if (e__ != cudaSuccess) return tce_fail_cuda(e__, what); \
    } while (0)

Ctx *tce_ctx_inner(tce_ctx *ctx) { return &ctx->c; }
int tce_ctx_attn_chunk(tce_ctx *ctx) { return ctx->attn_chunk; }

extern "C" {

int tce_version(void) { return 100; }
const char *tce_last_error(void) { return g_err.c_str(); }

int tce_zeros_width(int in_features, int group_size) {
    if (group_size != 128 && group_size != 64 && group_size != 32) return TCE_ERR_INVALID;
    return zeros_width(in_features, group_size);
}

static int env_int(const char *name, int dflt) {
    const char *v = getenv(name);
    return v ? atoi(v) : dflt;
}

int tce_ctx_create(int device, tce_ctx **out) {
    if (!out) return fail(TCE_ERR_INVALID, "tce_ctx_create: out is null");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return fail(TCE_ERR_CUDA, "no CUDA device: libtce_b200 has no CPU fallback (%s)", cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(TCE_ERR_INVALID, "device %d out of range (%d devices)", device, ndev);
    CK(cudaSetDevice(device), "cudaSetDevice");
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties");
    if (prop.major < 10) return fail(TCE_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    tce_ctx *ctx = new tce_ctx();
    Ctx &c = ctx->c;
    c.device = device;
    c.stream = nullptr;
    c.num_sms = prop.multiProcessorCount;
    c.smem_optin = (int)prop.sharedMemPerBlockOptin;
    c.gemv_impl = env_int("TCE_GEMV_IMPL", 1);
    c.gemv_ctas_per_sm = env_int("TCE_GEMV_CTAS_PER_SM", 1);
    c.gemv_consumer_warps = env_int("TCE_GEMV_CONSUMER_WARPS", 8);  // 8, 16, or 0 = per shape (16 for long rows: faster alone, not in the step)
    c.gemv_stages = env_int("TCE_GEMV_STAGES", 8);  // 8 vs 4: +3 % on the decode step once the consumers outran HBM (profiles/README.md)
    c.pdl_early = env_int("TCE_PDL_EARLY", 1);
    c.use_pdl = env_int("TCE_USE_PDL", 1) != 0;  // programmatic dependent launch, dependents resident from kernel entry: +3 % (profiles/r01_pdl_matrix.txt)
    ctx->attn_chunk = env_int("TCE_ATTN_CHUNK", 256);  // cached rows per CTA: 256 measured best (64: -8 %, 128: -2 %; profiles/README.md)
    c.gemv_max_ctas = c.num_sms * 4;
    c.gemv_max_tiles = 32768;
    c.attn_ws_bytes = (size_t)128 * 1024 * 130 * sizeof(float);  // heads * splits * (128 + 2): 128 heads x 1024 splits
    cudaError_t ie = cudaMalloc(&c.gemv_partials, (size_t)c.gemv_max_ctas * 2 * 16 * 8 * sizeof(float));
    if (ie == cudaSuccess) ie = cudaMalloc(&c.gemv_counters, (size_t)c.gemv_max_tiles * sizeof(unsigned));
    if (ie == cudaSuccess) ie = cudaMemset(c.gemv_counters, 0, (size_t)c.gemv_max_tiles * sizeof(unsigned));
    if (ie == cudaSuccess) ie = cudaMalloc(&c.attn_ws, c.attn_ws_bytes);
    if (ie == cudaSuccess) ie = cudaMalloc(&c.attn_counters, 1024 * sizeof(unsigned));
    if (ie == cudaSuccess) ie = cudaMemset(c.attn_counters, 0, 1024 * sizeof(unsigned));
    if (ie == cudaSuccess) ie = cudaDeviceSynchronize();
    if (ie != cudaSuccess) {  // a half-built context is released, not leaked (cudaFree(nullptr) is a no-op)
        tce_ctx_destroy(ctx);
        return tce_fail_cuda(ie, "tce_ctx_create: workspace allocation");
    }
    *out = ctx;
    return TCE_OK;
}

int tce_ctx_destroy(tce_ctx *ctx) {
    if (!ctx) return TCE_OK;
    cudaSetDevice(ctx->c.device);
    cudaFree(ctx->c.gemv_partials);
    cudaFree(ctx->c.gemv_counters);
    cudaFree(ctx->c.attn_ws);
    cudaFree(ctx->c.attn_counters);
    cudaFree(ctx->c.w16_scratch);
    cudaFree(ctx->c.gemv_dbg_keep);
    delete ctx;
    return TCE_OK;
}

int tce_ctx_set_stream(tce_ctx *ctx, void *s) {
    if (!ctx) return fail(TCE_ERR_INVALID, "null ctx");
    ctx->c.stream = (cudaStream_t)s;
    ctx->c.option_gen++;
    return TCE_OK;
}

int tce_ctx_synchronize(tce_ctx *ctx) {
    if (!ctx) return fail(TCE_ERR_INVALID, "null ctx");
    CK(cudaStreamSynchronize(ctx->c.stream), "cudaStreamSynchronize");
    return TCE_OK;
}

int tce_ctx_num_sms(tce_ctx *ctx) { return ctx ? ctx->c.num_sms : TCE_ERR_INVALID; }

int tce_ctx_read_gemv_timing(tce_ctx *ctx, unsigned long long *host_out, int max_ctas) {
    if (!ctx || !host_out || !ctx->c.gemv_dbg) return fail(TCE_ERR_INVALID, "gemv_debug option is off");
    const int n = max_ctas < ctx->c.gemv_max_ctas ? max_ctas : ctx->c.gemv_max_ctas;
    CK(cudaStreamSynchronize(ctx->c.stream), "sync");
    CK(cudaMemcpy(host_out, ctx->c.gemv_dbg, (size_t)n * 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost), "memcpy");
    return n;
}

int tce_ctx_set_option(tce_ctx *ctx, const char *name, int value) {
    if (!ctx || !name) return fail(TCE_ERR_INVALID, "null argument");
    if (!strcmp(name, "gemv_impl"))
        ctx->c.gemv_impl = value;
    else if (!strcmp(name, "gemv_ctas_per_sm"))
        ctx->c.gemv_ctas_per_sm = value < 1 ? 1 : (value > 4 ? 4 : value);
    else if (!strcmp(name, "gemv_consumer_warps"))
        ctx->c.gemv_consumer_warps = (value == 16) ? 16 : (value == 8 ? 8 : 0);
    else if (!strcmp(name, "gemv_stages"))
        ctx->c.gemv_stages = value < 0 ? 0 : value;
    else if (!strcmp(name, "gemv_debug")) {
        // the buffer is never freed before the context dies: CUDA graphs captured while the option was on keep writing to it
        if (value && !ctx->c.gemv_dbg) {
            if (!ctx->c.gemv_dbg_keep) {
                CK(cudaMalloc(&ctx->c.gemv_dbg_keep, (size_t)ctx->c.gemv_max_ctas * 8 * sizeof(unsigned long long)), "cudaMalloc dbg");
                CK(cudaMemset(ctx->c.gemv_dbg_keep, 0, (size_t)ctx->c.gemv_max_ctas * 8 * sizeof(unsigned long long)), "cudaMemset");
            }
            ctx->c.gemv_dbg = ctx->c.gemv_dbg_keep;
        } else if (!value) {
            ctx->c.gemv_dbg = nullptr;
        }
    } else if (!strcmp(name, "use_pdl"))
        ctx->c.use_pdl = value != 0;
    else if (!strcmp(name, "gemm_min_m"))  // smallest M served by the tcgen05 GEMMs (W4A16 prefill slot, W8A8); below it the weight-streaming kernels run
        ctx->c.gemm_min_m = value < 1 ? 1 : value;
    else if (!strcmp(name, "attn_cluster"))
        (void)value;  // accepted and ignored: the cluster flavour of the stand-alone decode attention was removed (measured slower)
    else if (!strcmp(name, "attn_chunk"))
        ctx->attn_chunk = value;
    else
        return fail(TCE_ERR_INVALID, "unknown option %s", name);
    ctx->c.option_gen++;  // graphs captured under the old settings are stale
    return TCE_OK;
}

// ---------------------------------------------------------------------------------------------- W4A16
static int w4a16_common(tce_ctx *ctx, const void *x, const void *w, const void *zeros, const void *scales, void *y, int M, int IC,
                        int OC, int group, const char *who) {
    if (!ctx || !x || !w || !zeros || !scales || !y) return fail(TCE_ERR_INVALID, "%s: null pointer", who);
    // the reference exits on any group size but 64/128 (gemv_cuda.cu:253-257) and is compiled with QK=128
    if (group == 64) {  // gemv_kernel_g64 (gemv_cuda.cu:68-123)
        if (M < 1 || IC < 64 || IC % 64 || OC < 1) return fail(TCE_ERR_INVALID, "%s: bad shape M=%d IC=%d OC=%d", who, M, IC, OC);
        CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
        CK(launch_w4a16_gemv_g64(&ctx->c, (const __half *)x, (const uint32_t *)w, (const uint32_t *)zeros, (const __half *)scales, (__half *)y, M, IC, OC), who);
        return TCE_OK;
    }
    if (group != kW4Group) return fail(TCE_ERR_INVALID, "%s: unsupported group size %d (the reference supports 64 and 128)", who, group);
    if (M < 1 || IC < kW4Group || IC % kW4Group || OC < 1) return fail(TCE_ERR_INVALID, "%s: bad shape M=%d IC=%d OC=%d", who, M, IC, OC);
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    const int zw = zeros_width(IC, group);
    // rows beyond the last multiple of 16 (the reference needs OC % 4 == 0; OC % 16 != 0 goes to the simple kernel)
    const int oc_main = (ctx->c.gemv_impl == 1) ? (OC / 16) * 16 : 0;
    for (int m0 = 0; m0 < M; m0 += 8) {
        const int mb = (M - m0 < 8) ? (M - m0) : 8;
        W4GemvParams p;
        p.nseg = 1;
        p.IC = IC;
        p.M = mb;
        p.x = (const __half *)x + (size_t)m0 * IC;
        p.ldx = IC;
        p.x_mode = X_HALF;
        p.epi = EPI_STORE_HALF;
        p.ldy = OC;
        if (oc_main > 0) {
            p.seg[0] = {(const uint32_t *)w, (const uint32_t *)zeros, (const __half *)scales, oc_main};
            p.y = (__half *)y + (size_t)m0 * OC;
            CK(launch_w4a16_gemv(&ctx->c, p), who);
        }
        if (oc_main < OC) {
            p.seg[0] = {(const uint32_t *)w + (size_t)oc_main * (IC / 8), (const uint32_t *)zeros + (size_t)oc_main * zw,
                        (const __half *)scales + (size_t)oc_main * zw * 8, OC - oc_main};
            p.y = (__half *)y + (size_t)m0 * OC + oc_main;
            CK(launch_w4a16_gemv_simple(&ctx->c, p), who);
        }
    }
    return TCE_OK;
}

int tce_w4a16_gemv(tce_ctx *ctx, const void *x, const void *w, const void *zeros, const void *scales, void *y, int M, int IC, int OC,
                   int group) {
    return w4a16_common(ctx, x, w, zeros, scales, y, M, IC, OC, group, "tce_w4a16_gemv");
}

int tce_w4a16_gemm(tce_ctx *ctx, const void *x, const void *w, const void *zeros, const void *scales, void *y, int M, int IC, int OC,
                   int group) {
    if (!ctx || M < ctx->c.gemm_min_m) return w4a16_common(ctx, x, w, zeros, scales, y, M, IC, OC, group, "tce_w4a16_gemm");  // weight-streaming GEMV passes
    if (!x || !w || !zeros || !scales || !y) return fail(TCE_ERR_INVALID, "tce_w4a16_gemm: null pointer");
    if (group != kW4Group) return fail(TCE_ERR_INVALID, "tce_w4a16_gemm: unsupported group size %d (QM_CUDA uses 128)", group);
    if (IC < kW4Group || IC % kW4Group || OC < 1) return fail(TCE_ERR_INVALID, "tce_w4a16_gemm: bad shape M=%d IC=%d OC=%d", M, IC, OC);
    if (((uintptr_t)x | (uintptr_t)w | (uintptr_t)y) & 15) return fail(TCE_ERR_INVALID, "tce_w4a16_gemm: x, w, y must be 16-byte aligned");
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    CK(w4_scratch_reserve(&ctx->c, (size_t)OC * IC), "w16 scratch");
    CK(launch_w4_expand(&ctx->c, (const uint32_t *)w, (const uint32_t *)zeros, (const __half *)scales, ctx->c.w16_scratch, OC, IC), "w4_expand");
    CK(launch_gemm_f16_pair(&ctx->c, (const __half *)x, IC, ctx->c.w16_scratch, IC, (__half *)y, OC, M, OC, IC, 0), "tce_w4a16_gemm");
    return TCE_OK;
}

int tce_naive_fp16_int4(tce_ctx *ctx, const void *A, const void *B, const void *scales, void *C, int M, int IC, int OC, int block) {
    if (!ctx || !A || !B || !scales || !C || M < 1 || IC < 1 || OC < 8 || OC % 8 || block < 1) return fail(TCE_ERR_INVALID, "tce_naive_fp16_int4: bad argument");
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    CK(launch_naive_fp16_int4(&ctx->c, (const __half *)A, (const int32_t *)B, (const __half *)scales, (__half *)C, M, IC, OC, block), "tce_naive_fp16_int4");
    return TCE_OK;
}

int tce_f32_matmul_transposed(tce_ctx *ctx, const float *A, const float *B, float *C, int M, int N, int K) {
    if (!ctx || !A || !B || !C || M < 1 || N < 1 || K < 1) return fail(TCE_ERR_INVALID, "tce_f32_matmul_transposed: bad argument");
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    CK(launch_f32_matmul_transposed(&ctx->c, A, B, C, M, N, K), "tce_f32_matmul_transposed");
    return TCE_OK;
}

// ---------------------------------------------------------------------------------------------- W8A8
int tce_w8a8_matmul(tce_ctx *ctx, int variant, int batch, const void *A, const void *B, const void *bias, void *C, int M, int N, int K,
                    float alpha, float beta, int q_min, int q_max) {
    if (!ctx || !A || !B || !C) return fail(TCE_ERR_INVALID, "tce_w8a8_matmul: null pointer");
    if (variant < 0 || variant > 3) return fail(TCE_ERR_INVALID, "tce_w8a8_matmul: variant %d", variant);
    if ((variant == W8_BIAS8_O8 || variant == W8_BIASF_OF32) && !bias) return fail(TCE_ERR_INVALID, "tce_w8a8_matmul: bias required");
    if (batch && (variant == W8_BIAS8_O8 || variant == W8_BIASF_OF32)) return fail(TCE_ERR_INVALID, "tce_w8a8_matmul: batch has no bias flavour");
    if (M < 1 || N < 1 || K < 1) return fail(TCE_ERR_INVALID, "tce_w8a8_matmul: bad shape");
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    W8A8Args a;
    a.A = (const int8_t *)A;
    a.B = (const int8_t *)B;
    a.bias8 = (const int8_t *)bias;
    a.biasf = (const float *)bias;
    a.C8 = (int8_t *)C;
    a.Cf = (float *)C;
    a.M = M;
    a.N = N;
    a.K = K;
    a.alpha = alpha;
    a.beta = beta;
    a.q_min = q_min;
    a.q_max = q_max;
    a.variant = variant;
    a.batch = batch ? 1 : 0;
    if (!a.batch && M >= ctx->c.gemm_min_m && K % 128 == 0 && !(((uintptr_t)A | (uintptr_t)B | (uintptr_t)C) & 15)) {
        CK(launch_w8a8_tc(&ctx->c, a), "tce_w8a8_matmul (tcgen05)");
        return TCE_OK;
    }
    CK(launch_w8a8_dp4a(&ctx->c, a), "tce_w8a8_matmul");
    return TCE_OK;
}

int tce_opt_int8_attention(tce_ctx *ctx, const void *q8, const void *k8, const void *v8, const void *past_k, const void *past_v, long long past_hs,
                           void *final_k, void *final_v, long long final_hs, const float *mask, float qk_alpha, float pv_alpha, int sqlen, int past,
                           int H, int hd, void *attn_out) {
    if (!ctx || !q8 || !k8 || !v8 || !final_k || !final_v || !attn_out) return fail(TCE_ERR_INVALID, "tce_opt_int8_attention: null pointer");
    if (sqlen < 1 || past < 0 || H < 1 || hd < 4 || hd % 4 || hd > 512) return fail(TCE_ERR_INVALID, "tce_opt_int8_attention: bad shape");
    if (past > 0 && (!past_k || !past_v || past_hs < (long long)past * hd)) return fail(TCE_ERR_INVALID, "tce_opt_int8_attention: bad past cache");
    if (final_hs < (long long)(past + sqlen) * hd || final_hs % 4) return fail(TCE_ERR_INVALID, "tce_opt_int8_attention: final_head_stride too small");
    if (((uintptr_t)q8 | (uintptr_t)final_k | (uintptr_t)final_v) & 3) return fail(TCE_ERR_INVALID, "tce_opt_int8_attention: pointers must be 4-byte aligned");
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    OptAttnParams p = {};
    p.q8 = (const int8_t *)q8;
    p.k8 = (const int8_t *)k8;
    p.v8 = (const int8_t *)v8;
    p.past_k = (const int8_t *)past_k;
    p.past_v = (const int8_t *)past_v;
    p.past_hs = past_hs;
    p.final_k = (int8_t *)final_k;
    p.final_v = (int8_t *)final_v;
    p.final_hs = final_hs;
    p.mask = mask;
    p.qk_alpha = qk_alpha;
    p.pv_alpha = pv_alpha;
    p.sqlen = sqlen;
    p.past = past;
    p.H = H;
    p.hd = hd;
    p.out = (int8_t *)attn_out;
    cudaError_t e = launch_opt_int8_attention(&ctx->c, p);
    if (e == cudaErrorInvalidValue) return fail(TCE_ERR_UNSUPPORTED, "tce_opt_int8_attention: context %d too long for one CTA's shared memory", past + sqlen);
    CK(e, "tce_opt_int8_attention");
    return TCE_OK;
}

// ---------------------------------------------------------------------------------------------- attention
int tce_attn_decode(tce_ctx *ctx, const void *qkv, void *k_cache, void *v_cache, const float *cosb, const float *sinb, const int *pos,
                    void *out, float alpha, int num_heads, int num_kv_heads, int head_dim, int max_ctx) {
    if (!ctx || !qkv || !k_cache || !v_cache || !cosb || !sinb || !pos || !out) return fail(TCE_ERR_INVALID, "tce_attn_decode: null pointer");
    if (head_dim != 128) return fail(TCE_ERR_UNSUPPORTED, "tce_attn_decode: head_dim %d (only 128)", head_dim);
    if (num_heads < 1 || num_kv_heads < 1 || num_heads % num_kv_heads || max_ctx < 1) return fail(TCE_ERR_INVALID, "tce_attn_decode: bad shape");
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    AttnDecodeArgs a = {};
    a.qkv = (const __half *)qkv;
    a.k_cache = (__half *)k_cache;
    a.v_cache = (__half *)v_cache;
    a.cos = cosb;
    a.sin = sinb;
    a.pos = pos;
    a.out = (__half *)out;
    a.alpha = alpha;
    a.num_heads = num_heads;
    a.num_kv_heads = num_kv_heads;
    a.head_dim = head_dim;
    a.max_ctx = max_ctx;
    a.chunk = ctx->attn_chunk;
    CK(launch_attn_decode(&ctx->c, a, false), "tce_attn_decode");
    return TCE_OK;
}

int tce_attn_prefill(tce_ctx *ctx, void *qkv, void *k_cache, void *v_cache, const float *cosb, const float *sinb, void *out, float alpha, int n, int pos0,
                     int num_heads, int num_kv_heads, int head_dim, int max_ctx) {
    if (!ctx || !qkv || !k_cache || !v_cache || !cosb || !sinb || !out) return fail(TCE_ERR_INVALID, "tce_attn_prefill: null pointer");
    if (head_dim != 128) return fail(TCE_ERR_UNSUPPORTED, "tce_attn_prefill: head_dim %d (only 128)", head_dim);
    if (num_heads < 1 || num_kv_heads < 1 || num_heads % num_kv_heads || n < 1 || pos0 < 0 || pos0 + n > max_ctx)
        return fail(TCE_ERR_INVALID, "tce_attn_prefill: bad shape n=%d pos0=%d max_ctx=%d", n, pos0, max_ctx);
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    AttnPrefillArgs a = {};
    a.qkv = (__half *)qkv;
    a.k_cache = (__half *)k_cache;
    a.v_cache = (__half *)v_cache;
    a.cos = cosb;
    a.sin = sinb;
    a.out = (__half *)out;
    a.alpha = alpha;
    a.n = n;
    a.pos0 = pos0;
    a.num_heads = num_heads;
    a.num_kv_heads = num_kv_heads;
    a.head_dim = head_dim;
    a.max_ctx = max_ctx;
    CK(launch_attn_prefill(&ctx->c, a), "tce_attn_prefill");
    return TCE_OK;
}

int tce_rmsnorm_f16(tce_ctx *ctx, const void *x, const float *gamma, void *y, int rows, int dim, float eps) {
    if (!ctx || !x || !gamma || !y || rows < 1 || dim < 1) return fail(TCE_ERR_INVALID, "tce_rmsnorm_f16: bad argument");
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    CK(launch_rmsnorm_f16(&ctx->c, (const __half *)x, gamma, (__half *)y, rows, dim, eps), "tce_rmsnorm_f16");
    return TCE_OK;
}

int tce_layernorm_q(tce_ctx *ctx, const float *x, const float *weight, const float *bias, void *out_int8, int rows, int dim) {
    if (!ctx || !x || !weight || !bias || !out_int8 || rows < 1 || dim < 1 || dim > 49000) return fail(TCE_ERR_INVALID, "tce_layernorm_q: bad argument");
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    CK(launch_layernorm_q(&ctx->c, x, weight, bias, (int8_t *)out_int8, rows, dim), "tce_layernorm_q");
    return TCE_OK;
}

int tce_add_f32(tce_ctx *ctx, const float *a, const float *b, float *out, long long n) {
    if (!ctx || !a || !b || !out || n < 1) return fail(TCE_ERR_INVALID, "tce_add_f32: bad argument");
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    CK(launch_add_f32(&ctx->c, a, b, out, n), "tce_add_f32");
    return TCE_OK;
}

int tce_argmax_f32(tce_ctx *ctx, const float *x, int n, int *out) {
    if (!ctx || !x || !out || n < 1) return fail(TCE_ERR_INVALID, "tce_argmax_f32: bad argument");
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    CK(launch_argmax(&ctx->c, x, n, out, false), "tce_argmax_f32");
    return TCE_OK;
}

// ---------------------------------------------------------------------------------------------- llama
int tce_llama_create(tce_ctx *ctx, const tce_llama_config *cfg, const tce_llama_weights *w, tce_llama **out) {
    if (!ctx || !cfg || !w || !out) return fail(TCE_ERR_INVALID, "tce_llama_create: null argument");
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    std::string err;
    LlamaDecoder *d = LlamaDecoder::create(&ctx->c, ctx->attn_chunk, *cfg, *w, &err);
    if (!d) return fail(TCE_ERR_INVALID, "tce_llama_create: %s", err.c_str());
    *out = reinterpret_cast<tce_llama *>(d);
    return TCE_OK;
}
int tce_llama_load_dir(tce_ctx *ctx, const char *dir, const tce_llama_config *cfg, tce_llama **out) {
    if (!ctx || !dir || !cfg || !out) return fail(TCE_ERR_INVALID, "tce_llama_load_dir: null argument");
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    std::string err;
    LlamaDecoder *d = load_llama_dir(&ctx->c, ctx->attn_chunk, dir, *cfg, &err);
    if (!d) return fail(TCE_ERR_INVALID, "tce_llama_load_dir: %s", err.c_str());
    *out = reinterpret_cast<tce_llama *>(d);
    return TCE_OK;
}
int tce_w4_import_x86(const void *qs_u8, const float *scales_f32, int oc, int ic, void *w_out, void *scales_f16_out, void *zeros_out) {
    if (!qs_u8 || !scales_f32 || !w_out || !scales_f16_out || !zeros_out) return fail(TCE_ERR_INVALID, "tce_w4_import_x86: null argument");
    if (import_x86(static_cast<const uint8_t *>(qs_u8), scales_f32, oc, ic, static_cast<uint32_t *>(w_out), static_cast<__half *>(scales_f16_out),
                   static_cast<uint32_t *>(zeros_out)))
        return fail(TCE_ERR_INVALID, "tce_w4_import_x86: ic must be a multiple of 128");
    return TCE_OK;
}
int tce_llama_destroy(tce_llama *m) {
    delete reinterpret_cast<LlamaDecoder *>(m);
    return TCE_OK;
}
int tce_llama_decode(tce_llama *m, const int *tokpos_dev) {
    if (!m || !tokpos_dev) return fail(TCE_ERR_INVALID, "tce_llama_decode: null argument");
    std::string err;
    cudaError_t e = reinterpret_cast<LlamaDecoder *>(m)->decode_device(tokpos_dev, &err);
    if (e != cudaSuccess) return fail(TCE_ERR_CUDA, "tce_llama_decode: %s (%s)", cudaGetErrorString(e), err.c_str());
    return TCE_OK;
}
int tce_llama_decode_host(tce_llama *m, int token, int pos, float *logits_host, int *next_token) {
    if (!m) return fail(TCE_ERR_INVALID, "tce_llama_decode_host: null argument");
    std::string err;
    cudaError_t e = reinterpret_cast<LlamaDecoder *>(m)->decode_host(token, pos, logits_host, next_token, &err);
    if (e != cudaSuccess) return fail(TCE_ERR_CUDA, "tce_llama_decode_host: %s (%s)", cudaGetErrorString(e), err.c_str());
    return TCE_OK;
}
int tce_llama_prefill(tce_llama *m, const int *tokens_host, int n, int pos0, float *logits_host, int *next_token) {
    if (!m || !tokens_host) return fail(TCE_ERR_INVALID, "tce_llama_prefill: null argument");
    std::string err;
    cudaError_t e = reinterpret_cast<LlamaDecoder *>(m)->prefill(tokens_host, n, pos0, logits_host, next_token, &err);
    if (e == cudaErrorNotSupported) return fail(TCE_ERR_UNSUPPORTED, "tce_llama_prefill: %s", err.c_str());
    if (e == cudaErrorInvalidValue) return fail(TCE_ERR_INVALID, "tce_llama_prefill: bad tokens / n=%d pos0=%d", n, pos0);
    if (e != cudaSuccess) return fail(TCE_ERR_CUDA, "tce_llama_prefill: %s (%s)", cudaGetErrorString(e), err.c_str());
    return TCE_OK;
}
int tce_llama_generate(tce_llama *m, int first_token, int pos0, int n_predict, const tce_sampling *cfg, const int *history_host, int n_history, int eos_id,
                       int *out_tokens_host, int *n_out) {
    if (!m || !cfg || !n_out) return fail(TCE_ERR_INVALID, "tce_llama_generate: null argument");
    std::string err;
    cudaError_t e = reinterpret_cast<LlamaDecoder *>(m)->generate(first_token, pos0, n_predict, *cfg, history_host, n_history, eos_id, out_tokens_host, n_out, &err);
    if (e == cudaErrorNotSupported) return fail(TCE_ERR_UNSUPPORTED, "tce_llama_generate: %s", err.c_str());
    if (e == cudaErrorInvalidValue) return fail(TCE_ERR_INVALID, "tce_llama_generate: bad token / position / count");
    if (e != cudaSuccess) return fail(TCE_ERR_CUDA, "tce_llama_generate: %s (%s)", cudaGetErrorString(e), err.c_str());
    return TCE_OK;
}
int tce_sample(tce_ctx *ctx, float *logits_dev, int n_vocab, const int *window_host, int n_window, const tce_sampling *cfg, unsigned long long draw_index,
               int *token_host, int *cand_ids_host, float *cand_probs_host, int *cand_count_host) {
    if (!ctx || !logits_dev || !cfg || !token_host || n_vocab < 1 || n_window < 0 || (n_window > 0 && !window_host))
        return fail(TCE_ERR_INVALID, "tce_sample: bad argument");
    CK(cudaSetDevice(ctx->c.device), "cudaSetDevice");
    const bool want_cand = cand_ids_host && cand_probs_host && cand_count_host;
    const int kcap = 1024;
    int *scratch = nullptr;  // [0] token, [1] head, [2] cand count, [4..] window, then cand ids, cand probs
    const size_t words = 4 + (size_t)(n_window > 0 ? n_window : 1) + 2 * (size_t)kcap;
    CK(cudaMalloc((void **)&scratch, words * sizeof(int)), "tce_sample: scratch");
    cudaStream_t s = ctx->c.stream;
    int *win = scratch + 4, *cids = win + (n_window > 0 ? n_window : 1);
    float *cprob = reinterpret_cast<float *>(cids + kcap);
    const int ctl[4] = {0, n_window, 0, 0};
    cudaError_t e = cudaMemcpyAsync(scratch, ctl, sizeof(ctl), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess && n_window > 0) e = cudaMemcpyAsync(win, window_host, (size_t)n_window * sizeof(int), cudaMemcpyHostToDevice, s);
    SampleArgs a{};
    a.logits = logits_dev;
    a.n_vocab = n_vocab;
    a.top_k = cfg->top_k;
    a.top_p = cfg->top_p;
    a.temp = cfg->temp;
    a.repeat_penalty = cfg->repeat_penalty;
    a.frequency_penalty = cfg->frequency_penalty;
    a.presence_penalty = cfg->presence_penalty;
    a.repeat_last_n = cfg->repeat_last_n;
    a.seed = cfg->seed;
    a.draw_index = draw_index;
    if (n_window > 0) {
        a.hist = win;
        a.hist_cap = n_window;
    }
    a.out_token = scratch;
    if (want_cand) {
        a.dbg_ids = cids;
        a.dbg_probs = cprob;
        a.dbg_size = scratch + 2;
    }
    // a fixed window: the ring is exactly full (head == capacity), and the draw index is not advanced by the head
    int *head = scratch + 1;
    a.hist_head = n_window > 0 ? head : nullptr;
    if (n_window > 0) a.draw_index = draw_index - (unsigned long long)n_window;
    if (e == cudaSuccess) e = launch_sample(&ctx->c, a, s);
    int out[4] = {0, 0, 0, 0};
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, scratch, sizeof(out), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e == cudaSuccess && want_cand && out[2] > 0) {
        e = cudaMemcpy(cand_ids_host, cids, (size_t)out[2] * sizeof(int), cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(cand_probs_host, cprob, (size_t)out[2] * sizeof(float), cudaMemcpyDeviceToHost);
    }
    cudaFree(scratch);
    if (e == cudaErrorNotSupported) return fail(TCE_ERR_UNSUPPORTED, "tce_sample: temp > 0 needs 1 <= top_k <= 1024");
    if (e != cudaSuccess) return fail(TCE_ERR_CUDA, "tce_sample: %s", cudaGetErrorString(e));
    *token_host = out[0];
    if (want_cand) *cand_count_host = out[2];
    return TCE_OK;
}
const float *tce_llama_logits(tce_llama *m) { return m ? reinterpret_cast<LlamaDecoder *>(m)->logits() : nullptr; }
void *tce_llama_kv_cache(tce_llama *m, int layer, int which) { return m ? reinterpret_cast<LlamaDecoder *>(m)->kv_cache(layer, which) : nullptr; }
int tce_llama_enqueue_gemvs(tce_llama *m) {
    if (!m) return fail(TCE_ERR_INVALID, "tce_llama_enqueue_gemvs: null argument");
    int n = 0;
    cudaError_t e = reinterpret_cast<LlamaDecoder *>(m)->enqueue_gemvs(&n);
    if (e != cudaSuccess) return tce_fail_cuda(e, "tce_llama_enqueue_gemvs");
    return n;
}
void *tce_llama_debug_buffer(tce_llama *m, int which) { return m ? reinterpret_cast<LlamaDecoder *>(m)->debug_buffer(which) : nullptr; }
int tce_llama_tp_handle(tce_llama *m, void *out) {
    if (!m || !out) return fail(TCE_ERR_INVALID, "tce_llama_tp_handle: null argument");
    cudaError_t e = reinterpret_cast<LlamaDecoder *>(m)->tp_handle(out);
    if (e != cudaSuccess) return tce_fail_cuda(e, "tce_llama_tp_handle");
    return TCE_OK;
}
int tce_llama_tp_connect(tce_llama *m, const void *handles) {
    if (!m || !handles) return fail(TCE_ERR_INVALID, "tce_llama_tp_connect: null argument");
    cudaError_t e = reinterpret_cast<LlamaDecoder *>(m)->tp_connect(handles);
    if (e != cudaSuccess) return tce_fail_cuda(e, "tce_llama_tp_connect");
    return TCE_OK;
}
int tce_llama_kernels_per_step(tce_llama *m) { return m ? reinterpret_cast<LlamaDecoder *>(m)->kernels_per_step() : TCE_ERR_INVALID; }

}  // extern "C"
