// kernels.h -- internal C++ launch interface of libtce_b200 (the public face is include/tce_b200.h).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

namespace tce {

// One context per (device, stream).  Owns the small workspaces the kernels need; never owns caller data.
struct Ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    int num_sms = 0;
    int smem_optin = 0;
    // stream-K fix-up workspace of the W4A16 GEMV: 2 partial records per CTA + one arrival counter per row tile
    float *gemv_partials = nullptr;
    unsigned *gemv_counters = nullptr;
    int gemv_max_ctas = 0;
    int gemv_max_tiles = 0;
    unsigned long long *gemv_dbg = nullptr;  // optional phase timestamps (option "gemv_debug")
    unsigned long long *gemv_dbg_keep = nullptr;  // its allocation (kept until the context is destroyed)
    // flash-decode workspace (partial m, l, o per (head, split))
    float *attn_ws = nullptr;
    size_t attn_ws_bytes = 0;
    unsigned *attn_counters = nullptr;
    unsigned option_gen = 0;       // bumped by every tce_ctx_set_option / set_stream: captured CUDA graphs hold the context by value and are rebuilt
    unsigned attn_seed_epoch = 0;  // calls of the int8 OPT attention so far (tags the in-kernel seed hand-off)
    // tunables (env overridable, see ctx.cu)
    int gemv_impl = 1;      // 0 = simple warp-per-row, 1 = TMA + mma.sync stream-K
    int gemv_ctas_per_sm = 1;
    int gemv_consumer_warps = 8;   // 8 or 16 consumer warps per CTA; 0 = chosen per shape
    int gemv_stages = 8;           // TMA ring depth (16 KiB stages, capped by the per-CTA shared-memory share); 0 = deepest that fits
    bool use_pdl = false;
    int pdl_early = 0;  // with use_pdl: 1 = dependents may become resident from the first instruction of each GEMV (2: and no 2-CTA/SM mode)
    // large-M (prefill) path: fp16 expansion of one int4 weight matrix, grown on demand; M >= gemm_min_m goes to the tcgen05 GEMM
    __half *w16_scratch = nullptr;
    size_t w16_scratch_elems = 0;
    int gemm_min_m = 16;
};

// One-time kernel attribute setup (cudaFuncSetAttribute) is per (kernel, DEVICE): a process may hold contexts on several devices, so each launch site
// keeps one bit per device instead of one flag per process.  Setting the attribute twice from two racing threads is harmless.
struct DeviceOnce {
    std::atomic<unsigned long long> mask{0};
    bool pending(int device) const { return !((mask.load(std::memory_order_acquire) >> (device & 63)) & 1ull); }
    void done(int device) { mask.fetch_or(1ull << (device & 63), std::memory_order_release); }
};

constexpr int kW4Group = 128;  // QK for QM_CUDA (llm/include/common.h:17-21)

inline int zeros_width(int ic, int group) {  // llm/src/nn_modules/cuda/utils.cu:162-178
    int mult = group >= 128 ? 1 : (group == 64 ? 2 : 4);
    int base = (ic / group + 7) / 8;
    return (base + mult - 1) / mult * mult;
}

enum XMode : int { X_HALF = 0, X_RMSNORM_F32 = 1 };
enum EpiMode : int { EPI_STORE_HALF = 0, EPI_STORE_F32 = 1, EPI_ADD_F32 = 2, EPI_SILU_MUL_HALF = 3, EPI_TP_SCATTER_F32 = 4 };
constexpr int kMaxTP = 8;

struct W4Seg {
    const uint32_t *w;       // [rows][IC/8]
    const uint32_t *zeros;   // [rows][zeros_w]
    const __half *scales;    // [rows][zeros_w*8]
    int rows;                // multiple of 16 (8 in pair mode)
};

struct W4GemvParams {
    W4Seg seg[3];
    int nseg = 1;
    int pair_mode = 0;  // 1: row tile = 8 rows of seg[0] (-> MMA rows 0-7) + the same 8 rows of seg[1] (rows 8-15)
    int IC = 0;
    int M = 1;          // activation rows (<= 8 per launch)
    const void *x = nullptr;
    int x_mode = X_HALF;
    int ldx = 0;        // elements between activation rows
    const float *gamma = nullptr;
    float eps = 0.f;
    void *y = nullptr;
    int epi = EPI_STORE_HALF;
    int ldy = 0;        // elements between output rows
    bool pdl = false;   // launch with programmatic stream serialization
    bool atomic_residual = false;  // EPI_ADD_F32 only: allow RED.ADD for split tiles (non-deterministic last bit)
    // ---- tensor parallel (tp_size > 1) ----
    int tp_size = 1;
    // prologue (X_RMSNORM_F32): x = resid + sum_p tp_in[p][:] once tp_flags[p] >= expected, written back to resid_out
    const float *tp_in = nullptr;        // local gather buffer [tp_size][IC] fp32 (peers store into it)
    const unsigned *tp_flags = nullptr;  // local arrival flags [tp_size]
    const int *tp_step = nullptr;        // device int: decode step index (flags carry step * tp_per_step + tp_k + 1)
    int tp_k = 0, tp_per_step = 1;
    float *resid_out = nullptr;
    // epilogue (EPI_TP_SCATTER_F32): the finished fp32 outputs are stored into slot `rank` of every peer's gather buffer
    float *tp_out[kMaxTP] = {};
    // ... and, once every CTA of the launch has stored (local arrival counter), the last one release-stores the step-stamped flag
    // into every peer's flag word: the collective needs no separate signal kernel
    unsigned *tp_sig_counter = nullptr;
    unsigned *tp_sig_flag[kMaxTP] = {};
    int tp_sig_k = 0;
};

cudaError_t launch_w4a16_gemv(Ctx *ctx, const W4GemvParams &p);
cudaError_t launch_w4a16_gemv_simple(Ctx *ctx, const W4GemvParams &p);
cudaError_t launch_w4a16_gemv_g64(Ctx *ctx, const __half *x, const uint32_t *w, const uint32_t *zeros, const __half *scales, __half *y, int M, int IC, int OC);
size_t w4a16_gemv_smem_bytes(int ncols, int consumer_warps, int IC);
cudaError_t encode_w4_tmap(CUtensorMap *out, const void *w, int rows, int IC, int sg, int box_rows);
cudaError_t encode_w4_tmap_units(CUtensorMap *out, const void *w, int rows, int IC, int sg, int box_rows);  // [group][row][64 B] boxes

cudaError_t launch_naive_fp16_int4(Ctx *ctx, const __half *A, const int32_t *B, const __half *scales, __half *C, int M, int IC, int OC, int block);
cudaError_t launch_f32_matmul_transposed(Ctx *ctx, const float *A, const float *B, float *C, int M, int N, int K);

// W4A16 prefill GEMM (gemm_tc2.cu): the int4 weights are expanded to fp16 (launch_w4_expand), then multiplied on CTA pairs
// (tcgen05.mma.cta_group::2, 256 x 256 tiles)
cudaError_t launch_w4_expand(Ctx *ctx, const uint32_t *w, const uint32_t *zeros, const __half *scales, __half *out, int OC, int IC);
cudaError_t launch_gemm_f16_pair(Ctx *ctx, const __half *X, long long ldx, const __half *W, long long ldw, void *C, long long ldc, int M, int N, int K, int add_f32);
cudaError_t launch_gemm_f16_pair_silu(Ctx *ctx, const __half *X, long long ldx, const __half *W, long long ldw, __half *act, long long ldc, int M, int F, int K);
cudaError_t w4_scratch_reserve(Ctx *ctx, size_t elems);  // grows ctx->w16_scratch (may synchronise the device)

// host-side mirror of the stream-K partition used by the kernel (unit-tested on the CPU)
struct StreamK {
    long long U;   // total units = tiles * groups
    int nc;        // CTAs
    int NG;        // groups per row tile
    int aligned = 0;  // cut at row-tile boundaries instead of unit boundaries
    int T = 0;        // row tiles (aligned mode)
    int gran = 1;     // unaligned mode: cuts fall on multiples of `gran` units (16 = whole pipeline stages; U % gran == 0)
    __host__ __device__ long long start(int c) const {
        const long long n = aligned ? (long long)T : U / gran;  // cut positions are n * c / nc, in tiles or in `gran` units
        const long long q = (n * nc < 0x7fffffffLL) ? (long long)(((unsigned)n * (unsigned)c) / (unsigned)nc) : (n * (long long)c) / nc;  // 32-bit divide when it fits
        return q * (aligned ? NG : gran);
    }
    // owner of unit u in unaligned mode: the largest c with start(c) <= u
    __host__ __device__ int cta_of(long long u) const {
        const long long Ug = U / gran, ug = u / gran;
        return (int)(((ug + 1) * nc + Ug - 1) / Ug - 1);
    }
};

}  // namespace tce
