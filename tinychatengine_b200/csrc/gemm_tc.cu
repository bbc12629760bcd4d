// gemm_tc.cu -- instantiations of the tcgen05 GEMM for the large-M W8A8 slot (mat_mul_accelerator_int8_fast_2x2_32unroll* at M >= 16,
// kernels/ref/matmul_ref_int8.cc:11-159): tcgen05 kind::i8 with int32 accumulation is exact, the float epilogue keeps the reference's
// evaluation order -> bit-identical int8 / fp32 outputs.  (The W4A16 prefill GEMM runs on CTA pairs: gemm_tc2.cu.)
#include "gemm_tc.cuh"
#include "kernels.h"
#include "kernels_w8a8.h"

namespace tce {
namespace {

using tc::GemmArgs;

// ------------------------------------------------------------------------------------------------ epilogues
template <int VARIANT>
struct EpiW8 {  // int32 accumulator -> the four W8A8 epilogues (same float op order as w8a8.cu / kernels/ref)
    TCE_DEVINL static void apply(const GemmArgs &a, int row, int col0, int n, const uint32_t (&v)[32]) {
        const size_t o = (size_t)row * a.ldc + col0;
        if constexpr (VARIANT == W8_BIAS8_O8 || VARIANT == W8_NOBIAS_O8) {
            int8_t *dst = reinterpret_cast<int8_t *>(a.C) + o;
            uint32_t packed[8];
#pragma unroll
            for (int i = 0; i < 32; i++) {
                float f = __fmul_rn((float)(int)v[i], a.alpha);
                if constexpr (VARIANT == W8_BIAS8_O8) f = __fadd_rn(f, __fmul_rn((float)(i < n ? a.bias8[col0 + i] : (int8_t)0), a.beta));
                int qv = (int)roundf(f);
                qv = min(max(qv, a.q_min), a.q_max);
                if ((i & 3) == 0) packed[i >> 2] = 0;
                packed[i >> 2] |= (uint32_t)(qv & 0xff) << (8 * (i & 3));
            }
            if (n == 32 && (a.ldc & 15) == 0) {
                reinterpret_cast<uint4 *>(dst)[0] = make_uint4(packed[0], packed[1], packed[2], packed[3]);
                reinterpret_cast<uint4 *>(dst)[1] = make_uint4(packed[4], packed[5], packed[6], packed[7]);
            } else {
#pragma unroll
                for (int i = 0; i < 32; i++)
                    if (i < n) dst[i] = (int8_t)((packed[i >> 2] >> (8 * (i & 3))) & 0xff);
            }
        } else {
            float *dst = reinterpret_cast<float *>(a.C) + o;
#pragma unroll
            for (int i = 0; i < 32; i++) {
                if (i < n) {
                    float f = __fmul_rn((float)(int)v[i], a.alpha);
                    if constexpr (VARIANT == W8_BIASF_OF32) f = __fadd_rn(f, a.biasf[col0 + i]);
                    dst[i] = f;
                }
            }
        }
    }
};

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                             const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

cudaError_t encode_kmajor(CUtensorMap *out, const void *base, long long rows, long long K, int box_rows) {  // int8 [rows][K]
    static EncodeFn fn = nullptr;
    if (!fn) {
        void *sym = nullptr;
        cudaDriverEntryPointQueryResult q;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q);
        if (e != cudaSuccess || !sym) return e != cudaSuccess ? e : cudaErrorNotSupported;
        fn = reinterpret_cast<EncodeFn>(sym);
    }
    const cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)K};
    const cuuint32_t box[2] = {(cuuint32_t)tc::kAtomBytes, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void *>(base), gdim, gstride, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}

template <int BLOCK_N, int STAGES, class Epi>
cudaError_t launch(Ctx *ctx, GemmArgs &a, const void *A, const void *B, int K) {
    cudaError_t e = encode_kmajor(&a.tmA, A, a.M, K, tc::kBlockM);
    if (e != cudaSuccess) return e;
    e = encode_kmajor(&a.tmB, B, a.N, K, BLOCK_N);
    if (e != cudaSuccess) return e;
    a.k_blocks = K / tc::kAtomBytes;
    a.m_blocks = (a.M + tc::kBlockM - 1) / tc::kBlockM;
    a.n_blocks = (a.N + BLOCK_N - 1) / BLOCK_N;
    auto kern = tc::gemm_tc_kernel<BLOCK_N, STAGES, Epi>;
    constexpr size_t smem = tc::smem_bytes<BLOCK_N, STAGES>();
    static DeviceOnce attr_once;  // per instantiation
    if (attr_once.pending(ctx->device)) {
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        attr_once.done(ctx->device);
    }
    const int tiles = a.m_blocks * a.n_blocks;
    const int grid = tiles < ctx->num_sms ? tiles : ctx->num_sms;
    kern<<<grid, tc::kThreads, smem, ctx->stream>>>(a);
    return cudaGetLastError();
}

// Tile width by wave quantisation: a persistent grid of `sms` CTAs needs ceil(tiles / sms) rounds, each costing ~BLOCK_N (the MMA
// time of one tile) times a small penalty for the narrower tiles (the 128-row A tile is re-read once per N block).
int pick_block_n(int M, int N, int sms) {
    const long long mb = (M + 127) / 128;
    const int bn[3] = {256, 192, 128};
    const double pen[3] = {1.00, 1.04, 1.12};
    int best = 256;
    double best_cost = 1e30;
    for (int i = 0; i < 3; i++) {
        const long long tiles = mb * ((N + bn[i] - 1) / bn[i]);
        const double cost = (double)((tiles + sms - 1) / sms) * bn[i] * pen[i];
        if (cost < best_cost) {
            best_cost = cost;
            best = bn[i];
        }
    }
    return best;
}

template <class Epi>
cudaError_t dispatch(Ctx *ctx, GemmArgs &a, const void *A, const void *B, int K) {
    switch (pick_block_n(a.M, a.N, ctx->num_sms)) {
        case 256: return launch<256, 4, Epi>(ctx, a, A, B, K);
        case 192: return launch<192, 5, Epi>(ctx, a, A, B, K);
        default: return launch<128, 6, Epi>(ctx, a, A, B, K);
    }
}

}  // namespace

// the four non-batched W8A8 variants on the int8 tensor cores.  K % 128 == 0 (one swizzle atom), pointers 16-byte aligned.
cudaError_t launch_w8a8_tc(Ctx *ctx, const W8A8Args &w) {
    if (w.batch || w.M < 1 || w.N < 1 || w.K < 128 || (w.K % 128)) return cudaErrorInvalidValue;
    GemmArgs a = {};
    a.M = w.M;
    a.N = w.N;
    a.ldc = w.N;
    a.bias8 = w.bias8;
    a.biasf = w.biasf;
    a.alpha = w.alpha;
    a.beta = w.beta;
    a.q_min = w.q_min;
    a.q_max = w.q_max;
    switch (w.variant) {
        case W8_BIAS8_O8: a.C = w.C8; return dispatch<EpiW8<W8_BIAS8_O8>>(ctx, a, w.A, w.B, w.K);
        case W8_NOBIAS_O8: a.C = w.C8; return dispatch<EpiW8<W8_NOBIAS_O8>>(ctx, a, w.A, w.B, w.K);
        case W8_BIASF_OF32: a.C = w.Cf; return dispatch<EpiW8<W8_BIASF_OF32>>(ctx, a, w.A, w.B, w.K);
        case W8_NOBIAS_OF32: a.C = w.Cf; return dispatch<EpiW8<W8_NOBIAS_OF32>>(ctx, a, w.A, w.B, w.K);
    }
    return cudaErrorInvalidValue;
}

}  // namespace tce
