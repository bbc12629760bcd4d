// gemm_tc2.cu -- the W4A16 prefill GEMM (MatmulOperator::gemm_forward_cuda, declared-but-undefined in the reference,
// kernels/matmul.h:142-145): the QM_CUDA int4 weights are expanded to fp16 ((q - z) * s, one rounding) by a bandwidth-bound pass, then
// C[M][N] = X[M][K] (fp16) * W[N][K]^T runs on CTA pairs with tcgen05.mma.cta_group::2 and fp32 accumulation in TMEM.  Expanding once
// per call instead of once per M tile keeps the CUDA-core dequant work at OC*IC instead of OC*IC*ceil(M/256).
//
// Two CTAs of a cluster (one TPC) own one 256 x 256 output tile.  Each CTA stages ITS 128 activation rows and ITS 128 weight rows of
// every 64-k block; one thread of the leader CTA issues M = 256 MMAs that read both CTAs' shared memory, so per CTA and k-block the
// tensor core pulls 32 KiB of operands for 128 x 256 x 64 MACs -- half of what a single-CTA 128 x 256 tile needs, which is what bounds
// a single-CTA kernel: there the operand reads + TMA writes exceed the 128 B/clk of one SM's shared memory long before the tensor pipe
// is busy (profiles/README.md, round 2).  Both operands arrive by TMA (cta_group::2 flavour: completion bytes are counted on the
// leader's mbarrier).
// Epilogue: every CTA reads its own 128 accumulator rows from its own TMEM (double-buffered accumulators), fp16 store or fp32 accumulate.
#include "gemm_tc.cuh"
#include "kernels.h"

namespace tce {
namespace {

using namespace tc;

constexpr int kPairN = 256;                 // output columns per tile (each CTA stages half of the weight rows)
constexpr int kHalfN = 128;
constexpr int kBHalfBytes = kHalfN * 128;   // 16 KiB fp16 operand tile per CTA and k-block
constexpr int kStages = 6;                  // ring of activation tiles + this CTA's fp16 weight tile in the same slot
constexpr int kSlotBytes = kABytes + kBHalfBytes;
constexpr int kPairThreads = 32 * 6;
constexpr size_t kPairSmem = 1024 + (size_t)kStages * kSlotBytes;
constexpr uint32_t kPeerMask = 0xFEFFFFFFu; // clears the CTA-rank bit of a shared::cluster address: "the same location in CTA 0"
constexpr uint64_t kEvictNormal = 0x1000000000000000ull;

struct PairArgs {
    alignas(64) CUtensorMap tmA;  // fp16 [M][K], box {64, 128}, SWIZZLE_128B
    alignas(64) CUtensorMap tmB;  // fp16 [N][K], box {64, pn / 2}, SWIZZLE_128B
    int M, N, k_blocks, m_blocks, n_blocks;  // blocks of 256
    void *C;
    long long ldc;
    int add_f32;
    int pn;      // output columns per tile of the fp16-weight kernel: 256, or 128 where 256-wide tiles quantise badly onto the 74 clusters (N = 5120:
                 // 160 tiles = 2.16 waves); each CTA stages pn / 2 weight rows.  The SiLU variant uses 256.
    int silu_F;  // > 0: W = [gate (F rows); up (F rows)], the pair's two halves are the SAME 128 channels of gate (CTA 0) and up (CTA 1), and the
                 // epilogue writes act[M][F] = SiLU(gate) * up (SiLuMul_half, llm/src/nn_modules/cuda/Int4llamaDecoderLayer.cu:12-30; fp32 math)
};

TCE_DEVINL uint32_t cluster_rank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
TCE_DEVINL uint32_t cluster_id_x() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
    return r;
}
TCE_DEVINL uint32_t num_clusters_x() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
    return r;
}
TCE_DEVINL void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the mbarrier at the same shared-memory offset in CTA `rank` of the cluster
TCE_DEVINL void mbar_arrive_cluster(uint64_t *bar, uint32_t rank) {
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(rank));
    // default semantics (release at CTA scope), as for a local arrive: the caller's tcgen05.fence::before_thread_sync orders its TMEM reads;
    // a cluster-scope release costs MEMBAR.ALL.GPU + ERRBAR per arrive (profiles/README.md)
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
// wait on a barrier whose arrivals come from both CTAs (plain try_wait: an acquire.cluster wait invalidates L1 on every poll)
TCE_DEVINL void mbar_wait_cl(uint64_t *bar, uint32_t parity) {
    const long long t0 = clock64();
    while (true) {
        uint32_t ok;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok)
                     : "r"(smem_u32(bar)), "r"(parity)
                     : "memory");
        if (ok) return;
        if (clock64() - t0 > 6000000000LL) __trap();  // a protocol bug surfaces as a launch failure, not as a hung GPU
    }
}
// TMA load whose completion bytes are counted on the LEADER's barrier (same offset in CTA 0); the data lands in this CTA
TCE_DEVINL void tma_load_2d_pair(void *dst_smem, const void *tmap, int x, int y, uint64_t *bar) {
    asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(tmap), "r"(x), "r"(y), "r"(smem_u32(bar) & kPeerMask), "l"(kEvictNormal)
                 : "memory");
}
TCE_DEVINL void tmem_alloc_pair(uint32_t *dst_smem, uint32_t ncols) {  // the same warp of BOTH CTAs
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
TCE_DEVINL void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// all MMAs issued so far by this thread complete -> one arrival on `bar` in BOTH CTAs
TCE_DEVINL void umma_commit_pair(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)), "h"((unsigned short)3)
                 : "memory");
}
TCE_DEVINL void umma_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc),
                 "r"(idesc), "r"(accumulate)
                 : "memory");
}

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kPairThreads, 1) gemm_pair_kernel(const __grid_constant__ PairArgs a) {
    constexpr int AS = kStages;
    extern __shared__ uint8_t smem_raw[];
    // barriers live at identical offsets in both CTAs (multicast commits and remote arrives address "the same barrier in the other CTA")
    __shared__ __align__(8) uint64_t a_full[AS], a_empty[AS], tfull_bar[2], tempty_bar[2];
    __shared__ uint32_t tmem_base_s;
    const uint32_t raw = smem_u32(smem_raw);
    uint8_t *sSlot = smem_raw + (((raw + 1023u) & ~1023u) - raw);  // [AS][A 16 KiB | B half fp16 16 KiB]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_rank();
    const bool leader = rank == 0;
    const int tiles_total = a.m_blocks * a.n_blocks;
    const int cl = (int)cluster_id_x(), ncl = (int)num_clusters_x();

    if (threadIdx.x == 0) {
        for (int s = 0; s < AS; s++) {
            mbar_init(&a_full[s], 1);                          // leader: its own expect_tx arrival; bytes from both CTAs
            mbar_init(&a_empty[s], 1);                         // multicast MMA commit
        }
        for (int s = 0; s < 2; s++) {
            mbar_init(&tfull_bar[s], 1);                       // multicast MMA commit
            mbar_init(&tempty_bar[s], 256);                    // leader: the epilogue threads of both CTAs
        }
        mbar_fence_init();
    }
    cluster_sync_all();  // barriers of both CTAs exist before anyone signals across
    if (warp == 1) tmem_alloc_pair(&tmem_base_s, 512);
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (warp == 0) {
        // ------------------------------------------------------------------------------- TMA producer (both CTAs)
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&a.tmA) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&a.tmB) : "memory");
            int s = 0;
            uint32_t ph = 0;
            for (int t = cl; t < tiles_total; t += ncl) {
                const int mb = t % a.m_blocks, nb = t / a.m_blocks;
                const int row0 = mb * 256 + (int)rank * kBlockM;
                const int pn = a.pn, hn = pn >> 1;
                const int wrow0 = a.silu_F > 0 ? nb * kHalfN + (int)rank * a.silu_F : nb * pn + (int)rank * hn;
                for (int kb = 0; kb < a.k_blocks; kb++) {
                    mbar_wait(&a_empty[s], ph ^ 1u);
                    uint8_t *dst = sSlot + (size_t)s * kSlotBytes;
                    if (leader) mbar_arrive_expect_tx(&a_full[s], 2 * (kABytes + hn * 128));
                    tma_load_2d_pair(dst, &a.tmA, kb * 64, row0, &a_full[s]);
                    tma_load_2d_pair(dst + kABytes, &a.tmB, kb * 64, wrow0, &a_full[s]);
                    if (++s == AS) {
                        s = 0;
                        ph ^= 1u;
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ------------------------------------------------------------------------------- MMA issuer (leader CTA only)
        if (leader && lane == 0) {
            const uint32_t idesc = (1u << 4) | ((uint32_t)(a.pn >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);  // F32 acc, f16 x f16, K-major, N, M 256
            int s = 0, it = 0;
            uint32_t ph = 0;
            for (int t = cl; t < tiles_total; t += ncl, it++) {
                const int acc = it & 1;
                const uint32_t acc_ph = (uint32_t)(it >> 1) & 1u;
                mbar_wait_cl(&tempty_bar[acc], acc_ph ^ 1u);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(acc * kPairN);
                for (int kb = 0; kb < a.k_blocks; kb++) {
                    mbar_wait(&a_full[s], ph);
                    tc_fence_after();
                    const uint64_t adesc = make_sw128_desc(smem_u32(sSlot + (size_t)s * kSlotBytes));
                    const uint64_t bdesc = make_sw128_desc(smem_u32(sSlot + (size_t)s * kSlotBytes + kABytes));
#pragma unroll
                    for (int k = 0; k < 4; k++) umma_pair(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
                    umma_commit_pair(&a_empty[s]);
                    if (++s == AS) {
                        s = 0;
                        ph ^= 1u;
                    }
                }
                umma_commit_pair(&tfull_bar[acc]);
            }
        }
        __syncwarp();
    } else {
        // ------------------------------------------------------------------------------- epilogue (both CTAs, own accumulator rows)
        const int q = warp & 3;
        int it = 0;
        for (int t = cl; t < tiles_total; t += ncl, it++) {
            const int mb = t % a.m_blocks, nb = t / a.m_blocks;
            const int acc = it & 1;
            const uint32_t acc_ph = (uint32_t)(it >> 1) & 1u;
            mbar_wait(&tfull_bar[acc], acc_ph);
            tc_fence_after();
            const int row = mb * 256 + (int)rank * kBlockM + q * 32 + lane;
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * kPairN);
            if (a.silu_F > 0) {
                // accumulator columns 0..127 = gate, 128..255 = up of output channels nb * 128 ..: act = SiLU(gate) * up
#pragma unroll 1
                for (int c = 0; c < kHalfN / 32; c++) {
                    uint32_t g[32], u[32];
                    tmem_ld32(taddr + (uint32_t)(c * 32), g);
                    tmem_ld32(taddr + (uint32_t)(kHalfN + c * 32), u);
                    tmem_ld_wait();
                    const int col0 = nb * kHalfN + c * 32;
                    if (row < a.M && col0 < a.silu_F) {
                        __half *dst = reinterpret_cast<__half *>(a.C) + (size_t)row * a.ldc + col0;
                        uint32_t o[16];
#pragma unroll
                        for (int i = 0; i < 16; i++) {
                            const float g0 = __uint_as_float(g[2 * i]), g1 = __uint_as_float(g[2 * i + 1]);
                            o[i] = pack_half2((g0 / (1.f + __expf(-g0))) * __uint_as_float(u[2 * i]), (g1 / (1.f + __expf(-g1))) * __uint_as_float(u[2 * i + 1]));
                        }
#pragma unroll
                        for (int i = 0; i < 4; i++) reinterpret_cast<uint4 *>(dst)[i] = make_uint4(o[4 * i], o[4 * i + 1], o[4 * i + 2], o[4 * i + 3]);
                    }
                }
                tc_fence_before();
                mbar_arrive_cluster(&tempty_bar[acc], 0);
                continue;
            }
            const int pn = a.pn;
#pragma unroll 1
            for (int c = 0; c < pn / 32; c++) {
                uint32_t v[32];
                tmem_ld32(taddr + (uint32_t)(c * 32), v);
                tmem_ld_wait();
                const int col0 = nb * pn + c * 32;
                if (row < a.M && col0 < a.N) {
                    const int n = min(32, a.N - col0);
                    if (a.add_f32) {
                        float *dst = reinterpret_cast<float *>(a.C) + (size_t)row * a.ldc + col0;
                        if (n == 32 && (a.ldc & 3) == 0) {
#pragma unroll
                            for (int i = 0; i < 8; i++) {
                                float4 cc = reinterpret_cast<float4 *>(dst)[i];
                                cc.x += __uint_as_float(v[4 * i + 0]);
                                cc.y += __uint_as_float(v[4 * i + 1]);
                                cc.z += __uint_as_float(v[4 * i + 2]);
                                cc.w += __uint_as_float(v[4 * i + 3]);
                                reinterpret_cast<float4 *>(dst)[i] = cc;
                            }
                        } else {
#pragma unroll
                            for (int i = 0; i < 32; i++)
                                if (i < n) dst[i] += __uint_as_float(v[i]);
                        }
                    } else {
                        __half *dst = reinterpret_cast<__half *>(a.C) + (size_t)row * a.ldc + col0;
                        if (n == 32 && (a.ldc & 7) == 0) {
#pragma unroll
                            for (int i = 0; i < 4; i++) {
                                uint4 o;
                                o.x = pack_half2(__uint_as_float(v[8 * i + 0]), __uint_as_float(v[8 * i + 1]));
                                o.y = pack_half2(__uint_as_float(v[8 * i + 2]), __uint_as_float(v[8 * i + 3]));
                                o.z = pack_half2(__uint_as_float(v[8 * i + 4]), __uint_as_float(v[8 * i + 5]));
                                o.w = pack_half2(__uint_as_float(v[8 * i + 6]), __uint_as_float(v[8 * i + 7]));
                                reinterpret_cast<uint4 *>(dst)[i] = o;
                            }
                        } else {
#pragma unroll
                            for (int i = 0; i < 32; i++)
                                if (i < n) dst[i] = __float2half_rn(__uint_as_float(v[i]));
                        }
                    }
                }
            }
            tc_fence_before();
            mbar_arrive_cluster(&tempty_bar[acc], 0);  // the leader's MMA thread may overwrite this accumulator (in both CTAs)
        }
    }
    tc_fence_before();
    cluster_sync_all();  // both CTAs are done with TMEM and with each other's shared memory
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc_pair(tmem_base, 512);
    }
}

// W4 -> fp16 expansion: // one thread per 32-bit word (8 sequential nibbles, weights 8c..8c+7 of row o) -> one 16-byte store
__global__ void w4_expand_kernel(const uint32_t *__restrict__ w, const uint32_t *__restrict__ zeros, const __half *__restrict__ scales, __half *__restrict__ out,
                                 int OC, int words_per_row, int zeros_w, int sf_w) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)OC * words_per_row) return;
    const int o = (int)(idx / words_per_row), c = (int)(idx % words_per_row);
    const int g = c >> 4;  // 16 words = 128 weights per group
    const uint32_t z = (zeros[(size_t)o * zeros_w + (g >> 3)] >> (4 * (g & 7))) & 0xFu;
    const __half s = scales[(size_t)o * sf_w + g];
    const __half2 s2 = __half2half2(s);
    const uint32_t zmagic = 0x64006400u | z | (z << 16);  // (1024 + z) in both halves
    const uint32_t word = w[idx];
    uint32_t r[4];
#pragma unroll
    for (int p = 0; p < 4; p++) {
        const uint32_t x = word >> (8 * p);
        const uint32_t qmagic = 0x64006400u | (x & 0xFu) | ((x & 0xF0u) << 12);  // (1024 + q) for weights 2p, 2p+1
        const __half2 d = __hsub2(*reinterpret_cast<const __half2 *>(&qmagic), *reinterpret_cast<const __half2 *>(&zmagic));  // exact
        const __half2 m = __hmul2(d, s2);                                                                                     // one rounding
        r[p] = *reinterpret_cast<const uint32_t *>(&m);
    }
    reinterpret_cast<uint4 *>(out)[idx] = make_uint4(r[0], r[1], r[2], r[3]);
}

typedef CUresult (*EncodeFn2)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                              const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeFn2 encoder2() {
    static EncodeFn2 fn = nullptr;
    if (!fn) {
        void *sym = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess && sym) fn = reinterpret_cast<EncodeFn2>(sym);
    }
    return fn;
}

bool encode_f16(CUtensorMap *out, const void *base, long long rows, long long K, long long ld, int box_rows = 128) {
    const cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {(cuuint64_t)(ld * 2)};
    const cuuint32_t box[2] = {64u, (cuuint32_t)box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return encoder2()(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void *>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

cudaError_t launch_pair(Ctx *ctx, PairArgs &a) {
    static DeviceOnce attr_once;
    if (attr_once.pending(ctx->device)) {
        cudaError_t e = cudaFuncSetAttribute(gemm_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPairSmem);
        if (e != cudaSuccess) return e;
        attr_once.done(ctx->device);
    }
    const int tiles = a.m_blocks * a.n_blocks;
    int clusters = ctx->num_sms / 2;
    if (clusters > tiles) clusters = tiles;
    gemm_pair_kernel<<<2 * clusters, kPairThreads, kPairSmem, ctx->stream>>>(a);
    return cudaGetLastError();
}

}  // namespace

cudaError_t w4_scratch_reserve(Ctx *ctx, size_t elems) {
    if (ctx->w16_scratch_elems >= elems) return cudaSuccess;
    if (ctx->w16_scratch) {  // rare: grows to the largest weight matrix seen (cudaFree synchronises)
        cudaError_t e = cudaFree(ctx->w16_scratch);
        ctx->w16_scratch = nullptr;
        ctx->w16_scratch_elems = 0;
        if (e != cudaSuccess) return e;
    }
    cudaError_t e = cudaMalloc(&ctx->w16_scratch, elems * sizeof(__half));
    if (e == cudaSuccess) ctx->w16_scratch_elems = elems;
    return e;
}

cudaError_t launch_w4_expand(Ctx *ctx, const uint32_t *w, const uint32_t *zeros, const __half *scales, __half *out, int OC, int IC) {
    const int wpr = IC / 8, zw = zeros_width(IC, kW4Group);
    const long long n = (long long)OC * wpr;
    w4_expand_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(w, zeros, scales, out, OC, wpr, zw, zw * 8);
    return cudaGetLastError();
}

// W fp16 [N][K] (ldw elements between rows)
cudaError_t launch_gemm_f16_pair(Ctx *ctx, const __half *X, long long ldx, const __half *W, long long ldw, void *C, long long ldc, int M, int N, int K, int add_f32) {
    if (M < 1 || N < 1 || K < 64 || (K % 64) || (ldx % 8) || (ldw % 8) || !encoder2()) return cudaErrorInvalidValue;
    PairArgs a = {};
    a.M = M;
    a.N = N;
    a.k_blocks = K / 64;
    a.m_blocks = (M + 255) / 256;
    // tile width by wave quantisation over the clusters: rounds x width (x a small penalty for the narrower tile: the activation tile is re-read per N block)
    const int clusters = ctx->num_sms / 2;
    auto cost = [&](int pn, double pen) {
        const long long tiles = (long long)a.m_blocks * ((N + pn - 1) / pn);
        return (double)((tiles + clusters - 1) / clusters) * pn * pen;
    };
    // measured: 128-wide tiles run at 0.70 of the 256-wide rate per FLOP (the activation tile is read twice as often from shared memory), which
    // costs more than the wave quantisation it removes (13B o / down: 919 / 973 -> 640 / 673 TFLOP/s): a penalty of 1.45 keeps them for tiny N only
    a.pn = cost(128, 1.45) < cost(256, 1.0) ? 128 : 256;
    if (!encode_f16(&a.tmA, X, M, K, ldx) || !encode_f16(&a.tmB, W, N, K, ldw, a.pn / 2)) return cudaErrorInvalidValue;
    a.n_blocks = (N + a.pn - 1) / a.pn;
    a.C = C;
    a.ldc = ldc;
    a.add_f32 = add_f32;
    return launch_pair(ctx, a);
}

// act[M][F] = SiLU(X Wg^T) * (X Wu^T), W = fp16 [2F][K] with the gate rows first; F % 128 == 0, ldc % 8 == 0
cudaError_t launch_gemm_f16_pair_silu(Ctx *ctx, const __half *X, long long ldx, const __half *W, long long ldw, __half *act, long long ldc, int M, int F, int K) {
    if (M < 1 || F < 128 || (F % kHalfN) || K < 64 || (K % 64) || (ldx % 8) || (ldw % 8) || (ldc % 8) || !encoder2()) return cudaErrorInvalidValue;
    PairArgs a = {};
    if (!encode_f16(&a.tmA, X, M, K, ldx) || !encode_f16(&a.tmB, W, 2LL * F, K, ldw)) return cudaErrorInvalidValue;
    a.M = M;
    a.N = F;
    a.k_blocks = K / 64;
    a.m_blocks = (M + 255) / 256;
    a.n_blocks = F / kHalfN;
    a.C = act;
    a.ldc = ldc;
    a.pn = kPairN;
    a.silu_F = F;
    return launch_pair(ctx, a);
}

}  // namespace tce
