// gemm_tc.cuh -- the large-M int8 GEMM of the path on the 5th-generation tensor cores:  C[M][N] = A[M][K] * B[N][K]^T with both operands
// K-major, which is the natural layout of the activations ([tokens][IC]) and of the weights ([OC][IC]) on this path.
//
//   * operands reach shared memory by 2-D TMA (128-byte swizzle, one 128-byte swizzle atom of K = 128 int8 per stage row),
//   * one elected thread issues tcgen05.mma.kind::i8 (cta_group::1, M = 128, N = BLOCK_N, K = 32 per instruction) straight from the
//     swizzled tiles through shared-memory matrix descriptors,
//   * the int32 accumulator lives in TMEM, double buffered (2 x BLOCK_N columns), so the epilogue of tile i overlaps the
//     main loop of tile i+1,
//   * four epilogue warps read their 32-lane quarter of TMEM with tcgen05.ld and apply the op's epilogue in registers.
// Persistent: one CTA per SM walks tiles m-fastest so that concurrently running CTAs share the same B (weight) tile in L2.
//
// Roles (6 warps): warp 0 = TMA producer, warp 1 = TMEM owner + MMA issuer, warps 2-5 = epilogue (warp w owns TMEM lanes
// 32*(w%4)..+31, the hardware's lane-quarter rule for tcgen05.ld).
#pragma once
#include <cuda.h>

#include "common.cuh"

namespace tce {
namespace tc {

constexpr int kBlockM = 128;
constexpr int kAtomBytes = 128;  // bytes of K per row per stage = one SWIZZLE_128B atom
constexpr int kThreads = 192;
constexpr int kABytes = kBlockM * kAtomBytes;  // 16 KiB

struct GemmArgs {
    alignas(64) CUtensorMap tmA;  // [M][K] box {128 B, 128 rows}
    alignas(64) CUtensorMap tmB;  // [N][K] box {128 B, BLOCK_N rows}
    int M, N;
    int k_blocks;                 // K / 128
    int m_blocks, n_blocks;
    // epilogue
    void *C;
    long long ldc;                // elements between output rows
    const int8_t *bias8;
    const float *biasf;
    float alpha, beta;
    int q_min, q_max;
};

TCE_DEVINL void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
TCE_DEVINL void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
TCE_DEVINL void tmem_alloc(uint32_t *dst_smem, uint32_t ncols) {  // whole warp
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
TCE_DEVINL void tmem_dealloc(uint32_t taddr, uint32_t ncols) {  // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// all previously issued tcgen05.mma of this thread complete -> one arrival on `bar` (implies fence::before_thread_sync)
TCE_DEVINL void umma_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
TCE_DEVINL void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d), "l"(adesc),
                 "l"(bdesc), "r"(idesc), "r"(accumulate)
                 : "memory");
}
// 32 lanes x 32 consecutive 32-bit columns: thread t of the warp receives row (lane quarter base + t), columns c..c+31
TCE_DEVINL void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, "
        "%23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]),
          "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]),
          "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
TCE_DEVINL void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

TCE_DEVINL void tma_load_2d(void *dst_smem, const void *tmap, int x, int y, uint64_t *bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(smem_u32(dst_smem)),
                 "l"(tmap), "r"(x), "r"(y), "r"(smem_u32(bar))
                 : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (sm_100 format): start address >> 4 in bits [0,14), leading byte offset
// (unused for swizzled K-major, set to 1) in [16,30), stride byte offset = 8 rows * 128 B = 1024 B (>> 4) in [32,46), version 1 in
// [46,48), layout type 2 (SWIZZLE_128B) in [61,64).  Tiles are 1024-byte aligned, so base_offset stays 0.
TCE_DEVINL uint64_t make_sw128_desc(uint32_t smem_addr) {
    const uint32_t lo = ((smem_addr >> 4) & 0x3FFFu) | (1u << 16);
    const uint32_t hi = 64u | (1u << 14) | (2u << 29);
    return ((uint64_t)hi << 32) | lo;
}

// instruction descriptor: c_format [4,6) (2 = S32), a_format [7,10), b_format [10,13) (INT8 signed = 1),
// a/b major bits 15/16 = 0 (K-major), N >> 3 in [17,23), M >> 4 in [24,29)
template <int BLOCK_N>
constexpr uint32_t make_idesc_i8() {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BLOCK_N >> 3) << 17) | ((uint32_t)(kBlockM >> 4) << 24);
}

template <int BLOCK_N, int STAGES>
constexpr size_t smem_bytes() {
    return 1024 + (size_t)STAGES * (kABytes + BLOCK_N * kAtomBytes);
}

// Epi::apply(args, row, col0, ncols_valid, v[32]) consumes 32 consecutive accumulator columns of one output row.
template <int BLOCK_N, int STAGES, class Epi>
__global__ void __launch_bounds__(kThreads, 1) gemm_tc_kernel(const __grid_constant__ GemmArgs a) {
    static_assert(BLOCK_N == 128 || BLOCK_N == 192 || BLOCK_N == 256, "BLOCK_N");
    constexpr int kBBytes = BLOCK_N * kAtomBytes;
    constexpr uint32_t kTmemCols = BLOCK_N == 128 ? 256 : 512;  // two accumulators; allocations are powers of two
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t full_bar[STAGES], empty_bar[STAGES], tfull_bar[2], tempty_bar[2];
    __shared__ uint32_t tmem_base_s;

    const uint32_t raw = smem_u32(smem_raw);
    uint8_t *tiles = smem_raw + (((raw + 1023u) & ~1023u) - raw);  // SWIZZLE_128B tiles need 1024-byte alignment
    uint8_t *sA = tiles, *sB = tiles + (size_t)STAGES * kABytes;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tiles_total = a.m_blocks * a.n_blocks;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; s++) {
            mbar_init(&full_bar[s], 1);
            mbar_init(&empty_bar[s], 1);
        }
        for (int s = 0; s < 2; s++) {
            mbar_init(&tfull_bar[s], 1);
            mbar_init(&tempty_bar[s], 128);
        }
        mbar_fence_init();
    }
    if (warp == 1) tmem_alloc(&tmem_base_s, kTmemCols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;

    if (warp == 0) {
        // ------------------------------------------------------------------------------- TMA producer
        if (lane == 0) {
            asm volatile("prefetch.tensormap [%0];" ::"l"(&a.tmA) : "memory");
            asm volatile("prefetch.tensormap [%0];" ::"l"(&a.tmB) : "memory");
            int s = 0;
            uint32_t ph = 0;
            for (int t = blockIdx.x; t < tiles_total; t += gridDim.x) {
                const int mb = t % a.m_blocks, nb = t / a.m_blocks;
                for (int kb = 0; kb < a.k_blocks; kb++) {
                    mbar_wait(&empty_bar[s], ph ^ 1u);
                    mbar_arrive_expect_tx(&full_bar[s], kABytes + kBBytes);
                    const int kx = kb * kAtomBytes;  // element coordinate along K
                    tma_load_2d(sA + (size_t)s * kABytes, &a.tmA, kx, mb * kBlockM, &full_bar[s]);
                    tma_load_2d(sB + (size_t)s * kBBytes, &a.tmB, kx, nb * BLOCK_N, &full_bar[s]);
                    if (++s == STAGES) {
                        s = 0;
                        ph ^= 1u;
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ------------------------------------------------------------------------------- MMA issuer
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc_i8<BLOCK_N>();
            int s = 0;
            uint32_t ph = 0;
            int it = 0;
            for (int t = blockIdx.x; t < tiles_total; t += gridDim.x, it++) {
                const int acc = it & 1;
                const uint32_t acc_ph = (uint32_t)(it >> 1) & 1u;
                mbar_wait(&tempty_bar[acc], acc_ph ^ 1u);  // epilogue has drained this accumulator
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BLOCK_N);
                for (int kb = 0; kb < a.k_blocks; kb++) {
                    mbar_wait(&full_bar[s], ph);
                    tc_fence_after();
                    const uint64_t adesc = make_sw128_desc(smem_u32(sA + (size_t)s * kABytes));
                    const uint64_t bdesc = make_sw128_desc(smem_u32(sB + (size_t)s * kBBytes));
#pragma unroll
                    for (int k = 0; k < kAtomBytes / 32; k++)  // 32 bytes of K per instruction; +2 in the (>>4) address field
                        umma_i8(tmem_d, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, (kb | k) != 0 ? 1u : 0u);
                    umma_commit(&empty_bar[s]);  // smem slot reusable once these MMAs have read it
                    if (++s == STAGES) {
                        s = 0;
                        ph ^= 1u;
                    }
                }
                umma_commit(&tfull_bar[acc]);  // accumulator complete
            }
        }
        __syncwarp();
    } else {
        // ------------------------------------------------------------------------------- epilogue
        const int q = warp & 3;  // TMEM lane quarter this warp may read
        int it = 0;
        for (int t = blockIdx.x; t < tiles_total; t += gridDim.x, it++) {
            const int mb = t % a.m_blocks, nb = t / a.m_blocks;
            const int acc = it & 1;
            const uint32_t acc_ph = (uint32_t)(it >> 1) & 1u;
            mbar_wait(&tfull_bar[acc], acc_ph);
            tc_fence_after();
            const int row = mb * kBlockM + q * 32 + lane;
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(acc * BLOCK_N);
#pragma unroll 1
            for (int c = 0; c < BLOCK_N / 32; c++) {
                uint32_t v[32];
                tmem_ld32(taddr + (uint32_t)(c * 32), v);
                tmem_ld_wait();
                const int col0 = nb * BLOCK_N + c * 32;
                if (row < a.M && col0 < a.N) Epi::apply(a, row, col0, min(32, a.N - col0), v);
            }
            tc_fence_before();
            mbar_arrive(&tempty_bar[acc]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem_base, kTmemCols);
    }
}

}  // namespace tc
}  // namespace tce
