// decode_persistent.cu -- one persistent cooperative kernel per decoded token (Llama, AWQ-INT4, batch 1) on sm_100a.
//
// Call sites restated (reference, CUDA build): Int4LlamaForCausalLM::forward (cuda/Int4llamaForCausalLM.cu:17-50) ->
// Int4llamaDecoder::forward (cuda/Int4llamaDecoder.cu:57-112) -> 32 x Int4llamaDecoderLayer::forward (cuda/Int4llamaDecoderLayer.cu:73-115)
// -> Int4llamaAttention::forward (cuda/Int4llamaAttention.cu:116-229): ~19 kernels + 128 memcpys per layer on stream 0.  Here the whole
// token is ONE kernel of one CTA per SM whose warp roles persist across all phases (5 per layer + lm_head):
//
//   producer (1 warp, 1 elected lane)  walks the phases in order and keeps a ring of `nst` TMA stages full.  A stage is either
//        [16 rows x <=32 groups] of packed int4 weights (two 2-D UTMALDG boxes of 16 KiB) + the stage's repacked scales|zeros record (one
//        1280 B UBLKCP), or 64 cached K rows + 64 cached V rows of the attention phase (four 128B-swizzled 2-D boxes).  It depends on
//        nothing but static data and the token position, so it runs ahead across every phase boundary.
//   consumers (16 warps)  per phase: spin on the flag-carrying words of their input vector, quantise it (fused RMSNorm, four int8 planes
//        per 128-group), run the integer-MMA GEMV over this CTA's tiles (two 128-k groups per warp and stage), or run flash-decoding
//        attention straight out of the ring stages (mma.sync m16n8k16, ldmatrix on the swizzled K/V rows).
//   epilogue (1 warp)  reduces the 16 consumer partials of every tile and publishes the results as {value, phase tag} words.
//
// There is NO grid barrier between phases.  Every vector that crosses CTAs (q|k|v, attention partials and outputs, SiLU*mul
// activations, the o_proj / down_proj outputs) is an array of 8-byte words {payload, tag} written with one 8-byte store and read with
// 8/16-byte loads: a reader spins until the tag of the phase it waits for appears, so the hand-off costs one L2 write + one L2 read
// instead of fence + arrive + poll + fence.  The fp32 residual stream never leaves the SM: every CTA keeps its own copy in shared
// memory and adds the (identical) o_proj / down_proj outputs to it in the same order -- which is also the tensor-parallel
// all-reduce: with P ranks every rank stores its partial outputs into slot `rank` of every rank's buffer (NVLink peer stores of
// 8-byte words, flag included) and every reader sums the P slots in rank order.
// All waits are bounded: a protocol bug surfaces as a launch failure within seconds, not as a hung GPU.
#include <stdio.h>

#include "attention_impl.cuh"
#include "persistent.h"
#include "w4a16_gemv_impl.cuh"

namespace tce {
namespace pk {

namespace {

// ------------------------------------------------------------------------------------------------------------ small helpers
TCE_DEVINL unsigned ld_acquire_gpu(const unsigned *p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
TCE_DEVINL void red_release_gpu(unsigned *p) { asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(p) : "memory"); }

// {payload, tag} words.  8-byte aligned 8-byte accesses are single transactions: payload and tag always travel together.
TCE_DEVINL void st_ll(uint2 *p, uint32_t data, uint32_t tag, bool sys) {
    if (sys)
        asm volatile("st.relaxed.sys.global.v2.b32 [%0], {%1, %2};" ::"l"(p), "r"(data), "r"(tag) : "memory");
    else
        asm volatile("st.relaxed.gpu.global.v2.b32 [%0], {%1, %2};" ::"l"(p), "r"(data), "r"(tag) : "memory");
}
TCE_DEVINL uint4 ld_ll2(const uint2 *p, bool sys) {  // two consecutive words (16-byte aligned)
    uint4 r;
    if (sys)
        asm volatile("ld.relaxed.sys.global.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
    else
        asm volatile("ld.relaxed.gpu.global.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p) : "memory");
    return r;
}
TCE_DEVINL uint2 ld_ll1(const uint2 *p, bool sys) {
    uint2 r;
    if (sys)
        asm volatile("ld.relaxed.sys.global.v2.b32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p) : "memory");
    else
        asm volatile("ld.relaxed.gpu.global.v2.b32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p) : "memory");
    return r;
}
// A failed poll waits this long before it asks L2 again: thousands of threads spinning without a pause fill the L2 request queues and
// stretch every round trip (their own and the producers' stores) to ~0.5 us (profiles/README.md, run 11).
// Back-off 0 / 30 / 100 / 250 ns on one B200: 652 / 652 / 651 / 643 tok/s (profiles/README.md).
constexpr unsigned kPollBackoffNs = 100;
constexpr long long kSpinLimit = 20000000000LL;  // ~10 s: a peer rank may legitimately start its kernel later
// spin until both words of the pair carry `tag`
TCE_DEVINL uint4 wait_ll2(const uint2 *p, uint32_t tag, bool sys) {
    uint4 r = ld_ll2(p, sys);
    if (r.y == tag && r.w == tag) return r;
    const long long t0 = clock64();
    while (true) {
        __nanosleep(kPollBackoffNs);
        r = ld_ll2(p, sys);
        if (r.y == tag && r.w == tag) return r;
        if (clock64() - t0 > kSpinLimit) __trap();
    }
}
TCE_DEVINL uint32_t wait_ll1(const uint2 *p, uint32_t tag, bool sys) {
    uint2 r = ld_ll1(p, sys);
    if (r.y == tag) return r.x;
    const long long t0 = clock64();
    while (true) {
        __nanosleep(kPollBackoffNs);
        r = ld_ll1(p, sys);
        if (r.y == tag) return r.x;
        if (clock64() - t0 > kSpinLimit) __trap();
    }
}
// N consecutive 16-byte pairs: all loads are issued before the first tag is examined (one L2 round trip when the data is there)
template <int N>
TCE_DEVINL void wait_ll2xN(const uint2 *p, uint32_t tag, bool sys, uint4 (&r)[N]) {
    long long t0 = 0;
    while (true) {
        bool ok = true;
#pragma unroll
        for (int i = 0; i < N; i++) r[i] = ld_ll2(p + 2 * i, sys);
#pragma unroll
        for (int i = 0; i < N; i++) ok = ok && (r[i].y == tag) && (r[i].w == tag);
        if (ok) return;
        if (t0 == 0) t0 = clock64();
        if (clock64() - t0 > kSpinLimit) __trap();
        __nanosleep(kPollBackoffNs);
    }
}

TCE_DEVINL float2 h2_to_f2(uint32_t u) { return __half22float2(*reinterpret_cast<const __half2 *>(&u)); }

// shared-memory accesses by 32-bit shared address (no generic-address conversion inside the hot loops)
TCE_DEVINL uint4 lds_u4(uint32_t a) {
    uint4 r;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(a) : "memory");
    return r;
}
TCE_DEVINL uint2 lds_u2(uint32_t a) {
    uint2 r;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(r.x), "=r"(r.y) : "r"(a) : "memory");
    return r;
}
TCE_DEVINL uint32_t lds_u32(uint32_t a) {
    uint32_t r;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r) : "r"(a) : "memory");
    return r;
}
TCE_DEVINL float lds_f32(uint32_t a) { return __uint_as_float(lds_u32(a)); }
TCE_DEVINL uint32_t lds_u16(uint32_t a) {
    unsigned short r;
    asm volatile("ld.shared.u16 %0, [%1];" : "=h"(r) : "r"(a) : "memory");
    return (uint32_t)r;
}
TCE_DEVINL bool mbar_try_wait_u32(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
TCE_DEVINL void mbar_wait_u32(uint32_t bar, uint32_t parity) {
    if (mbar_try_wait_u32(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait_u32(bar, parity)) {
        if (clock64() - t0 > kSpinLimit) __trap();
    }
}
TCE_DEVINL void mbar_arrive_u32(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }

TCE_DEVINL int lds_volatile_i32(const int *p) {
    int v;
    asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(v) : "r"(smem_u32(p)) : "memory");
    return v;
}

TCE_DEVINL void stamp(const Args &a, int cta, int nphase, int p, int k) {  // one thread
    if (a.dbg) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        a.dbg[((size_t)cta * nphase + p) * 8 + k] = t;
    }
}

TCE_DEVINL unsigned long long argmax_key(float v, int idx) {
    unsigned b = __float_as_uint(v);
    b = (b & 0x80000000u) ? ~b : (b | 0x80000000u);  // monotone map float -> uint
    return ((unsigned long long)b << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)idx);  // ties: lowest index wins (arg_max.cc)
}

struct PSmem {
    uint8_t *ring;      // [nst][kStageBytes], 1024-B aligned
    uint8_t *xs;        // activation planes (4 * IC bytes) | attention scratch
    float *resid;       // [E] this CTA's copy of the fp32 residual stream
    float *gx;          // [max_ng] group steps
    int *gsum;          // [max_ng][2] group sums
    float *red;         // [kRedBufs][kCW][16] tile partials
    float *rms;         // [kCW]
    float *rope;        // cos[128] | sin[128] of the token position
    uint64_t *full, *empty, *red_full, *red_empty;
    uint64_t *rx;       // pair staging: counts the bytes the partner has mirrored into this CTA for the current staging
    int *free_gen;      // pair staging: written by the partner: the number of phases it has finished (its buffers may be overwritten)
    uint32_t ring_u32, xs_u32, gx_u32, gsum_u32, full_u32, empty_u32, redfull_u32, redempty_u32;
    int nst;
};

TCE_DEVINL PSmem carve(uint8_t *raw, const Args &a) {
    PSmem s;
    uint8_t *base = raw + ((1024u - (smem_u32(raw) & 1023u)) & 1023u);
    s.nst = a.nst;
    s.ring = base;
    uint8_t *p = base + (size_t)a.nst * kStageBytes;
    s.xs = p;
    p += a.xs_bytes;
    s.resid = reinterpret_cast<float *>(p);
    p += (size_t)a.E * 4;
    s.gx = reinterpret_cast<float *>(p);
    p += (size_t)a.max_ng * 4;
    s.gsum = reinterpret_cast<int *>(p);
    p += (size_t)a.max_ng * 8;
    s.red = reinterpret_cast<float *>(p);
    p += (size_t)kRedBufs * kCW * 16 * 4;
    s.rms = reinterpret_cast<float *>(p);
    p += 32 * 4;
    s.rope = reinterpret_cast<float *>(p);
    p += 256 * 4;
    s.full = reinterpret_cast<uint64_t *>(p);
    s.empty = s.full + a.nst;
    s.red_full = s.empty + a.nst;
    s.red_empty = s.red_full + kRedBufs;
    s.rx = s.red_empty + kRedBufs;
    s.free_gen = reinterpret_cast<int *>(s.rx + 1);
    s.ring_u32 = smem_u32(s.ring);
    s.xs_u32 = smem_u32(s.xs);
    s.gx_u32 = smem_u32(s.gx);
    s.gsum_u32 = smem_u32(s.gsum);
    s.full_u32 = smem_u32(s.full);
    s.empty_u32 = smem_u32(s.empty);
    s.redfull_u32 = smem_u32(s.red_full);
    s.redempty_u32 = smem_u32(s.red_empty);
    return s;
}

struct Ring {
    int stage = 0;
    uint32_t phase = 0;
    TCE_DEVINL void advance(int nst) {
        if (++stage == nst) {
            stage = 0;
            phase ^= 1;
        }
    }
};
struct Red {
    int rb = 0;
    uint32_t rphase = 0;
    TCE_DEVINL void advance() {
        if (++rb == kRedBufs) {
            rb = 0;
            rphase ^= 1;
        }
    }
};

// this CTA's tile range of one GEMV op: cut at tile boundaries (every output has exactly one writer)
TCE_DEVINL void partition(const GemvOp &op, int cta, int ncta, int &t0, int &t1) {
    const unsigned T = (unsigned)op.num_tiles;
    t0 = (int)((T * (unsigned)cta) / (unsigned)ncta);
    t1 = (int)((T * (unsigned)(cta + 1)) / (unsigned)ncta);
}

// attention work split: the visible positions [0, T) in chunks of kKvChunk; every KV head gets NS = #CTAs / KVH consecutive CTAs,
// each takes `cps` consecutive chunks (the fewest that cover the context: see kAttnCps)
struct AttnSplit {
    int kvh, split, ch0, ch1, nsplit;  // ch0 >= ch1: nothing to do
};
TCE_DEVINL AttnSplit attn_split(int cta, int ncta, int KVH, int pos) {
    AttnSplit s;
    const int T = pos + 1;
    const int nch = (T + kKvChunk - 1) / kKvChunk;
    int NS = ncta / KVH;
    if (NS < 1) NS = 1;
    int cps = (nch + NS - 1) / NS;
    const int want = nch < kAttnCps ? nch : kAttnCps;
    if (cps < want) cps = want;
    if (cps * 32 < nch) cps = (nch + 31) / 32;  // the split merge keeps one split per lane
    s.nsplit = (nch + cps - 1) / cps;
    s.kvh = cta / NS;
    s.split = cta - s.kvh * NS;
    if (s.kvh >= KVH || s.split >= s.nsplit) {
        s.ch0 = s.ch1 = 0;
        s.kvh = 0;
    } else {
        s.ch0 = s.split * cps;
        s.ch1 = min(nch, s.ch0 + cps);
    }
    return s;
}

// ------------------------------------------------------------------------------------------------------------ producer
// The loader walks (tile, stage, box) in consumption order and moves every stage into the ring as soon as its slot is free.
TCE_DEVINL void produce_gemv(const GemvOp &op, const CUtensorMap *m0, const uint8_t *meta, const PSmem &sm, Ring &rs, int cta, int ncta, uint32_t leader,
                             uint64_t policy) {
    int t0, t1;
    partition(op, cta, ncta, t0, t1);
    const bool ragged = (op.NG % kStageGroups) != 0;
    for (int tile = t0; tile < t1; tile++) {
        for (int s = 0; s < op.S; s++) {
            const BoxPlan &pl = op.plan[(ragged && s == op.S - 1) ? 1 : 0];
            mbar_wait(&sm.empty[rs.stage], rs.phase ^ 1);
            uint64_t *bar = &sm.full[rs.stage];
            uint8_t *dst = sm.ring + (size_t)rs.stage * kStageBytes;
            mbar_arrive_expect_tx_pred(bar, (uint32_t)pl.bytes + kMetaBytes, leader);
#pragma unroll 1
            for (int b = 0; b < pl.nbox; b++) {
                const int xw = (kStageGroups * s + pl.b0[b]) * 16;  // first 32-bit word of the box within the row
                uint8_t *d = dst + pl.off[b];
                if (op.pair) {  // matrices of an op are kMapsPerMat maps apart
                    if (op.unit) {
                        tma_load_3d_pred(d, m0 + pl.map[b], 0, tile * 8, xw >> 4, bar, policy, leader);
                        tma_load_3d_pred(d + 8 * pl.bw[b] * 64, m0 + kMapsPerMat + pl.map[b], 0, tile * 8, xw >> 4, bar, policy, leader);
                    } else {
                        tma_load_2d_pred(d, m0 + pl.map[b], xw, tile * 8, bar, policy, leader);
                        tma_load_2d_pred(d + 8 * pl.bw[b] * 64, m0 + kMapsPerMat + pl.map[b], xw, tile * 8, bar, policy, leader);
                    }
                } else {
                    int row = tile * 16;
                    const CUtensorMap *m = m0;
                    if (op.nseg > 1 && row >= op.rows0) {
                        row -= op.rows0;
                        m = m0 + kMapsPerMat;
                        if (op.nseg > 2 && row >= op.rows1) {
                            row -= op.rows1;
                            m = m0 + 2 * kMapsPerMat;
                        }
                    }
                    if (op.unit)
                        tma_load_3d_pred(d, m + pl.map[b], 0, row, xw >> 4, bar, policy, leader);
                    else
                        tma_load_2d_pred(d, m + pl.map[b], xw, row, bar, policy, leader);
                }
            }
            const uint8_t *mrec = meta + ((size_t)tile * op.S + s) * kMetaBytes;
            bulk_g2s_pred(dst + kMetaOff, mrec, kMetaBytes, bar, policy, leader);
            __syncwarp();
            rs.advance(sm.nst);
        }
    }
}

TCE_DEVINL void produce_attn(const Args &a, const LayerDesc &L, const CUtensorMap *kvmap, const PSmem &sm, Ring &rs, int cta, int ncta, int pos,
                             uint32_t leader, uint64_t policy) {
    const AttnSplit sp = attn_split(cta, ncta, a.KVH, pos);
    for (int c = sp.ch0; c < sp.ch1; c++) {
        mbar_wait(&sm.empty[rs.stage], rs.phase ^ 1);
        uint64_t *bar = &sm.full[rs.stage];
        uint8_t *dst = sm.ring + (size_t)rs.stage * kStageBytes;
        const int krow = L.k_row0 + sp.kvh * a.max_ctx + c * kKvChunk, vrow = L.v_row0 + sp.kvh * a.max_ctx + c * kKvChunk;
        mbar_arrive_expect_tx_pred(bar, 2u * kHalfBytes, leader);
        tma_load_2d_pred(dst, kvmap, 0, krow, bar, policy, leader);
        tma_load_2d_pred(dst + 8192, kvmap, 64, krow, bar, policy, leader);
        tma_load_2d_pred(dst + kHalfBytes, kvmap, 0, vrow, bar, policy, leader);
        tma_load_2d_pred(dst + kHalfBytes + 8192, kvmap, 64, vrow, bar, policy, leader);
        __syncwarp();
        rs.advance(sm.nst);
    }
}

// the producer role (warp 0)
TCE_DEVINL void producer_walk(const Args &a, const PSmem &sm, int cta, int ncta, int pos, int lane) {
    Ring rs;
    const uint64_t policy = l2_policy_evict_first();
    const uint32_t leader = (lane == 0) ? 1u : 0u;
    const int Lyr = a.num_layers, nphase = 5 * Lyr + 1;
    const CUtensorMap *kvmap = a.maps + ((size_t)Lyr * 7 + 1) * kMapsPerMat;
#pragma unroll 1
    for (int p = 0; p < nphase; p++) {
        const int l = p / 5, k = p - 5 * l;
        if (l == Lyr) {
            produce_gemv(a.op[OPI_LMHEAD], a.maps + (size_t)Lyr * 7 * kMapsPerMat, a.lm_meta, sm, rs, cta, ncta, leader, policy);
        } else if (k == 1) {
            produce_attn(a, a.layers[l], kvmap, sm, rs, cta, ncta, pos, leader, policy);
        } else {
            const int oi = (k == 0) ? OPI_QKV : (k - 1);       // k = 2,3,4 -> OPI_O, OPI_GATEUP, OPI_DOWN
            const int mi = (k == 0) ? 0 : (k == 2 ? 3 : (k == 3 ? 4 : 6));  // first tensor map of the op within the layer's seven
            produce_gemv(a.op[oi], a.maps + ((size_t)l * 7 + mi) * kMapsPerMat, a.layers[l].meta[oi], sm, rs, cta, ncta, leader, policy);
        }
    }
}

// ------------------------------------------------------------------------------------------------------------ pair staging (clusters of two CTAs)
// Every CTA needs the whole quantised input vector of a GEMV phase.  In pair mode the two CTAs of a cluster split that work: CTA `rank` polls and
// quantises the 128-groups g = rank (mod 2) and mirrors planes / steps / sums into its partner with st.async (remote shared-memory stores that
// complete transaction bytes on the partner's `rx` mbarrier: no fence, no flag).  A CTA tells its partner when its buffers may be overwritten
// (`free_gen` = phases finished, a relaxed remote store: it only orders the partner's writes after this CTA's reads).
struct PairCtx {
    bool on = false;
    uint32_t rank = 0;
    gemv::PairDst dst = {0u, 0u, 0u, 0u};
    uint32_t r_rms = 0, r_free = 0;  // partner's rms[16..31] and free_gen
    uint32_t nstage = 0;             // stagings done so far (parity of the rx barrier)
};
TCE_DEVINL uint32_t map_to_cta(uint32_t local_u32, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_u32), "r"(rank));
    return r;
}
TCE_DEVINL void st_cluster_u32(uint32_t raddr, uint32_t v) { asm volatile("st.relaxed.cluster.shared::cluster.u32 [%0], %1;" ::"r"(raddr), "r"(v) : "memory"); }
// groups a CTA stages itself / expects from its partner
TCE_DEVINL int own_groups(const PairCtx &pc, int NG) { return pc.on ? (NG + 1 - (int)pc.rank) / 2 : NG; }
TCE_DEVINL int peer_groups(const PairCtx &pc, int NG) { return pc.on ? (NG + (int)pc.rank) / 2 : 0; }
// before the first mirrored store of phase p: the partner has finished phase p - 1 (it no longer reads the buffers this CTA writes into)
TCE_DEVINL void wait_partner_free(const PSmem &sm, const PairCtx &pc, int p) {
    if (!pc.on || p == 0) return;
    const long long t0 = clock64();
    while (lds_volatile_i32(sm.free_gen) < p) {
        if (clock64() - t0 > kSpinLimit) __trap();
    }
}
// arm the rx barrier for this staging (one thread) / wait for the partner's bytes (every consumer thread)
TCE_DEVINL void rx_expect(const PSmem &sm, const PairCtx &pc, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(sm.rx)), "r"(bytes) : "memory");
}
TCE_DEVINL void rx_wait(const PSmem &sm, PairCtx &pc) {
    mbar_wait_u32(smem_u32(sm.rx), pc.nstage & 1u);
    pc.nstage++;
}

// ------------------------------------------------------------------------------------------------------------ consumers: staging
// unit rotation: CTA c starts its walk over the input vector `rot` groups further on, so that the 148 CTAs do not all pull the same
// L2 lines at the same moment.  Whole groups (16 units) keep the half-warp amax shuffles of emit_unit intact.
TCE_DEVINL int rot_unit(int u, int units, int cta) {
    const int ng = units >> 4;
    int g = (u >> 4) + (cta % ng);
    if (g >= ng) g -= ng;
    return (g << 4) | (u & 15);
}

// fp16 input vector (attention output / SiLU*mul activations) published as {half2, tag} words -> activation planes
TCE_DEVINL void stage_half(const Args &a, const GemvOp &op, const PSmem &sm, PairCtx &pc, const uint2 *src, uint32_t tag, int cta, int ctid, int lane, int p,
                           int nphase) {
    const int ng_own = own_groups(pc, op.NG);
    const int units = ng_own * 16;  // 8 halfs = 4 words = 32 B per unit; this CTA's groups only (pair mode: every other group)
    if (pc.on) {
        if (ctid == 0) rx_expect(sm, pc, (uint32_t)peer_groups(pc, op.NG) * 524u);  // 16 units x 32 B of planes + step + two sums per group
        wait_partner_free(sm, pc, p);
    }
    constexpr int PRE = 4;        // iterations whose words are requested together: one L2 round trip for up to 4 * 512 units
    for (int ub = 0; ub < units; ub += PRE * kConsumerThreads) {
        uint4 w[PRE][2];
        int ui[PRE];
#pragma unroll
        for (int k = 0; k < PRE; k++) {
            const int u = ub + k * kConsumerThreads + ctid;
            ui[k] = -1;
            if (u < units) {
                const int ru = rot_unit(u, units, cta);  // index among this CTA's groups
                ui[k] = pc.on ? (((ru >> 4) * 2 + (int)pc.rank) << 4) | (ru & 15) : ru;
            }
            w[k][0] = w[k][1] = make_uint4(0u, tag, 0u, tag);
            if (ui[k] >= 0) {
                w[k][0] = ld_ll2(src + (size_t)ui[k] * 4, false);
                w[k][1] = ld_ll2(src + (size_t)ui[k] * 4 + 2, false);
            }
        }
        {
            long long t0 = 0;
            while (true) {  // every word of the block that is not there yet is asked for again in the same round
                bool ok = true;
#pragma unroll
                for (int k = 0; k < PRE; k++) ok = ok && w[k][0].y == tag && w[k][0].w == tag && w[k][1].y == tag && w[k][1].w == tag;
                if (ok) break;
                if (t0 == 0) t0 = clock64();
                if (clock64() - t0 > kSpinLimit) __trap();
                __nanosleep(kPollBackoffNs);
#pragma unroll
                for (int k = 0; k < PRE; k++) {
                    if (ui[k] >= 0 && !(w[k][0].y == tag && w[k][0].w == tag && w[k][1].y == tag && w[k][1].w == tag)) {
                        w[k][0] = ld_ll2(src + (size_t)ui[k] * 4, false);
                        w[k][1] = ld_ll2(src + (size_t)ui[k] * 4 + 2, false);
                    }
                }
            }
            __syncwarp();
        }
        if (ub == 0 && ctid == 0) stamp(a, cta, nphase, p, 4);
#pragma unroll
        for (int k = 0; k < PRE; k++) {
            if (ub + k * kConsumerThreads >= units) break;  // warp-uniform
            const bool valid = ui[k] >= 0;
            float v[8];
            const float2 f0 = h2_to_f2(w[k][0].x), f1 = h2_to_f2(w[k][0].z), f2 = h2_to_f2(w[k][1].x), f3 = h2_to_f2(w[k][1].z);
            v[0] = f0.x; v[1] = f0.y; v[2] = f1.x; v[3] = f1.y;
            v[4] = f2.x; v[5] = f2.y; v[6] = f3.x; v[7] = f3.y;
            if (pc.on)
                gemv::emit_unit<1, true>(sm.xs, op.IC, sm.gx, sm.gsum, valid ? ui[k] : 0, valid, v, lane, &pc.dst);
            else
                gemv::emit_unit<1>(sm.xs, op.IC, sm.gx, sm.gsum, valid ? ui[k] : 0, valid, v, lane);
        }
    }
    if (ctid == 0) stamp(a, cta, nphase, p, 5);
    named_bar_sync(1, kConsumerThreads);
    if (pc.on) rx_wait(sm, pc);
}

// Tensor parallel: x[0..7] += the eight output words of every rank's slot, in rank order (bit-identical on all ranks).  The slots of two ranks
// are requested together: one L2 round trip per pair of ranks instead of one per rank (measured at P = 8: the per-rank round trips made 8 GPUs
// slower than 4; a batch of four needs 64 payload registers and pushed the whole kernel into spills).
TCE_DEVINL void tp_accumulate(float (&x)[8], const uint2 *slot0, int tp_size, int E, uint32_t tag) {
    int pr = 0;
    for (; pr + 2 <= tp_size; pr += 2) {
        const uint2 *pa = slot0 + (size_t)pr * E, *pb = pa + E;
        uint4 wa[4], wb[4];
        long long t0 = 0;
        while (true) {  // both slots are (re)requested in every round: one round trip when the words are there
            bool ok = true;
#pragma unroll
            for (int i = 0; i < 4; i++) wa[i] = ld_ll2(pa + 2 * i, true);
#pragma unroll
            for (int i = 0; i < 4; i++) wb[i] = ld_ll2(pb + 2 * i, true);
#pragma unroll
            for (int i = 0; i < 4; i++) ok = ok && wa[i].y == tag && wa[i].w == tag && wb[i].y == tag && wb[i].w == tag;
            if (ok) break;
            if (t0 == 0) t0 = clock64();
            if (clock64() - t0 > kSpinLimit) __trap();
            __nanosleep(kPollBackoffNs);
        }
        x[0] += __uint_as_float(wa[0].x); x[1] += __uint_as_float(wa[0].z); x[2] += __uint_as_float(wa[1].x); x[3] += __uint_as_float(wa[1].z);
        x[4] += __uint_as_float(wa[2].x); x[5] += __uint_as_float(wa[2].z); x[6] += __uint_as_float(wa[3].x); x[7] += __uint_as_float(wa[3].z);
        x[0] += __uint_as_float(wb[0].x); x[1] += __uint_as_float(wb[0].z); x[2] += __uint_as_float(wb[1].x); x[3] += __uint_as_float(wb[1].z);
        x[4] += __uint_as_float(wb[2].x); x[5] += __uint_as_float(wb[2].z); x[6] += __uint_as_float(wb[3].x); x[7] += __uint_as_float(wb[3].z);
    }
    if (pr < tp_size) {
        uint4 w[4];
        wait_ll2xN<4>(slot0 + (size_t)pr * E, tag, true, w);
        x[0] += __uint_as_float(w[0].x); x[1] += __uint_as_float(w[0].z); x[2] += __uint_as_float(w[1].x); x[3] += __uint_as_float(w[1].z);
        x[4] += __uint_as_float(w[2].x); x[5] += __uint_as_float(w[2].z); x[6] += __uint_as_float(w[3].x); x[7] += __uint_as_float(w[3].z);
    }
}

// fp32 residual stream with fused RMSNorm.  Every CTA holds the stream in shared memory; `delta` (o_proj or down_proj outputs of all
// tensor-parallel ranks, {float, tag} words) is added to it here by every CTA in the same (rank) order.  Returns 1/rms: y = inv * W (x . gamma).
TCE_DEVINL float stage_rms(const Args &a, const GemvOp &op, const PSmem &sm, PairCtx &pc, const uint2 *delta, uint32_t tag, const float *gamma, int token,
                           bool first, bool emit, int cta, int ctid, int cw, int lane, int p, int nphase) {
    const int units = own_groups(pc, op.NG) * 16;  // pair mode: this CTA keeps (and normalises) every other 128-group of the residual stream
    const bool sys = a.tp_size > 1;
    if (pc.on && emit) {
        if (ctid == 0) rx_expect(sm, pc, (uint32_t)peer_groups(pc, op.NG) * 524u + (uint32_t)kCW * 4u);  // + the partner's 16 partial sums of squares
        wait_partner_free(sm, pc, p);
    }
    float ss = 0.f;
    for (int ui0 = 0; ui0 < units; ui0 += kConsumerThreads) {  // warp-uniform trip count
        const int u = ui0 + ctid;
        const bool valid = u < units;
        int ui = 0;
        if (valid) {
            const int ru = rot_unit(u, units, cta);
            ui = pc.on ? (((ru >> 4) * 2 + (int)pc.rank) << 4) | (ru & 15) : ru;
        }
        float x[8], v[8];
#pragma unroll
        for (int i = 0; i < 8; i++) x[i] = 0.f;
        float4 g0 = make_float4(0.f, 0.f, 0.f, 0.f), g1 = g0;
        if (valid) {
            g0 = *reinterpret_cast<const float4 *>(gamma + (size_t)ui * 8);  // static: requested before the spin
            g1 = *reinterpret_cast<const float4 *>(gamma + (size_t)ui * 8 + 4);
            if (first) {
                // the token's embedding row is the residual stream (reference: CPU Embedding, cuda/Int4llamaDecoder.cu:62-69)
                const uint4 raw = *reinterpret_cast<const uint4 *>(a.embed + (size_t)token * a.E + (size_t)ui * 8);
                const __half2 *h2 = reinterpret_cast<const __half2 *>(&raw);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    const float2 f = __half22float2(h2[i]);
                    x[2 * i] = f.x;
                    x[2 * i + 1] = f.y;
                }
            } else {
                const float4 r0 = *reinterpret_cast<const float4 *>(sm.resid + (size_t)ui * 8);
                const float4 r1 = *reinterpret_cast<const float4 *>(sm.resid + (size_t)ui * 8 + 4);
                x[0] = r0.x; x[1] = r0.y; x[2] = r0.z; x[3] = r0.w;
                x[4] = r1.x; x[5] = r1.y; x[6] = r1.z; x[7] = r1.w;
                // residual += sum over ranks, in rank order (bit-identical everywhere).  The slots of up to four ranks are requested together:
                // one L2 round trip per batch instead of one per rank (measured at P = 8: the per-rank round trips made 8 GPUs slower than 4)
                if (a.tp_size == 1) {
                    uint4 w[4];
                    wait_ll2xN<4>(delta + (size_t)ui * 8, tag, false, w);
                    x[0] += __uint_as_float(w[0].x); x[1] += __uint_as_float(w[0].z); x[2] += __uint_as_float(w[1].x); x[3] += __uint_as_float(w[1].z);
                    x[4] += __uint_as_float(w[2].x); x[5] += __uint_as_float(w[2].z); x[6] += __uint_as_float(w[3].x); x[7] += __uint_as_float(w[3].z);
                } else {
                    tp_accumulate(x, delta + (size_t)ui * 8, a.tp_size, a.E, tag);
                }
                if (ui0 == 0 && ctid == 0) stamp(a, cta, nphase, p, 4);
            }
            *reinterpret_cast<float4 *>(sm.resid + (size_t)ui * 8) = make_float4(x[0], x[1], x[2], x[3]);
            *reinterpret_cast<float4 *>(sm.resid + (size_t)ui * 8 + 4) = make_float4(x[4], x[5], x[6], x[7]);
        }
        if (emit) {
#pragma unroll
            for (int i = 0; i < 8; i++) ss += x[i] * x[i];
            v[0] = x[0] * g0.x; v[1] = x[1] * g0.y; v[2] = x[2] * g0.z; v[3] = x[3] * g0.w;
            v[4] = x[4] * g1.x; v[5] = x[5] * g1.y; v[6] = x[6] * g1.z; v[7] = x[7] * g1.w;
            if (pc.on)
                gemv::emit_unit<1, true>(sm.xs, op.IC, sm.gx, sm.gsum, ui, valid, v, lane, &pc.dst);
            else
                gemv::emit_unit<1>(sm.xs, op.IC, sm.gx, sm.gsum, ui, valid, v, lane);
        }
    }
    if (!emit) return 1.f;
    ss = warp_sum(ss);
    // partial sums of squares: slot (staging rank, warp) on both CTAs of a pair, so that both add them in the same order
    if (lane == 0) {
        sm.rms[pc.rank * kCW + cw] = ss;
        if (pc.on) gemv::st_async_b32(pc.r_rms + (uint32_t)(pc.rank * kCW + cw) * 4u, __float_as_uint(ss), pc.dst.bar);
    }
    if (ctid == 0) stamp(a, cta, nphase, p, 5);
    named_bar_sync(1, kConsumerThreads);
    if (pc.on) rx_wait(sm, pc);
    float tot = 0.f;
    const int nparts = pc.on ? 2 * kCW : kCW;
    for (int w = 0; w < nparts; w++) tot += sm.rms[w];
    return rsqrtf(tot / (float)op.IC + a.eps);  // LlamaRMSNorm (llm/src/ops/LlamaRMSNorm.cc): x / sqrt(mean(x^2) + eps) * weight
}

// ------------------------------------------------------------------------------------------------------------ consumers: GEMV
// one (16 rows x 128 k) unit; see gemv::unit1 (w4a16_gemv_impl.cuh) for the arithmetic.  All operands by shared address; the loads
// of both units of a stage are issued before either is consumed.
struct UnitRegs {
    uint4 wa, wb, xe, xo;
    uint32_t z;   // zero points of rows g (bits 0..7) and g + 8 (bits 8..15)
    uint32_t sc;  // half2: scales of rows g, g + 8
    int sxv;
    float st;
};
TCE_DEVINL void unit_load(UnitRegs &u, uint32_t w_addr, uint32_t rp8, uint32_t x_addr, uint32_t meta_addr, int gi, int g, int G, uint32_t gx_u32,
                          uint32_t gsum_u32, int gsel) {
    u.wa = lds_u4(w_addr);
    u.wb = lds_u4(w_addr + rp8);
    u.xe = u.xo = make_uint4(0u, 0u, 0u, 0u);
    if (g < 4) {  // MMA columns 4..7 are don't-cares: half of the warp skips the activation loads (half the shared-memory wavefronts)
        u.xe = lds_u4(x_addr + (uint32_t)G * 256u);
        u.xo = lds_u4(x_addr + (uint32_t)G * 256u + 128u);
    }
    u.sc = lds_u32(meta_addr + (uint32_t)(gi * 8 + g) * 4u);
    u.z = lds_u16(meta_addr + 1024u + (uint32_t)(gi * 8 + g) * 2u);
    u.sxv = (int)lds_u32(gsum_u32 + (uint32_t)(2 * G + gsel) * 4u);
    u.st = lds_f32(gx_u32 + (uint32_t)G * 4u);
}
TCE_DEVINL void unit_compute(const UnitRegs &u, float lscale, float &totA, float &totB) {
    constexpr uint32_t ML = 0x0f0f0f0fu, MH = 0xf0f0f0f0u;
    int accL[4], accH[4];
    mma_m16n8k32_u8s8_z(accL, u.wa.x & ML, u.wb.x & ML, u.wa.y & ML, u.wb.y & ML, u.xe.x, u.xe.y);
    mma_m16n8k32_u8s8_z(accH, u.wa.x & MH, u.wb.x & MH, u.wa.y & MH, u.wb.y & MH, u.xo.x, u.xo.y);
    mma_m16n8k32_u8s8(accL, u.wa.z & ML, u.wb.z & ML, u.wa.w & ML, u.wb.w & ML, u.xe.z, u.xe.w);
    mma_m16n8k32_u8s8(accH, u.wa.z & MH, u.wb.z & MH, u.wa.w & MH, u.wb.w & MH, u.xo.z, u.xo.w);
    const float2 sc = h2_to_f2(u.sc);
    const float st = u.st * lscale;
    const int zAq = (int)(u.z & 0xFFu), zBq = (int)(u.z >> 8);
    // X = 2^24*p3 + 2^16*p2 + 2^8*p1 + p0; odd slots carry 16 x nibble (exact multiple of 16): c0 * 256 + c1 per parity, then q*X - z*sum X
    const int vA = (accL[0] << 8) + accL[1] + (((accH[0] << 8) + accH[1]) >> 4) - zAq * u.sxv;
    const int vB = (accL[2] << 8) + accL[3] + (((accH[2] << 8) + accH[3]) >> 4) - zBq * u.sxv;
    totA += (sc.x * st) * (float)vA;
    totB += (sc.y * st) * (float)vB;
}

// where group `gi` of a stage lives: byte offset of (row g, this lane's 16-byte chunk) and the distance to row g + 8
TCE_DEVINL void locate(const BoxPlan &pl, int gi, int g, int t, uint32_t &off, uint32_t &rp8) {
    int b = 0;
#pragma unroll
    for (int i = 1; i < kMaxBoxes; i++)
        if (i < pl.nbox && gi >= pl.b0[i]) b = i;
    const uint32_t rp = (uint32_t)pl.bw[b] * 64u;
    off = (uint32_t)pl.off[b] + (uint32_t)g * rp + (uint32_t)(gi - pl.b0[b]) * 64u + (uint32_t)t * 16u;
    rp8 = 8u * rp;
}

// Fast path for dense boxes of 16 groups (NG >= 16: every Llama width): within a stage every operand address is a per-lane constant
// plus the slot base, and the second unit of a warp sits at fixed distances (+16 KiB weights, +4 KiB planes, +512 B scales ...), so the
// inner loop carries almost no address arithmetic (the ALU pipe is what bounds this loop, profiles/README.md).
TCE_DEVINL void consume_gemv_dense(const GemvOp &op, const PSmem &sm, Ring &rs, Red &cs, float inv, int cta, int ncta, int cw, int lane) {
    const int g = lane >> 2, t = lane & 3;
    int t0, t1;
    partition(op, cta, ncta, t0, t1);
    const int NG = op.NG, S = op.S;
    // row g of group cw, this lane's 16-byte chunk.  Row-major boxes: rows 1 KiB apart (2-way bank conflict between rows g, g + 1 of a quarter-warp);
    // unit boxes: the 16 rows of a group 64 B apart (conflict free), gate | up pairs as two 8-row regions
    const uint32_t w_lane = op.unit ? (uint32_t)cw * (op.pair ? 512u : 1024u) + (uint32_t)g * 64u + (uint32_t)t * 16u : (uint32_t)g * 1024u + (uint32_t)t * 16u + (uint32_t)cw * 64u;
    const uint32_t wb_off = op.unit ? (op.pair ? 8192u : 512u) : 8192u;  // row g + 8
    const uint32_t m_lane = (uint32_t)kMetaOff + (uint32_t)(cw * 8 + g) * 4u;                            // scales of rows g, g + 8 of group cw
    const uint32_t z_lane = (uint32_t)kMetaOff + 1024u + (uint32_t)(cw * 8 + g) * 2u;
    const uint32_t x_lane = sm.xs_u32 + (uint32_t)((g >> 1) & 1) * (uint32_t)op.IC * 2u + (uint32_t)(t * 2 + (g & 1)) * 16u + (uint32_t)cw * 256u;
    const uint32_t s_lane = sm.gsum_u32 + (uint32_t)(2 * cw + (t & 1)) * 4u;
    const uint32_t q_lane = sm.gx_u32 + (uint32_t)cw * 4u;
    const float lscale = (t == 0) ? 65536.f : (t == 1 ? 1.f : 0.f);
    const bool xl = g < 4;  // MMA columns 4..7 are don't-cares
    for (int tile = t0; tile < t1; tile++) {
        float totA = 0.f, totB = 0.f;
        for (int s = 0; s < S; s++) {
            const bool two = kStageGroups * s + 16 < NG;  // the stage carries groups 16..31 as well (warp-uniform)
            mbar_wait_u32(sm.full_u32 + (uint32_t)rs.stage * 8u, rs.phase);
            const uint32_t base = sm.ring_u32 + (uint32_t)rs.stage * (uint32_t)kStageBytes;
            const uint32_t wb_ = base + w_lane, mb_ = base + m_lane, zb_ = base + z_lane;
            const uint32_t xb_ = x_lane + (uint32_t)s * (kStageGroups * 256u), sb_ = s_lane + (uint32_t)s * (kStageGroups * 8u), qb_ = q_lane + (uint32_t)s * (kStageGroups * 4u);
            UnitRegs u0, u1;
            u0.wa = lds_u4(wb_);
            u0.wb = lds_u4(wb_ + wb_off);
            u0.xe = u0.xo = u1.xe = u1.xo = make_uint4(0u, 0u, 0u, 0u);
            if (xl) {
                u0.xe = lds_u4(xb_);
                u0.xo = lds_u4(xb_ + 128u);
            }
            u0.sc = lds_u32(mb_);
            u0.z = lds_u16(zb_);
            u0.sxv = (int)lds_u32(sb_);
            u0.st = lds_f32(qb_);
            if (two) {
                u1.wa = lds_u4(wb_ + 16384u);
                u1.wb = lds_u4(wb_ + 16384u + wb_off);
                if (xl) {
                    u1.xe = lds_u4(xb_ + 4096u);
                    u1.xo = lds_u4(xb_ + 4096u + 128u);
                }
                u1.sc = lds_u32(mb_ + 512u);
                u1.z = lds_u16(zb_ + 256u);
                u1.sxv = (int)lds_u32(sb_ + 128u);
                u1.st = lds_f32(qb_ + 64u);
            }
            unit_compute(u0, lscale, totA, totB);
            if (two) unit_compute(u1, lscale, totA, totB);
            __syncwarp();
            if (lane == 0) mbar_arrive_u32(sm.empty_u32 + (uint32_t)rs.stage * 8u);
            rs.advance(sm.nst);
        }
        // ---- hand the tile sums to the epilogue warp ----
        totA += __shfl_xor_sync(0xffffffffu, totA, 1);  // (p3, p2) share of t = 0 + (p1, p0) share of t = 1
        totB += __shfl_xor_sync(0xffffffffu, totB, 1);
        mbar_wait_u32(sm.redempty_u32 + (uint32_t)cs.rb * 8u, cs.rphase ^ 1);
        float *rbuf = sm.red + ((size_t)cs.rb * kCW + cw) * 16;
        if (t == 0) {
            rbuf[g] = totA * inv;
            rbuf[g + 8] = totB * inv;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive_u32(sm.redfull_u32 + (uint32_t)cs.rb * 8u);
        cs.advance();
    }
}

TCE_DEVINL void consume_gemv(const GemvOp &op, const PSmem &sm, Ring &rs, Red &cs, float inv, int cta, int ncta, int cw, int lane) {
    const int g = lane >> 2, t = lane & 3;
    int t0, t1;
    partition(op, cta, ncta, t0, t1);
    const int NG = op.NG, S = op.S;
    const bool ragged = (NG % kStageGroups) != 0;
    // lane-constant weight operands of this warp's two groups (cw, cw + 16), for a full stage and for the ragged last stage of a tile
    uint32_t wf0, rf0, wf1, rf1, wl0 = 0, rl0 = 0, wl1 = 0, rl1 = 0;
    locate(op.plan[0], cw, g, t, wf0, rf0);
    locate(op.plan[0], cw + 16, g, t, wf1, rf1);
    if (ragged) {
        locate(op.plan[1], cw, g, t, wl0, rl0);
        locate(op.plan[1], cw + 16, g, t, wl1, rl1);
    }
    // lane-constant activation operands: MMA column g & 3 supplies plane 3 - (g & 3)
    const uint32_t x_lane = sm.xs_u32 + (uint32_t)((g >> 1) & 1) * (uint32_t)op.IC * 2u + (uint32_t)(t * 2 + (g & 1)) * 16u;
    const float lscale = (t == 0) ? 65536.f : (t == 1 ? 1.f : 0.f);
    const int gsel = t & 1;
    const uint32_t gx_u32 = sm.gx_u32, gsum_u32 = sm.gsum_u32;
    for (int tile = t0; tile < t1; tile++) {
        float totA = 0.f, totB = 0.f;
        for (int s = 0; s < S; s++) {
            const int n = min(kStageGroups, NG - kStageGroups * s);  // groups this stage carries
            const bool last = ragged && s == S - 1;
            mbar_wait_u32(sm.full_u32 + (uint32_t)rs.stage * 8u, rs.phase);
            const uint32_t base = sm.ring_u32 + (uint32_t)rs.stage * (uint32_t)kStageBytes;
            UnitRegs u0, u1;
            const bool has0 = cw < n, has1 = cw + 16 < n;
            if (has0) unit_load(u0, base + (last ? wl0 : wf0), last ? rl0 : rf0, x_lane, base + kMetaOff, cw, g, kStageGroups * s + cw, gx_u32, gsum_u32, gsel);
            if (has1) unit_load(u1, base + (last ? wl1 : wf1), last ? rl1 : rf1, x_lane, base + kMetaOff, cw + 16, g, kStageGroups * s + cw + 16, gx_u32, gsum_u32, gsel);
            if (has0) unit_compute(u0, lscale, totA, totB);
            if (has1) unit_compute(u1, lscale, totA, totB);
            __syncwarp();
            if (lane == 0) mbar_arrive_u32(sm.empty_u32 + (uint32_t)rs.stage * 8u);
            rs.advance(sm.nst);
        }
        // ---- hand the tile sums to the epilogue warp ----
        totA += __shfl_xor_sync(0xffffffffu, totA, 1);  // (p3, p2) share of t = 0 + (p1, p0) share of t = 1
        totB += __shfl_xor_sync(0xffffffffu, totB, 1);
        mbar_wait_u32(sm.redempty_u32 + (uint32_t)cs.rb * 8u, cs.rphase ^ 1);
        float *rbuf = sm.red + ((size_t)cs.rb * kCW + cw) * 16;
        if (t == 0) {
            rbuf[g] = totA * inv;
            rbuf[g + 8] = totB * inv;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive_u32(sm.redfull_u32 + (uint32_t)cs.rb * 8u);
        cs.advance();
    }
}

// ------------------------------------------------------------------------------------------------------------ epilogue warp
struct EpiState {
    unsigned long long best;  // PE_LOGITS: running arg-max key of this warp
};

TCE_DEVINL void epilogue_gemv(const Args &a, const GemvOp &op, const PSmem &sm, Red &es, EpiState &st, uint2 *out_ll, int which, uint32_t tag, int cta, int ncta,
                              int lane) {
    int t0, t1;
    partition(op, cta, ncta, t0, t1);
    const bool tp = a.tp_size > 1;
    for (int tile = t0; tile < t1; tile++) {
        mbar_wait_u32(sm.redfull_u32 + (uint32_t)es.rb * 8u, es.rphase);
        const float *rbuf = sm.red + (size_t)es.rb * kCW * 16;
        // lane l < 16 sums consumer warps 0..7 of row l, lane l + 16 warps 8..15
        float v = 0.f;
        {
            const int row = lane & 15, w0 = (lane >> 4) * 8;
#pragma unroll
            for (int w = 0; w < 8; w++) v += rbuf[(w0 + w) * 16 + row];
        }
        v += __shfl_down_sync(0xffffffffu, v, 16);
        __syncwarp();
        if (lane == 0) mbar_arrive_u32(sm.redempty_u32 + (uint32_t)es.rb * 8u);
        es.advance();
        switch (op.epi) {
            case PE_DELTA_LL:
                // o_proj / down_proj output rows: one {float, tag} word each, into slot `rank` of every rank's buffer (NVLink peer stores
                // when tensor parallel) -- the residual add happens in every reader (stage_rms)
                if (lane < 16) {
                    const size_t o = (size_t)a.tp_rank * a.E + (size_t)tile * 16 + lane;
                    if (tp) {
                        for (int pr = 0; pr < a.tp_size; pr++) st_ll(a.tp_delta[which][pr] + o, __float_as_uint(v), tag, true);
                    } else {
                        st_ll(out_ll + o, __float_as_uint(v), tag, false);
                    }
                }
                break;
            case PE_HALF_LL: {
                const float hi = __shfl_down_sync(0xffffffffu, v, 1);
                if (lane < 16 && !(lane & 1)) st_ll(out_ll + (size_t)tile * 8 + (lane >> 1), pack_half2(v, hi), tag, false);
                break;
            }
            case PE_SILU_LL: {
                // rows 0-7 = gate, rows 8-15 = up of the same output channels: y = SiLU(gate) * up
                // (reference SiLuMul_half, llm/src/nn_modules/cuda/Int4llamaDecoderLayer.cu:21-30; fp32 here)
                const float up = __shfl_down_sync(0xffffffffu, v, 8);
                const float y = v / (1.f + __expf(-v)) * up;
                const float yhi = __shfl_down_sync(0xffffffffu, y, 1);
                if (lane < 8 && !(lane & 1)) st_ll(out_ll + (size_t)tile * 4 + (lane >> 1), pack_half2(y, yhi), tag, false);
                break;
            }
            case PE_LOGITS:
                if (lane < 16) {
                    const int idx = tile * 16 + lane;
                    a.logits[idx] = v;
                    const unsigned long long key = argmax_key(v, a.vocab_base + idx);
                    st.best = key > st.best ? key : st.best;
                }
                break;
        }
    }
}

// ------------------------------------------------------------------------------------------------------------ consumers: attention
// byte offset of (row r, 16-byte chunk c of the 256-byte row) inside the K or V half of a stage: two [64 rows][128 B] boxes, 128B-swizzled
TCE_DEVINL uint32_t kv_off(int r, int c) { return (uint32_t)((c >> 3) * 8192 + r * 128 + (((c & 7) ^ (r & 7)) << 4)); }

// RoPE (llm/src/ops/RotaryPosEmb.cc:7-69, rotate-half) of one {half2, tag} word pair: word j holds dims (2j, 2j+1), its partner word j +- 32
TCE_DEVINL float2 rope_pair(const uint2 *vec, int j, uint32_t tag, const float *cosr, const float *sinr) {
    const uint2 *pa = vec + j, *pb = vec + (j < 32 ? j + 32 : j - 32);
    uint2 wa = ld_ll1(pa, false), wb = ld_ll1(pb, false);  // both requests in flight before either tag is examined
    if (wa.y != tag) wa.x = wait_ll1(pa, tag, false);
    if (wb.y != tag) wb.x = wait_ll1(pb, tag, false);
    const float2 x = h2_to_f2(wa.x), xp = h2_to_f2(wb.x);
    const float sgn = (j < 32) ? -1.f : 1.f;
    const int d = 2 * j;
    return make_float2(x.x * cosr[d] + sgn * xp.x * sinr[d], x.y * cosr[d + 1] + sgn * xp.y * sinr[d + 1]);
}

TCE_DEVINL void attention_phase(const Args &a, const LayerDesc &L, const PSmem &sm, Ring &rs, uint32_t tag_qkv, uint32_t tag_part, uint32_t tag_out, int cta,
                                int ncta, int pos, int ctid, int cw, int lane, int p, int nphase) {
    const AttnSplit sp = attn_split(cta, ncta, a.KVH, pos);
    const int nrep = a.nrep;
    const int g = lane >> 2, t = lane & 3;
    if (sp.ch0 < sp.ch1) {
        // scratch (the activation-plane buffer is idle during this phase)
        __half *sQ = reinterpret_cast<__half *>(sm.xs);                        // [8][136] q * alpha after RoPE, rows >= nrep zero
        float *sO = reinterpret_cast<float *>(sm.xs + 8 * 136 * 2);            // [kCW][nrep][128] per-warp unnormalised outputs
        float *sML = sO + (size_t)kCW * nrep * 128;                            // [kCW][nrep][2] per-warp (max, sum)
        const float *cosr = sm.rope, *sinr = sm.rope + 128;  // the position's table rows, staged once per kernel
        // ---- RoPE on the nrep query heads of this KV head (fp32), one {half2} word per thread and pass ----
        for (int i = ctid; i < 8 * 64; i += kConsumerThreads) {
            const int r = i >> 6, j = i & 63;
            float2 v = make_float2(0.f, 0.f);
            if (r < nrep) {
                v = rope_pair(a.qkv_ll + (size_t)(sp.kvh * nrep + r) * 64, j, tag_qkv, cosr, sinr);
                v.x *= a.alpha;
                v.y *= a.alpha;
            }
            *reinterpret_cast<__half2 *>(sQ + r * 136 + 2 * j) = __floats2half2_rn(v.x, v.y);
        }
        named_bar_sync(1, kConsumerThreads);
        if (ctid == 0) stamp(a, cta, nphase, p, 4);
        uint32_t qa[8][2];  // A operand: q[head g][dims], all 8 k-steps (rows 8..15 of the MMA tile are zero)
#pragma unroll
        for (int ks = 0; ks < 8; ks++) {
            qa[ks][0] = *reinterpret_cast<const uint32_t *>(sQ + g * 136 + ks * 16 + t * 2);
            qa[ks][1] = *reinterpret_cast<const uint32_t *>(sQ + g * 136 + ks * 16 + 8 + t * 2);
        }
        float m_run = -INFINITY, l_run = 0.f;  // of head row g (replicated over t)
        bool have = false;
        float *myO = sO + (size_t)cw * nrep * 128;
        const int kb = cw & 3;  // 16-key block of the chunk this warp owns
        for (int c = sp.ch0; c < sp.ch1; c++) {
            const int kbase = c * kKvChunk + kb * 16;  // first key of the block
            const bool mine = (((c - sp.ch0) & 3) == (cw >> 2)) && (kbase <= pos);
            const bool has_new = mine && pos < kbase + 16;
            mbar_wait_u32(sm.full_u32 + (uint32_t)rs.stage * 8u, rs.phase);
            if (c == sp.ch0 && ctid == 0) stamp(a, cta, nphase, p, 7);
            if (mine) {
                uint8_t *kst = sm.ring + (size_t)rs.stage * kStageBytes, *vst = kst + kHalfBytes;
                if (has_new) {
                    // the token's own key / value: RoPE(k), round to fp16, append to the cache and patch the (stale) rows of the stage
                    const uint2 *kw = a.qkv_ll + (size_t)a.H * 64 + (size_t)sp.kvh * 64, *vw = a.qkv_ll + (size_t)(a.H + a.KVH) * 64 + (size_t)sp.kvh * 64;
                    const int r = pos - c * kKvChunk;
#pragma unroll
                    for (int i = 0; i < 2; i++) {
                        const int j = lane * 2 + i;  // word j = dims 2j, 2j+1
                        const float2 kr = rope_pair(kw, j, tag_qkv, cosr, sinr);
                        const __half2 kh = __floats2half2_rn(kr.x, kr.y);
                        const uint32_t vv = wait_ll1(vw + j, tag_qkv, false);
                        *reinterpret_cast<__half2 *>(kst + kv_off(r, j >> 2) + (j & 3) * 4) = kh;
                        *reinterpret_cast<uint32_t *>(vst + kv_off(r, j >> 2) + (j & 3) * 4) = vv;
                        *reinterpret_cast<__half2 *>(L.k_cache + ((size_t)sp.kvh * a.max_ctx + pos) * 128 + 2 * j) = kh;
                        *reinterpret_cast<uint32_t *>(L.v_cache + ((size_t)sp.kvh * a.max_ctx + pos) * 128 + 2 * j) = vv;
                    }
                    // V rows of the block beyond the token were never written for this sequence: finite zeros (0 * garbage must not be NaN)
                    for (int rr = r + 1; rr < kb * 16 + 16; rr++)
                        *reinterpret_cast<uint2 *>(vst + kv_off(rr, lane >> 1) + (lane & 1) * 8) = make_uint2(0u, 0u);
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic writes into a stage the TMA unit will refill
                    __syncwarp();
                }
                // ---- scores: S[head][key] = q . K ----
                float s0[4] = {0.f, 0.f, 0.f, 0.f}, s1[4] = {0.f, 0.f, 0.f, 0.f};
                {
                    const int lr = (lane & 7) + ((lane >> 4) << 3);  // ldmatrix row supplied by this lane (key within the block)
                    const int lc = (lane >> 3) & 1;                  // ... and which 8-dim half of the k-step
#pragma unroll
                    for (int ks = 0; ks < 8; ks++) {
                        uint32_t b0, b1, b2, b3;
                        attn::ldmatrix_x4(b0, b1, b2, b3, kst + kv_off(kb * 16 + lr, 2 * ks + lc));
                        mma_m16n8k16(s0, qa[ks][0], 0u, qa[ks][1], 0u, b0, b1);  // keys 0..7 of the block
                        mma_m16n8k16(s1, qa[ks][0], 0u, qa[ks][1], 0u, b2, b3);  // keys 8..15
                    }
                }
                // thread (g, t): head row g, keys kbase + {2t, 2t+1} (s0) and kbase + 8 + {2t, 2t+1} (s1)
                const int k0 = kbase + 2 * t;
                float e0 = (k0 <= pos) ? s0[0] : -INFINITY, e1 = (k0 + 1 <= pos) ? s0[1] : -INFINITY;
                float e2 = (k0 + 8 <= pos) ? s1[0] : -INFINITY, e3 = (k0 + 9 <= pos) ? s1[1] : -INFINITY;
                float mb = fmaxf(fmaxf(e0, e1), fmaxf(e2, e3));
                mb = fmaxf(mb, __shfl_xor_sync(0xffffffffu, mb, 1));
                mb = fmaxf(mb, __shfl_xor_sync(0xffffffffu, mb, 2));
                const float m_new = fmaxf(m_run, mb);  // finite: key kbase is visible
                e0 = __expf(e0 - m_new);
                e1 = __expf(e1 - m_new);
                e2 = __expf(e2 - m_new);
                e3 = __expf(e3 - m_new);
                float lb = (e0 + e1) + (e2 + e3);
                lb += __shfl_xor_sync(0xffffffffu, lb, 1);
                lb += __shfl_xor_sync(0xffffffffu, lb, 2);
                const float sc_old = have ? __expf(m_run - m_new) : 0.f;
                l_run = l_run * sc_old + lb;
                m_run = m_new;
                const uint32_t pa0 = pack_half2(e0, e1), pa2 = pack_half2(e2, e3);  // A operand: P[head g][keys], rows 8..15 zero
                const int lr = (lane & 7) + (((lane >> 3) & 1) << 3);  // ldmatrix.trans row = key within the block
                const int lc = lane >> 4;                                // ... which of the two 8-dim n-tiles
#pragma unroll
                for (int h = 0; h < 2; h++) {  // dims 64h .. 64h + 63
                    float oacc[8][4];
#pragma unroll
                    for (int j = 0; j < 8; j++) oacc[j][0] = oacc[j][1] = oacc[j][2] = oacc[j][3] = 0.f;
#pragma unroll
                    for (int jp = 0; jp < 4; jp++) {
                        uint32_t b0, b1, b2, b3;
                        attn::ldmatrix_x4_t(b0, b1, b2, b3, vst + kv_off(kb * 16 + lr, 8 * h + 2 * jp + lc));
                        mma_m16n8k16(oacc[2 * jp], pa0, 0u, pa2, 0u, b0, b1);
                        mma_m16n8k16(oacc[2 * jp + 1], pa0, 0u, pa2, 0u, b2, b3);
                    }
                    if (g < nrep) {
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            float2 *dst = reinterpret_cast<float2 *>(myO + g * 128 + 64 * h + 8 * j + 2 * t);
                            float2 nv = make_float2(oacc[j][0], oacc[j][1]);
                            if (have) {
                                const float2 old = *dst;
                                nv.x += old.x * sc_old;
                                nv.y += old.y * sc_old;
                            }
                            *dst = nv;
                        }
                    }
                }
                have = true;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive_u32(sm.empty_u32 + (uint32_t)rs.stage * 8u);
            rs.advance(sm.nst);
        }
        if (ctid == 0) stamp(a, cta, nphase, p, 5);
        if (t == 0 && g < nrep) {
            sML[(cw * nrep + g) * 2] = have ? m_run : -INFINITY;
            sML[(cw * nrep + g) * 2 + 1] = have ? l_run : 0.f;
        }
        named_bar_sync(1, kConsumerThreads);
        // ---- merge the 16 warp partials of this CTA: thread i < nrep * 128 owns (head r, dim d) ----
        const int r = ctid >> 7, d = ctid & 127;
        if (ctid < nrep * 128) {  // whole warps: nrep * 128 is a multiple of 32
            float o = 0.f, M = -INFINITY, Lsum = 0.f;
            for (int w = 0; w < kCW; w++) M = fmaxf(M, sML[(w * nrep + r) * 2]);
            for (int w = 0; w < kCW; w++) {
                const float mw = sML[(w * nrep + r) * 2];
                if (mw != -INFINITY) {
                    const float wt = __expf(mw - M);
                    Lsum += wt * sML[(w * nrep + r) * 2 + 1];
                    o += wt * sO[((size_t)w * nrep + r) * 128 + d];
                }
            }
            const int head = sp.kvh * nrep + r;
            if (sp.nsplit == 1) {
                const float y = o / Lsum;
                const float yhi = __shfl_down_sync(0xffffffffu, y, 1);
                if (!(d & 1)) st_ll(a.attn_ll + (size_t)head * 64 + (d >> 1), pack_half2(y, yhi), tag_out, false);
            } else {
                uint2 *rec = a.part_ll + ((size_t)head * a.nsplit_max + sp.split) * 130;
                st_ll(rec + d, __float_as_uint(o), tag_part, false);
                if (d == 0) {
                    st_ll(rec + 128, __float_as_uint(M), tag_part, false);
                    st_ll(rec + 129, __float_as_uint(Lsum), tag_part, false);
                }
            }
        }
    }
    if (ctid == 0) stamp(a, cta, nphase, p, 6);
    if (sp.nsplit == 1) return;
    // ---- split merge, spread over the grid: task = (head, block of 32 dims), one warp each ----
    const int ntask = a.H * 4;
    for (int task = cta + cw * ncta; task < ntask; task += ncta * kCW) {
        const int head = task >> 2, d = ((task & 3) << 5) + lane;
        const uint2 *base = a.part_ll + (size_t)head * a.nsplit_max * 130;
        // lane s < nsplit fetches (m, l) of split s; the maximum and the weights are formed with shuffles.  All requests of a round
        // (the statistics and up to kRound partial outputs) are in flight together: one L2 round trip when the partials are there.
        constexpr int kRound = 20;
        uint2 wm = make_uint2(0u, tag_part), wl = wm;
        uint2 ow[kRound];
#pragma unroll
        for (int i = 0; i < kRound; i++) ow[i] = make_uint2(0u, tag_part);
        {
            const bool stat = lane < sp.nsplit;
            if (stat) wm.y = wl.y = tag_part + 1u;  // "not here yet"
#pragma unroll
            for (int i = 0; i < kRound; i++)
                if (i < sp.nsplit) ow[i].y = tag_part + 1u;
            long long t0 = 0;
            while (true) {
                if (wm.y != tag_part) wm = ld_ll1(base + (size_t)lane * 130 + 128, false);
                if (wl.y != tag_part) wl = ld_ll1(base + (size_t)lane * 130 + 129, false);
#pragma unroll
                for (int i = 0; i < kRound; i++)
                    if (ow[i].y != tag_part) ow[i] = ld_ll1(base + (size_t)i * 130 + d, false);
                bool ok = wm.y == tag_part && wl.y == tag_part;
#pragma unroll
                for (int i = 0; i < kRound; i++) ok = ok && ow[i].y == tag_part;
                if (ok) break;
                if (t0 == 0) t0 = clock64();
                if (clock64() - t0 > kSpinLimit) __trap();
                __nanosleep(kPollBackoffNs);
            }
            __syncwarp();
        }
        const float ms = (lane < sp.nsplit) ? __uint_as_float(wm.x) : -INFINITY, ls = (lane < sp.nsplit) ? __uint_as_float(wl.x) : 0.f;
        const float M = warp_max(ms);
        const float wgt = (lane < sp.nsplit) ? __expf(ms - M) : 0.f;
        const float Lt = warp_sum(wgt * ls);
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < kRound; i++) acc += __shfl_sync(0xffffffffu, wgt, i) * __uint_as_float(ow[i].x);
        for (int s0 = kRound; s0 < sp.nsplit; s0++)
            acc += __shfl_sync(0xffffffffu, wgt, s0) * __uint_as_float(wait_ll1(base + (size_t)s0 * 130 + d, tag_part, false));
        const float y = acc / Lt;
        const float yhi = __shfl_down_sync(0xffffffffu, y, 1);
        if (!(lane & 1)) st_ll(a.attn_ll + (size_t)head * 64 + (d >> 1), pack_half2(y, yhi), tag_out, false);
    }
}

// ------------------------------------------------------------------------------------------------------------ the kernel
__global__ void __launch_bounds__(kThreads, 1) decode_persistent_kernel(const __grid_constant__ Args a) {
    extern __shared__ uint8_t smem_raw[];
    const PSmem sm = carve(smem_raw, a);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int cta = blockIdx.x, ncta = gridDim.x;
    const int Lyr = a.num_layers;
    const int token = a.tokpos[0], pos = a.tokpos[1];
    if (token < 0 || token >= a.embed_rows || pos < 0 || pos >= a.max_ctx) {  // uniform over the grid: nobody starts
        if (cta == 0 && tid == 0) {
            *a.error = 1;
            *a.next_token = -1;
        }
        return;
    }
    if (warp == 0) {
        if (lane < a.nst) {
            mbar_init(&sm.full[lane], 1);
            mbar_init(&sm.empty[lane], kCW);
        } else if (lane >= 16 && lane < 16 + kRedBufs) {
            mbar_init(&sm.red_full[lane - 16], kCW);
            mbar_init(&sm.red_empty[lane - 16], 1);
        }
        if (lane == 30) {
            mbar_init(sm.rx, 1);
            *sm.free_gen = 0;
        }
        mbar_fence_init();
    }
    __syncthreads();
    PairCtx pc;
    if (a.pair) {
        // both CTAs of the cluster have initialised their barriers before either sends
        asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
        asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
        pc.on = true;
        asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(pc.rank));
        const uint32_t peer = pc.rank ^ 1u;
        pc.dst.xs = map_to_cta(sm.xs_u32, peer);
        pc.dst.gx = map_to_cta(sm.gx_u32, peer);
        pc.dst.gsum = map_to_cta(sm.gsum_u32, peer);
        pc.dst.bar = map_to_cta(smem_u32(sm.rx), peer);
        pc.r_rms = map_to_cta(smem_u32(sm.rms), peer);
        pc.r_free = map_to_cta(smem_u32(sm.free_gen), peer);
    }
    // phase p = 5 * layer + k, k: 0 RMSNorm + q|k|v, 1 attention, 2 o_proj, 3 RMSNorm + gate|up, 4 down_proj; p = 5 * Lyr: lm_head
    const int nphase = 5 * Lyr + 1;
    const unsigned epoch = *a.epoch;
    const uint32_t tag_base = epoch * (uint32_t)(2 * nphase + 2) + 1u;  // tag of (phase p, sub-result s) = tag_base + 2p + s: unique over launches, never 0

    // register budget: 20 warps x 96 registers at launch; warpgroup 0 (producer, epilogue, two spare warps) gives most of its share back
    // and the 16 consumer warps grow to 112 (per scheduler: 32 + 4 x 112 <= 5 x 96 registers per lane)
    if (warp < kAuxWarps) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 32;" ::: "memory");
        if (warp >= 2) return;
        if (warp == 0) {
            // ================= loader: every byte this CTA needs from HBM, in consumption order =================
            producer_walk(a, sm, cta, ncta, pos, lane);
            return;
        }
    if (warp == 1) {
        // ================= epilogue warp =================
        Red es;
        EpiState st;
        st.best = 0ull;
#pragma unroll 1
        for (int p = 0; p < nphase; p++) {
            const int l = p / 5, k = p - 5 * l;
            if (l < Lyr && k == 1) continue;  // attention publishes its own results
            const int oi = (l == Lyr) ? OPI_LMHEAD : ((k == 0) ? OPI_QKV : (k - 1));
            uint2 *out = (oi == OPI_QKV) ? a.qkv_ll : (oi == OPI_GATEUP ? a.act_ll : (oi == OPI_O ? a.delta_ll[0] : a.delta_ll[1]));
            epilogue_gemv(a, a.op[oi], sm, es, st, out, (oi == OPI_DOWN) ? 1 : 0, tag_base + 2u * (uint32_t)p, cta, ncta, lane);
            if (lane == 0) stamp(a, cta, nphase, p, 3);
        }
        unsigned long long key = st.best;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, key, off);
            key = other > key ? other : key;
        }
        if (lane == 0 && key) atomicMax(a.argmax_cell, key);
        // the logits and the arg-max contribution of this CTA are visible device-wide before the arrival
        __threadfence();
        __syncwarp();
        if (lane == 0) red_release_gpu(a.done);
        return;
    }
        return;  // (not reached: every warp of warpgroup 0 has returned above)
    }
    asm volatile("setmaxnreg.inc.sync.aligned.u32 112;" ::: "memory");

    // ================= consumers =================
    const int ctid = tid - 32 * kAuxWarps;
    const int cw = warp - kAuxWarps;
    Ring rs;
    Red cs;
    if (ctid < 256) sm.rope[ctid] = (ctid < 128) ? a.cos[(size_t)pos * 128 + ctid] : a.sin[(size_t)pos * 128 + ctid - 128];  // visible after the first phase's barrier
#pragma unroll 1
    for (int p = 0; p < nphase; p++) {
        const int l = p / 5, k = p - 5 * l;
        const uint32_t tag_in = tag_base + 2u * (uint32_t)(p - 1);  // primary result of the previous phase
        if (ctid == 0) stamp(a, cta, nphase, p, 0);
        if (l < Lyr && k == 1) {
            // ---- RoPE + KV append + attention ----
            attention_phase(a, a.layers[l], sm, rs, tag_in, tag_base + 2u * (uint32_t)p + 1u, tag_base + 2u * (uint32_t)p, cta, ncta, pos, ctid, cw, lane, p, nphase);
            if (ctid == 0) stamp(a, cta, nphase, p, 2);
            named_bar_sync(1, kConsumerThreads);  // the scratch aliases the activation planes of the next phase
            if (pc.on && ctid == 0) st_cluster_u32(pc.r_free, (uint32_t)(p + 1));  // the partner may mirror the next phase's planes into this CTA
            continue;
        }
        const int oi = (l == Lyr) ? OPI_LMHEAD : ((k == 0) ? OPI_QKV : (k - 1));
        const GemvOp &op = a.op[oi];
        int t0, t1;
        partition(op, cta, ncta, t0, t1);
        const bool work = t1 > t0;
        bool stage = work;  // pair mode: a CTA stages its half whenever either CTA of the pair has tiles in this phase
        if (pc.on) {
            int u0, u1;
            partition(op, cta ^ 1, ncta, u0, u1);
            stage = work || u1 > u0;
        }
        float inv = 1.f;
        if (oi == OPI_O) {
            if (stage) stage_half(a, op, sm, pc, a.attn_ll, tag_in, cta, ctid, lane, p, nphase);
        } else if (oi == OPI_DOWN) {
            if (stage) stage_half(a, op, sm, pc, a.act_ll, tag_in, cta, ctid, lane, p, nphase);
        } else {
            // the residual copy of this CTA must see every o_proj / down_proj output, whether or not the CTA owns tiles of this phase
            const float *gamma = (oi == OPI_LMHEAD) ? a.final_norm : (oi == OPI_QKV ? a.layers[l].input_norm : a.layers[l].post_norm);
            const uint2 *delta = (oi == OPI_GATEUP) ? a.delta_ll[0] : a.delta_ll[1];
            inv = stage_rms(a, op, sm, pc, delta, tag_in, gamma, token, p == 0, stage, cta, ctid, cw, lane, p, nphase);
        }
        if (ctid == 0) stamp(a, cta, nphase, p, 1);
        if (work) {
            if (op.plan[0].bw[0] == 16 && (op.NG & 15) == 0)
                consume_gemv_dense(op, sm, rs, cs, inv, cta, ncta, cw, lane);
            else
                consume_gemv(op, sm, rs, cs, inv, cta, ncta, cw, lane);
        }
        if (ctid == 0) stamp(a, cta, nphase, p, 2);
        named_bar_sync(1, kConsumerThreads);  // every warp is done with the planes before the next phase overwrites them
        if (pc.on && ctid == 0 && p + 1 < nphase) st_cluster_u32(pc.r_free, (uint32_t)(p + 1));  // (not after the last phase: the partner may be gone)
    }
    // ---- greedy token: decoded once every CTA's epilogue has contributed its maximum ----
    if (cta == 0 && ctid == 0) {
        const unsigned target = (epoch + 1u) * (unsigned)ncta;
        const long long t0 = clock64();
        while ((int)(ld_acquire_gpu(a.done) - target) < 0) {
            if (clock64() - t0 > kSpinLimit) __trap();
        }
        unsigned long long key = *reinterpret_cast<volatile unsigned long long *>(a.argmax_cell);
        if (a.tp_size > 1) {
            // vocabulary shards: publish the local key to every rank as two tagged words, take the global maximum
            const uint32_t tag = tag_base + 2u * (uint32_t)nphase;
            for (int pr = 0; pr < a.tp_size; pr++) {
                st_ll(a.tp_keys[pr] + (size_t)a.tp_rank * 2, (uint32_t)(key >> 32), tag, true);
                st_ll(a.tp_keys[pr] + (size_t)a.tp_rank * 2 + 1, (uint32_t)key, tag, true);
            }
            key = 0ull;
            for (int pr = 0; pr < a.tp_size; pr++) {
                const uint32_t hi = wait_ll1(a.tp_keys[a.tp_rank] + (size_t)pr * 2, tag, true), lo = wait_ll1(a.tp_keys[a.tp_rank] + (size_t)pr * 2 + 1, tag, true);
                const unsigned long long k2 = ((unsigned long long)hi << 32) | lo;
                key = k2 > key ? k2 : key;
            }
        }
        *a.next_token = (int)(0xFFFFFFFFu - (unsigned)(key & 0xFFFFFFFFull));
        *a.argmax_cell = 0ull;  // re-armed for the next launch (every CTA has arrived: nobody touches it any more)
        *a.epoch = epoch + 1u;
    }
}

// ------------------------------------------------------------------------------------------------------------ repack kernel
// scales half[rows][sf_w] + zeros u32[rows][zeros_w] (QM_CUDA, llm/tools/quantize_methods.py:370-442) -> one 1280-byte record per
// (16-row tile, 32-group stage): scales half[32 groups][8][2] (rows g and g + 8 adjacent), then zero points u8[32 groups][8][2] in the same order.
__global__ void repack_meta_kernel(W4Seg s0, W4Seg s1, W4Seg s2, int nseg, int pair, int NG, int zeros_w, int sf_w, int S, int num_tiles, uint8_t *out) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;  // (tile, s, gi)
    if (idx >= num_tiles * S * kStageGroups) return;
    const int gi = idx % kStageGroups, su = idx / kStageGroups;
    const int tile = su / S, s = su - tile * S;
    const int G = kStageGroups * s + gi;
    uint8_t *rec = out + (size_t)su * kMetaBytes;
    __half *so = reinterpret_cast<__half *>(rec) + gi * 16;  // [g][2]: rows g and g + 8 adjacent
    uint8_t *zo = rec + 1024 + gi * 16;                        // zero points, same order, one byte each
    for (int r = 0; r < 16; r++) {
        const W4Seg *seg = &s0;
        int row;
        if (pair) {
            seg = (r < 8) ? &s0 : &s1;
            row = tile * 8 + (r & 7);
        } else {
            row = tile * 16 + r;
            if (nseg > 1 && row >= s0.rows) {
                row -= s0.rows;
                seg = &s1;
                if (nseg > 2 && row >= s1.rows) {
                    row -= s1.rows;
                    seg = &s2;
                }
            }
        }
        const int slot = (r & 7) * 2 + (r >> 3);
        if (G < NG) {
            so[slot] = seg->scales[(size_t)row * sf_w + G];
            zo[slot] = (uint8_t)((seg->zeros[(size_t)row * zeros_w + (G >> 3)] >> ((G & 7) * 4)) & 0xFu);
        } else {
            so[slot] = __float2half(0.f);
            zo[slot] = 0;
        }
    }
}

}  // namespace

BoxPlan make_box_plan(int n, int *widths, int *nwidths) {
    BoxPlan pl{};
    int w[kMaxBoxes], nb = 0;
    // Dense boxes of up to 16 groups: their rows are whole 128-byte L2 lines (odd widths, conflict-free but not line-aligned, measured
    // 25 % slower end to end, profiles/README.md).
    w[nb++] = n < 16 ? n : 16;
    if (n > 16) w[nb++] = n - 16;
    int g0 = 0, off = 0;
    for (int i = 0; i < nb; i++) {
        pl.b0[i] = g0;
        pl.bw[i] = w[i];
        pl.off[i] = off;
        int m = -1;
        for (int k = 0; k < *nwidths; k++)
            if (widths[k] == w[i]) m = k;
        if (m < 0 && *nwidths < kMapsPerMat) {
            m = (*nwidths)++;
            widths[m] = w[i];
        }
        pl.map[i] = m;  // -1: more distinct widths than maps (caller rejects)
        g0 += w[i];
        off += 16 * w[i] * 64;
        pl.bytes += 16 * w[i] * 64;
    }
    pl.nbox = nb;
    return pl;
}

int attn_scratch_bytes(int nrep) { return 8 * 136 * 2 + kCW * nrep * 128 * 4 + kCW * nrep * 2 * 4; }

int attn_nsplit_max(int ncta, int KVH, int max_ctx) {
    int NS = ncta / KVH;
    if (NS < 1) NS = 1;
    const int nch = (max_ctx + kKvChunk - 1) / kKvChunk;
    return NS < nch ? NS : nch;
}

// everything next to the ring; the 16 bytes after the barriers hold the rx barrier and free_gen (padded)
static size_t fixed_bytes(int xs_bytes, int max_ng, int E) {
    return (size_t)xs_bytes + (size_t)E * 4 + (size_t)max_ng * 12 + (size_t)kRedBufs * kCW * 16 * 4 + 32 * 4 + 256 * 4 + (size_t)(2 * kMaxStages + 2 * kRedBufs) * 8 + 16 + 1024;
}
int pick_stages(int smem_optin, int xs_bytes, int max_ng, int E) {
    const long long avail = (long long)smem_optin - (long long)fixed_bytes(xs_bytes, max_ng, E);
    long long n = avail / kStageBytes;
    if (n > kMaxStages) n = kMaxStages;
    return n < 2 ? 0 : (int)n;
}
size_t smem_bytes(const Args &a) { return fixed_bytes(a.xs_bytes, a.max_ng, a.E) + (size_t)a.nst * kStageBytes; }

cudaError_t repack_meta(Ctx *ctx, const W4Seg *segs, int nseg, int pair, int IC, uint8_t *out, cudaStream_t stream) {
    const int NG = IC / kW4Group, S = (NG + kStageGroups - 1) / kStageGroups;
    int rows = 0;
    for (int i = 0; i < nseg; i++) rows += segs[i].rows;
    const int num_tiles = rows / 16;
    const int zw = zeros_width(IC, kW4Group);
    const int total = num_tiles * S * kStageGroups;
    if (total == 0) return cudaSuccess;
    repack_meta_kernel<<<(total + 127) / 128, 128, 0, stream>>>(segs[0], segs[nseg > 1 ? 1 : 0], segs[nseg > 2 ? 2 : 0], nseg, pair, NG, zw, zw * 8, S, num_tiles, out);
    (void)ctx;
    return cudaGetLastError();
}

cudaError_t encode_kv_tmap(CUtensorMap *out, const void *kv, long long rows) {
    typedef CUresult (*EncodeFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                 const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    void *sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q);
    if (e != cudaSuccess || !sym) return e != cudaSuccess ? e : cudaErrorNotSupported;
    const cuuint64_t gdim[2] = {128, (cuuint64_t)rows};
    const cuuint64_t gstride[1] = {256};
    const cuuint32_t box[2] = {64, (cuuint32_t)kKvChunk};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = reinterpret_cast<EncodeFn>(sym)(out, CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, const_cast<void *>(kv), gdim, gstride, box, estr,
                                                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? cudaSuccess : cudaErrorInvalidValue;
}

// can the grid run as co-resident clusters of two CTAs (one per TPC)?
bool pair_supported(Ctx *ctx, const Args &a) {
    if (ctx->num_sms % 2) return false;
    const size_t smem = smem_bytes(a);
    if (cudaFuncSetAttribute(decode_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smem_optin) != cudaSuccess) return false;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(ctx->num_sms);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int nclusters = 0;
    if (cudaOccupancyMaxActiveClusters(&nclusters, decode_persistent_kernel, &cfg) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return nclusters * 2 >= ctx->num_sms;
}

cudaError_t launch(Ctx *ctx, const Args &a, cudaStream_t stream) {
    const size_t smem = smem_bytes(a);
    if ((int)smem > ctx->smem_optin) return cudaErrorInvalidConfiguration;
    cudaError_t e = cudaFuncSetAttribute(decode_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->smem_optin);
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(ctx->num_sms);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeCooperative;  // all CTAs must be co-resident: they wait for each other's results
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    static bool pair_refused = false;  // a cluster launch was refused once in this process
    if (a.pair && !pair_refused) {
        // Clusters of two CTAs (one TPC) share the activation staging over distributed shared memory.  Launched with the cluster attribute ALONE:
        // profilers (ncu) cannot intercept a launch that is both cooperative and clustered (LaunchFailed), and co-residency -- what the cooperative
        // attribute would assert -- is established instead by pair_supported(): one CTA per SM fits for all num_sms / 2 clusters, and the step is the only
        // work on its stream.  A CTA that were not resident would surface through the bounded spins (__trap after ~10 s), not as a silent hang.
        cudaLaunchAttribute cattr[1];
        cattr[0].id = cudaLaunchAttributeClusterDimension;
        cattr[0].val.clusterDim.x = 2;
        cattr[0].val.clusterDim.y = 1;
        cattr[0].val.clusterDim.z = 1;
        cfg.attrs = cattr;
        cfg.numAttrs = 1;
        e = cudaLaunchKernelEx(&cfg, decode_persistent_kernel, a);
        if (e == cudaSuccess) return e;
        cudaGetLastError();  // a launch-configuration error is not sticky: run without clusters (every CTA stages the whole vector itself)
        pair_refused = true;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
    }
    Args single = a;
    single.pair = 0;
    return cudaLaunchKernelEx(&cfg, decode_persistent_kernel, single);
}

}  // namespace pk
}  // namespace tce
