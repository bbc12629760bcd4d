// persistent.h -- host/device interface of the persistent Llama decode kernel (decode_persistent.cu).
//
// One cooperative kernel per decoded token, one CTA per SM.  Everything a token needs from HBM -- packed weights, their repacked
// scales/zeros, and the K/V cache rows -- flows through ONE ring of TMA stages per CTA that is filled by a producer warp which depends
// on nothing but static data, so it runs ahead across all phase boundaries.  Phases hand their results to each other through
// flag-carrying 8-byte words (value + phase tag, stored and loaded as one unit): there is no grid barrier, fence or counter between
// the five phases of a layer -- a consumer simply spins on the words it needs.
#pragma once
#include "kernels.h"

namespace tce {
namespace pk {

constexpr int kCW = 16;                          // consumer warps
constexpr int kAuxWarps = 4;                     // warpgroup 0: loader warp, epilogue warp, two spare warps that only donate their registers
constexpr int kThreads = 32 * (kAuxWarps + kCW); // 640
constexpr int kConsumerThreads = 32 * kCW;       // 512
constexpr int kStageGroups = 32;                 // 128-k groups per ring stage: every consumer warp owns two of them
constexpr int kHalfBytes = 16384;                // 64 K rows or 64 V rows (one half of an attention stage)
constexpr int kMaxBoxes = 4;                     // TMA boxes per weight stage
constexpr int kMapsPerMat = 4;                   // tensor maps per weight matrix (one per distinct box width)
constexpr int kMetaOff = 2 * kHalfBytes;         // scales half[32 groups][8][2] (rows g, g+8 adjacent; 1 KiB) then zero points u8[32 groups][8][2] (512 B)
constexpr int kMetaBytes = 1536;
constexpr int kStageBytes = 34816;               // 32 KiB + 1.5 KiB meta (+ pad), 1 KiB multiple (128B-swizzle atoms of the K/V boxes)
constexpr int kMaxStages = 6;
constexpr int kRedBufs = 3;
constexpr int kKvChunk = 64;                     // cached positions per ring stage (K rows in the first half, V rows in the second)
constexpr int kAttnCps = 1;                      // least chunks per attention CTA: as many CTAs as the context has chunks take part, so that a CTA's K/V stages
                                                 // fit the ring slots left free by the tail of the q|k|v GEMV (a 4-chunk CTA waited ~3 us for its last stage)

enum XMode : int { PX_HALF = 0, PX_RMS_F32 = 1 };
enum Epi : int { PE_HALF_LL = 0, PE_DELTA_LL = 1, PE_SILU_LL = 2, PE_LOGITS = 3 };
enum OpIdx : int { OPI_QKV = 0, OPI_O = 1, OPI_GATEUP = 2, OPI_DOWN = 3, OPI_LMHEAD = 4, OPI_COUNT = 5 };

// shape of one GEMV op; identical for every layer, so it lives in the kernel parameter block
// A stage's <= 32 groups arrive as one or two dense TMA boxes of up to 16 groups (see make_box_plan).
struct BoxPlan {
    int nbox;
    int b0[kMaxBoxes];   // first group of the box within the stage
    int bw[kMaxBoxes];   // width in groups (<= 16)
    int off[kMaxBoxes];  // byte offset of the box inside the stage (1 KiB multiple)
    int map[kMaxBoxes];  // which of the matrix's tensor maps has this box width
    int bytes;           // sum over boxes of 16 * bw * 64
};
struct GemvOp {
    int IC, NG;          // input channels, 128-groups per row
    BoxPlan plan[2];     // [0] a full stage (min(32, NG) groups), [1] the last stage of a tile when NG % 32 != 0
    int S;               // stages per 16-row tile = ceil(NG / 32)
    int num_tiles;       // 16-row tiles (pair mode: 8 gate rows + 8 up rows)
    int nseg, pair;      // row segments (q|k|v = 3); pair = gate/up interleave
    int rows0, rows1;    // rows of segments 0 and 1 (tile -> segment)
    int x_mode, epi;
    int unit;            // 1: the op's tensor maps are the 3-D [group][row][64 B] views: a (tile, group) unit is 1 KiB contiguous in the stage
};

struct LayerDesc {       // per layer, global memory
    const uint8_t *meta[4];      // repacked scales|zeros of qkv, o, gate_up, down: [tile][S][1536 B]
    const float *input_norm, *post_norm;
    __half *k_cache, *v_cache;   // [KVH][max_ctx][128] of this layer (append)
    int k_row0, v_row0;          // first row of this layer's K / V slab in the cache tensor map
    int pad[2];
};

struct Args {
    GemvOp op[OPI_COUNT];
    const LayerDesc *layers;
    int num_layers;
    const CUtensorMap *maps;     // [num_layers][7 (q k v o gate up down)][kMapsPerMat], then lm_head [kMapsPerMat], then the KV cache map
    const uint8_t *lm_meta;
    const float *final_norm;
    const __half *embed;         // [rows][E]
    int embed_rows;
    // phase-to-phase hand-off buffers: 8-byte words {payload, tag}
    uint2 *delta_ll[2];          // [tp][E] o_proj (0) / down_proj (1) outputs per rank slot: fp32 payload (added to the residual by every reader)
    uint2 *qkv_ll;               // [(H + 2 KVH) * 64]  half2 payload
    uint2 *attn_ll;              // [H * 64]            half2 payload
    uint2 *act_ll;               // [F / 2]             half2 payload
    uint2 *part_ll;              // [H][nsplit_max][130] fp32 payload: flash-decode partials (o[128], m, l)
    float *logits;
    const int *tokpos;           // {token, position}
    int *next_token;
    unsigned long long *argmax_cell;
    unsigned *done;              // monotonic arrival counter of the final phase
    unsigned *epoch;             // launches completed so far
    int *error;                  // device error word (bad token / position)
    const float *cos, *sin;      // [max_ctx][128]
    float alpha, eps;
    int H, KVH, nrep, max_ctx, E, V, F;
    int nsplit_max;
    int nst;                     // ring depth
    int pair;                    // 1: launched as clusters of two CTAs that share the activation staging: each polls and quantises every other
                                 // 128-group and mirrors the result into its partner's shared memory (st.async over DSMEM)
    int xs_bytes;                // activation-plane buffer (also the attention scratch)
    int max_ng;
    // tensor parallel (tp_size > 1): every rank writes its o_proj / down_proj outputs into slot `tp_rank` of every rank's delta buffers
    int tp_size, tp_rank;
    uint2 *tp_delta[2][kMaxTP];  // [which][peer]: that peer's delta_ll[which] base
    uint2 *tp_keys[kMaxTP];      // every rank's arg-max key words [P][2]
    int vocab_base;              // global index of this rank's first vocabulary row
    unsigned long long *dbg;     // optional (TCE_PK_DEBUG=1): globaltimer stamps [cta][phase][8]: 0 phase entered, 1 staged, 2 consumed, 3 results written, 4.. sub-steps
};

size_t smem_bytes(const Args &a);
// ring depth that fits `smem_optin` next to the fixed buffers (0 = does not fit)
int pick_stages(int smem_optin, int xs_bytes, int max_ng, int E);
int attn_scratch_bytes(int nrep);
int attn_nsplit_max(int ncta, int KVH, int max_ctx);
cudaError_t launch(Ctx *ctx, const Args &a, cudaStream_t stream);
bool pair_supported(Ctx *ctx, const Args &a);  // the grid fits as co-resident clusters of two CTAs
// one-off repack of a (possibly multi-segment / gate-up paired) matrix's scales and zeros into per-stage records
cudaError_t repack_meta(Ctx *ctx, const W4Seg *segs, int nseg, int pair, int IC, uint8_t *out, cudaStream_t stream);
cudaError_t encode_kv_tmap(CUtensorMap *out, const void *kv, long long rows);
// split n <= 32 groups into dense boxes of at most 16 groups; `widths` collects the distinct widths (<= kMapsPerMat) of the op
BoxPlan make_box_plan(int n, int *widths, int *nwidths);

}  // namespace pk
}  // namespace tce
