// llama_decoder.cu -- one-token decode of an AWQ-INT4 Llama as a single CUDA graph.
//
// Call sites restated (reference, CUDA build): Int4LlamaForCausalLM::forward (cuda/Int4llamaForCausalLM.cu:17-50)
// -> Int4llamaDecoder::forward (cuda/Int4llamaDecoder.cu:57-112) -> 32 x Int4llamaDecoderLayer::forward
// (cuda/Int4llamaDecoderLayer.cu:73-115) -> Int4llamaAttention::forward (cuda/Int4llamaAttention.cu:116-229).
// The reference issues ~19 kernels + 128 memcpys per layer on stream 0; here a layer is 5 kernels
// (RMSNorm+QKV GEMV | RoPE+append+attention | o_proj+residual | RMSNorm+gate/up+SiLU*mul | down+residual),
// chained with programmatic dependent launch so each GEMV prefetches its weights while its predecessor drains.
// The residual stream is kept in fp32 (the reference's CUDA build keeps it in fp16, its CPU build in fp32).
#include "llama_decoder.h"

#include "kernels_tp.h"
#include "persistent.h"

#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

namespace tce {

#define DCK(call)                              \
    do {                                       \
        cudaError_t e__ = (call);              \
        if (e__ != cudaSuccess) return e__;    \
    } while (0)

static bool w4_ok(const tce_w4_tensor &t, int oc, int ic) { return t.w && t.zeros && t.scales && t.oc == oc && t.ic == ic; }

LlamaDecoder *LlamaDecoder::create(Ctx *ctx, int attn_chunk, const tce_llama_config &cfg, const tce_llama_weights &w, std::string *err) {
    auto bad = [&](const char *m) {
        *err = m;
        return (LlamaDecoder *)nullptr;
    };
    if (cfg.head_dim != 128) return bad("head_dim must be 128");
    if (cfg.num_layers < 1 || cfg.num_heads < 1 || cfg.num_kv_heads < 1 || cfg.num_heads % cfg.num_kv_heads) return bad("bad head configuration");
    if (cfg.embed_dim % 128 || cfg.hidden_dim % 128) return bad("embed_dim / hidden_dim must be multiples of the 128 group");
    if (cfg.tp_size > kMaxTP || cfg.tp_size < 0 || (cfg.tp_size > 1 && (cfg.tp_rank < 0 || cfg.tp_rank >= cfg.tp_size))) return bad("bad tensor-parallel rank/size");
    const int E = cfg.embed_dim, F = cfg.hidden_dim, H = cfg.num_heads, KVH = cfg.num_kv_heads, hd = cfg.head_dim, V = cfg.vocab_size;
    if (!w.embed_f16 || !w.layers || !w.final_norm) return bad("missing weights");
    if (!w4_ok(w.lm_head, V, E) || V % 16) return bad("lm_head shape");
    for (int l = 0; l < cfg.num_layers; l++) {
        const tce_llama_layer &L = w.layers[l];
        if (!w4_ok(L.q, H * hd, E) || !w4_ok(L.k, KVH * hd, E) || !w4_ok(L.v, KVH * hd, E) || !w4_ok(L.o, E, H * hd) || !w4_ok(L.gate, F, E) ||
            !w4_ok(L.up, F, E) || !w4_ok(L.down, E, F) || !L.input_norm || !L.post_norm)
            return bad("layer weight shape");
    }
    LlamaDecoder *d = new LlamaDecoder();
    d->ctx_ = ctx;
    d->attn_chunk_ = attn_chunk;
    d->cfg_ = cfg;
    d->w_ = w;
    d->layers_.assign(w.layers, w.layers + cfg.num_layers);
    d->w_.layers = d->layers_.data();
    d->use_graphs_ = getenv("TCE_NO_GRAPH") == nullptr;
    d->atomic_residual_ = getenv("TCE_DETERMINISTIC") == nullptr;
    const size_t kv_elems = (size_t)cfg.num_layers * 2 * KVH * cfg.max_ctx * hd;
    cudaError_t e = cudaSuccess;
    auto A = [&](void **p, size_t bytes) {
        if (e == cudaSuccess) e = cudaMalloc(p, bytes);
    };
    A((void **)&d->d_kv_, kv_elems * sizeof(__half));
    A((void **)&d->d_resid_, (size_t)2 * E * sizeof(float));  // two buffers: the tensor-parallel path ping-pongs the residual
    A((void **)&d->d_qkv_, (size_t)(H + 2 * KVH) * hd * sizeof(__half));
    A((void **)&d->d_attn_, (size_t)H * hd * sizeof(__half));
    A((void **)&d->d_act_, (size_t)F * sizeof(__half));
    A((void **)&d->d_logits_, (size_t)V * sizeof(float));
    A((void **)&d->d_tokpos_, 4 * sizeof(int));
    A((void **)&d->d_next_, sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(d->d_kv_, 0, kv_elems * sizeof(__half));
    if (e == cudaSuccess) e = cudaMemset(d->d_tokpos_, 0, 4 * sizeof(int));  // [3] = tensor-parallel step counter, advanced on the device
    if (e == cudaSuccess) e = cudaMalloc((void **)&d->d_tokpos_safe_, 4 * sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(d->d_tokpos_safe_, 0, 4 * sizeof(int));
    if (e == cudaSuccess) e = cudaMallocHost((void **)&d->h_tokpos_, 4 * sizeof(int));
    if (e == cudaSuccess) e = cudaMallocHost((void **)&d->h_logits_, (size_t)V * sizeof(float));
    if (e == cudaSuccess) e = cudaMallocHost((void **)&d->h_next_, sizeof(int));
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&d->cap_stream_, cudaStreamNonBlocking);
    if (e == cudaSuccess) {
        if (w.rope_cos && w.rope_sin) {
            d->d_cos_ = const_cast<float *>(w.rope_cos);
            d->d_sin_ = const_cast<float *>(w.rope_sin);
        } else {
            // HF rotate-half tables: cos/sin(pos * theta^(-2i/hd)) duplicated over both halves
            std::vector<float> hc((size_t)cfg.max_ctx * hd), hs((size_t)cfg.max_ctx * hd);
            const double theta = cfg.rope_theta > 0 ? cfg.rope_theta : 10000.0;
            for (int p = 0; p < cfg.max_ctx; p++)
                for (int i = 0; i < hd / 2; i++) {
                    const double inv = 1.0 / pow(theta, (2.0 * i) / hd);
                    const double ang = p * inv;
                    hc[(size_t)p * hd + i] = hc[(size_t)p * hd + i + hd / 2] = (float)cos(ang);
                    hs[(size_t)p * hd + i] = hs[(size_t)p * hd + i + hd / 2] = (float)sin(ang);
                }
            A((void **)&d->d_cos_, hc.size() * sizeof(float));
            A((void **)&d->d_sin_, hs.size() * sizeof(float));
            d->own_rope_ = true;
            if (e == cudaSuccess) e = cudaMemcpy(d->d_cos_, hc.data(), hc.size() * sizeof(float), cudaMemcpyHostToDevice);
            if (e == cudaSuccess) e = cudaMemcpy(d->d_sin_, hs.data(), hs.size() * sizeof(float), cudaMemcpyHostToDevice);
        }
    }
    if (e != cudaSuccess) {
        *err = std::string("allocation failed: ") + cudaGetErrorString(e);
        delete d;
        return nullptr;
    }
    d->persistent_ = getenv("TCE_PERSISTENT") ? atoi(getenv("TCE_PERSISTENT")) != 0 : true;
    d->tp_ = cfg.tp_size > 1 ? cfg.tp_size : 1;
    if (d->tp_ > 1) {
        // tensor parallel: one peer-visible allocation [gather A|B: 2 x P x E fp32][flags: 3 x P u32 (256-B padded)][keys: P u64]
        d->tp_gather_floats_ = (size_t)2 * d->tp_ * E;
        d->tp_bytes_ = d->tp_gather_floats_ * sizeof(float) + 256 + (size_t)kMaxTP * sizeof(unsigned long long);
        // persistent kernel layout: two delta buffers of P x E {float, tag} words + P x 2 key words
        const size_t pk_bytes = ((size_t)2 * d->tp_ * E + (size_t)2 * d->tp_) * sizeof(uint2);
        if (d->tp_bytes_ < pk_bytes) d->tp_bytes_ = pk_bytes;
        if (cudaMalloc((void **)&d->tp_buf_, d->tp_bytes_) != cudaSuccess || cudaMemset(d->tp_buf_, 0, d->tp_bytes_) != cudaSuccess) {
            *err = "tensor-parallel buffer allocation failed";
            delete d;
            return nullptr;
        }
        cudaDeviceSynchronize();
        d->kernels_per_step_ = d->persistent_ ? 1 : 1 + 7 * cfg.num_layers + 4;
        return d;  // the op list needs the peers' pointers: built in tp_connect()
    }
    d->build_ops();
    if (d->persistent_) {
        std::string why;
        cudaError_t me = d->build_persistent(&why);
        if (me == cudaErrorNotSupported) {
            d->persistent_ = false;  // shape outside the persistent kernel's envelope: one kernel per op
        } else if (me != cudaSuccess) {
            *err = std::string("persistent kernel setup failed: ") + why + " " + cudaGetErrorString(me);
            delete d;
            return nullptr;
        }
    }
    d->kernels_per_step_ = d->persistent_ ? 1 : 1 + 5 * cfg.num_layers + 2;
    return d;
}

LlamaDecoder::~LlamaDecoder() {
    if (g_host_) cudaGraphExecDestroy(g_host_);
    if (g_dev_) cudaGraphExecDestroy(g_dev_);
    if (cap_stream_) cudaStreamDestroy(cap_stream_);
    cudaFree(d_kv_);
    cudaFree(d_resid_);
    cudaFree(d_qkv_);
    cudaFree(d_attn_);
    cudaFree(d_act_);
    cudaFree(d_logits_);
    cudaFree(d_tokpos_);
    cudaFree(d_gen_);
    cudaFree(d_tokpos_safe_);
    for (int b = 0; b < 2; b++) {
        cudaFree(pf_w16_[b]);
        if (pf_expanded_[b]) cudaEventDestroy(pf_expanded_[b]);
        if (pf_consumed_[b]) cudaEventDestroy(pf_consumed_[b]);
    }
    if (pf_side_) cudaStreamDestroy(pf_side_);
    cudaFree(d_next_);
    cudaFree(pf_x_);
    cudaFree(pf_xn_);
    cudaFree(pf_qkv_);
    cudaFree(pf_att_);
    cudaFree(pf_gu_);
    cudaFree(pf_act_);
    cudaFree(pf_tok_);
    for (void *p : pk_allocs_) cudaFree(p);
    for (int p = 0; p < tp_; p++)
        if (p != cfg_.tp_rank && tp_peer_[p]) cudaIpcCloseMemHandle(tp_peer_[p]);
    cudaFree(tp_buf_);
    if (own_rope_) {
        cudaFree(d_cos_);
        cudaFree(d_sin_);
    }
    if (h_tokpos_) cudaFreeHost(h_tokpos_);
    if (h_logits_) cudaFreeHost(h_logits_);
    if (h_next_) cudaFreeHost(h_next_);
}

void *LlamaDecoder::kv_cache(int layer, int which) const {
    if (layer < 0 || layer >= cfg_.num_layers || which < 0 || which > 1) return nullptr;
    const size_t per = (size_t)cfg_.num_kv_heads * cfg_.max_ctx * cfg_.head_dim;
    return d_kv_ + ((size_t)layer * 2 + which) * per;
}

static W4Seg seg_of(const tce_w4_tensor &t) { return W4Seg{(const uint32_t *)t.w, (const uint32_t *)t.zeros, (const __half *)t.scales, t.oc}; }

cudaError_t LlamaDecoder::enqueue_gemvs(int *count) {
    if (tp_ > 1) return cudaErrorNotSupported;  // the GEMVs of a tensor-parallel step poll their peers: without the rest of the step they would spin
    *count = 4 * cfg_.num_layers + 1;
    return enqueue_step(d_tokpos_, ctx_->stream, false, true);
}

cudaError_t LlamaDecoder::tp_handle(void *out64) {
    if (tp_ <= 1 || !tp_buf_) return cudaErrorInvalidValue;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle size");
    return cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t *>(out64), tp_buf_);
}

cudaError_t LlamaDecoder::tp_connect(const void *handles) {
    if (tp_ <= 1) return cudaErrorInvalidValue;
    const cudaIpcMemHandle_t *h = reinterpret_cast<const cudaIpcMemHandle_t *>(handles);
    for (int p = 0; p < tp_; p++) {
        if (p == cfg_.tp_rank) {
            tp_peer_[p] = tp_buf_;
        } else {
            DCK(cudaIpcOpenMemHandle((void **)&tp_peer_[p], h[p], cudaIpcMemLazyEnablePeerAccess));
        }
    }
    tp_connected_ = true;
    build_ops();
    if (persistent_) {
        std::string why;
        cudaError_t e = build_persistent(&why);
        if (e == cudaErrorNotSupported) {
            persistent_ = false;
            kernels_per_step_ = 1 + 7 * cfg_.num_layers + 4;
        } else if (e != cudaSuccess) {
            return e;
        }
    }
    return cudaSuccess;
}

// The op list of one decode step (built once): the graph path launches one kernel per op, the persistent kernel
// turns the same list into its phase table.
void LlamaDecoder::build_ops() {
    const int E = cfg_.embed_dim, F = cfg_.hidden_dim, H = cfg_.num_heads, KVH = cfg_.num_kv_heads, hd = cfg_.head_dim;
    ops_.clear();
    StepOp emb;
    emb.type = OP_EMBED;
    ops_.push_back(emb);
    // ---- tensor-parallel plumbing (tp_ == 1: every helper below is a no-op) ----
    const int P = tp_, per_step = 2 * cfg_.num_layers + 1;
    float *resid[2] = {d_resid_, d_resid_ + E};
    int cur = 0;  // residual buffer holding the stream
    auto gather_of = [&](int peer, int buf) { return reinterpret_cast<float *>(tp_peer_[peer]) + ((size_t)buf * P) * E; };            // [P][E]
    auto flags_of = [&](int peer, int buf) { return reinterpret_cast<unsigned *>(reinterpret_cast<float *>(tp_peer_[peer]) + tp_gather_floats_) + buf * kMaxTP; };
    auto keys_of = [&](int peer) { return reinterpret_cast<unsigned long long *>(reinterpret_cast<uint8_t *>(tp_peer_[peer]) + tp_gather_floats_ * sizeof(float) + 256); };
    const int me = cfg_.tp_rank;
    // receive side of collective k (the buffer it used): fold the gathered partials into the residual in this prologue
    auto tp_recv = [&](W4GemvParams &p, int buf, int k) {
        if (P <= 1) return;
        p.tp_size = P;
        p.x = resid[cur];
        p.tp_in = gather_of(me, buf);
        p.tp_flags = flags_of(me, buf);
        p.tp_step = d_tokpos_ + 3;
        p.tp_k = k;
        p.tp_per_step = per_step;
        p.resid_out = resid[cur ^ 1];
        cur ^= 1;
    };
    // send side: scatter epilogue + signal op
    auto tp_send = [&](W4GemvParams &p, int buf, int k) {
        p.tp_size = P;
        p.tp_sig_counter = flags_of(me, 0) + 32 + buf;  // spare words of the local flag block
        for (int q = 0; q < P; q++) p.tp_sig_flag[q] = flags_of(q, buf) + me;
        p.tp_sig_k = k;
        p.tp_step = d_tokpos_ + 3;
        p.tp_per_step = per_step;
        p.epi = EPI_TP_SCATTER_F32;
        p.atomic_residual = false;
        p.y = nullptr;
        for (int q = 0; q < P; q++) p.tp_out[q] = gather_of(q, buf) + (size_t)me * E;
    };
    auto push_signal = [&](int buf, int k) {
        StepOp op;
        op.type = OP_TP_SIGNAL;
        op.sig = TpSignalArgs{};
        for (int q = 0; q < P; q++) op.sig.peer_flag[q] = flags_of(q, buf) + me;
        op.sig.tp_size = P;
        op.sig.step = d_tokpos_ + 3;
        op.sig.k = k;
        op.sig.per_step = per_step;
        ops_.push_back(op);
    };
    for (int l = 0; l < cfg_.num_layers; l++) {
        const tce_llama_layer &L = layers_[l];
        {  // RMSNorm(input_layernorm) + fused q|k|v projection
            StepOp op;
            op.type = OP_GEMV;
            W4GemvParams &p = op.g;
            p.nseg = 3;
            p.seg[0] = seg_of(L.q);
            p.seg[1] = seg_of(L.k);
            p.seg[2] = seg_of(L.v);
            p.IC = E;
            p.M = 1;
            p.x = d_resid_;
            p.x_mode = X_RMSNORM_F32;
            p.ldx = E;
            p.gamma = L.input_norm;
            p.eps = cfg_.rms_eps;
            p.y = d_qkv_;
            p.epi = EPI_STORE_HALF;
            p.x = resid[cur];
            if (l > 0) tp_recv(p, 1, 2 * (l - 1) + 1);
            ops_.push_back(op);
        }
        {  // RoPE + in-place KV append + attention over the cache
            StepOp op;
            op.type = OP_ATTN;
            AttnDecodeArgs &a = op.at;
            a = AttnDecodeArgs{};
            a.qkv = d_qkv_;
            a.k_cache = (__half *)kv_cache(l, 0);
            a.v_cache = (__half *)kv_cache(l, 1);
            a.cos = d_cos_;
            a.sin = d_sin_;
            a.out = d_attn_;
            a.alpha = cfg_.qk_alpha > 0 ? cfg_.qk_alpha : 1.0f / sqrtf((float)hd);
            a.num_heads = H;
            a.num_kv_heads = KVH;
            a.head_dim = hd;
            a.max_ctx = cfg_.max_ctx;
            a.chunk = attn_chunk_;
            ops_.push_back(op);
        }
        {  // o_proj, accumulated straight into the residual stream
            StepOp op;
            op.type = OP_GEMV;
            W4GemvParams &p = op.g;
            p.nseg = 1;
            p.seg[0] = seg_of(L.o);
            p.IC = H * hd;
            p.M = 1;
            p.x = d_attn_;
            p.x_mode = X_HALF;
            p.y = resid[cur];
            p.epi = EPI_ADD_F32;
            p.atomic_residual = atomic_residual_;
            if (P > 1) tp_send(p, 0, 2 * l);
            ops_.push_back(op);
        }
        {  // RMSNorm(post_attention_layernorm) + gate/up with SiLU(gate)*up epilogue
            StepOp op;
            op.type = OP_GEMV;
            W4GemvParams &p = op.g;
            p.nseg = 2;
            p.pair_mode = 1;
            p.seg[0] = seg_of(L.gate);
            p.seg[1] = seg_of(L.up);
            p.IC = E;
            p.M = 1;
            p.x = resid[cur];
            p.x_mode = X_RMSNORM_F32;
            p.gamma = L.post_norm;
            p.eps = cfg_.rms_eps;
            p.y = d_act_;
            p.epi = EPI_SILU_MUL_HALF;
            p.ldy = F;
            tp_recv(p, 0, 2 * l);
            ops_.push_back(op);
        }
        {  // down_proj + residual
            StepOp op;
            op.type = OP_GEMV;
            W4GemvParams &p = op.g;
            p.nseg = 1;
            p.seg[0] = seg_of(L.down);
            p.IC = F;
            p.M = 1;
            p.x = d_act_;
            p.x_mode = X_HALF;
            p.y = resid[cur];
            p.epi = EPI_ADD_F32;
            p.atomic_residual = atomic_residual_;
            if (P > 1) tp_send(p, 1, 2 * l + 1);
            ops_.push_back(op);
        }
    }
    {  // final RMSNorm + lm_head -> fp32 logits (reference: lm_head GEMV + half2float, cuda/Int4llamaForCausalLM.cu:33-38)
        StepOp op;
        op.type = OP_GEMV;
        W4GemvParams &p = op.g;
        p.nseg = 1;
        p.seg[0] = seg_of(w_.lm_head);
        p.IC = E;
        p.M = 1;
        p.x = resid[cur];
        p.x_mode = X_RMSNORM_F32;
        p.gamma = w_.final_norm;
        p.eps = cfg_.rms_eps;
        p.y = d_logits_;
        p.epi = EPI_STORE_F32;
        tp_recv(p, 1, 2 * (cfg_.num_layers - 1) + 1);
        ops_.push_back(op);
    }
    if (P > 1) {
        // greedy token over the vocabulary shards: scatter the local key, signal, pick the global maximum
        StepOp sc;
        sc.type = OP_TP_ARGMAX_SCATTER;
        sc.am = TpArgmaxArgs{};
        sc.am.logits = d_logits_;
        sc.am.n_local = cfg_.vocab_size;
        sc.am.index_base = me * cfg_.vocab_size;
        for (int q = 0; q < P; q++) sc.am.peer_key[q] = keys_of(q) + me;
        sc.am.tp_size = P;
        ops_.push_back(sc);
        push_signal(2, 2 * cfg_.num_layers);
        StepOp fin;
        fin.type = OP_TP_ARGMAX_FINISH;
        fin.amf = TpArgmaxFinishArgs{};
        fin.amf.keys = keys_of(me);
        fin.amf.flags = flags_of(me, 2);
        fin.amf.step = d_tokpos_ + 3;
        fin.amf.k = 2 * cfg_.num_layers;
        fin.amf.per_step = per_step;
        fin.amf.tp_size = P;
        fin.amf.next_token = d_next_;
        ops_.push_back(fin);
    } else {
        StepOp am;
        am.type = OP_ARGMAX;
        ops_.push_back(am);
    }
}

// Everything the persistent decode kernel (decode_persistent.cu) needs beyond the caller's weights: one 2-D tensor map per packed
// matrix, the per-stage scales|zeros records (a one-off repack of the QM_CUDA scales / zeros arrays into the order the TMA ring
// consumes them: SURVEY.md 8(f)2 "repack once into the TMA-friendly interleave"), the layer table and the tagged hand-off buffers.
cudaError_t LlamaDecoder::build_persistent(std::string *err) {
    const int E = cfg_.embed_dim, F = cfg_.hidden_dim, H = cfg_.num_heads, KVH = cfg_.num_kv_heads, hd = cfg_.head_dim, V = cfg_.vocab_size;
    const int Lyr = cfg_.num_layers, ncta = ctx_->num_sms;
    const int nrep = H / KVH;
    auto no = [&](const char *m) {
        if (err) *err = m;
        return cudaErrorNotSupported;
    };
    if (hd != 128 || nrep > 4 || ncta < KVH || F % 16 || V % 16) return no("shape outside the persistent kernel's envelope");
    int coop = 0;
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, ctx_->device);
    if (!coop) return no("device cannot launch cooperative kernels");
    pk::Args a{};
    auto mk = [&](int IC, int rows, int nseg, int pair, int rows0, int rows1, int x_mode, int epi) {
        pk::GemvOp o{};
        o.IC = IC;
        o.NG = IC / kW4Group;
        o.S = (o.NG + pk::kStageGroups - 1) / pk::kStageGroups;
        o.num_tiles = rows / 16;
        o.nseg = nseg;
        o.pair = pair;
        o.rows0 = rows0;
        o.rows1 = rows1;
        o.x_mode = x_mode;
        o.epi = epi;
        return o;
    };
    // TMA box plans (see make_box_plan) and the distinct widths each op needs a tensor map for
    int widths[pk::OPI_COUNT][pk::kMapsPerMat] = {}, nwidths[pk::OPI_COUNT] = {};
    const bool tp = tp_ > 1;
    a.op[pk::OPI_QKV] = mk(E, (H + 2 * KVH) * hd, 3, 0, H * hd, KVH * hd, pk::PX_RMS_F32, pk::PE_HALF_LL);
    a.op[pk::OPI_O] = mk(H * hd, E, 1, 0, E, 0, pk::PX_HALF, pk::PE_DELTA_LL);
    a.op[pk::OPI_GATEUP] = mk(E, 2 * F, 2, 1, F, F, pk::PX_RMS_F32, pk::PE_SILU_LL);
    a.op[pk::OPI_DOWN] = mk(F, E, 1, 0, E, 0, pk::PX_HALF, pk::PE_DELTA_LL);
    a.op[pk::OPI_LMHEAD] = mk(E, V, 1, 0, V, 0, pk::PX_RMS_F32, pk::PE_LOGITS);
    int max_ic = 0, max_ng = 0;
    for (int i = 0; i < pk::OPI_COUNT; i++) {
        const int NG = a.op[i].NG, full = NG < pk::kStageGroups ? NG : pk::kStageGroups, rem = NG % pk::kStageGroups;
        a.op[i].plan[0] = pk::make_box_plan(full, widths[i], &nwidths[i]);
        a.op[i].plan[1] = (NG > pk::kStageGroups && rem) ? pk::make_box_plan(rem, widths[i], &nwidths[i]) : a.op[i].plan[0];
        for (int k = 0; k < pk::kMaxBoxes; k++)
            if ((k < a.op[i].plan[0].nbox && a.op[i].plan[0].map[k] < 0) || (k < a.op[i].plan[1].nbox && a.op[i].plan[1].map[k] < 0)) return no("too many box widths");
        // unit boxes ([group][row][64 B], conflict-free LDS.128: +1.3 %, profiles/README.md) where the dense consumer applies (every stage made
        // of 16-group boxes)
        a.op[i].unit = (a.op[i].plan[0].bw[0] == 16 && (NG & 15) == 0) ? 1 : 0;
        if (a.op[i].IC > max_ic) max_ic = a.op[i].IC;
        if (a.op[i].NG > max_ng) max_ng = a.op[i].NG;
        if (a.op[i].IC % kW4Group || a.op[i].num_tiles < 1) return no("bad GEMV shape");
    }
    max_ng = (max_ng + 3) & ~3;
    int xs = 4 * max_ic;  // four int8 activation planes
    if (xs < pk::attn_scratch_bytes(nrep)) xs = pk::attn_scratch_bytes(nrep);
    xs = (xs + 15) & ~15;
    a.xs_bytes = xs;
    a.max_ng = max_ng;
    a.E = E;
    a.nst = pk::pick_stages(ctx_->smem_optin, xs, max_ng, E);
    if (a.nst < 2) return no("shared memory too small for the persistent kernel");
    a.pair = 0;  // decided below, once the shared-memory footprint is known

    auto dalloc = [&](size_t bytes) -> void * {
        void *p = nullptr;
        if (cudaMalloc(&p, bytes ? bytes : 16) != cudaSuccess) return nullptr;
        pk_allocs_.push_back(p);
        return p;
    };
    cudaStream_t s = ctx_->stream;
    // ---- tensor maps: [Lyr][7] + lm_head + KV cache ----
    std::vector<CUtensorMap> maps(((size_t)Lyr * 7 + 1) * pk::kMapsPerMat + 1);
    memset(maps.data(), 0, maps.size() * sizeof(CUtensorMap));
    std::vector<pk::LayerDesc> descs(Lyr);
    const size_t per_kv = (size_t)KVH * cfg_.max_ctx;  // rows per (layer, K|V) slab
    for (int l = 0; l < Lyr; l++) {
        const tce_llama_layer &L = layers_[l];
        const tce_w4_tensor *t7[7] = {&L.q, &L.k, &L.v, &L.o, &L.gate, &L.up, &L.down};
        const int opi[7] = {pk::OPI_QKV, pk::OPI_QKV, pk::OPI_QKV, pk::OPI_O, pk::OPI_GATEUP, pk::OPI_GATEUP, pk::OPI_DOWN};
        for (int i = 0; i < 7; i++) {
            const pk::GemvOp &o = a.op[opi[i]];
            for (int k = 0; k < nwidths[opi[i]]; k++)
                DCK((o.unit ? encode_w4_tmap_units : encode_w4_tmap)(&maps[((size_t)l * 7 + i) * pk::kMapsPerMat + k], t7[i]->w, t7[i]->oc, t7[i]->ic, widths[opi[i]][k],
                                                                   o.pair ? 8 : 16));
        }
        pk::LayerDesc &D = descs[l];
        memset(&D, 0, sizeof(D));
        const W4Seg qkv[3] = {seg_of(L.q), seg_of(L.k), seg_of(L.v)}, o1[1] = {seg_of(L.o)}, gu[2] = {seg_of(L.gate), seg_of(L.up)}, d1[1] = {seg_of(L.down)};
        const W4Seg *segs[4] = {qkv, o1, gu, d1};
        const int nsegs[4] = {3, 1, 2, 1}, pairs[4] = {0, 0, 1, 0};
        const int ops4[4] = {pk::OPI_QKV, pk::OPI_O, pk::OPI_GATEUP, pk::OPI_DOWN};
        for (int i = 0; i < 4; i++) {
            const pk::GemvOp &o = a.op[ops4[i]];
            uint8_t *m = (uint8_t *)dalloc((size_t)o.num_tiles * o.S * pk::kMetaBytes);
            if (!m) return cudaErrorMemoryAllocation;
            DCK(pk::repack_meta(ctx_, segs[i], nsegs[i], pairs[i], o.IC, m, s));
            D.meta[i] = m;
        }
        D.input_norm = L.input_norm;
        D.post_norm = L.post_norm;
        D.k_cache = (__half *)kv_cache(l, 0);
        D.v_cache = (__half *)kv_cache(l, 1);
        D.k_row0 = (int)(((size_t)l * 2 + 0) * per_kv);
        D.v_row0 = (int)(((size_t)l * 2 + 1) * per_kv);
    }
    {
        const pk::GemvOp &o = a.op[pk::OPI_LMHEAD];
        for (int k = 0; k < nwidths[pk::OPI_LMHEAD]; k++)
            DCK((o.unit ? encode_w4_tmap_units : encode_w4_tmap)(&maps[(size_t)Lyr * 7 * pk::kMapsPerMat + k], w_.lm_head.w, w_.lm_head.oc, w_.lm_head.ic,
                                                               widths[pk::OPI_LMHEAD][k], 16));
        uint8_t *m = (uint8_t *)dalloc((size_t)o.num_tiles * o.S * pk::kMetaBytes);
        if (!m) return cudaErrorMemoryAllocation;
        const W4Seg lm[1] = {seg_of(w_.lm_head)};
        DCK(pk::repack_meta(ctx_, lm, 1, 0, o.IC, m, s));
        a.lm_meta = m;
        DCK(pk::encode_kv_tmap(&maps[((size_t)Lyr * 7 + 1) * pk::kMapsPerMat], d_kv_, (long long)Lyr * 2 * per_kv));
    }
    CUtensorMap *dmaps = (CUtensorMap *)dalloc(maps.size() * sizeof(CUtensorMap));
    pk::LayerDesc *ddesc = (pk::LayerDesc *)dalloc(descs.size() * sizeof(pk::LayerDesc));
    a.nsplit_max = pk::attn_nsplit_max(ncta, KVH, cfg_.max_ctx);
    // hand-off buffers ({payload, tag} words; tag 0 = never written)
    const size_t n_qkv = (size_t)(H + 2 * KVH) * 64, n_attn = (size_t)H * 64, n_act = (size_t)F / 2, n_part = (size_t)H * a.nsplit_max * 130;
    const size_t ll_words = n_qkv + n_attn + n_act + n_part + (tp ? 0 : (size_t)2 * E);
    uint2 *ll = (uint2 *)dalloc(ll_words * sizeof(uint2));
    // [arg-max cell u64][epoch u32][error i32][done u32]
    uint8_t *ctl = (uint8_t *)dalloc(32);
    if (!dmaps || !ddesc || !ll || !ctl) return cudaErrorMemoryAllocation;
    DCK(cudaMemcpyAsync(dmaps, maps.data(), maps.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice, s));
    DCK(cudaMemcpyAsync(ddesc, descs.data(), descs.size() * sizeof(pk::LayerDesc), cudaMemcpyHostToDevice, s));
    DCK(cudaMemsetAsync(ll, 0, ll_words * sizeof(uint2), s));
    DCK(cudaMemsetAsync(ctl, 0, 32, s));
    DCK(cudaStreamSynchronize(s));  // `maps` / `descs` are host temporaries
    a.layers = ddesc;
    a.num_layers = Lyr;
    a.maps = dmaps;
    a.final_norm = w_.final_norm;
    a.embed = (const __half *)w_.embed_f16;
    a.embed_rows = V * tp_;
    a.qkv_ll = ll;
    a.attn_ll = a.qkv_ll + n_qkv;
    a.act_ll = a.attn_ll + n_attn;
    a.part_ll = a.act_ll + n_act;
    a.logits = d_logits_;
    a.tokpos = d_tokpos_;
    a.next_token = d_next_;
    a.argmax_cell = reinterpret_cast<unsigned long long *>(ctl);
    a.epoch = reinterpret_cast<unsigned *>(ctl + 8);
    a.error = reinterpret_cast<int *>(ctl + 12);
    a.done = reinterpret_cast<unsigned *>(ctl + 16);
    a.cos = d_cos_;
    a.sin = d_sin_;
    a.alpha = cfg_.qk_alpha > 0 ? cfg_.qk_alpha : 1.0f / sqrtf((float)hd);
    a.eps = cfg_.rms_eps;
    a.H = H;
    a.KVH = KVH;
    a.nrep = nrep;
    a.max_ctx = cfg_.max_ctx;
    a.V = V;
    a.F = F;
    a.tp_size = tp_;
    a.tp_rank = tp ? cfg_.tp_rank : 0;
    a.vocab_base = tp ? cfg_.tp_rank * V : 0;
    if (tp) {
        // peer-visible allocation of every rank: [delta 0: P x E words][delta 1: P x E words][keys: P x 2 words]
        for (int q = 0; q < tp_; q++) {
            uint2 *base = reinterpret_cast<uint2 *>(tp_peer_[q]);
            a.tp_delta[0][q] = base;
            a.tp_delta[1][q] = base + (size_t)tp_ * E;
            a.tp_keys[q] = base + (size_t)2 * tp_ * E;
        }
        a.delta_ll[0] = a.tp_delta[0][a.tp_rank];
        a.delta_ll[1] = a.tp_delta[1][a.tp_rank];
    } else {
        a.delta_ll[0] = a.part_ll + n_part;
        a.delta_ll[1] = a.delta_ll[0] + E;
    }
    if (getenv("TCE_PK_DEBUG") && atoi(getenv("TCE_PK_DEBUG"))) {
        const size_t n = (size_t)ncta * ((size_t)5 * Lyr + 1) * 8 * sizeof(unsigned long long);
        a.dbg = (unsigned long long *)dalloc(n);
        if (!a.dbg) return cudaErrorMemoryAllocation;
        DCK(cudaMemset(a.dbg, 0, n));
    }
    if ((int)pk::smem_bytes(a) > ctx_->smem_optin) return no("shared memory");
    // pair staging (clusters of two CTAs share the activation staging over DSMEM): on unless switched off or the device cannot co-schedule
    // num_sms / 2 such clusters (+3 % on one B200, profiles/README.md)
    a.pair = (!getenv("TCE_PK_PAIR") || atoi(getenv("TCE_PK_PAIR")) != 0) && pk::pair_supported(ctx_, a) ? 1 : 0;
    pargs_ = a;
    return cudaSuccess;
}

cudaError_t LlamaDecoder::enqueue_step(const int *tokpos, cudaStream_t s, bool pdl, bool gemv_only) {
    if (persistent_ && !gemv_only) {
        pk::Args m = pargs_;
        m.tokpos = tokpos;
        return pk::launch(ctx_, m, s);
    }
    Ctx local = *ctx_;  // same workspaces, but launch on `s`
    local.stream = s;
    Ctx *c = &local;
    bool first = true;
    for (const StepOp &op : ops_) {
        const bool use_pdl = pdl && !first && tp_ == 1;  // TP steps keep plain edges around the peer-flag kernels
        switch (op.type) {
            case OP_EMBED:
                // also range-checks the device-resident {token, position} and publishes the clamped pair for the attention launches of this step
                if (!gemv_only)
                    DCK(launch_embedding(c, (const __half *)w_.embed_f16, tokpos, d_resid_, cfg_.embed_dim, false, cfg_.vocab_size * tp_, cfg_.max_ctx, d_tokpos_safe_));
                break;
            case OP_GEMV: {
                W4GemvParams p = op.g;
                p.pdl = use_pdl;
                DCK(launch_w4a16_gemv(c, p));
                break;
            }
            case OP_ATTN:
                if (!gemv_only) {
                    AttnDecodeArgs a = op.at;
                    a.pos = d_tokpos_safe_ + 1;  // the position after the embedding kernel's range check
                    DCK(launch_attn_decode(c, a, use_pdl));
                }
                break;
            case OP_ARGMAX:
                if (!gemv_only) DCK(launch_argmax(c, d_logits_, cfg_.vocab_size, d_next_, use_pdl));
                break;
            case OP_TP_SIGNAL:
                if (!gemv_only) DCK(launch_tp_signal(c, op.sig));
                break;
            case OP_TP_ARGMAX_SCATTER:
                if (!gemv_only) DCK(launch_tp_argmax_scatter(c, op.am));
                break;
            case OP_TP_ARGMAX_FINISH:
                if (!gemv_only) DCK(launch_tp_argmax_finish(c, op.amf));
                break;
        }
        first = false;
    }
    return cudaSuccess;
}

cudaError_t LlamaDecoder::build_graphs(std::string *err) {
    // one eager step first: loads the modules and sets the kernels' shared-memory attributes outside of capture
    // (re-running a step at the same position is idempotent: the same K/V row is rewritten).  Work queued on the caller's stream
    // (an asynchronous decode_device) touches the same buffers: drain it before switching to the capture stream.
    DCK(cudaStreamSynchronize(ctx_->stream));
    DCK(cudaMemcpyAsync(d_tokpos_, h_tokpos_, 3 * sizeof(int), cudaMemcpyHostToDevice, cap_stream_));
    DCK(enqueue_step(d_tokpos_, cap_stream_, false));
    DCK(cudaStreamSynchronize(cap_stream_));
    // try PDL edges first; if capture/instantiate refuses them, fall back to plain edges
    for (int attempt = 0; attempt < 2; attempt++) {
        const bool pdl = ctx_->use_pdl && attempt == 0;
        cudaGraph_t g = nullptr;
        cudaError_t e = cudaStreamBeginCapture(cap_stream_, cudaStreamCaptureModeThreadLocal);
        if (e != cudaSuccess) return e;
        e = cudaMemcpyAsync(d_tokpos_, h_tokpos_, 3 * sizeof(int), cudaMemcpyHostToDevice, cap_stream_);
        if (e == cudaSuccess) e = enqueue_step(d_tokpos_, cap_stream_, pdl);
        if (e == cudaSuccess) e = cudaMemcpyAsync(h_logits_, d_logits_, (size_t)cfg_.vocab_size * sizeof(float), cudaMemcpyDeviceToHost, cap_stream_);
        if (e == cudaSuccess) e = cudaMemcpyAsync(h_next_, d_next_, sizeof(int), cudaMemcpyDeviceToHost, cap_stream_);
        cudaError_t e2 = cudaStreamEndCapture(cap_stream_, &g);
        if (e == cudaSuccess) e = e2;
        if (e == cudaSuccess) e = cudaGraphInstantiate(&g_host_, g, 0);
        if (g) cudaGraphDestroy(g);
        if (e == cudaSuccess) {
            graphs_ok_ = true;
            graphs_gen_ = ctx_->option_gen;
            if (!pdl) ctx_->use_pdl = false;
            return cudaSuccess;
        }
        cudaGetLastError();
        if (err) *err = std::string("graph capture failed (pdl=") + (pdl ? "1" : "0") + "): " + cudaGetErrorString(e);
        g_host_ = nullptr;
        if (!ctx_->use_pdl) return e;
    }
    return cudaErrorUnknown;
}

cudaError_t LlamaDecoder::decode_host(int token, int pos, float *logits_host, int *next_token, std::string *err) {
    const int tp = cfg_.tp_size > 1 ? cfg_.tp_size : 1;
    if (pos < 0 || pos >= cfg_.max_ctx || token < 0 || token >= cfg_.vocab_size * tp) return cudaErrorInvalidValue;
    if (tp > 1 && !tp_connected_) return cudaErrorNotReady;
    h_tokpos_[0] = token;
    h_tokpos_[1] = pos;
    h_tokpos_[2] = 0;
    cudaStream_t s = ctx_->stream;
    if (graphs_ok_ && graphs_gen_ != ctx_->option_gen) {  // an option or the stream changed since capture: the graph holds the old context by value
        cudaGraphExecDestroy(g_host_);
        g_host_ = nullptr;
        graphs_ok_ = false;
    }
    if (use_graphs_ && !graphs_ok_) {
        cudaError_t e = build_graphs(err);
        if (e != cudaSuccess) use_graphs_ = false;
    }
    if (use_graphs_ && graphs_ok_) {
        DCK(cudaGraphLaunch(g_host_, s));
    } else {
        DCK(cudaMemcpyAsync(d_tokpos_, h_tokpos_, 3 * sizeof(int), cudaMemcpyHostToDevice, s));
        DCK(enqueue_step(d_tokpos_, s, ctx_->use_pdl));
        DCK(cudaMemcpyAsync(h_logits_, d_logits_, (size_t)cfg_.vocab_size * sizeof(float), cudaMemcpyDeviceToHost, s));
        DCK(cudaMemcpyAsync(h_next_, d_next_, sizeof(int), cudaMemcpyDeviceToHost, s));
    }
    DCK(cudaStreamSynchronize(s));
    if (logits_host) memcpy(logits_host, h_logits_, (size_t)cfg_.vocab_size * sizeof(float));
    if (next_token) *next_token = *h_next_;
    return cudaSuccess;
}

// Generate loop (LLaMAGenerate.cu:67-252 without the tokenizer / console parts): every token is one decode step plus one sampler launch, both
// enqueued back to back; the sampler writes the next step's {token, position} on the device.  The host only looks at the stop flag every
// few tokens, and copies the generated ids out at the end.
cudaError_t LlamaDecoder::generate(int first_token, int pos0, int n_predict, const tce_sampling &sc, const int *history_host, int n_history, int eos_id,
                                   int *out_tokens_host, int *n_out, std::string *err) {
    if (cfg_.tp_size > 1) {
        if (err) *err = "generate: single GPU only (the vocabulary is sharded under tensor parallelism)";
        return cudaErrorNotSupported;
    }
    const int cap = cfg_.max_ctx;
    if (first_token < 0 || first_token >= cfg_.vocab_size || pos0 < 0 || pos0 >= cap || n_predict < 0 || n_history < 0 || n_history > cap || !n_out ||
        (n_predict > 0 && !out_tokens_host))
        return cudaErrorInvalidValue;
    if (sc.temp > 0.f && (sc.top_k <= 0 || sc.top_k > 1024) && cfg_.vocab_size > 1024) {
        if (err) *err = "generate: temp > 0 needs 1 <= top_k <= 1024";
        return cudaErrorNotSupported;
    }
    if (n_predict > cap - pos0) n_predict = cap - pos0;
    cudaStream_t s = ctx_->stream;
    if (!d_gen_) DCK(cudaMalloc((void **)&d_gen_, (size_t)(4 + 2 * cap) * sizeof(int)));
    int *hist = d_gen_ + 4, *out_list = d_gen_ + 4 + cap;
    DCK(cudaMemsetAsync(d_gen_, 0, (size_t)(4 + 2 * cap) * sizeof(int), s));
    if (n_history > 0) DCK(cudaMemcpyAsync(hist, history_host, (size_t)n_history * sizeof(int), cudaMemcpyHostToDevice, s));
    const int ctl0[4] = {n_history, 0, 0, 0};
    DCK(cudaMemcpyAsync(d_gen_, ctl0, sizeof(ctl0), cudaMemcpyHostToDevice, s));
    h_tokpos_[0] = first_token;
    h_tokpos_[1] = pos0;
    h_tokpos_[2] = 0;
    DCK(cudaMemcpyAsync(d_tokpos_, h_tokpos_, 3 * sizeof(int), cudaMemcpyHostToDevice, s));
    SampleArgs a{};
    a.logits = d_logits_;
    a.n_vocab = cfg_.vocab_size;
    a.top_k = sc.top_k;
    a.top_p = sc.top_p;
    a.temp = sc.temp;
    a.repeat_penalty = sc.repeat_penalty;
    a.frequency_penalty = sc.frequency_penalty;
    a.presence_penalty = sc.presence_penalty;
    a.repeat_last_n = sc.repeat_last_n;
    a.seed = sc.seed;
    a.draw_index = 0;
    a.hist = hist;
    a.hist_head = d_gen_;
    a.hist_cap = cap;
    a.eos_id = eos_id;
    a.tokpos = d_tokpos_;
    a.out_list = out_list;
    a.out_count = d_gen_ + 1;
    a.out_cap = cap;
    a.stop = d_gen_ + 2;
    int ctl[4] = {0, 0, 0, 0};
    constexpr int kCheckEvery = 16;
    for (int i = 0; i < n_predict; i++) {
        DCK(enqueue_step(d_tokpos_, s, ctx_->use_pdl));
        DCK(launch_sample(ctx_, a, s));
        if ((i + 1) % kCheckEvery == 0 && i + 1 < n_predict) {
            DCK(cudaMemcpyAsync(ctl, d_gen_, sizeof(ctl), cudaMemcpyDeviceToHost, s));
            DCK(cudaStreamSynchronize(s));
            if (ctl[2]) break;
        }
    }
    DCK(cudaMemcpyAsync(ctl, d_gen_, sizeof(ctl), cudaMemcpyDeviceToHost, s));
    DCK(cudaStreamSynchronize(s));
    const int n = ctl[1] < cap ? ctl[1] : cap;
    if (n > 0) DCK(cudaMemcpy(out_tokens_host, out_list, (size_t)n * sizeof(int), cudaMemcpyDeviceToHost));
    *n_out = n;
    return cudaSuccess;
}

cudaError_t LlamaDecoder::decode_device(const int *tokpos_dev, std::string *err) {
    cudaStream_t s = ctx_->stream;
    if (tp_ > 1 && !tp_connected_) return cudaErrorNotReady;
    if (use_graphs_ && (g_dev_ == nullptr || g_dev_src_ != tokpos_dev || g_dev_gen_ != ctx_->option_gen)) {
        if (g_dev_) {
            cudaGraphExecDestroy(g_dev_);
            g_dev_ = nullptr;
        }
        DCK(cudaStreamSynchronize(s));
        DCK(enqueue_step(tokpos_dev, cap_stream_, false));  // eager warm-up outside of capture (idempotent)
        DCK(cudaStreamSynchronize(cap_stream_));
        for (int attempt = 0; attempt < 2 && !g_dev_; attempt++) {
            const bool pdl = ctx_->use_pdl && attempt == 0;
            cudaGraph_t g = nullptr;
            cudaError_t e = cudaStreamBeginCapture(cap_stream_, cudaStreamCaptureModeThreadLocal);
            if (e == cudaSuccess) e = enqueue_step(tokpos_dev, cap_stream_, pdl);
            cudaError_t e2 = cudaStreamEndCapture(cap_stream_, &g);
            if (e == cudaSuccess) e = e2;
            if (e == cudaSuccess) e = cudaGraphInstantiate(&g_dev_, g, 0);
            if (g) cudaGraphDestroy(g);
            if (e != cudaSuccess) {
                cudaGetLastError();
                g_dev_ = nullptr;
                if (err) *err = std::string("graph capture failed: ") + cudaGetErrorString(e);
                if (!pdl) use_graphs_ = false;
            } else if (!pdl) {
                ctx_->use_pdl = false;
            }
        }
        g_dev_src_ = tokpos_dev;
        g_dev_gen_ = ctx_->option_gen;
    }
    if (use_graphs_ && g_dev_) return cudaGraphLaunch(g_dev_, s);
    return enqueue_step(tokpos_dev, s, ctx_->use_pdl);
}

}  // namespace tce

// ------------------------------------------------------------------------------------------------ prompt processing
// n tokens at once (sqlen > 1 in the reference's Int4LlamaForCausalLM::forward): every linear runs as one tensor-core GEMM over the
// [n][.] activation block (int4 weights expanded to fp16 once per GEMM), attention as one causal flash kernel over the KV cache.
namespace tce {

cudaError_t LlamaDecoder::prefill_reserve(int n) {
    if (n <= pf_cap_) return cudaSuccess;
    DCK(cudaStreamSynchronize(ctx_->stream));
    cudaFree(pf_x_);
    cudaFree(pf_xn_);
    cudaFree(pf_qkv_);
    cudaFree(pf_att_);
    cudaFree(pf_gu_);
    cudaFree(pf_act_);
    cudaFree(pf_tok_);
    pf_x_ = nullptr; pf_xn_ = nullptr; pf_qkv_ = nullptr; pf_att_ = nullptr; pf_gu_ = nullptr; pf_act_ = nullptr; pf_tok_ = nullptr;
    pf_cap_ = 0;
    const size_t E = cfg_.embed_dim, F = cfg_.hidden_dim, Q = (size_t)(cfg_.num_heads + 2 * cfg_.num_kv_heads) * cfg_.head_dim,
                 A = (size_t)cfg_.num_heads * cfg_.head_dim;
    DCK(cudaMalloc(&pf_x_, n * E * sizeof(float)));
    DCK(cudaMalloc(&pf_xn_, n * E * sizeof(__half)));
    DCK(cudaMalloc(&pf_qkv_, n * Q * sizeof(__half)));
    DCK(cudaMalloc(&pf_att_, n * A * sizeof(__half)));
    DCK(cudaMalloc(&pf_gu_, n * 2 * F * sizeof(__half)));
    DCK(cudaMalloc(&pf_act_, n * F * sizeof(__half)));
    DCK(cudaMalloc(&pf_tok_, n * sizeof(int)));
    pf_cap_ = n;
    return cudaSuccess;
}

// C[n][sum oc] (row-major, leading dimension ldc) = X[n][ic] * [deq(t0); deq(t1); ...]^T : the `count` weight matrices (same ic) of the
// prompt pass's next job were expanded into consecutive row ranges of one fp16 scratch half, and ONE GEMM multiplies them (q|k|v and
// gate|up share their input).  Called in the order of pf_jobs_.
cudaError_t LlamaDecoder::prefill_linear(const tce_w4_tensor *const *ts, int count, const __half *x, void *C, long long ldc, int n, bool add_f32, bool silu) {
    const int ic = ts[0]->ic;
    size_t rows = 0;
    for (int i = 0; i < count; i++) rows += (size_t)ts[i]->oc;
    // this job's weights were expanded on the side stream while the previous GEMM ran; queue the next job's expansion, then run
    const int j = pf_next_job_++;
    const int b = j & 1;
    if (j + 1 < (int)pf_jobs_.size()) DCK(pf_expand_job(j + 1));
    DCK(cudaStreamWaitEvent(ctx_->stream, pf_expanded_[b], 0));
    if (silu)
        DCK(launch_gemm_f16_pair_silu(ctx_, x, ic, pf_w16_[b], ic, (__half *)C, ldc, n, (int)(rows / 2), ic));
    else
        DCK(launch_gemm_f16_pair(ctx_, x, ic, pf_w16_[b], ic, C, ldc, n, (int)rows, ic, add_f32 ? 1 : 0));
    return cudaEventRecord(pf_consumed_[b], ctx_->stream);
}

// expansion of job j into scratch half (j & 1) on the side stream, after the GEMM that last read that half
cudaError_t LlamaDecoder::pf_expand_job(int j) {
    const PfJob &job = pf_jobs_[j];
    const int b = j & 1;
    Ctx side = *ctx_;
    side.stream = pf_side_;
    if (j >= 2) DCK(cudaStreamWaitEvent(pf_side_, pf_consumed_[b], 0));
    size_t r0 = 0;
    const int ic = job.ts[0]->ic;
    for (int i = 0; i < job.count; i++) {
        const tce_w4_tensor &t = *job.ts[i];
        DCK(launch_w4_expand(&side, (const uint32_t *)t.w, (const uint32_t *)t.zeros, (const __half *)t.scales, pf_w16_[b] + r0 * ic, t.oc, ic));
        r0 += (size_t)t.oc;
    }
    return cudaEventRecord(pf_expanded_[b], pf_side_);
}

cudaError_t LlamaDecoder::prefill(const int *tokens_host, int n, int pos0, float *logits_host, int *next_token, std::string *err) {
    if (tp_ > 1) {
        if (err) *err = "prefill is single-GPU in this build (tensor-parallel ranks process the prompt with decode steps)";
        return cudaErrorNotSupported;
    }
    if (!tokens_host || n < 1 || pos0 < 0 || pos0 + n > cfg_.max_ctx) return cudaErrorInvalidValue;
    for (int i = 0; i < n; i++)
        if (tokens_host[i] < 0 || tokens_host[i] >= cfg_.vocab_size) return cudaErrorInvalidValue;
    DCK(prefill_reserve(n));
    if (pf_jobs_.empty()) {
        size_t need = 0;
        for (int l = 0; l < cfg_.num_layers; l++) {
            const tce_llama_layer &L = layers_[l];
            pf_jobs_.push_back(PfJob{{&L.q, &L.k, &L.v}, 3});
            pf_jobs_.push_back(PfJob{{&L.o, nullptr, nullptr}, 1});
            pf_jobs_.push_back(PfJob{{&L.gate, &L.up, nullptr}, 2});
            pf_jobs_.push_back(PfJob{{&L.down, nullptr, nullptr}, 1});
        }
        for (const PfJob &jb : pf_jobs_) {
            size_t e = 0;
            for (int i = 0; i < jb.count; i++) e += (size_t)jb.ts[i]->oc * jb.ts[i]->ic;
            need = e > need ? e : need;
        }
        for (int b = 0; b < 2; b++) {
            DCK(cudaMalloc((void **)&pf_w16_[b], need * sizeof(__half)));
            DCK(cudaEventCreateWithFlags(&pf_expanded_[b], cudaEventDisableTiming));
            DCK(cudaEventCreateWithFlags(&pf_consumed_[b], cudaEventDisableTiming));
        }
        pf_w16_elems_ = need;
        DCK(cudaStreamCreateWithFlags(&pf_side_, cudaStreamNonBlocking));
    }
    pf_next_job_ = 0;
    // the side stream starts after everything already queued on the main stream (a previous prompt's GEMMs read the scratch)
    DCK(cudaEventRecord(pf_consumed_[0], ctx_->stream));
    DCK(cudaStreamWaitEvent(pf_side_, pf_consumed_[0], 0));
    DCK(pf_expand_job(0));
    cudaStream_t s = ctx_->stream;
    const int E = cfg_.embed_dim, F = cfg_.hidden_dim, H = cfg_.num_heads, KVH = cfg_.num_kv_heads, hd = cfg_.head_dim;
    const long long Q = (long long)(H + 2 * KVH) * hd;
    DCK(cudaMemcpyAsync(pf_tok_, tokens_host, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, s));
    DCK(launch_embedding_rows(ctx_, (const __half *)w_.embed_f16, pf_tok_, pf_x_, n, E));
    for (int l = 0; l < cfg_.num_layers; l++) {
        const tce_llama_layer &L = layers_[l];
        DCK(launch_rmsnorm_rows_f32(ctx_, pf_x_, L.input_norm, pf_xn_, n, E, cfg_.rms_eps));
        const tce_w4_tensor *qkv[3] = {&L.q, &L.k, &L.v}, *gu[2] = {&L.gate, &L.up}, *o1[1] = {&L.o}, *d1[1] = {&L.down};
        DCK(prefill_linear(qkv, 3, pf_xn_, pf_qkv_, Q, n, false));
        AttnPrefillArgs a{};
        a.qkv = pf_qkv_;
        a.k_cache = (__half *)kv_cache(l, 0);
        a.v_cache = (__half *)kv_cache(l, 1);
        a.cos = d_cos_;
        a.sin = d_sin_;
        a.out = pf_att_;
        a.alpha = cfg_.qk_alpha > 0 ? cfg_.qk_alpha : 1.0f / sqrtf((float)hd);
        a.n = n;
        a.pos0 = pos0;
        a.num_heads = H;
        a.num_kv_heads = KVH;
        a.head_dim = hd;
        a.max_ctx = cfg_.max_ctx;
        DCK(launch_attn_prefill(ctx_, a));
        DCK(prefill_linear(o1, 1, pf_att_, pf_x_, E, n, true));  // residual add in the GEMM epilogue
        DCK(launch_rmsnorm_rows_f32(ctx_, pf_x_, L.post_norm, pf_xn_, n, E, cfg_.rms_eps));
        if ((F % 128) == 0) {
            DCK(prefill_linear(gu, 2, pf_xn_, pf_act_, F, n, false, true));  // SiLU(gate) * up in the GEMM epilogue: gate|up never reach HBM
        } else {
            DCK(prefill_linear(gu, 2, pf_xn_, pf_gu_, 2LL * F, n, false));
            DCK(launch_silu_mul_rows(ctx_, pf_gu_, pf_act_, n, F));
        }
        DCK(prefill_linear(d1, 1, pf_act_, pf_x_, E, n, true));
    }
    // only the last position feeds the sampler: final RMSNorm + lm_head as the decode step's last GEMV, then arg-max
    DCK(cudaMemcpyAsync(d_resid_, pf_x_ + (size_t)(n - 1) * E, (size_t)E * sizeof(float), cudaMemcpyDeviceToDevice, s));
    const StepOp *lm = nullptr;
    for (const StepOp &op : ops_)
        if (op.type == OP_GEMV) lm = &op;
    if (!lm) return cudaErrorUnknown;
    DCK(launch_w4a16_gemv(ctx_, lm->g));
    DCK(launch_argmax(ctx_, d_logits_, cfg_.vocab_size, d_next_, false));
    if (logits_host) DCK(cudaMemcpyAsync(h_logits_, d_logits_, (size_t)cfg_.vocab_size * sizeof(float), cudaMemcpyDeviceToHost, s));
    DCK(cudaMemcpyAsync(h_next_, d_next_, sizeof(int), cudaMemcpyDeviceToHost, s));
    DCK(cudaStreamSynchronize(s));
    if (logits_host) memcpy(logits_host, h_logits_, (size_t)cfg_.vocab_size * sizeof(float));
    if (next_token) *next_token = *h_next_;
    return cudaSuccess;
}

}  // namespace tce
