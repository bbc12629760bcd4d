// llama_decoder.h -- host-side runner of the fused Llama decode step (one CUDA graph per token).
#pragma once
#include <string>
#include <vector>

#include "../../include/tce_b200.h"
#include "kernels.h"
#include "kernels_attn.h"
#include "kernels_tp.h"
#include "persistent.h"

namespace tce {

class LlamaDecoder {
   public:
    static LlamaDecoder *create(Ctx *ctx, int attn_chunk, const tce_llama_config &cfg, const tce_llama_weights &w, std::string *err);
    ~LlamaDecoder();
    cudaError_t decode_device(const int *tokpos_dev, std::string *err);
    cudaError_t decode_host(int token, int pos, float *logits_host, int *next_token, std::string *err);
    cudaError_t generate(int first_token, int pos0, int n_predict, const tce_sampling &sc, const int *history_host, int n_history, int eos_id,
                         int *out_tokens_host, int *n_out, std::string *err);
    // prompt processing: n tokens at positions pos0..pos0+n-1 in one pass (tensor-core GEMMs + causal flash attention)
    cudaError_t prefill(const int *tokens_host, int n, int pos0, float *logits_host, int *next_token, std::string *err);
    const float *logits() const { return d_logits_; }
    void *kv_cache(int layer, int which) const;
    int kernels_per_step() const { return kernels_per_step_; }
    void *debug_buffer(int which) const {
        switch (which) {
            case 0: return d_resid_;
            case 1: return d_qkv_;
            case 2: return d_attn_;
            case 3: return d_act_;
            case 4: return pargs_.dbg;  // persistent-kernel phase timestamps (TCE_PK_DEBUG=1), [#CTAs][5 * layers + 1][4] u64 ns
            default: return nullptr;
        }
    }
    cudaError_t enqueue_gemvs(int *count);
    cudaError_t tp_handle(void *out64);
    cudaError_t tp_connect(const void *handles);
    void adopt(void *device_allocation) { pk_allocs_.push_back(device_allocation); }  // freed with the model (loader.cu)

   private:
    LlamaDecoder() = default;
    cudaError_t prefill_reserve(int n);
    cudaError_t prefill_linear(const tce_w4_tensor *const *ts, int count, const __half *x, void *C, long long ldc, int n, bool add_f32, bool silu = false);
    cudaError_t enqueue_step(const int *tokpos, cudaStream_t s, bool pdl, bool gemv_only = false);  // raw kernel sequence
    cudaError_t build_graphs(std::string *err);
    void build_ops();
    cudaError_t build_persistent(std::string *err);

    enum OpType { OP_EMBED, OP_GEMV, OP_ATTN, OP_ARGMAX, OP_TP_SIGNAL, OP_TP_ARGMAX_SCATTER, OP_TP_ARGMAX_FINISH };
    struct StepOp {
        OpType type;
        W4GemvParams g;
        AttnDecodeArgs at;
        TpSignalArgs sig;
        TpArgmaxArgs am;
        TpArgmaxFinishArgs amf;
    };
    // tensor parallel state
    int tp_ = 1;
    bool tp_connected_ = false;
    uint8_t *tp_buf_ = nullptr;          // peer-visible allocation of this rank
    size_t tp_bytes_ = 0, tp_gather_floats_ = 0;
    uint8_t *tp_peer_[kMaxTP] = {};      // every rank's allocation as mapped into this process
    int step_index_ = 0;
    std::vector<StepOp> ops_;
    // persistent decode kernel (default; TCE_PERSISTENT=0 selects one kernel per op inside a CUDA graph)
    bool persistent_ = false;
    pk::Args pargs_{};
    std::vector<void *> pk_allocs_;     // repacked scales|zeros, tensor maps, layer table, counters

    Ctx *ctx_ = nullptr;
    int attn_chunk_ = 128;
    tce_llama_config cfg_{};
    std::vector<tce_llama_layer> layers_;
    tce_llama_weights w_{};
    // device state
    __half *d_kv_ = nullptr;        // [L][2][KVH][max_ctx][hd]
    float *d_resid_ = nullptr;      // fp32 residual stream [E]
    __half *d_qkv_ = nullptr;       // [(H+2KVH)*hd]
    __half *d_attn_ = nullptr;      // [H*hd]
    __half *d_act_ = nullptr;       // [F] SiLU(gate)*up
    float *d_logits_ = nullptr;     // [V]
    int *d_tokpos_ = nullptr;       // {token, pos} staged for the host entry point
    int *d_next_ = nullptr;         // greedy arg-max
    int *d_gen_ = nullptr;          // generate loop: [0] history head, [1] output count, [2] stop flag, then history ring [max_ctx], output list [max_ctx]
    float *d_cos_ = nullptr, *d_sin_ = nullptr;
    bool own_rope_ = false;
    // prompt-processing activations, [pf_cap_] rows each (allocated on first use)
    int pf_cap_ = 0;
    float *pf_x_ = nullptr;         // fp32 residual stream [n][E]
    __half *pf_xn_ = nullptr;       // RMSNorm output [n][E]
    __half *pf_qkv_ = nullptr;      // [n][(H+2KVH)*hd]
    __half *pf_att_ = nullptr;      // [n][H*hd]
    __half *pf_gu_ = nullptr;       // [n][2F] gate | up
    __half *pf_act_ = nullptr;      // [n][F]
    int *pf_tok_ = nullptr;
    // the int4 -> fp16 expansion of the NEXT linear runs on a side stream into the other half of a double-buffered scratch while the
    // tensor cores work on the current one (the expansion is HBM-bound, the GEMM tensor-bound)
    __half *pf_w16_[2] = {nullptr, nullptr};
    size_t pf_w16_elems_ = 0;
    cudaStream_t pf_side_ = nullptr;
    cudaEvent_t pf_expanded_[2] = {nullptr, nullptr}, pf_consumed_[2] = {nullptr, nullptr};
    struct PfJob { const tce_w4_tensor *ts[3]; int count; };
    std::vector<PfJob> pf_jobs_;
    int pf_next_job_ = 0;
    cudaError_t pf_expand_job(int j);
    // pinned host staging for the end-to-end entry point
    int *h_tokpos_ = nullptr;
    float *h_logits_ = nullptr;
    int *h_next_ = nullptr;
    // graphs
    cudaStream_t cap_stream_ = nullptr;
    cudaGraphExec_t g_host_ = nullptr;    // H2D(tokpos) + step + argmax + D2H(logits,next)
    cudaGraphExec_t g_dev_ = nullptr;     // copy tokpos (D2D) + step
    const int *g_dev_src_ = nullptr;
    bool graphs_ok_ = false;
    unsigned graphs_gen_ = 0, g_dev_gen_ = 0;       // ctx_->option_gen at capture time
    int *d_tokpos_safe_ = nullptr;  // kernel-per-op path: {token, position} after the device-side range check (+ [2] unused, [3] TP step counter alias)
    bool use_graphs_ = true;
    bool atomic_residual_ = true;  // o_proj/down_proj partial tiles use RED.ADD (TCE_DETERMINISTIC=1 turns it off)
    int kernels_per_step_ = 0;
};

// loader.cu: the reference's on-disk INT4 tree -> a model that owns its device copies
LlamaDecoder *load_llama_dir(Ctx *ctx, int attn_chunk, const char *dir, tce_llama_config cfg, std::string *err);
int import_x86(const uint8_t *qs, const float *scales_f32, int oc, int ic, uint32_t *w_out, __half *scales_out, uint32_t *zeros_out);

}  // namespace tce
