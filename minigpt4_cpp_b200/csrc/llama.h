// llama.h — device-resident LLaMA/Vicuna step (the path behind llama_eval / llama_eval_embd,
// called by the reference at minigpt4.cpp:2373 and :2412).
//
// Data layout in HBM (owned by this engine; algorithmic bytes == file bytes):
//   * every quantised matrix is repacked at load into SoA planes so that each warp-level access is a
//     128-bit aligned vector (Q4_1/Q4_0: row-packed [nb x 16 B nibbles][nb x half2{d,m} | half d] so a run of rows is ONE contiguous range for cp.async.bulk;
//     Q5_K: row-packed [nsb x 128 B qs][nsb x 32 B qh][nsb x 16 B {scales[12],d,dmin}]; Q6_K: ql 128 B + qh 64 B + scales 16 B + half d)
//   * wq|wk|wv are concatenated row-wise (one launch), w1/w3 are row-interleaved (gate r, up r adjacent)
//   * KV cache: F16 [layer][n_ctx][n_embd_local] for K and V (token-major; values as in ggml's cache)
//   * activations between kernels are F32 vectors; each consumer re-quantises them to the weight type's
//     vec_dot type (Q8_0/Q8_1/Q8_K/F16) in its prologue — the integer-dot formulation ggml uses (SURVEY §A.3)
#pragma once
#include "formats.h"

namespace mg4 {

struct TPLink;  // tensor-parallel communicator (tp.h)

struct QMat {          // one repacked weight matrix (or a fused group of matrices of one type)
    int type = -1;     // GGType
    int rows = 0, cols = 0;
    void *p0 = nullptr, *p1 = nullptr, *p2 = nullptr, *p3 = nullptr;
    size_t bytes = 0;  // algorithmic bytes (rows * row_bytes)
    int row_bytes = 0; // row-packed layouts (p0 holds rows of row_bytes each): Q4_0 / Q4_1 [nb x 16 B nibbles][nb x scales]; Q5_K [nsb x 128 B qs][nsb x 32 B qh][nsb x 16 B {scales, d, dmin}]
};

struct PQMat {         // prefill operand cache of one Q4_0 / Q4_1 matrix (llama_prefill.cuh): int8, class-major, + {d, m} in the same order
    int rows = 0, rows_pad = 0, cols = 0, nb = 0, S = 0; bool q41 = false;
    signed char *q = nullptr; void *sc = nullptr;
    alignas(64) unsigned char tm[128];  // CUtensorMap over q
};

struct LlamaDims { int n_vocab, n_embd, n_head, n_layer, n_ff, n_ctx, head_dim; };

struct DeviceState {   // lives in device memory; kernels read positions/tokens from here so graphs are position independent
    int n_past;
    int n_tok;
    int tokens[8];
    unsigned long long argmax_key;
    int argmax_id;
    int pad[3];
};

class LlamaDevice {
public:
    LlamaDevice();
    ~LlamaDevice();
    bool load(const LlamaFile &f, int n_ctx, TPLink *tp);
    const LlamaDims &dims() const { return d_; }
    // Evaluate `n` mixed token / embedding rows (ids < 0: row -1 - id of emb_host) starting at position n_past. Afterwards logits
    // of the last row are on device and the arg-max id is known.  Returns false if the context would overflow.
    bool eval_rows(const int32_t *ids, int n, const float *emb_host, int n_emb, int n_past);
    void logits_to_host(float *dst);   // n_vocab floats, synchronous
    int32_t argmax();                  // greedy id of the current logits (already in pinned host memory after a sync)
    void sync();
    void sync_decode();              // stream sync that reports the megakernel's spin-guard reason code if the launch failed
    int sm_count() const { return sm_count_; }
    bool uses_megakernel() const { return mega_; }
    bool uses_prefill_gemm() const { return pf_ready_; }
    static constexpr int kPrefillMax = 512;   // rows per prefill pass (the reference's default n_batch)
    int mega_generation() const { return mega_ ? 6 : 0; }   // llama_mega6.cuh
    int mega_trace(long long *out, int max_values);  // debug: per-op clock64 stamps of the last megakernel launch (env MINIGPT4_B200_MEGA_TRACE)
    // one decode step through the captured CUDA graph: feeds `id` (or, if id < 0, the on-device arg-max of the
    // previous step), leaves new logits/arg-max on device.
    bool decode_step(int32_t id, int n_past);
    // bench leg: `steps` chained greedy steps with no host round trip; returns device ms for the loop.
    float decode_chain(int steps, int n_past, int32_t *ids_out);
    // measurement seam: average CUDA-event duration (ms) of one launch of the decode matvec of `kind`
    // (0 qkv, 1 wo, 2 gate/up, 3 down, 4 output) cycling through all layers so every launch streams cold weights.
    float time_matvec(int kind, int reps, double *bytes_per_launch);
    float time_allreduce(int reps);   // us per [1, n_embd] all-reduce on the tensor-parallel path in use (0 without tensor parallelism)
    bool tp_peer_path() const;
    // test taps
    void hidden_to_host(float *dst, int n);  // residual stream after the last evaluated chunk (n rows)
    size_t weight_bytes_per_token() const { return bytes_per_token_; }
    unsigned long long kernel_launches() const { return launches_; }
    cudaStream_t stream() const { return stream_; }

    // kernel-level test hook: y[n][rows] = W x (W given as raw ggml blocks on host), through the same
    // repack + matvec kernels the engine uses.
    static void test_matvec(int gg, int rows, int cols, const void *w_host, const float *x_host, int n, float *y_host);

private:
    struct Layer { QMat qkv, wq, wk, wv, wo, w13, w2; bool fused_qkv; float *attn_norm, *ffn_norm; PQMat pqkv, pwo, pw13, pw2; };
    bool build_prefill();            // tensor-core prefill (llama_prefill.cuh): homogeneous Q4_0 / Q4_1 layers, single GPU
    void prefill_chunk(int n, bool want_logits);   // n <= kPrefillMax rows that sit in x_
    bool pf_ready_ = false; int pf_S_e_ = 0, pf_S_ff_ = 0;
    signed char *pf_q8_ = nullptr; void *pf_sc_ = nullptr; int32_t *tok_ids_ = nullptr; void *pf_part_ = nullptr; size_t pf_part_bytes_ = 0;
    alignas(64) unsigned char pf_tmB_e_[128], pf_tmS_e_[128], pf_tmB_ff_[128], pf_tmS_ff_[128];
    void launch_layers(int nt, int ntok, bool want_logits);
    void build_graph();
    bool build_mega();               // persistent one-launch-per-token decode (homogeneous Q4_0/Q4_1, single GPU)
    void launch_mega();
    const void *mega_fn() const;
    LlamaDims d_{};
    int n_head_local_ = 0, n_embd_local_ = 0, n_ff_local_ = 0;
    TPLink *tp_ = nullptr;
    std::vector<Layer> layers_;
    QMat output_;
    float *final_norm_ = nullptr;
    void *tok_raw_ = nullptr; int tok_type_ = -1;  // tok_embeddings kept as raw ggml blocks (row gather only)
    __half *kcache_ = nullptr, *vcache_ = nullptr;
    float2 *rope_ = nullptr;                        // [n_ctx][head_dim/2] {cos, sin}, host-computed with libm like ggml
    __half *tab_exp_ = nullptr, *tab_silu_ = nullptr;  // ggml's fp16 LUTs
    float *x_ = nullptr, *q_ = nullptr, *att_ = nullptr, *act_ = nullptr, *logits_ = nullptr, *partial_ = nullptr;
    float *embd_in_ = nullptr;
    unsigned char *qact_ = nullptr;                 // per-op staged (quantised) activations for the per-op kernels
    DeviceState *state_ = nullptr;
    DeviceState *h_state_ = nullptr;  // pinned
    int32_t *h_argmax_ = nullptr;     // pinned
    cudaStream_t stream_ = nullptr;
    cudaGraphExec_t graph_ = nullptr;
    cudaEvent_t ev0_ = nullptr, ev1_ = nullptr;
    size_t bytes_per_token_ = 0;
    unsigned long long launches_ = 0;
    int graph_kernels_ = 0;
    long long *mega_trace_ = nullptr; int mega_n_ops_ = 0;
    void *mega6_params_ = nullptr; int mega6_nbl_ = 0;  // generation 6 (llama_mega6.cuh)
    bool h_state_busy_ = false;
    bool mega_ = false; unsigned *mega_barrier_ = nullptr; size_t mega_smem_ = 0; int mega_type_ = -1;
    int sm_count_ = 148;
};

}  // namespace mg4
