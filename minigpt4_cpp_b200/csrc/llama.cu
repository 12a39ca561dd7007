// llama.cu — host side of the device-resident LLaMA step (see llama.h, llama_kernels.cuh).
#include "llama_kernels.cuh"
#include "llama_mega6.cuh"
#include "llama_prefill.cuh"
#include "tp.h"
#include <stdlib.h>
#include <math.h>
#include <string.h>
#include <algorithm>

namespace mg4 {
using namespace k;

static size_t g_max_dyn_smem = 0;

template <int WT, int NT>
static void launch_mv(const MatvecArgs &a, int grid, size_t smem, cudaStream_t s) {
    static bool configured[64] = {};   // the attribute is per device (minigpt4_b200_set_device: several contexts of one process may sit on different GPUs)
    int dev = 0; cudaGetDevice(&dev);
    if (!configured[dev & 63]) {
        CUDA_CHECK(cudaFuncSetAttribute(matvec_kernel<WT, NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g_max_dyn_smem));
        configured[dev & 63] = true;
    }
    matvec_kernel<WT, NT><<<grid, kThreads, smem, s>>>(a);
}
template <int WT>
static void launch_mv_nt(int nt, const MatvecArgs &a, int grid, size_t smem, cudaStream_t s) {
    switch (nt) {
        case 1: launch_mv<WT, 1>(a, grid, smem, s); break;
        case 2: launch_mv<WT, 2>(a, grid, smem, s); break;
        case 4: launch_mv<WT, 4>(a, grid, smem, s); break;
        default: launch_mv<WT, 8>(a, grid, smem, s); break;
    }
}
static int nt_for(int ntok) { return ntok <= 1 ? 1 : ntok <= 2 ? 2 : ntok <= 4 ? 4 : 8; }

static void launch_stage(const MatvecArgs &a, cudaStream_t s, unsigned long long *counter) {
    const int act = act_of(a.w.type);
    const size_t astride = act_bytes(act, a.w.cols);
    switch (act) {
        case ACT_Q8_0: stage_kernel<ACT_Q8_0><<<a.ntok, kThreads, 0, s>>>(a.x, a.x_stride, a.norm_w, a.w.cols, a.staged, astride); break;
        case ACT_Q8_1: stage_kernel<ACT_Q8_1><<<a.ntok, kThreads, 0, s>>>(a.x, a.x_stride, a.norm_w, a.w.cols, a.staged, astride); break;
        case ACT_Q8_K: stage_kernel<ACT_Q8_K><<<a.ntok, kThreads, 0, s>>>(a.x, a.x_stride, a.norm_w, a.w.cols, a.staged, astride); break;
        default: stage_kernel<ACT_F16><<<a.ntok, kThreads, 0, s>>>(a.x, a.x_stride, a.norm_w, a.w.cols, a.staged, astride); break;
    }
    CUDA_CHECK(cudaGetLastError());
    if (counter) ++*counter;
}
// restage = false when the previous launch staged the same input in the same format (unfused q/k/v of one type)
static void launch_matvec(MatvecArgs a, int nt, int sm_count, cudaStream_t s, unsigned long long *counter, bool restage = true) {
    if (restage) launch_stage(a, s, counter);
    const int rows = a.w.rows;
    const int target = 2 * sm_count * kWarps;
    int rpw = (rows + target - 1) / target;
    rpw = std::max(2, (rpw + 1) & ~1);
    a.rows_per_warp = rpw;
    const int grid = (rows + kWarps * rpw - 1) / (kWarps * rpw);
    const size_t smem = (size_t)nt * act_bytes(act_of(a.w.type), a.w.cols);
    if (smem > g_max_dyn_smem) MG4_PANIC("activation staging needs %zu B of shared memory (> %zu)", smem, g_max_dyn_smem);
    switch (a.w.type) {
        case GG_Q4_0: launch_mv_nt<GG_Q4_0>(nt, a, grid, smem, s); break;
        case GG_Q4_1: launch_mv_nt<GG_Q4_1>(nt, a, grid, smem, s); break;
        case GG_Q5_K: launch_mv_nt<GG_Q5_K>(nt, a, grid, smem, s); break;
        case GG_Q4_K: launch_mv_nt<GG_Q4_K>(nt, a, grid, smem, s); break;
        case GG_Q5_0: launch_mv_nt<GG_Q5_0>(nt, a, grid, smem, s); break;
        case GG_Q5_1: launch_mv_nt<GG_Q5_1>(nt, a, grid, smem, s); break;
        case GG_Q8_0: launch_mv_nt<GG_Q8_0>(nt, a, grid, smem, s); break;
        case GG_Q6_K: launch_mv_nt<GG_Q6_K>(nt, a, grid, smem, s); break;
        case GG_F16: launch_mv_nt<GG_F16>(nt, a, grid, smem, s); break;
        default: MG4_PANIC("no matvec kernel for ggml type %d", a.w.type);
    }
    CUDA_CHECK(cudaGetLastError());
    if (counter) ++*counter;
}

// ------------------------------------------------------------------------------------------------
// weight upload + repack
// ------------------------------------------------------------------------------------------------
static bool type_supported(int t) {  // (Q4_K, Q5_0, Q5_1, Q8_0: tests/test_block_types_gpu.py)
    return t == GG_Q4_0 || t == GG_Q4_1 || t == GG_Q4_K || t == GG_Q5_K || t == GG_Q6_K || t == GG_F16 || t == GG_Q5_0 || t == GG_Q5_1 || t == GG_Q8_0;
}

static void qmat_alloc(QMat &m, int type, int rows, int cols) {
    m.type = type; m.rows = (rows + 1) & ~1; m.cols = cols;
    const size_t R = (size_t)m.rows;
    auto zalloc = [](void **p, size_t n) { CUDA_CHECK(cudaMalloc(p, n)); CUDA_CHECK(cudaMemset(*p, 0, n)); };
    switch (type) {
        case GG_Q4_0: m.row_bytes = (cols / 32 * 18 + 15) & ~15; zalloc(&m.p0, R * m.row_bytes + 256); break;
        case GG_Q4_1: m.row_bytes = (cols / 32 * 20 + 15) & ~15; zalloc(&m.p0, R * m.row_bytes + 256); break;
        case GG_Q5_K: m.row_bytes = cols / 256 * 176; zalloc(&m.p0, R * m.row_bytes + 256); break;   // row-packed: [nsb x 128 B qs][nsb x 32 B qh][nsb x 16 B scales, d, dmin]
        case GG_Q4_K: zalloc(&m.p0, R * cols / 256 * 128); zalloc(&m.p2, R * cols / 256 * 16); break;
        case GG_Q8_0: zalloc(&m.p0, R * cols / 32 * 32); zalloc(&m.p2, R * cols / 32 * 2); break;
        case GG_Q5_0: zalloc(&m.p0, R * cols / 32 * 16); zalloc(&m.p1, R * cols / 32 * 4); zalloc(&m.p2, R * cols / 32 * 2); break;
        case GG_Q5_1: zalloc(&m.p0, R * cols / 32 * 16); zalloc(&m.p1, R * cols / 32 * 4); zalloc(&m.p2, R * cols / 32 * 4); break;
        case GG_Q6_K: zalloc(&m.p0, R * cols / 256 * 128); zalloc(&m.p1, R * cols / 256 * 64); zalloc(&m.p2, R * cols / 256 * 16); zalloc(&m.p3, R * cols / 256 * 2); break;
        case GG_F16: zalloc(&m.p0, R * cols * 2); break;
        default: MG4_PANIC("unsupported weight type %d", type);
    }
    m.bytes = (size_t)rows * gg_row_bytes(type, (size_t)cols);
}
static void qmat_free(QMat &m) {
    for (void **p : {&m.p0, &m.p1, &m.p2, &m.p3}) if (*p) { cudaFree(*p); *p = nullptr; }
}

struct Stager {  // raw tensor bytes -> device scratch
    unsigned char *dev = nullptr; size_t cap = 0;
    unsigned char *put(const void *host, size_t n) {
        if (n > cap) { if (dev) cudaFree(dev); cap = n + (n >> 2); CUDA_CHECK(cudaMalloc((void **)&dev, cap)); }
        CUDA_CHECK(cudaMemcpy(dev, host, n, cudaMemcpyHostToDevice));
        return dev;
    }
    ~Stager() { if (dev) cudaFree(dev); }
};

// copy rows [row0,row0+nrows) x column range [col0,col0+ncols) of src into dst at dst_row = r*row_mul + row_off, dst_col0
static void repack_into(QMat &dst, const HostTensor &src, Stager &st, int row0, int nrows, int col0, int ncols, int row_mul, int row_off, int dst_col0) {
    const int src_cols = (int)src.ne[0];
    const size_t rb = gg_row_bytes(src.gg, (size_t)src_cols);
    const unsigned char *raw = st.put(src.data + (size_t)row0 * rb, (size_t)nrows * rb);
    const int be = (int)gg_block_elems(src.gg);
    const int src_nb = src_cols / be, blk0 = col0 / be, nblk = ncols / be, dst_nb = dst.cols / be, dblk0 = dst_col0 / be;
    const size_t n = (size_t)nrows * nblk;
    const int th = 256; const unsigned gr = (unsigned)((n + th - 1) / th);
    switch (src.gg) {
        case GG_Q4_0: repack_q4<<<gr, th>>>(raw, src_nb, blk0, nblk, nrows, false, (unsigned char *)dst.p0, dst_nb, dst.row_bytes, row_mul, row_off, dblk0); break;
        case GG_Q4_1: repack_q4<<<gr, th>>>(raw, src_nb, blk0, nblk, nrows, true, (unsigned char *)dst.p0, dst_nb, dst.row_bytes, row_mul, row_off, dblk0); break;
        case GG_Q5_K: repack_q5k<<<gr, th>>>(raw, src_nb, blk0, nblk, nrows, (unsigned char *)dst.p0, dst_nb, dst.row_bytes, row_mul, row_off, dblk0); break;
        case GG_Q4_K: repack_q4k<<<gr, th>>>(raw, src_nb, blk0, nblk, nrows, (unsigned char *)dst.p0, (unsigned char *)dst.p2, dst_nb, row_mul, row_off, dblk0); break;
        case GG_Q5_0: case GG_Q5_1: case GG_Q8_0:
            repack_b32<<<gr, th>>>(src.gg, raw, src_nb, blk0, nblk, nrows, (unsigned char *)dst.p0, (unsigned char *)dst.p1, (unsigned char *)dst.p2, dst_nb, row_mul, row_off, dblk0); break;
        case GG_Q6_K: repack_q6k<<<gr, th>>>(raw, src_nb, blk0, nblk, nrows, (unsigned char *)dst.p0, (unsigned char *)dst.p1, (unsigned char *)dst.p2, (unsigned short *)dst.p3, dst_nb, row_mul, row_off, dblk0); break;
        case GG_F16: repack_f16<<<gr, th>>>((const unsigned short *)raw, src_cols, col0, ncols, nrows, (unsigned short *)dst.p0, dst.cols, row_mul, row_off, dst_col0); break;
        default: MG4_PANIC("unsupported weight type %d", src.gg);
    }
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaDeviceSynchronize());  // the stager is reused by the next tensor
}

static float *upload_f32(const HostTensor &t) {
    if (t.gg != GG_F32) MG4_PANIC("tensor %s must be F32", t.name.c_str());
    float *d; CUDA_CHECK(cudaMalloc((void **)&d, t.nbytes)); CUDA_CHECK(cudaMemcpy(d, t.data, t.nbytes, cudaMemcpyHostToDevice));
    return d;
}

// ------------------------------------------------------------------------------------------------
LlamaDevice::LlamaDevice() {}
LlamaDevice::~LlamaDevice() {
    if (graph_) cudaGraphExecDestroy(graph_);
    for (auto &L : layers_) { qmat_free(L.qkv); qmat_free(L.wq); qmat_free(L.wk); qmat_free(L.wv); qmat_free(L.wo); qmat_free(L.w13); qmat_free(L.w2); cudaFree(L.attn_norm); cudaFree(L.ffn_norm); }
    qmat_free(output_);
    for (void *p : {(void *)final_norm_, tok_raw_, (void *)kcache_, (void *)vcache_, (void *)rope_, (void *)tab_exp_, (void *)tab_silu_, (void *)x_, (void *)q_, (void *)att_,
                    (void *)act_, (void *)logits_, (void *)partial_, (void *)qact_, (void *)embd_in_, (void *)state_}) if (p) cudaFree(p);
    for (auto &L : layers_) for (PQMat *m : {&L.pqkv, &L.pwo, &L.pw13, &L.pw2}) { if (m->q) cudaFree(m->q); if (m->sc) cudaFree(m->sc); }
    for (void *p : {(void *)pf_q8_, pf_sc_, (void *)tok_ids_, pf_part_}) if (p) cudaFree(p);
    if (mega_barrier_) cudaFree(mega_barrier_);
    if (mega_trace_) cudaFree(mega_trace_);
    delete (mk6::Params6 *)mega6_params_;
    if (h_state_) cudaFreeHost(h_state_);
    if (h_argmax_) cudaFreeHost(h_argmax_);
    if (ev0_) cudaEventDestroy(ev0_);
    if (ev1_) cudaEventDestroy(ev1_);
    if (stream_) cudaStreamDestroy(stream_);
}

static inline unsigned short f2h_bits(float f) { __half h = __float2half_rn(f); unsigned short u; memcpy(&u, &h, 2); return u; }
static inline float h2f_bits(unsigned short u) { __half h; memcpy(&h, &u, 2); return __half2float(h); }

bool LlamaDevice::load(const LlamaFile &f, int n_ctx, TPLink *tp) {
    tp_ = tp;
    const int world = tp ? tp->world : 1, rank = tp ? tp->rank : 0;
    d_.n_vocab = (int)f.n_vocab; d_.n_embd = (int)f.n_embd; d_.n_head = (int)f.n_head; d_.n_layer = (int)f.n_layer;
    d_.n_ff = (int)f.n_ff(); d_.n_ctx = n_ctx; d_.head_dim = d_.n_embd / d_.n_head;
    if (d_.head_dim != 128 || (int)f.n_rot != 128) { MG4_ERR("only head_dim 128 LLaMA models are supported (got %d)", d_.head_dim); return false; }
    if (n_ctx < 8 || n_ctx > 32768) { MG4_ERR("n_ctx %d is outside the supported range 8 .. 32768 (attention scratch = 6 n_ctx bytes of shared memory)", n_ctx); return false; }
    if (d_.n_head % world || d_.n_ff % (32 * world)) { MG4_ERR("tensor-parallel degree %d does not divide the model", world); return false; }
    n_head_local_ = d_.n_head / world; n_embd_local_ = n_head_local_ * 128; n_ff_local_ = d_.n_ff / world;
    const int E = d_.n_embd, El = n_embd_local_, FF = d_.n_ff, FFl = n_ff_local_;

    int dev = 0; CUDA_CHECK(cudaGetDevice(&dev));
    cudaDeviceProp prop; CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
    sm_count_ = prop.multiProcessorCount;
    g_max_dyn_smem = std::min<size_t>(prop.sharedMemPerBlockOptin, 220 * 1024) - 1024;
    CUDA_CHECK(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
    CUDA_CHECK(cudaEventCreate(&ev0_)); CUDA_CHECK(cudaEventCreate(&ev1_));

    Stager st;
    bytes_per_token_ = 0;
    layers_.resize((size_t)d_.n_layer);
    for (int il = 0; il < d_.n_layer; ++il) {
        Layer &L = layers_[(size_t)il];
        const std::string p = "layers." + std::to_string(il) + ".";
        const HostTensor &wq = f.get(p + "attention.wq.weight"), &wk = f.get(p + "attention.wk.weight"), &wv = f.get(p + "attention.wv.weight");
        const HostTensor &wo = f.get(p + "attention.wo.weight");
        const HostTensor &w1 = f.get(p + "feed_forward.w1.weight"), &w2 = f.get(p + "feed_forward.w2.weight"), &w3 = f.get(p + "feed_forward.w3.weight");
        for (const HostTensor *t : {&wq, &wk, &wv, &wo, &w1, &w2, &w3}) {
            if (!type_supported(t->gg)) { MG4_ERR("tensor %s has unsupported type %d", t->name.c_str(), t->gg); return false; }
            const int be = (int)gg_block_elems(t->gg);
            if (world > 1 && be > 1 && ((El % be) || (FFl % be))) { MG4_ERR("tensor-parallel split of %s is not aligned to its %d-element quant blocks", t->name.c_str(), be); return false; }
        }
        if (wq.ne[0] != E || wq.ne[1] != E || w1.ne[1] != FF || w2.ne[0] != FF) { MG4_ERR("unexpected tensor shapes in layer %d", il); return false; }
        if (w1.gg != w3.gg) { MG4_ERR("w1/w3 of layer %d differ in type", il); return false; }
        L.fused_qkv = wq.gg == wk.gg && wk.gg == wv.gg;
        if (L.fused_qkv) {
            qmat_alloc(L.qkv, wq.gg, 3 * El, E);
            repack_into(L.qkv, wq, st, rank * El, El, 0, E, 1, 0, 0);
            repack_into(L.qkv, wk, st, rank * El, El, 0, E, 1, El, 0);
            repack_into(L.qkv, wv, st, rank * El, El, 0, E, 1, 2 * El, 0);
            bytes_per_token_ += L.qkv.bytes;
        } else {
            qmat_alloc(L.wq, wq.gg, El, E); repack_into(L.wq, wq, st, rank * El, El, 0, E, 1, 0, 0);
            qmat_alloc(L.wk, wk.gg, El, E); repack_into(L.wk, wk, st, rank * El, El, 0, E, 1, 0, 0);
            qmat_alloc(L.wv, wv.gg, El, E); repack_into(L.wv, wv, st, rank * El, El, 0, E, 1, 0, 0);
            bytes_per_token_ += L.wq.bytes + L.wk.bytes + L.wv.bytes;
        }
        qmat_alloc(L.wo, wo.gg, E, El); repack_into(L.wo, wo, st, 0, E, rank * El, El, 1, 0, 0);
        qmat_alloc(L.w13, w1.gg, 2 * FFl, E);
        repack_into(L.w13, w1, st, rank * FFl, FFl, 0, E, 2, 0, 0);
        repack_into(L.w13, w3, st, rank * FFl, FFl, 0, E, 2, 1, 0);
        qmat_alloc(L.w2, w2.gg, E, FFl); repack_into(L.w2, w2, st, 0, E, rank * FFl, FFl, 1, 0, 0);
        bytes_per_token_ += L.wo.bytes + L.w13.bytes + L.w2.bytes;
        L.attn_norm = upload_f32(f.get(p + "attention_norm.weight"));
        L.ffn_norm = upload_f32(f.get(p + "ffn_norm.weight"));
    }
    {
        const HostTensor &out = f.get("output.weight");
        if (!type_supported(out.gg)) { MG4_ERR("output.weight has unsupported type %d", out.gg); return false; }
        qmat_alloc(output_, out.gg, d_.n_vocab, E);
        repack_into(output_, out, st, 0, d_.n_vocab, 0, E, 1, 0, 0);
        bytes_per_token_ += output_.bytes;
        final_norm_ = upload_f32(f.get("norm.weight"));
        const HostTensor &tok = f.get("tok_embeddings.weight");
        tok_type_ = tok.gg;
        if (!(type_supported(tok.gg) || tok.gg == GG_F32)) { MG4_ERR("tok_embeddings has unsupported type %d", tok.gg); return false; }
        CUDA_CHECK(cudaMalloc(&tok_raw_, tok.nbytes));
        CUDA_CHECK(cudaMemcpy(tok_raw_, tok.data, tok.nbytes, cudaMemcpyHostToDevice));
    }
    // ggml's fp16 lookup tables (ggml_init): exp and silu, computed with the host libm exactly as ggml does
    {
        std::vector<unsigned short> te(65536), ts(65536);
        for (int i = 0; i < 65536; ++i) { const float x = h2f_bits((unsigned short)i); te[(size_t)i] = f2h_bits(expf(x)); ts[(size_t)i] = f2h_bits(x / (1.0f + expf(-x))); }
        CUDA_CHECK(cudaMalloc((void **)&tab_exp_, 131072)); CUDA_CHECK(cudaMemcpy(tab_exp_, te.data(), 131072, cudaMemcpyHostToDevice));
        CUDA_CHECK(cudaMalloc((void **)&tab_silu_, 131072)); CUDA_CHECK(cudaMemcpy(tab_silu_, ts.data(), 131072, cudaMemcpyHostToDevice));
    }
    // RoPE table, mode 0: theta_i = pos * 10000^(-2i/n_rot) formed by repeated multiplication, cosf/sinf from libm (ggml_rope_f32)
    {
        const int hd2 = 64;
        std::vector<float2> tab((size_t)n_ctx * hd2);
        const float theta_scale = powf(10000.0f, -2.0f / 128.0f);
        for (int p = 0; p < n_ctx; ++p) { float theta = (float)p; for (int i = 0; i < hd2; ++i) { tab[(size_t)p * hd2 + i] = make_float2(cosf(theta), sinf(theta)); theta *= theta_scale; } }
        CUDA_CHECK(cudaMalloc((void **)&rope_, tab.size() * sizeof(float2)));
        CUDA_CHECK(cudaMemcpy(rope_, tab.data(), tab.size() * sizeof(float2), cudaMemcpyHostToDevice));
    }
    const size_t kv = (size_t)d_.n_layer * n_ctx * El;
    CUDA_CHECK(cudaMalloc((void **)&kcache_, kv * 2)); CUDA_CHECK(cudaMemset(kcache_, 0, kv * 2));
    CUDA_CHECK(cudaMalloc((void **)&vcache_, kv * 2)); CUDA_CHECK(cudaMemset(vcache_, 0, kv * 2));
    const size_t R = (size_t)kPrefillMax;  // rows of one prefill pass (the per-op path uses the first 8)
    CUDA_CHECK(cudaMalloc((void **)&x_, R * E * 4));
    CUDA_CHECK(cudaMalloc((void **)&q_, R * El * 4));
    CUDA_CHECK(cudaMalloc((void **)&att_, R * El * 4));
    CUDA_CHECK(cudaMalloc((void **)&act_, R * FFl * 4));
    CUDA_CHECK(cudaMalloc((void **)&partial_, (size_t)8 * E * 4));
    CUDA_CHECK(cudaMalloc((void **)&tok_ids_, R * 4));
    CUDA_CHECK(cudaMalloc((void **)&qact_, (size_t)8 * ((size_t)std::max(E, FF) * 2 + 4096)));
    CUDA_CHECK(cudaMalloc((void **)&logits_, (size_t)(d_.n_vocab + 1) * 4));
    CUDA_CHECK(cudaMalloc((void **)&embd_in_, (size_t)512 * E * 4));
    CUDA_CHECK(cudaMalloc((void **)&state_, sizeof(DeviceState))); CUDA_CHECK(cudaMemset(state_, 0, sizeof(DeviceState)));
    CUDA_CHECK(cudaHostAlloc((void **)&h_state_, sizeof(DeviceState), cudaHostAllocDefault)); memset(h_state_, 0, sizeof(DeviceState));
    CUDA_CHECK(cudaHostAlloc((void **)&h_argmax_, 64, cudaHostAllocDefault)); *h_argmax_ = 0;
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaFuncSetAttribute(attn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, std::max(49152, d_.n_ctx * 6)));
    if (tp_ && tp_->world > 1) tp_->setup_peers(E, stream_);
    pf_ready_ = build_prefill();
    build_graph();
    MG4_INFO("LLaMA on device: %d layers, n_embd %d, n_ff %d, vocab %d, %.1f MB streamed per token, tp %d/%d", d_.n_layer, E, FF, d_.n_vocab,
             bytes_per_token_ / 1048576.0, rank, world);
    return true;
}

// ------------------------------------------------------------------------------------------------
// one pass of all layers over `ntok` (<= nt) rows that sit in x_; positions/tokens come from *state_
// ------------------------------------------------------------------------------------------------
void LlamaDevice::launch_layers(int nt, int ntok, bool want_logits) {
    const int E = d_.n_embd, El = n_embd_local_, FFl = n_ff_local_, C = d_.n_ctx;
    const bool tp = tp_ && tp_->world > 1;
    const float kq_scale = 1.0f / sqrtf((float)d_.n_embd / (float)d_.n_head);
    const size_t attn_smem = (size_t)C * 6;
    // wo / down: x_ += W x, the residual added in the matvec epilogue or, under tensor parallelism, after the partial sums are all-reduced
    auto matvec_resid = [&](const QMat &w, const float *x, int x_stride) {
        MatvecArgs b{};
        b.w = w; b.x = x; b.x_stride = x_stride; b.norm_w = nullptr; b.ntok = ntok; b.n_valid = b.w.rows; b.state = state_; b.tab_silu = tab_silu_; b.staged = qact_;
        if (!tp) { b.epi = EPI_RESID; b.out = x_; b.out_stride = E; b.resid = x_; launch_matvec(b, nt, sm_count_, stream_, &launches_); }
        else if (tp_->peers_ready()) {   // partial -> this rank's exchange buffer; ONE kernel: signal peers, wait, sum all partials + residual out of peer memory
            b.epi = EPI_PLAIN; b.out = tp_->partial_out(); b.out_stride = E; launch_matvec(b, nt, sm_count_, stream_, &launches_);
            tp_->all_reduce_resid(x_, x_, (size_t)ntok * E, stream_); ++launches_;
        } else {
            b.epi = EPI_PLAIN; b.out = partial_; b.out_stride = E; launch_matvec(b, nt, sm_count_, stream_, &launches_);
            tp_->all_reduce_sum(partial_, (size_t)ntok * E, stream_);
            add_kernel<<<(ntok * E + 255) / 256, 256, 0, stream_>>>(x_, partial_, ntok * E); ++launches_;
        }
    };
    for (int il = 0; il < d_.n_layer; ++il) {
        Layer &L = layers_[(size_t)il];
        __half *kc = kcache_ + (size_t)il * C * El, *vc = vcache_ + (size_t)il * C * El;
        MatvecArgs a{};
        a.x = x_; a.x_stride = E; a.norm_w = L.attn_norm; a.ntok = ntok; a.epi = EPI_QKV; a.staged = qact_;
        a.q_out = q_; a.kcache = kc; a.vcache = vc; a.rope = rope_; a.e_local = El; a.half_dim = 64; a.state = state_; a.tab_silu = tab_silu_;
        if (L.fused_qkv) { a.w = L.qkv; a.part = -1; a.n_valid = a.w.rows; launch_matvec(a, nt, sm_count_, stream_, &launches_); }
        else {
            const QMat *ms[3] = {&L.wq, &L.wk, &L.wv};
            for (int part = 0; part < 3; ++part) {
                const bool same = part > 0 && act_of(ms[part]->type) == act_of(ms[part - 1]->type);
                a.w = *ms[part]; a.part = part; a.n_valid = a.w.rows; launch_matvec(a, nt, sm_count_, stream_, &launches_, !same);
            }
        }
        attn_kernel<<<dim3((unsigned)n_head_local_, (unsigned)ntok), 256, attn_smem, stream_>>>(q_, kc, vc, att_, state_, El, C, kq_scale, tab_exp_);
        CUDA_CHECK(cudaGetLastError()); ++launches_;
        matvec_resid(L.wo, att_, El);
        MatvecArgs c{};
        c.w = L.w13; c.x = x_; c.x_stride = E; c.norm_w = L.ffn_norm; c.ntok = ntok; c.epi = EPI_SWIGLU; c.out = act_; c.out_stride = FFl; c.n_valid = c.w.rows;
        c.state = state_; c.tab_silu = tab_silu_; c.staged = qact_;
        launch_matvec(c, nt, sm_count_, stream_, &launches_);
        matvec_resid(L.w2, act_, FFl);
    }
    if (want_logits) {
        MatvecArgs o{};
        o.w = output_; o.x = x_ + (size_t)(ntok - 1) * E; o.x_stride = E; o.norm_w = final_norm_; o.ntok = 1; o.epi = EPI_LOGITS; o.out = logits_; o.n_valid = d_.n_vocab;
        o.state = state_; o.tab_silu = tab_silu_; o.staged = qact_;
        launch_matvec(o, 1, sm_count_, stream_, &launches_);
    }
    finalize_kernel<<<1, 32, 0, stream_>>>(state_, want_logits ? 1 : 0, nullptr); ++launches_;
    CUDA_CHECK(cudaGetLastError());
    // 4-byte result of the step for the greedy fast path (pinned; valid after the next stream sync)
    if (want_logits) CUDA_CHECK(cudaMemcpyAsync(h_argmax_, &state_->argmax_id, 4, cudaMemcpyDeviceToHost, stream_));
}

// One or more passes over `n` mixed rows starting at position n_past: ids[i] >= 0 is a token, ids[i] < 0 is row -1 - ids[i] of emb_host
// (n_emb rows of n_embd floats).  The engine collects consecutive add_tokens / add_embedding calls of a chat turn (reference call sites
// minigpt4.cpp:2365-2382 and :2399-2415 evaluate each piece separately; results are batch invariant) and evaluates them together, so the
// weights stream once per kPrefillMax rows instead of once per piece.
bool LlamaDevice::eval_rows(const int32_t *ids, int n, const float *emb_host, int n_emb, int n_past) {
    if (n <= 0) return true;
    if (n_past + n > d_.n_ctx) { MG4_ERR("context overflow: %d + %d > n_ctx %d", n_past, n, d_.n_ctx); return false; }
    if (n_emb > 512) { MG4_ERR("eval_rows: at most 512 embedding rows per call"); return false; }
    for (int i = 0; i < n; ++i) if (ids[i] >= d_.n_vocab || ids[i] < -n_emb) { MG4_ERR("token id %d out of range", ids[i]); return false; }
    if (n_emb > 0) CUDA_CHECK(cudaMemcpyAsync(embd_in_, emb_host, (size_t)n_emb * d_.n_embd * 4, cudaMemcpyHostToDevice, stream_));
    const int step = pf_ready_ ? kPrefillMax : 8;
    for (int i = 0; i < n; i += step) {
        const int c = std::min(step, n - i);
        const bool last = i + c == n;
        CUDA_CHECK(cudaStreamSynchronize(stream_));  // h_state_ (pinned) of the previous pass / decode step has been consumed
        h_state_->n_past = n_past + i; h_state_->n_tok = c;
        CUDA_CHECK(cudaMemcpyAsync(state_, h_state_, offsetof(DeviceState, argmax_key), cudaMemcpyHostToDevice, stream_));
        CUDA_CHECK(cudaMemcpyAsync(tok_ids_, ids + i, (size_t)c * 4, cudaMemcpyHostToDevice, stream_));
        embed_rows_kernel<<<c, 256, 0, stream_>>>(tok_type_, (const unsigned char *)tok_raw_, gg_row_bytes(tok_type_, (size_t)d_.n_embd), d_.n_embd, tok_ids_, embd_in_, x_);
        ++launches_;
        if (pf_ready_ && c >= 2) prefill_chunk(c, last);
        else launch_layers(nt_for(c), c, last);
    }
    CUDA_CHECK(cudaStreamSynchronize(stream_));
    return true;
}
void LlamaDevice::logits_to_host(float *dst) {
    CUDA_CHECK(cudaMemcpyAsync(dst, logits_, (size_t)d_.n_vocab * 4, cudaMemcpyDeviceToHost, stream_));
    CUDA_CHECK(cudaStreamSynchronize(stream_));
}
void LlamaDevice::sync_decode() {
    CUDA_CHECK(cudaStreamSynchronize(stream_));
    h_state_busy_ = false;
}
int32_t LlamaDevice::argmax() {
    sync_decode();
    return *h_argmax_;
}
void LlamaDevice::sync() { CUDA_CHECK(cudaStreamSynchronize(stream_)); h_state_busy_ = false; }
void LlamaDevice::hidden_to_host(float *dst, int n) {
    CUDA_CHECK(cudaMemcpyAsync(dst, x_, (size_t)n * d_.n_embd * 4, cudaMemcpyDeviceToHost, stream_));
    CUDA_CHECK(cudaStreamSynchronize(stream_));
}

// ------------------------------------------------------------------------------------------------
// tensor-core prefill (llama_prefill.cuh)
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tm_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr; cudaDriverEntryPointQueryResult qr;
        CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr));
        if (!p || qr != cudaDriverEntryPointSuccess) MG4_PANIC("cuTensorMapEncodeTiled is not available from this driver");
        fn = (EncodeTiledFn)p;
    }
    return fn;
}
// bytes [rows][pitch] -> boxes of box_bytes x box_rows
static void make_map_u8(void *tm, const void *ptr, size_t rows, size_t pitch, int box_bytes, int box_rows, bool swizzle128) {
    cuuint64_t dims[2] = {(cuuint64_t)pitch, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)pitch};
    cuuint32_t box[2] = {(cuuint32_t)box_bytes, (cuuint32_t)box_rows};
    cuuint32_t es[2] = {1, 1};
    CUresult r = tm_encode_fn()((CUtensorMap *)tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, (void *)ptr, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) MG4_PANIC("cuTensorMapEncodeTiled failed (%d) for [%zu x %zu] box %d x %d", (int)r, rows, pitch, box_bytes, box_rows);
}
static int pf_slots(int cols) { const int nbl = (cols / 32 + 31) / 32; return 4 * ((nbl + 3) / 4); }

static void pq_build(PQMat &p, const QMat &m) {
    p.rows = m.rows; p.rows_pad = (m.rows + 127) & ~127; p.cols = m.cols; p.nb = m.cols / 32; p.S = pf_slots(m.cols); p.q41 = m.type == GG_Q4_1;
    const size_t pitch = (size_t)32 * p.S * 32;
    CUDA_CHECK(cudaMalloc((void **)&p.q, (size_t)p.rows_pad * pitch)); CUDA_CHECK(cudaMemset(p.q, 0, (size_t)p.rows_pad * pitch));
    CUDA_CHECK(cudaMalloc(&p.sc, (size_t)p.rows_pad * 32 * p.S * 4)); CUDA_CHECK(cudaMemset(p.sc, 0, (size_t)p.rows_pad * 32 * p.S * 4));
    const size_t n = (size_t)m.rows * p.nb;
    pf::expand_q4_classmajor<<<(unsigned)((n + 255) / 256), 256>>>((const unsigned char *)m.p0, m.row_bytes, m.rows, p.nb, p.q41 ? 1 : 0, p.S, p.q, (__half2 *)p.sc);
    CUDA_CHECK(cudaGetLastError());
    make_map_u8(p.tm, p.q, (size_t)p.rows_pad, pitch, 128, pf::kRows, true);
}

bool LlamaDevice::build_prefill() {
    if (getenv("MINIGPT4_B200_NO_PREFILL_GEMM")) return false;
    if (tp_ && tp_->world > 1) return false;  // (tensor-parallel ranks keep the per-op prefill path for now)
    for (auto &L : layers_) {   // (each matrix stages its own input: mixed Q4_0 / Q4_1 layers are fine)
        if (!L.fused_qkv) return false;
        for (const QMat *m : {&L.qkv, &L.wo, &L.w13, &L.w2}) if (m->type != GG_Q4_0 && m->type != GG_Q4_1) return false;
    }
    const int E = d_.n_embd, FF = d_.n_ff;
    size_t free_b = 0, total_b = 0; CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
    const size_t need = (size_t)d_.n_layer * ((size_t)4 * E * E + (size_t)3 * E * (size_t)32 * pf_slots(FF) * 32 / 1) + ((size_t)1 << 30);
    if (need > free_b) { MG4_INFO("prefill operand cache (%.1f GB) does not fit: per-op prefill path", need / 1073741824.0); return false; }
    for (auto &L : layers_) { pq_build(L.pqkv, L.qkv); pq_build(L.pwo, L.wo); pq_build(L.pw13, L.w13); pq_build(L.pw2, L.w2); }
    pf_S_e_ = pf_slots(E); pf_S_ff_ = pf_slots(FF);
    const size_t pitch_e = (size_t)32 * pf_S_e_ * 32, pitch_ff = (size_t)32 * pf_S_ff_ * 32, R = (size_t)kPrefillMax;
    CUDA_CHECK(cudaMalloc((void **)&pf_q8_, R * std::max(pitch_e, pitch_ff))); CUDA_CHECK(cudaMemset(pf_q8_, 0, R * std::max(pitch_e, pitch_ff)));
    CUDA_CHECK(cudaMalloc(&pf_sc_, R * std::max(pitch_e, pitch_ff) / 4)); CUDA_CHECK(cudaMemset(pf_sc_, 0, R * std::max(pitch_e, pitch_ff) / 4));
    make_map_u8(pf_tmB_e_, pf_q8_, R, pitch_e, 128, pf::kTok, true);
    make_map_u8(pf_tmS_e_, pf_sc_, R, pitch_e / 4, 32, pf::kTok, false);
    make_map_u8(pf_tmB_ff_, pf_q8_, R, pitch_ff, 128, pf::kTok, true);
    make_map_u8(pf_tmS_ff_, pf_sc_, R, pitch_ff / 4, 32, pf::kTok, false);
    pf_part_bytes_ = (size_t)96 << 20;   // roots of K-split slices: [slice][token][row] {d-tree, m-tree}
    CUDA_CHECK(cudaMalloc(&pf_part_, pf_part_bytes_));
    const size_t smem = 1024 + (size_t)pf::kStages * pf::kStageBytes + pf::kStackBytes + 256;
    CUDA_CHECK(cudaFuncSetAttribute(pf::prefill_gemm_q4<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CUDA_CHECK(cudaFuncSetAttribute(pf::prefill_gemm_q4<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    CUDA_CHECK(cudaDeviceSynchronize());
    MG4_INFO("tensor-core prefill: int8 class-major operand cache built (%d / %d slots per class)", pf_S_e_, pf_S_ff_);
    return true;
}

// one pass of all layers over n (<= kPrefillMax) rows in x_; positions from *state_ (n_past), KV rows appended, logits of the last row
void LlamaDevice::prefill_chunk(int n, bool want_logits) {
    const int E = d_.n_embd, El = n_embd_local_, FFl = n_ff_local_, C = d_.n_ctx;
    const float kq_scale = 1.0f / sqrtf((float)d_.n_embd / (float)d_.n_head);
    const size_t smem = 1024 + (size_t)pf::kStages * pf::kStageBytes + pf::kStackBytes + 256;
    const unsigned ty = (unsigned)((n + pf::kTok - 1) / pf::kTok);
    auto stage = [&](const QMat &w, const float *x, int x_stride, const float *nw, int S) {
        const int act = act_of(w.type);
        const size_t sm = act_bytes(act, w.cols);
        if (act == ACT_Q8_1) pf::stage_rows_classmajor<ACT_Q8_1><<<n, 256, sm, stream_>>>(x, x_stride, nw, w.cols, S, pf_q8_, (float2 *)pf_sc_);
        else pf::stage_rows_classmajor<ACT_Q8_0><<<n, 256, sm, stream_>>>(x, x_stride, nw, w.cols, S, pf_q8_, (float2 *)pf_sc_);
        ++launches_;
    };
    auto gemm = [&](const PQMat &p, bool ff_wide, pf::PrefillArgs a) {
        a.rows = p.rows; a.n_tok = n; a.nb = p.nb; a.S = p.S; a.wsc = (const __half2 *)p.sc; a.state = state_; a.tab_silu = tab_silu_;
        const CUtensorMap *tb = (const CUtensorMap *)(ff_wide ? pf_tmB_ff_ : pf_tmB_e_), *ts = (const CUtensorMap *)(ff_wide ? pf_tmS_ff_ : pf_tmS_e_);
        // K split over subtrees of the class butterfly so that matrices with few 128-row tiles (wo / down: 32) still fill the machine
        const int tiles = p.rows_pad / pf::kRows;
        int nz = 1;
        if (!getenv("MINIGPT4_B200_PREFILL_NO_KSPLIT")) {   // waves of CTAs x work per CTA (+ a little per-CTA overhead), smallest wins
            double best = 1e30;
            for (int c = 1; c <= 8; c *= 2) {
                if ((size_t)c * n * p.rows_pad * sizeof(float2) > pf_part_bytes_ && c > 1) break;
                const int ctas = tiles * (int)ty * c;
                const double cost = (double)((ctas + sm_count_ - 1) / sm_count_) / c + 0.02 * c;
                if (cost < best - 1e-9) { best = cost; nz = c; }
            }
        }
        a.jr_per_z = 32 / nz; a.partial = (float2 *)pf_part_; a.part_tok = n; a.part_rows = p.rows_pad;
        const dim3 grid((unsigned)tiles, ty, (unsigned)nz);
        if (p.q41) pf::prefill_gemm_q4<true><<<grid, pf::kThreads, smem, stream_>>>(*(const CUtensorMap *)p.tm, *tb, *ts, a);
        else pf::prefill_gemm_q4<false><<<grid, pf::kThreads, smem, stream_>>>(*(const CUtensorMap *)p.tm, *tb, *ts, a);
        ++launches_;
        if (nz > 1) { const size_t work = (size_t)n * (p.rows / 2); pf::prefill_combine<<<(unsigned)((work + 255) / 256), 256, 0, stream_>>>(a, nz); ++launches_; }
    };
    for (int il = 0; il < d_.n_layer; ++il) {
        Layer &L = layers_[(size_t)il];
        __half *kc = kcache_ + (size_t)il * C * El, *vc = vcache_ + (size_t)il * C * El;
        stage(L.qkv, x_, E, L.attn_norm, pf_S_e_);
        { pf::PrefillArgs a{}; a.epi = EPI_QKV; a.q_out = q_; a.kcache = kc; a.vcache = vc; a.rope = rope_; a.e_local = El; a.half_dim = 64; gemm(L.pqkv, false, a); }
        attn_kernel<<<dim3((unsigned)n_head_local_, (unsigned)n), 256, (size_t)C * 6, stream_>>>(q_, kc, vc, att_, state_, El, C, kq_scale, tab_exp_); ++launches_;
        stage(L.wo, att_, El, nullptr, pf_S_e_);
        { pf::PrefillArgs a{}; a.epi = EPI_RESID; a.out = x_; a.out_stride = E; a.resid = x_; gemm(L.pwo, false, a); }
        stage(L.w13, x_, E, L.ffn_norm, pf_S_e_);
        { pf::PrefillArgs a{}; a.epi = EPI_SWIGLU; a.out = act_; a.out_stride = FFl; gemm(L.pw13, false, a); }
        stage(L.w2, act_, FFl, nullptr, pf_S_ff_);
        { pf::PrefillArgs a{}; a.epi = EPI_RESID; a.out = x_; a.out_stride = E; a.resid = x_; gemm(L.pw2, true, a); }
    }
    CUDA_CHECK(cudaGetLastError());
    if (want_logits) {
        MatvecArgs o{};
        o.w = output_; o.x = x_ + (size_t)(n - 1) * E; o.x_stride = E; o.norm_w = final_norm_; o.ntok = 1; o.epi = EPI_LOGITS; o.out = logits_; o.n_valid = d_.n_vocab;
        o.state = state_; o.tab_silu = tab_silu_; o.staged = qact_;
        launch_matvec(o, 1, sm_count_, stream_, &launches_);
    }
    finalize_kernel<<<1, 32, 0, stream_>>>(state_, want_logits ? 1 : 0, nullptr); ++launches_;
    CUDA_CHECK(cudaGetLastError());
    if (want_logits) CUDA_CHECK(cudaMemcpyAsync(h_argmax_, &state_->argmax_id, 4, cudaMemcpyDeviceToHost, stream_));
}

// ------------------------------------------------------------------------------------------------
// decode step as a CUDA graph: embed(tokens[0]) -> layers -> logits/arg-max -> finalize (n_past++, tokens[0] = arg-max)
// positions and the token come from *state_, so the same graph serves every step
// ------------------------------------------------------------------------------------------------
// ------------------------------------------------------------------------------------------------
// persistent megakernel program (llama_mega6.cuh)
// ------------------------------------------------------------------------------------------------
bool LlamaDevice::build_mega() {
    if (getenv("MINIGPT4_B200_NO_MEGAKERNEL")) return false;
    const bool tp = tp_ && tp_->world > 1;
    if (tp && (!tp_->peers_ready() || getenv("MINIGPT4_B200_TP_PER_OP"))) return false;   // the in-kernel all-reduce needs the peer mappings
    const int wt = output_.type;
    if (wt != GG_Q4_0 && wt != GG_Q4_1 && wt != GG_Q5_K) return false;   // homogeneous Q4_0 / Q4_1 / Q5_K files (the reference README's q5_k download has a Q6_K output matrix: per-op path)
    for (auto &L : layers_) if (!L.fused_qkv || L.qkv.type != wt || L.wo.type != wt || L.w13.type != wt || L.w2.type != wt) return false;
    // OP_EMBED gathers through dequant_elem, which has no Q4_K / Q5_0 / Q5_1 / Q8_0 case (such tok_embeddings: per-op graph)
    if (tok_type_ != GG_F32 && tok_type_ != GG_F16 && tok_type_ != GG_Q4_0 && tok_type_ != GG_Q4_1 && tok_type_ != GG_Q5_K && tok_type_ != GG_Q6_K) return false;
    if (d_.n_embd % 256 || d_.n_ff % 32 || d_.n_embd > 1024 * mk6::kNormItems || d_.n_ff > 4 * mk6::kConsumerThreads * mk6::kPlainItems) return false;
    if (d_.head_dim != 128 || d_.n_head > sm_count_ || 7 * d_.n_layer + 3 > mk6::kMaxOps) return false;
    if (tp && (n_embd_local_ % 32 || n_ff_local_ % 32)) return false;
    int coop = 0, dev = 0; CUDA_CHECK(cudaGetDevice(&dev));
    CUDA_CHECK(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
    if (!coop) return false;
    mega_type_ = wt;
    CUDA_CHECK(cudaMalloc((void **)&mega_barrier_, 64)); CUDA_CHECK(cudaMemset(mega_barrier_, 0, 64));
    mega_n_ops_ = (tp ? 7 : 5) * d_.n_layer + 3;
    if (getenv("MINIGPT4_B200_MEGA_TRACE")) { CUDA_CHECK(cudaMalloc((void **)&mega_trace_, (size_t)(mega_n_ops_ + 1) * 32 * sizeof(long long))); CUDA_CHECK(cudaMemset(mega_trace_, 0, (size_t)(mega_n_ops_ + 1) * 32 * sizeof(long long))); }

    // generation 6: self-refilled per-warp streams (llama_mega6.cuh)
    using namespace mk6;
    const int E = d_.n_embd, FF = n_ff_local_;   // (tensor parallel: this rank's feed-forward columns)
    size_t act_b = mega_type_ == GG_Q5_K ? std::max(act_bytes(ACT_Q8_K, FF), act_bytes(ACT_Q8_K, E)) : std::max(act6_bytes(FF), act6_bytes(E));
    act_b = std::max(act_b, (size_t)d_.n_ctx * 6);  // the attention op (which stages no activations) uses the region as its scratch
    act_b = (act_b + 127) & ~(size_t)127;
    if (mega_type_ == GG_Q5_K && (E % 256 || FF % 256 || FF > 256 * kConsumerWarps * kQ8kRounds || E > 256 * kConsumerWarps * 2)) return false;
    const int rb_e = layers_[0].qkv.row_bytes, rb_ff = layers_[0].w2.row_bytes;
    // a slot holds a row pair of an n_embd-wide matrix or ONE row of an n_ff-wide matrix (whose pair then takes both slots of the warp)
    int slot = std::max(2 * rb_e, rb_ff);
    slot = (slot + 15) & ~15;
    cudaDeviceProp prop; CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
    const size_t stat = 10240;  // static shared memory of decode_megakernel6 (red, redf, qh, part) + slack
    const long long room = (long long)prop.sharedMemPerBlockOptin - (long long)stat - (long long)act_b - 2 * kConsumerWarps * 8;
    int W = (int)std::min<long long>(kConsumerWarps, room / (2LL * slot));
    if (getenv("MINIGPT4_B200_MEGA_W")) W = std::min(W, atoi(getenv("MINIGPT4_B200_MEGA_W")));
    if (W < 4) return false;
    Params6 *P = new Params6();
    memset(P, 0, sizeof(Params6));
    int n = 0; bool uniform = true;   // every layer's matrices have the same shapes (the CTA's share of a kind is computed once)
    auto add = [&](int kind, int layer, const QMat *m, const float *norm) {
        Op6 &o = P->ops[n++]; o.kind = (unsigned char)kind; o.layer = (unsigned short)layer; o.norm_w = norm;
        if (m) {
            o.cols = m->cols; o.row_bytes = m->row_bytes; o.w = (const unsigned char *)m->p0;
            o.parts = (unsigned char)(2 * m->row_bytes <= slot ? 1 : 2);
            o.n_su = m->rows / 2;
            if ((2 * m->row_bytes / o.parts) % 16) uniform = false;   // every slot-load is a 16-byte aligned, 16-byte multiple bulk copy
            if (P->n_su_kind[kind] && P->n_su_kind[kind] != o.n_su) uniform = false;
            P->n_su_kind[kind] = o.n_su;
        }
    };
    add(OP_EMBED, 0, nullptr, nullptr);
    for (int il = 0; il < d_.n_layer; ++il) {
        Layer &L = layers_[(size_t)il];
        add(OP_QKV, il, &L.qkv, L.attn_norm);
        add(OP_ATTN, il, nullptr, nullptr);
        add(OP_WO, il, &L.wo, nullptr);
        if (tp) add(OP_REDUCE, 0, nullptr, nullptr);   // (`layer` = exchange buffer: 0 after wo, 1 after down)
        add(OP_GATEUP, il, &L.w13, L.ffn_norm);
        add(OP_DOWN, il, &L.w2, nullptr);
        if (tp) add(OP_REDUCE, 1, nullptr, nullptr);
    }
    add(OP_OUTPUT, 0, &output_, final_norm_);
    add(OP_FINAL, 0, nullptr, nullptr);
    if (!uniform) { delete P; return false; }
    P->n_ops = n; P->W = W; P->slot_bytes = slot; P->act_bytes = (int)act_b;
    P->E = E; P->FF = FF; P->n_head = n_head_local_; P->n_ctx = d_.n_ctx; P->n_vocab = d_.n_vocab;
    P->El = n_embd_local_;
    if (tp) { P->tp = tp_->peers; P->tp_seq = tp_->seq_dev; } else { P->tp.world = 1; P->tp.rank = 0; }
    P->flags = getenv("MINIGPT4_B200_MEGA_FLAGS") ? atoi(getenv("MINIGPT4_B200_MEGA_FLAGS")) : 1;
    P->kq_scale = 1.0f / sqrtf((float)d_.n_embd / (float)d_.n_head);
    P->E_pow2 = (E & (E - 1)) == 0; P->inv_E = 1.0 / (double)E;
    P->x = x_; P->q = q_; P->att = att_; P->act = act_; P->logits = logits_; P->kcache = kcache_; P->vcache = vcache_;
    P->rope = rope_; P->tab_exp = tab_exp_; P->tab_silu = tab_silu_;
    P->tok = (const unsigned char *)tok_raw_; P->tok_type = tok_type_; P->tok_row_bytes = gg_row_bytes(tok_type_, (size_t)E);
    P->state = state_; P->barrier = mega_barrier_; P->trace = mega_trace_;
    mega6_params_ = P;
    mega6_nbl_ = (getenv("MINIGPT4_B200_MEGA_NOREG") || mega_type_ == GG_Q5_K) ? 0 : E == 4096 ? 4 : E == 5120 ? 5 : 0;
    mega_smem_ = (size_t)2 * W * slot + act_b + (size_t)2 * W * 8;
    MG4_INFO("decode megakernel (generation 6): %d ops/token, %d stream warps x 2 slots x %d B, act %zu B, %zu B dynamic shared per CTA, register-resident blocks per lane %d, grid %d",
             n, W, slot, act_b, mega_smem_, mega6_nbl_, sm_count_);
    const void *fn = mega_fn();
    CUDA_CHECK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)mega_smem_));
    int occ = 0;
    CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, fn, mk6::kThreads, mega_smem_));
    if (occ < 1) { MG4_ERR("megakernel does not fit on an SM (smem %zu)", mega_smem_); return false; }
    return true;
}

const void *LlamaDevice::mega_fn() const {
    const bool t = mega_trace_ != nullptr, q41 = mega_type_ == GG_Q4_1;
    using namespace mk6;
    if (mega_type_ == GG_Q5_K) return t ? (const void *)decode_megakernel6<GG_Q5_K, 0, true> : (const void *)decode_megakernel6<GG_Q5_K, 0, false>;
#define MG4_M6(NBL) (q41 ? (t ? (const void *)decode_megakernel6<GG_Q4_1, NBL, true> : (const void *)decode_megakernel6<GG_Q4_1, NBL, false>) \
                         : (t ? (const void *)decode_megakernel6<GG_Q4_0, NBL, true> : (const void *)decode_megakernel6<GG_Q4_0, NBL, false>))
    return mega6_nbl_ == 4 ? MG4_M6(4) : mega6_nbl_ == 5 ? MG4_M6(5) : MG4_M6(0);
#undef MG4_M6
}
void LlamaDevice::launch_mega() {
    CUDA_CHECK(cudaMemsetAsync(mega_barrier_, 0, 4, stream_));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)sm_count_); cfg.blockDim = dim3(mk6::kThreads); cfg.dynamicSmemBytes = mega_smem_; cfg.stream = stream_;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative; at[0].val.cooperative = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    void *args[1] = {mega6_params_};
    CUDA_CHECK(cudaLaunchKernelExC(&cfg, mega_fn(), args));
    ++launches_;
    CUDA_CHECK(cudaMemcpyAsync(h_argmax_, &state_->argmax_id, 4, cudaMemcpyDeviceToHost, stream_));
}

void LlamaDevice::build_graph() {
    cudaGraph_t g = nullptr;
    const unsigned long long before = launches_;
    mega_ = build_mega();
    CUDA_CHECK(cudaStreamBeginCapture(stream_, cudaStreamCaptureModeThreadLocal));
    if (mega_) launch_mega();
    else {
        embed_rows_kernel<<<1, 256, 0, stream_>>>(tok_type_, (const unsigned char *)tok_raw_, gg_row_bytes(tok_type_, (size_t)d_.n_embd), d_.n_embd, state_->tokens, nullptr, x_);
        launch_layers(1, 1, true);
    }
    CUDA_CHECK(cudaStreamEndCapture(stream_, &g));
    CUDA_CHECK(cudaGraphInstantiate(&graph_, g, 0));
    CUDA_CHECK(cudaGraphDestroy(g));
    graph_kernels_ = (int)(launches_ - before) + (mega_ ? 0 : 1);
    launches_ = before;
}
bool LlamaDevice::decode_step(int32_t id, int n_past) {
    if (n_past + 1 > d_.n_ctx) { MG4_ERR("context overflow at %d", n_past); return false; }
    if (id >= 0) {
        if (h_state_busy_) CUDA_CHECK(cudaStreamSynchronize(stream_));  // the previous step's copy out of the pinned state may not have run yet
        h_state_->n_past = n_past; h_state_->n_tok = 1; h_state_->tokens[0] = id;
        CUDA_CHECK(cudaMemcpyAsync(state_, h_state_, offsetof(DeviceState, argmax_key), cudaMemcpyHostToDevice, stream_));
        h_state_busy_ = true;
    }
    CUDA_CHECK(cudaGraphLaunch(graph_, stream_));
    launches_ += (unsigned long long)graph_kernels_;
    return true;
}
float LlamaDevice::decode_chain(int steps, int n_past, int32_t *ids_out) {
    if (n_past + steps > d_.n_ctx) { MG4_ERR("context overflow"); return -1.f; }
    // the chain starts from the device state left by the previous eval: tokens[0] = arg-max, n_past up to date
    int32_t *ids_dev = nullptr;
    CUDA_CHECK(cudaMalloc((void **)&ids_dev, (size_t)steps * 4));
    CUDA_CHECK(cudaEventRecord(ev0_, stream_));
    for (int i = 0; i < steps; ++i) {
        CUDA_CHECK(cudaMemcpyAsync(ids_dev + i, &state_->tokens[0], 4, cudaMemcpyDeviceToDevice, stream_));  // the id being fed
        CUDA_CHECK(cudaGraphLaunch(graph_, stream_));
    }
    CUDA_CHECK(cudaEventRecord(ev1_, stream_));
    sync_decode();
    launches_ += (unsigned long long)graph_kernels_ * steps;
    float ms = 0.f; CUDA_CHECK(cudaEventElapsedTime(&ms, ev0_, ev1_));
    if (ids_out) CUDA_CHECK(cudaMemcpy(ids_out, ids_dev, (size_t)steps * 4, cudaMemcpyDeviceToHost));
    cudaFree(ids_dev);
    return ms;
}

// measurement seam: average CUDA-event duration (us) of one all-reduce of a [1, n_embd] partial on the tensor-parallel path in use
// (one-shot peer kernel, or ncclAllReduce + add); every rank must call it with the same reps (even)
bool LlamaDevice::tp_peer_path() const { return tp_ && tp_->world > 1 && tp_->peers_ready(); }
float LlamaDevice::time_allreduce(int reps) {
    if (!tp_ || tp_->world <= 1) return 0.f;
    reps = std::max(2, reps & ~1);
    const int E = d_.n_embd;
    auto one = [&]() {
        if (tp_->peers_ready()) { CUDA_CHECK(cudaMemsetAsync(tp_->partial_out(), 0, (size_t)E * 4, stream_)); tp_->all_reduce_resid(partial_, partial_, (size_t)E, stream_); }
        else { tp_->all_reduce_sum(partial_, (size_t)E, stream_); add_kernel<<<(E + 255) / 256, 256, 0, stream_>>>(partial_, partial_, E); }
    };
    for (int i = 0; i < 4; ++i) one();
    CUDA_CHECK(cudaEventRecord(ev0_, stream_));
    for (int i = 0; i < reps; ++i) one();
    CUDA_CHECK(cudaEventRecord(ev1_, stream_));
    CUDA_CHECK(cudaStreamSynchronize(stream_));
    float ms = 0.f; CUDA_CHECK(cudaEventElapsedTime(&ms, ev0_, ev1_));
    return ms * 1e3f / (float)reps;
}
int LlamaDevice::mega_trace(long long *out, int max_values) {
    if (!mega_trace_) return 0;
    const int n = std::min(max_values, mega_n_ops_ * 32);
    CUDA_CHECK(cudaStreamSynchronize(stream_));
    CUDA_CHECK(cudaMemcpy(out, mega_trace_, (size_t)n * sizeof(long long), cudaMemcpyDeviceToHost));
    return n;
}
float LlamaDevice::time_matvec(int kind, int reps, double *bytes_per_launch) {
    const int E = d_.n_embd, El = n_embd_local_, FFl = n_ff_local_, C = d_.n_ctx;
    void *flush = nullptr; const size_t flush_bytes = 256u << 20;
    if (kind == 4) CUDA_CHECK(cudaMalloc(&flush, flush_bytes));
    h_state_->n_past = 0; h_state_->n_tok = 1; h_state_->tokens[0] = 1;
    CUDA_CHECK(cudaMemcpyAsync(state_, h_state_, offsetof(DeviceState, argmax_key), cudaMemcpyHostToDevice, stream_));
    double total_ms = 0.0, bytes = 0.0; long launches = 0;
    auto one = [&](int il) {
        Layer &L = layers_[(size_t)(kind == 4 ? 0 : il)];
        MatvecArgs a{};
        a.ntok = 1; a.state = state_; a.tab_silu = tab_silu_; a.staged = qact_;
        switch (kind) {
            case 0: a.w = L.fused_qkv ? L.qkv : L.wq; a.x = x_; a.x_stride = E; a.norm_w = L.attn_norm; a.epi = EPI_QKV; a.q_out = q_;
                    a.kcache = kcache_ + (size_t)il * C * El; a.vcache = vcache_ + (size_t)il * C * El; a.rope = rope_; a.e_local = El; a.half_dim = 64; a.part = L.fused_qkv ? -1 : 0; break;
            case 1: a.w = L.wo; a.x = att_; a.x_stride = El; a.epi = EPI_PLAIN; a.out = partial_; a.out_stride = E; break;
            case 2: a.w = L.w13; a.x = x_; a.x_stride = E; a.norm_w = L.ffn_norm; a.epi = EPI_SWIGLU; a.out = act_; a.out_stride = FFl; break;
            case 3: a.w = L.w2; a.x = act_; a.x_stride = FFl; a.epi = EPI_PLAIN; a.out = partial_; a.out_stride = E; break;
            default: a.w = output_; a.x = x_; a.x_stride = E; a.norm_w = final_norm_; a.epi = EPI_LOGITS; a.out = logits_; a.n_valid = d_.n_vocab; break;
        }
        if (kind != 4) a.n_valid = a.w.rows;
        bytes = (double)a.w.bytes;
        launch_matvec(a, 1, sm_count_, stream_, &launches_);
    };
    for (int il = 0; il < d_.n_layer; ++il) one(il);  // warm-up pass (instruction cache, smem attributes)
    CUDA_CHECK(cudaStreamSynchronize(stream_));
    for (int r = 0; r < reps; ++r) {
        if (kind == 4) {
            for (int i = 0; i < 8; ++i) {
                CUDA_CHECK(cudaMemsetAsync(flush, i, flush_bytes, stream_));  // evict the 126 MB L2
                CUDA_CHECK(cudaEventRecord(ev0_, stream_)); one(0); CUDA_CHECK(cudaEventRecord(ev1_, stream_));
                CUDA_CHECK(cudaStreamSynchronize(stream_));
                float ms = 0.f; CUDA_CHECK(cudaEventElapsedTime(&ms, ev0_, ev1_)); total_ms += ms; ++launches;
            }
        } else {
            CUDA_CHECK(cudaEventRecord(ev0_, stream_));
            for (int il = 0; il < d_.n_layer; ++il) one(il);
            CUDA_CHECK(cudaEventRecord(ev1_, stream_));
            CUDA_CHECK(cudaStreamSynchronize(stream_));
            float ms = 0.f; CUDA_CHECK(cudaEventElapsedTime(&ms, ev0_, ev1_)); total_ms += ms; launches += d_.n_layer;
        }
    }
    if (flush) cudaFree(flush);
    CUDA_CHECK(cudaMemsetAsync(&state_->argmax_key, 0, 8, stream_));
    CUDA_CHECK(cudaStreamSynchronize(stream_));
    if (bytes_per_launch) *bytes_per_launch = bytes;
    return (float)(total_ms / (double)launches);
}

// ------------------------------------------------------------------------------------------------
void LlamaDevice::test_matvec(int gg, int rows, int cols, const void *w_host, const float *x_host, int n, float *y_host) {
    if (!type_supported(gg)) MG4_PANIC("test_matvec: unsupported type %d", gg);
    int dev = 0; CUDA_CHECK(cudaGetDevice(&dev));
    cudaDeviceProp prop; CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
    if (!g_max_dyn_smem) g_max_dyn_smem = std::min<size_t>(prop.sharedMemPerBlockOptin, 220 * 1024) - 1024;
    HostTensor t; t.gg = gg; t.n_dims = 2; t.ne[0] = cols; t.ne[1] = rows; t.data = (const uint8_t *)w_host; t.nbytes = (size_t)rows * gg_row_bytes(gg, (size_t)cols);
    QMat m; Stager st;
    qmat_alloc(m, gg, rows, cols);
    repack_into(m, t, st, 0, rows, 0, cols, 1, 0, 0);
    float *x, *y; DeviceState *stt; unsigned char *stg;
    CUDA_CHECK(cudaMalloc((void **)&stg, (size_t)8 * ((size_t)cols * 2 + 4096)));
    CUDA_CHECK(cudaMalloc((void **)&x, (size_t)n * cols * 4)); CUDA_CHECK(cudaMalloc((void **)&y, (size_t)n * m.rows * 4));
    CUDA_CHECK(cudaMalloc((void **)&stt, sizeof(DeviceState))); CUDA_CHECK(cudaMemset(stt, 0, sizeof(DeviceState)));
    CUDA_CHECK(cudaMemcpy(x, x_host, (size_t)n * cols * 4, cudaMemcpyHostToDevice));
    for (int i = 0; i < n; i += 8) {
        const int c = std::min(8, n - i);
        MatvecArgs a{};
        a.w = m; a.x = x + (size_t)i * cols; a.x_stride = cols; a.ntok = c; a.epi = EPI_PLAIN; a.out = y + (size_t)i * m.rows; a.out_stride = m.rows; a.n_valid = rows; a.state = stt; a.staged = stg;
        launch_matvec(a, nt_for(c), prop.multiProcessorCount, 0, nullptr);
    }
    CUDA_CHECK(cudaDeviceSynchronize());
    std::vector<float> tmp((size_t)n * m.rows);
    CUDA_CHECK(cudaMemcpy(tmp.data(), y, tmp.size() * 4, cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i) memcpy(y_host + (size_t)i * rows, tmp.data() + (size_t)i * m.rows, (size_t)rows * 4);
    cudaFree(x); cudaFree(y); cudaFree(stt); cudaFree(stg); qmat_free(m);
}

}  // namespace mg4
