// engine.cpp — see engine.h.
#include "engine.h"
#include "../../include/minigpt4.h"
#include <string.h>
#include <algorithm>
#include <exception>

namespace mg4 {

TPConfig g_tp_config;

Engine::~Engine() {
    llm_.reset();
    vis_lanes_.clear();   // (lanes borrow the first lane's weights)
    vis_.reset();
    tp.destroy();
}

Error Engine::init(const std::string &path, const std::string &llm_path, int verbosity, int seed, int n_ctx, int n_batch, bool /*numa: CPU-only notion*/) {
    g_verbosity = verbosity;
    n_batch_ = n_batch > 0 ? n_batch : 512;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        // No CPU fallback exists: the hot path is CUDA only.  Reported at every verbosity - a caller must never mistake this for a slow success.
        cudaGetLastError();
        fprintf(stderr, "[minigpt4-b200][error] no CUDA device available; this engine has no CPU path\n");
        return ErrLoadLanguageModel;
    }
    Error where = ErrLoadLanguageModel;
    try {
        LoadScope loading;   // failed checks below throw LoadFailure instead of aborting the host process (common.h)
        if (g_tp_config.set && g_tp_config.world > 1) tp.init(g_tp_config.rank, g_tp_config.world, g_tp_config.id);
        {
            const double t0 = now_ms();
            LlamaFile lf;
            if (!lf.load(llm_path)) { MG4_ERR("failed to read language model %s", llm_path.c_str()); return ErrLoadLanguageModel; }
            tok_.init(lf.vocab);
            llm_.reset(new LlamaDevice());
            if (!llm_->load(lf, n_ctx > 0 ? n_ctx : 2048, tp.world > 1 ? &tp : nullptr)) return ErrLoadLanguageModel;
            MG4_INFO("Load language model took %.0f ms", now_ms() - t0);
        }
        if (!path.empty()) {
            where = ErrLoadModelFileHeader;
            const double t0 = now_ms();
            vfile_.reset(new VisionFile());   // (kept mapped: further encode lanes are built from it on demand)
            VisionFile &vf = *vfile_;
            if (Error e = vf.load(path)) return e;
            vis_.reset(new VisionDevice());
            if (Error e = vis_->load(vf)) return e;
            if (vis_->dims().n_embd_llm != llm_->dims().n_embd)
                MG4_ERR("warning: llama_proj width %d != language model n_embd %d", vis_->dims().n_embd_llm, llm_->dims().n_embd);
            MG4_INFO("Load model from file took %.0f ms", now_ms() - t0);
        }
    } catch (const LoadFailure &f) {
        fprintf(stderr, "[minigpt4-b200][error] %s\n", f.msg);
        return where;
    } catch (const std::exception &e) {   // (host memory exhausted while reading a file, ...)
        fprintf(stderr, "[minigpt4-b200][error] %s\n", e.what());
        return where;
    }
    sampler_.reset(new Sampler(seed));
    logits_.resize((size_t)llm_->dims().n_vocab);
    return ErrNone;
}

// input validation = reference minigpt4.cpp:2130-2138
Error Engine::encode_image(const ::MiniGPT4Image *image, ::MiniGPT4Embedding *out) {
    if (!vis_) MG4_PANIC("encode_image on a context loaded without a vision model");
    if ((long)image->width * image->height * image->channels != 224L * 224 * 3) return ErrImageNot224_244_3;
    if (image->format != MINIGPT4_IMAGE_FORMAT_F32) return ErrImageNotF32;
    const size_t n = (size_t)32 * vis_->dims().n_embd_llm;
    out->elements = n;
    out->data = new float[n];
    last_encode_ms = vis_->encode((const float *)image->data, out->data);
    MG4_INFO("Encoding image took %.3f ms on device", last_encode_ms);
    return ErrNone;
}

// Batched encode (extension; the reference encodes one image per call, minigpt4.cpp:2094): up to kEncodeLanes images are in flight at once, each on
// its own lane = its own activations, CUDA graph and stream over the SHARED weights.  One image's graph leaves most SMs idle most of the time
// (its GEMMs are 44-144 CTAs, its attention 144, the Q-Former a handful), so concurrent graphs interleave on the machine; every image goes
// through exactly the single-image graph, so each embedding is bit-identical to minigpt4_encode_image's.
Error Engine::encode_images(const ::MiniGPT4Image *images, size_t n, ::MiniGPT4Embedding *out, float *total_ms) {
    if (!vis_) MG4_PANIC("encode_images on a context loaded without a vision model");
    for (size_t i = 0; i < n; ++i) {
        if ((long)images[i].width * images[i].height * images[i].channels != 224L * 224 * 3) return ErrImageNot224_244_3;
        if (images[i].format != MINIGPT4_IMAGE_FORMAT_F32) return ErrImageNotF32;
    }
    const size_t lanes = std::min<size_t>(n, (size_t)kEncodeLanes);
    while (vis_lanes_.size() + 1 < lanes) {
        std::unique_ptr<VisionDevice> l(new VisionDevice());
        try {
            LoadScope loading;   // (a lane that does not fit in device memory is an error code, not an abort)
            if (Error e = l->load(*vfile_, vis_.get())) return e;
        } catch (const LoadFailure &f) {
            fprintf(stderr, "[minigpt4-b200][error] encode lane %zu: %s\n", vis_lanes_.size() + 1, f.msg);
            return ErrLoadModelFileHeader;
        }
        vis_lanes_.push_back(std::move(l));
    }
    auto lane = [&](size_t k) { return k == 0 ? vis_.get() : vis_lanes_[k - 1].get(); };
    const size_t ne = (size_t)32 * vis_->dims().n_embd_llm;
    const double t0 = now_ms();
    for (size_t base = 0; base < n; base += lanes) {
        const size_t c = std::min(lanes, n - base);
        for (size_t k = 0; k < c; ++k) lane(k)->encode_begin((const float *)images[base + k].data);
        for (size_t k = 0; k < c; ++k) {
            out[base + k].elements = ne; out[base + k].data = new float[ne];
            last_encode_ms = lane(k)->encode_end(out[base + k].data);
        }
    }
    if (total_ms) *total_ms = (float)(now_ms() - t0);
    return ErrNone;
}

// add_tokens (minigpt4.cpp:2365-2382) / add_embedding (:2399-2415).  The reference evaluates every piece of a chat turn separately
// (system prompt, "Human: <Img>", the 32 image rows, "</Img> ", the question, "### Assistant:" = six passes over the weights).  Results are
// batch invariant (every row is quantised and reduced on its own), so the pieces are only QUEUED here and evaluated together - one pass over
// the weights per LlamaDevice::kPrefillMax rows - when something needs the model state (sampling, logits, a decode step, the hidden state).
// Validation happens at queue time, so the error codes of the reference's call sites are unchanged.  A single token on an empty queue is
// the decode loop: it goes straight through the captured decode graph.
Error Engine::add_tokens(const std::vector<int32_t> &tokens) {
    if (tokens.empty()) return ErrNone;
    const int n = (int)tokens.size(), n_vocab = llm_->dims().n_vocab;
    bool ok = n_past_ + n <= llm_->dims().n_ctx;
    if (!ok) MG4_ERR("context overflow: %d + %d > n_ctx %d", n_past_, n, llm_->dims().n_ctx);
    for (int i = 0; ok && i < n; ++i) if (tokens[(size_t)i] < 0 || tokens[(size_t)i] >= n_vocab) { MG4_ERR("token id %d out of range", tokens[(size_t)i]); ok = false; }
    if (ok) {
        if (n == 1 && pend_ids_.empty()) ok = llm_->decode_step(tokens[0], n_past_);   // asynchronous: the next sample / flush synchronises
        else {
            for (int i = 0; ok && i < n; i += kMaxPending) {   // a queue never exceeds kMaxPending rows
                const int c = std::min(kMaxPending, n - i);
                if ((int)pend_ids_.size() + c > kMaxPending) ok = flush();
                if (pend_ids_.empty()) pend_base_ = n_past_ + i;
                pend_ids_.insert(pend_ids_.end(), tokens.begin() + i, tokens.begin() + i + c);
            }
        }
    }
    if (!ok) { MG4_ERR("Failed to add string"); return ErrFailedToAddString; }
    n_past_ += n;
    return ErrNone;
}
// add_strings (minigpt4.cpp:2384-2397): add_bos is ALWAYS true
Error Engine::add_strings(const char *s) { return add_tokens(tok_.encode(s ? s : "", true)); }

Error Engine::add_embedding(const float *rows, int n_rows) {
    if (n_rows <= 0) return ErrNone;
    const size_t E = (size_t)llm_->dims().n_embd;
    bool ok = n_rows <= kMaxPending && n_past_ + n_rows <= llm_->dims().n_ctx;
    if (ok && (int)pend_ids_.size() + n_rows > kMaxPending) ok = flush();
    if (ok) {
        if (pend_ids_.empty()) pend_base_ = n_past_;
        const int k0 = (int)(pend_emb_.size() / E);
        for (int i = 0; i < n_rows; ++i) pend_ids_.push_back(-1 - (k0 + i));
        pend_emb_.insert(pend_emb_.end(), rows, rows + (size_t)n_rows * E);
    }
    if (!ok) { MG4_ERR("Failed to add embedding"); return ErrFailedToAddEmbedding; }
    n_past_ += n_rows;
    return ErrNone;
}
// evaluate the queued rows (no-op when the queue is empty)
bool Engine::flush() {
    if (pend_ids_.empty()) return true;
    const bool ok = llm_->eval_rows(pend_ids_.data(), (int)pend_ids_.size(), pend_emb_.data(), (int)(pend_emb_.size() / (size_t)llm_->dims().n_embd), pend_base_);
    pend_ids_.clear(); pend_emb_.clear();
    if (!ok) MG4_ERR("deferred evaluation of the queued prompt rows failed");
    return ok;
}

int32_t Engine::sample_token(const SamplingParams &p) {
    flush();
    if (p.temp <= 0) return llm_->argmax();  // greedy: arg-max was computed on device with the logits
    llm_->logits_to_host(logits_.data());
    return sampler_->sample(logits_.data(), (int)logits_.size(), p);
}
const char *Engine::id_to_token(int32_t id) const {  // minigpt4.cpp:2485-2497
    if (id == 2) return "</s>";
    return tok_.piece(id);
}

}  // namespace mg4
