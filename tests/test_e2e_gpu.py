"""End-to-end parity (GPU) on seeded tiny models: vision graph, LLaMA step, chat flow through the reference ABI.
Bars (north_star): logits within 1e-2 relative of the CPU path; greedy ids bit-identical for 32 tokens."""
import ctypes

import numpy as np
import pytest

from conftest import rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx(lib, tiny):
    c = lib.minigpt4_model_load(tiny["vision"], tiny["q4_1"].replace("tiny-q4_1", "tiny-q4_1"), 1, 1337, 512, 8, 0)
    assert c.ptr
    yield c
    lib.minigpt4_free(c)


@pytest.fixture(scope="module")
def big_llm(tmp_path_factory, mg):
    """LLaMA with n_embd 4096 (so the 4096-wide projected embedding can be fed), 2 layers."""
    p = str(tmp_path_factory.mktemp("m4096") / "llama-4096.bin")
    mg.write_llama_ggjt(p, mg.LlamaSpec(n_vocab=2048, n_embd=4096, n_head=32, n_layer=2, wtype="q4_1"))
    return p


def test_encode_image_matches_oracle(lib, ext, orc, mg, tiny, big_llm):
    c = lib.minigpt4_model_load(tiny["vision"], big_llm, 1, 1, 256, 8, 0)
    img = mg.synth_image()
    got = ext.encode_array(c, img)
    e = orc.OracleEngine(tiny["vision"], None)
    want = e.encode_image(img)
    assert got.shape == want.shape == (32, 4096)
    assert rel_err(got, want) < 1e-2, rel_err(got, want)
    # validation errors (reference minigpt4.cpp:2130-2138)
    import minigpt4_cpp_b200 as m
    bad = m.MiniGPT4Image(img.ctypes.data_as(ctypes.c_void_p), 224, 224, 4, m.ImageFormat.F32)
    with pytest.raises(RuntimeError, match="ImageNot224_244_3"):
        lib.minigpt4_encode_image(c, bad)
    bad = m.MiniGPT4Image(img.ctypes.data_as(ctypes.c_void_p), 224, 224, 3, m.ImageFormat.U8)
    with pytest.raises(RuntimeError, match="ImageNotF32"):
        lib.minigpt4_encode_image(c, bad)
    lib.minigpt4_free(c)


@pytest.mark.parametrize("wt", ["q4_1", "q4_0", "q5_k", "q6_k", "f16", "mixed"])
def test_llama_eval_matches_oracle(ext, orc, tiny, wt):
    c = ext.llm_load(tiny[wt], n_ctx=256)
    e = orc.OracleEngine(None, tiny[wt], n_ctx=256)
    rng = np.random.default_rng(11)
    ids = rng.integers(3, e.n_vocab, size=21).tolist()
    ext.eval_tokens(c, ids)
    want = e.eval_tokens(ids).copy()
    got = ext.logits(c)
    assert rel_err(got, want) < 1e-2 and int(np.argmax(got)) == int(np.argmax(want))  # the north_star bar
    assert np.array_equal(got, want), rel_err(got, want)  # canonical reduction order on both sides -> bit-identical logits
    # embedding rows (llama_eval_embd) continue the same context
    rows = rng.standard_normal((5, e.n_embd)).astype(np.float32)
    ext.eval_embd(c, rows)
    want = e.eval_embd(rows).copy()
    assert np.array_equal(ext.logits(c), want)
    assert ext.n_past(c) == e.n_past == 26
    # greedy continuation: 32 ids bit-identical
    a, b = [], []
    for _ in range(32):
        tid = ext.greedy_id(c); a.append(tid); ext.eval_tokens(c, [tid])
        b.append(e.end_chat_greedy()[0])
    assert a == b
    ext.base.minigpt4_free(c)


def test_batch_invariance_and_chain(ext, tiny):
    """size-independent properties: chunked prefill == token-by-token; device-chained greedy == host-driven greedy."""
    ids = list(range(5, 30))
    c1 = ext.llm_load(tiny["q4_1"], n_ctx=256); ext.eval_tokens(c1, ids); l1 = ext.logits(c1)
    c2 = ext.llm_load(tiny["q4_1"], n_ctx=256)
    for t in ids:
        ext.eval_tokens(c2, [t])
    l2 = ext.logits(c2)
    assert np.array_equal(l1, l2)
    chain, ms = ext.decode_chain(c1, 16)
    host = []
    for _ in range(16):
        tid = ext.greedy_id(c2); host.append(tid); ext.eval_tokens(c2, [tid])
    assert chain.tolist() == host and ms > 0
    assert ext.n_past(c1) == ext.n_past(c2)
    assert np.array_equal(ext.logits(c1), ext.logits(c2))
    ext.base.minigpt4_free(c1); ext.base.minigpt4_free(c2)


def test_megakernel_equals_per_op_path(ext, orc, tiny, monkeypatch):
    """The persistent one-launch-per-token megakernel (homogeneous Q4_0 / Q4_1 / Q5_K) and the per-op graph are the same function."""
    for wt in ("q4_1", "q4_0", "q5_k"):
        ids = list(range(7, 19))
        monkeypatch.setenv("MINIGPT4_B200_NO_MEGAKERNEL", "1")
        c1 = ext.llm_load(tiny[wt], n_ctx=128)
        monkeypatch.delenv("MINIGPT4_B200_NO_MEGAKERNEL")
        c2 = ext.llm_load(tiny[wt], n_ctx=128)
        assert ext.stats(c1).decode_megakernel == 0 and ext.stats(c2).decode_megakernel >= 6
        e = orc.OracleEngine(None, tiny[wt], n_ctx=128)
        ext.eval_tokens(c1, ids); ext.eval_tokens(c2, ids); e.eval_tokens(ids)
        for _ in range(24):  # single-token steps go through the decode graph: per-op kernels (c1) vs megakernel (c2)
            t1, t2 = ext.greedy_id(c1), ext.greedy_id(c2)
            assert t1 == t2 == int(np.argmax(e.logits))
            ext.eval_tokens(c1, [t1]); ext.eval_tokens(c2, [t2]); e.eval_tokens([t1])
            assert np.array_equal(ext.logits(c1), ext.logits(c2)) and np.array_equal(ext.logits(c2), e.logits)
        ch, _ = ext.decode_chain(c2, 8)
        host = []
        for _ in range(8):
            t = ext.greedy_id(c1); host.append(t); ext.eval_tokens(c1, [t])
        assert ch.tolist() == host
        ext.base.minigpt4_free(c1); ext.base.minigpt4_free(c2)


def test_vision_gemm_grid_variants(lib, ext, mg, tiny, big_llm, monkeypatch):
    """The encode runs its 257-token GEMMs token-split over grid.y (each output element keeps its K order: bit-identical to one CTA per weight
    slab) and proj / fc2 as three split-K slices folded into the residual stream by the following LayerNorm in slice order (a different float
    association: equal to a few ulps, deterministic).  MINIGPT4_B200_VISION_TSPLIT=0 / _SPLITK=1 select the plain grids."""
    img = mg.synth_image(5)
    c_def = lib.minigpt4_model_load(tiny["vision"], big_llm, 1, 1, 64, 8, 0)
    monkeypatch.setenv("MINIGPT4_B200_VISION_SPLITK", "1")
    c_ts = lib.minigpt4_model_load(tiny["vision"], big_llm, 1, 1, 64, 8, 0)        # token split only
    monkeypatch.setenv("MINIGPT4_B200_VISION_TSPLIT", "0")
    c_plain = lib.minigpt4_model_load(tiny["vision"], big_llm, 1, 1, 64, 8, 0)     # one CTA per 128-feature slab
    monkeypatch.delenv("MINIGPT4_B200_VISION_TSPLIT"); monkeypatch.delenv("MINIGPT4_B200_VISION_SPLITK")
    a, b, c = ext.encode_array(c_plain, img), ext.encode_array(c_ts, img), ext.encode_array(c_def, img)
    assert np.array_equal(a, b), float(np.abs(a - b).max())
    assert rel_err(c, a) < 2e-3, rel_err(c, a)   # (F32 sums differ in the last bits; a few LayerNorm outputs then round to the other F16 neighbour)
    assert np.array_equal(c, ext.encode_array(c_def, img))   # no atomics: the same bits every time
    for x in (c_def, c_ts, c_plain): lib.minigpt4_free(x)


def test_batched_encode_equals_single_encodes(lib, ext, mg, tiny, big_llm):
    """minigpt4_b200_encode_images runs the images concurrently on lanes (own activations / graph / stream, shared weights): every embedding must be
    the bits minigpt4_encode_image produces for that image, for batches smaller than, equal to and larger than the lane count."""
    c = lib.minigpt4_model_load(tiny["vision"], big_llm, 1, 1, 64, 8, 0)
    imgs = [mg.synth_image(s) for s in range(11)]
    single = [ext.encode_array(c, im) for im in imgs]
    for n in (1, 3, 8, 11):
        got, _ = ext.encode_batch(c, imgs[:n])
        assert len(got) == n
        for a, b in zip(got, single): assert np.array_equal(a, b)
    assert np.array_equal(ext.encode_array(c, imgs[2]), single[2])   # lane 0 still serves minigpt4_encode_image
    lib.minigpt4_free(c)


def check_queued_pieces(ext, llm):
    """The pieces of one chat turn queued (one pass over the weights at the end) versus flushed one by one: same logits, same greedy ids."""
    c1, c2 = ext.llm_load(llm, n_ctx=512), ext.llm_load(llm, n_ctx=512)
    rng = np.random.default_rng(3)
    rows = rng.standard_normal((32, ext.L.minigpt4_b200_n_embd(c1.ptr))).astype(np.float32)
    pieces = [("t", list(range(5, 25))), ("t", [7, 9, 11]), ("e", rows), ("t", [4]), ("t", list(range(30, 47))), ("t", [3, 3, 8])]
    for kind, p in pieces:
        (ext.eval_tokens if kind == "t" else ext.eval_embd)(c1, p)                      # queued: one pass over the weights at the end
        (ext.eval_tokens if kind == "t" else ext.eval_embd)(c2, p); ext.flush(c2)      # forced: one pass per piece
    assert ext.n_past(c1) == ext.n_past(c2) == sum(len(p) for _, p in pieces)
    assert np.array_equal(ext.logits(c1), ext.logits(c2))
    a, b = [], []
    for _ in range(6):
        t1, t2 = ext.greedy_id(c1), ext.greedy_id(c2); a.append(t1); b.append(t2)
        ext.eval_tokens(c1, [t1]); ext.eval_tokens(c2, [t2])
    assert a == b
    with pytest.raises(RuntimeError, match="FailedToAddString"):   # validated when queued, not when flushed
        ext.eval_tokens(c1, [10 ** 9])
    ext.base.minigpt4_free(c1); ext.base.minigpt4_free(c2)


def test_queued_prompt_pieces_equal_piecewise_evaluation(ext, tiny):
    """The engine queues consecutive add_tokens / add_embedding calls and evaluates them in one pass (the reference evaluates each piece on its own,
    minigpt4.cpp:2365-2415).  Rows are batch invariant, so the logits must not change by a single bit; errors are still raised at queue time."""
    for wt in ("q4_1", "q5_k"):
        check_queued_pieces(ext, tiny[wt])


def test_context_overflow_is_an_error(ext, tiny):
    c = ext.llm_load(tiny["q4_1"], n_ctx=16)
    with pytest.raises(RuntimeError, match="FailedToAddString"):
        ext.eval_tokens(c, list(range(3, 3 + 17)))
    ext.base.minigpt4_free(c)


def test_damaged_model_is_an_error_not_an_abort(ext, tiny, tmp_path):
    """A load-time failure (here: a tensor the graph needs is missing) returns NULL like the reference; the process and the device stay usable."""
    raw = open(tiny["q4_1"], "rb").read()
    name = b"layers.1.ffn_norm.weight"
    assert raw.count(name) == 1
    bad = tmp_path / "missing-tensor.bin"
    bad.write_bytes(raw.replace(name, b"layers.1.ffn_norx.weight"))
    assert ext.L.minigpt4_b200_llm_load(str(bad).encode(), 64, 1, 0) is None
    c = ext.llm_load(tiny["q4_1"], n_ctx=64)
    ext.eval_tokens(c, [3, 4, 5])
    assert np.isfinite(ext.logits(c)).all()
    ext.base.minigpt4_free(c)


def test_image_file_to_embedding_through_the_abi(lib, ext, tiny, big_llm, tmp_path):
    """examples/main.cpp's flow (reference :207-240): minigpt4_image_load_from_file -> minigpt4_preprocess_image -> minigpt4_encode_image on a PNG of
    arbitrary size == encoding the Pillow-resized, CLIP-normalised tensor directly."""
    from PIL import Image
    rng = np.random.default_rng(11)
    yy, xx = np.mgrid[0:300, 0:420]
    rgb = ((np.stack([xx * 2 + yy, xx + yy * 3, 255 - xx], -1) % 256) + rng.integers(-20, 20, (300, 420, 3))).clip(0, 255).astype(np.uint8)
    path = tmp_path / "photo.png"
    Image.fromarray(rgb).save(path)
    c = lib.minigpt4_model_load(tiny["vision"], big_llm, 1, 1337, 256, 8, 0)
    img = lib.minigpt4_image_load_from_file(c, str(path), 0)
    pre = lib.minigpt4_preprocess_image(c, img, 0)
    emb = lib.minigpt4_encode_image(c, pre, 0)
    got = np.ctypeslib.as_array(emb.data, shape=(32 * 4096,)).copy()
    small = np.asarray(Image.fromarray(rgb).resize((224, 224), Image.BICUBIC))
    f = small.astype(np.float32) * np.float32(1.0 / 255.0)
    d = (f.astype(np.float64) - np.array([0.48145466, 0.4578275, 0.40821073])).astype(np.float32)
    chw = np.ascontiguousarray((d.astype(np.float64) / np.array([0.26862954, 0.26130258, 0.27577711])).astype(np.float32).transpose(2, 0, 1))
    want = ext.encode_array(c, chw).reshape(-1)
    assert np.array_equal(got, want)
    lib.minigpt4_free_embedding(emb)
    lib.minigpt4_free_image(img); lib.minigpt4_free_image(pre)
    lib.minigpt4_free(c)


def test_chat_flow_through_reference_abi(lib, ext, orc, mg, tiny, big_llm):
    """system prompt -> begin_chat_image -> 32 x end_chat_image (greedy) == oracle engine, token for token."""
    c = lib.minigpt4_model_load(tiny["vision"], big_llm, 1, 1337, 512, 8, 0)
    e = orc.OracleEngine(tiny["vision"], big_llm, n_ctx=512)
    img = mg.synth_image(7)
    import minigpt4_cpp_b200 as m
    mi = m.MiniGPT4Image(img.ctypes.data_as(ctypes.c_void_p), 224, 224, 3, m.ImageFormat.F32)
    emb = lib.minigpt4_encode_image(c, mi)
    assert emb.n_embeddings == 32 * 4096
    lib.minigpt4_system_prompt(c)
    lib.minigpt4_begin_chat_image(c, emb, "what is this?")
    # the oracle consumes the embedding the GPU produced, so this isolates the language path + chat flow
    gemb = np.ctypeslib.as_array(emb.data, shape=(32 * 4096,)).copy().reshape(32, 4096)
    e.system_prompt(); e.begin_chat_image(gemb, "what is this?")
    assert ext.n_past(c) == e.n_past
    assert np.array_equal(ext.logits(c), e.logits)
    got = [lib.minigpt4_end_chat_image(c, temp=0.0) for _ in range(32)]
    want = [e.end_chat_greedy()[1].decode("utf-8", errors="ignore") for _ in range(32)]
    assert got == want
    # text-only turn + reset
    lib.minigpt4_begin_chat(c, "and the color?"); e.begin_chat("and the color?")
    assert lib.minigpt4_end_chat(c, temp=0.0) == e.end_chat_greedy()[1].decode("utf-8", errors="ignore")
    lib.minigpt4_reset_chat(c)
    assert ext.n_past(c) == 0
    # wrong embedding size (reference minigpt4.cpp:2682-2686)
    bad = m.MiniGPT4Embedding(emb.data, 100)
    with pytest.raises(RuntimeError, match="LLamaProjectionEmbeddingInvalidSize"):
        lib.minigpt4_begin_chat_image(c, bad, "x")
    lib.minigpt4_free_embedding(emb)
    assert not emb.data
    # sampling path (temp > 0) returns valid tokens
    lib.minigpt4_reset_chat(c); lib.minigpt4_begin_chat(c, "hi")
    toks = [lib.minigpt4_end_chat(c, temp=0.8, top_k=40, top_p=0.9) for _ in range(4)]
    assert all(isinstance(t, str) for t in toks)
    st = ext.stats(c)
    assert st.kernel_launches > 0 and st.n_layer == 2 and st.tp_world == 1
    lib.minigpt4_free(c)
