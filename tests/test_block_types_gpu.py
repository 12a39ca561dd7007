"""Device paths of the remaining ggjt block types - Q4_K (dot2_q4k) and Q5_0 / Q5_1 / Q8_0 (dot2_b32), their repack and token-embedding kernels:
bit-identical to the CPU oracle (first run on hardware in round 2: 68 cases green, profiles/r2_call_block_types.txt)."""
import os

import numpy as np
import pytest

from test_e2e_gpu import check_queued_pieces

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("shape", [(64, 512), (130, 4096), (48, 11008 - 11008 % 256), (33, 256)])
@pytest.mark.parametrize("n", [1, 3, 8, 11])
def test_q4_k_matvec_is_bit_identical(ext, orc, mg, shape, n):
    """Q4_K device path (dot2_q4k, repack_q4k): the Q5_K kernel minus the fifth bits."""
    rows, cols = shape
    rng = np.random.default_rng(rows * 7 + cols + n)
    raw = mg.synth_quant(rng, 12, rows, cols, 0.02)
    x = rng.standard_normal((n, cols)).astype(np.float32)
    x[0, :256] = 0.0
    assert np.array_equal(ext.op_matvec(12, raw, rows, cols, x), orc.mul_mat(12, raw, rows, cols, x))


def test_q4_k_llama_file_matches_oracle(ext, orc, mg, tmp_path):
    llm = str(tmp_path / "llama-q4_k.bin")
    mg.write_llama_ggjt(llm, mg.LlamaSpec(n_vocab=1024, n_embd=512, n_head=4, n_layer=2, wtype="q4_k", output_type="q6_k"))
    c = ext.llm_load(llm, n_ctx=256)
    e = orc.OracleEngine(None, llm, n_ctx=256)
    ids = np.random.default_rng(11).integers(3, 1024, size=21).tolist()
    ext.eval_tokens(c, ids)
    assert np.array_equal(ext.logits(c), e.eval_tokens(ids))
    a, b = [], []
    for _ in range(32):
        t = ext.greedy_id(c); a.append(t); ext.eval_tokens(c, [t]); b.append(e.end_chat_greedy()[0])
    assert a == b
    ext.base.minigpt4_free(c)


@pytest.mark.parametrize("name,gt", [("q5_0", 6), ("q5_1", 7), ("q8_0", 8)])
@pytest.mark.parametrize("shape", [(64, 512), (130, 4096), (48, 11008), (34, 32)])
@pytest.mark.parametrize("n", [1, 3, 8, 11])
def test_b32_family_matvec_is_bit_identical(ext, orc, mg, name, gt, shape, n):
    """Q5_0 / Q5_1 / Q8_0 device path (dot2_b32, repack_b32) against the oracle's canonical order
    (the fifth-bit reconstruction was checked by a CPU emulation of the dp4a arithmetic)."""
    rows, cols = shape
    rng = np.random.default_rng(rows * 7 + cols + n + gt)
    raw = mg.synth_quant(rng, gt, rows, cols, 0.02)
    x = rng.standard_normal((n, cols)).astype(np.float32)
    x[0, :32] = 0.0
    assert np.array_equal(ext.op_matvec(gt, raw, rows, cols, x), orc.mul_mat(gt, raw, rows, cols, x))


@pytest.mark.parametrize("name", ["q5_0", "q5_1", "q8_0"])
def test_b32_family_llama_file_matches_oracle(ext, orc, mg, tmp_path, name):
    llm = str(tmp_path / f"llama-{name}.bin")
    mg.write_llama_ggjt(llm, mg.LlamaSpec(n_vocab=1024, n_embd=512, n_head=4, n_layer=2, wtype=name))
    c = ext.llm_load(llm, n_ctx=256)
    e = orc.OracleEngine(None, llm, n_ctx=256)
    ids = np.random.default_rng(11).integers(3, 1024, size=21).tolist()
    ext.eval_tokens(c, ids)
    assert np.array_equal(ext.logits(c), e.eval_tokens(ids))
    a, b = [], []
    for _ in range(32):
        t = ext.greedy_id(c); a.append(t); ext.eval_tokens(c, [t]); b.append(e.end_chat_greedy()[0])
    assert a == b
    ext.base.minigpt4_free(c)


@pytest.mark.parametrize("name", ["q4_k", "q5_0", "q5_1", "q8_0"])
def test_prompt_rows_of_every_block_type_match_oracle(ext, orc, mg, tmp_path, name):
    """Token and embedding rows of these files take the queued prompt path of every other type: tokens then embedding rows against the
    oracle, and the pieces of a chat turn queued against one pass per piece."""
    llm = str(tmp_path / f"llama-{name}.bin")
    mg.write_llama_ggjt(llm, mg.LlamaSpec(n_vocab=1024, n_embd=512, n_head=4, n_layer=2, wtype=name, output_type="q6_k" if name == "q4_k" else None))
    c = ext.llm_load(llm, n_ctx=256)
    e = orc.OracleEngine(None, llm, n_ctx=256)
    rng = np.random.default_rng(11)
    ids = rng.integers(3, 1024, size=21).tolist()
    ext.eval_tokens(c, ids)
    assert np.array_equal(ext.logits(c), e.eval_tokens(ids))
    rows = rng.standard_normal((5, 512)).astype(np.float32)
    ext.eval_embd(c, rows)
    assert np.array_equal(ext.logits(c), e.eval_embd(rows))
    assert ext.n_past(c) == e.n_past == 26
    ext.base.minigpt4_free(c)
    check_queued_pieces(ext, llm)


@pytest.mark.parametrize("tok", ["q4_k", "q5_0", "q5_1", "q8_0"])
def test_q4_1_layers_with_foreign_token_embeddings(ext, orc, mg, tmp_path, tok):
    """Q4_1 layers whose tok_embeddings the decode megakernel cannot gather: tensor-core prefill, then the per-op decode graph."""
    llm = str(tmp_path / f"llama-q4_1-tok-{tok}.bin")
    mg.write_llama_ggjt(llm, mg.LlamaSpec(n_vocab=1024, n_embd=512, n_head=4, n_layer=2, wtype="q4_1", tok_type=tok))
    c = ext.llm_load(llm, n_ctx=256)
    st = ext.stats(c)
    assert st.decode_megakernel == 0 and st.prefill_gemm == 1
    e = orc.OracleEngine(None, llm, n_ctx=256)
    ids = np.random.default_rng(11).integers(3, 1024, size=21).tolist()
    ext.eval_tokens(c, ids)
    assert np.array_equal(ext.logits(c), e.eval_tokens(ids))
    a, b = [], []
    for _ in range(32):
        t = ext.greedy_id(c); a.append(t); ext.eval_tokens(c, [t]); b.append(e.end_chat_greedy()[0])
    assert a == b
    ext.base.minigpt4_free(c)
