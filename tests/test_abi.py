"""C-ABI surface: the library loads and exports every symbol include/*.h declares; GPU-free entry points behave like
the reference (error strings minigpt4.cpp:97-119, EOS helpers :2764-2782, image entry points :2576-2651)."""
import ctypes
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
ERRORS = ["None", "LoadModelFileHeader", "LoadModelFileVersion", "LoadModelMiniGPT4DataType", "LoadLanguageModel", "OpenImage", "ImageSize",
          "MmapSupport", "FailedToAddString", "LLamaProjectionEmbeddingInvalidSize", "FailedToAddEmbedding", "EosToken", "Eos", "ImageNot224_244_3",
          "ImageNotF32", "ImageChannelsExpectedRGB", "ImageFormatExpectedU8", "PathDoesNotExist", "DumpModelFileOpen", "OpenCVNotLinked"]


def declared_symbols():
    names = []
    for h in (ROOT / "include").glob("*.h"):
        names += re.findall(r"MINIGPT4_API[^;]*?\b(minigpt4_\w+)\s*\(", h.read_text())
    return sorted(set(names))


def test_header_declares_the_18_reference_symbols():
    import minigpt4_cpp_b200.minigpt4_library as ml
    base = [s for s in declared_symbols() if not s.startswith("minigpt4_b200_")]
    assert sorted(base) == sorted(ml.ABI_SYMBOLS) and len(base) == 18


def test_library_exports_every_declared_symbol(lib):
    for name in declared_symbols():
        assert hasattr(lib.library, name), name


def test_extension_table_matches_header():
    import minigpt4_cpp_b200.minigpt4_library as ml
    ext = [s for s in declared_symbols() if s.startswith("minigpt4_b200_")]
    assert sorted(ext) == sorted(ml.EXT_SYMBOLS)


def test_error_strings(lib):
    for code, name in enumerate(ERRORS):
        assert lib.minigpt4_error_code_to_string(code) == name


def test_eos_helpers(lib):
    assert lib.library.minigpt4_contains_eos_token(b"##") == 11
    assert lib.library.minigpt4_contains_eos_token(b"###") == 0
    assert lib.library.minigpt4_is_eos(b"hello###") == 12
    assert lib.library.minigpt4_is_eos(b"##") == 0
    assert lib.minigpt4_is_eos("a ###") and not lib.minigpt4_is_eos("### a")


def test_image_entry_points_validate_like_the_reference(lib):
    """minigpt4.cpp:2598-2615: 3 channels and U8 or an error code; a file that cannot be read is OpenImage (tests/test_image_cpu.py has the rest)."""
    import minigpt4_cpp_b200 as m
    with pytest.raises(RuntimeError, match="OpenImage"):
        lib.minigpt4_image_load_from_file(m.MiniGPT4Context(None), "/nonexistent/x.png", 0)
    with pytest.raises(RuntimeError, match="OpenImage"):
        lib.minigpt4_preprocess_image(m.MiniGPT4Context(None), m.MiniGPT4Image())


def test_struct_layouts_match_header():
    import minigpt4_cpp_b200 as m
    assert ctypes.sizeof(m.MiniGPT4Image) == 24 and m.MiniGPT4Image.width.offset == 8 and m.MiniGPT4Image.format.offset == 20
    assert ctypes.sizeof(m.MiniGPT4Embedding) == 16 and m.MiniGPT4Embedding.n_embeddings.offset == 8


def test_model_load_missing_path_returns_null(lib):
    ctx = lib.library.minigpt4_model_load(b"/nonexistent/a.bin", b"/nonexistent/b.bin", 0, 1, 128, 8, False)
    assert ctx is None


def test_quantize_missing_input(lib):
    with pytest.raises(RuntimeError, match="PathDoesNotExist"):
        lib.minigpt4_quantize_model("/nonexistent/in.bin", "/tmp/out.bin", 5)


def test_reference_binding_binds_unmodified(lib):
    """The original project's ctypes binding (minigpt4/minigpt4_library.py) must bind to the new .so without edits.  What it
    declares - every prototype, both struct layouts - and what its GPU-free calls returned are recorded in
    tests/golden/reference_binding.json (tools/make_reference_fixtures.py); here they are applied to the library as the binding does."""
    import json
    import minigpt4_cpp_b200 as m
    rec = json.loads((ROOT / "tests" / "golden" / "reference_binding.json").read_text())
    ours = {"MiniGPT4Image": m.MiniGPT4Image, "MiniGPT4Embedding": m.MiniGPT4Embedding}
    for name, s in rec["structs"].items():
        S = ours[name]
        assert ctypes.sizeof(S) == s["size"]
        assert [[f, t.__name__, getattr(S, f).offset] for f, t in S._fields_] == s["fields"], name
    types = {t.__name__: t for t in (ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_ulong)}
    types.update(LP_c_char=ctypes.POINTER(ctypes.c_char), LP_LP_c_char=ctypes.POINTER(ctypes.POINTER(ctypes.c_char)),
                 LP_c_float=ctypes.POINTER(ctypes.c_float), LP_MiniGPT4Image=ctypes.POINTER(m.MiniGPT4Image),
                 LP_MiniGPT4Embedding=ctypes.POINTER(m.MiniGPT4Embedding))
    L = ctypes.cdll.LoadLibrary(lib.library._name)  # its own handle, like the binding's: these prototypes stay out of the session-wide one
    assert len(rec["prototypes"]) == 18
    for name, p in rec["prototypes"].items():
        fn = getattr(L, name)
        if p["argtypes"] is not None:
            fn.argtypes = [types[t] for t in p["argtypes"]]
        fn.restype = None if p["restype"] is None else types[p["restype"]]
    for name, cases in rec["calls"].items():
        for s, want in cases.items():
            assert bool(getattr(L, name)(s.encode("utf-8"))) == want, (name, s)


def test_null_arguments_are_harmless(lib):
    """The reference dereferences NULL in these entry points (minigpt4.cpp:2764-2809); here a null is 'nothing to do' / 'no such path'."""
    import ctypes
    L = ctypes.CDLL(lib.library._name)  # a private handle: the prototypes set below must not leak into the session-wide binding
    for name in ("minigpt4_free", "minigpt4_free_image", "minigpt4_free_embedding"):
        fn = getattr(L, name); fn.argtypes = [ctypes.c_void_p]; fn.restype = ctypes.c_int
        assert fn(None) == 0
    for name in ("minigpt4_contains_eos_token", "minigpt4_is_eos"):
        fn = getattr(L, name); fn.argtypes = [ctypes.c_char_p]; fn.restype = ctypes.c_int
        assert fn(None) == 0
    L.minigpt4_quantize_model.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int]
    assert L.minigpt4_quantize_model(None, None, 5) == 17  # PathDoesNotExist


def test_model_load_without_a_device_is_an_error_code_not_an_abort(lib, tmp_path):
    """No CUDA device: the engine has no CPU path, says so on stderr and returns NULL (the ABI's failure value) - the host process survives."""
    import minigpt4_cpp_b200 as m
    from minigpt4_cpp_b200 import modelgen as mg
    ext = m.B200(lib)
    if ext.L.minigpt4_b200_device_count() > 0:
        pytest.skip("this box has a CUDA device")
    p = str(tmp_path / "llama.bin")
    mg.write_llama_ggjt(p, mg.LlamaSpec(n_vocab=1024, n_embd=128, n_head=1, n_layer=1, wtype="q4_1"))
    assert ext.L.minigpt4_b200_llm_load(p.encode(), 32, 1, 0) is None
