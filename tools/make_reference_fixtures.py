#!/usr/bin/env python
"""Write the fixtures under tests/golden/ that come from the original minigpt4.cpp project, so that the tests using them
need nothing outside this repository:

  golden/reference_binding.json   what the original project's ctypes binding (minigpt4/minigpt4_library.py) declares for the
                                  18 ABI symbols and its two structs, and what its GPU-free calls return against build/libminigpt4.so
  golden/images/llama.png         the original project's sample images (minigpt4/images/): llama.png as shipped;
  golden/images/story_rows84-147.png   story.png (421 KB) cut to rows 84..147.  The band starts on a Sub-filtered row, so
                                  its filtered scanlines are the original bytes (Sub / Up / Paeth rows), re-deflated.

Run on a CPU box after build():  python tools/make_reference_fixtures.py /path/to/minigpt4.cpp
"""
from __future__ import annotations

import ctypes
import importlib.util
import json
import re
import shutil
import struct
import sys
import zlib
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
GOLD = ROOT / "tests" / "golden"
STORY_BAND = (84, 64)   # first row, rows
EOS_CASES = ["x###", "hello###", "### a", "a ###", "##", "#", ""]


def type_name(t) -> str | None:
    return None if t is None else t.__name__


def record_binding(ref: Path) -> dict:
    from minigpt4_cpp_b200 import build, minigpt4_library as ml
    spec = importlib.util.spec_from_file_location("ref_minigpt4_library", ref / "minigpt4" / "minigpt4_library.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    rlib = mod.MiniGPT4SharedLibrary(str(build.build()))
    protos = {}
    for name in sorted(ml.ABI_SYMBOLS):
        fn = getattr(rlib.library, name)
        protos[name] = {"argtypes": None if fn.argtypes is None else [type_name(a) for a in fn.argtypes], "restype": type_name(fn.restype)}
    structs = {s.__name__: {"size": ctypes.sizeof(s), "fields": [[f, type_name(t), getattr(s, f).offset] for f, t in s._fields_]}
               for s in (mod.MiniGPT4Image, mod.MiniGPT4Embedding)}
    calls = {"minigpt4_is_eos": {s: bool(rlib.minigpt4_is_eos(s)) for s in EOS_CASES},
             "minigpt4_contains_eos_token": {s: bool(rlib.minigpt4_contains_eos_token(s)) for s in EOS_CASES}}
    return {"source": "minigpt4.cpp minigpt4/minigpt4_library.py (MiniGPT4SharedLibrary.__init__ and its wrappers)",
            "prototypes": protos, "structs": structs, "calls": calls}


def png_chunks(data: bytes):
    i = 8
    while i < len(data):
        n, = struct.unpack(">I", data[i:i + 4])
        yield data[i + 4:i + 8], data[i + 8:i + 8 + n]
        i += 12 + n


def png_chunk(kind: bytes, body: bytes) -> bytes:
    return struct.pack(">I", len(body)) + kind + body + struct.pack(">I", zlib.crc32(kind + body))


def row_band(data: bytes, first: int, rows: int) -> bytes:
    """rows first..first+rows-1 of an 8-bit non-interlaced PNG; the first kept row must not depend on the row above it"""
    chunks = list(png_chunks(data))
    assert chunks[0][0] == b"IHDR"
    w, h, depth, ctype, comp, filt, interlace = struct.unpack(">IIBBBBB", chunks[0][1])
    assert depth == 8 and interlace == 0 and first + rows <= h
    stride = 1 + w * {2: 3, 6: 4, 0: 1, 4: 2}[ctype]
    raw = zlib.decompress(b"".join(body for kind, body in chunks if kind == b"IDAT"))
    assert raw[first * stride] in (0, 1), "band must start on a None / Sub row"
    z = zlib.compress(raw[first * stride:(first + rows) * stride], 9)
    out = [png_chunk(b"IHDR", struct.pack(">IIBBBBB", w, rows, depth, ctype, comp, filt, interlace))]
    out += [png_chunk(kind, body) for kind, body in chunks if kind not in (b"IHDR", b"IDAT", b"IEND")]
    out += [png_chunk(b"IDAT", z[i:i + 65536]) for i in range(0, len(z), 65536)]
    return data[:8] + b"".join(out) + png_chunk(b"IEND", b"")


def main():
    ref = Path(sys.argv[1])
    text = json.dumps(record_binding(ref), indent=1)
    text = re.sub(r"\[\s+([^\[\]{}]*?)\s+\]", lambda mt: "[" + " ".join(mt.group(1).split()) + "]", text)   # lists of scalars on one line
    (GOLD / "reference_binding.json").write_text(text + "\n")
    img = GOLD / "images"
    img.mkdir(parents=True, exist_ok=True)
    shutil.copyfile(ref / "minigpt4" / "images" / "llama.png", img / "llama.png")
    first, rows = STORY_BAND
    band = row_band((ref / "minigpt4" / "images" / "story.png").read_bytes(), first, rows)
    (img / f"story_rows{first}-{first + rows - 1}.png").write_bytes(band)


if __name__ == "__main__":
    main()
