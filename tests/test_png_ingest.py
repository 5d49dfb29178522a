"""Texture ingest (SURVEY §8f.3): rtnw_host_load_png replaces the reference's stbi_load("picture.png") (PSC/main.cpp:93).
The decoder is checked against PNG files written here with zlib (every colour type, every row filter), against the
reference's own picture.png when RTNW_REFERENCE names a checkout of the reference project, and through the "earth@<file>" scene builder."""
import importlib
import os
import struct
import sys
import zlib
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
rtnw = importlib.import_module("peter-shirley-ray-tracing-the-next-week_b200")


def _chunk(kind: bytes, data: bytes) -> bytes:
    return struct.pack(">I", len(data)) + kind + data + struct.pack(">I", zlib.crc32(kind + data) & 0xffffffff)


def _paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = abs(p - a), abs(p - b), abs(p - c)
    return a if pa <= pb and pa <= pc else (b if pb <= pc else c)


def write_png(path, samples: np.ndarray, ctype: int, depth: int = 8, filters=None, palette=None, idat_split=1):
    """samples: (h, w, channels) of uint8 (depth 8) or uint16 (depth 16); rows are filtered with filters[r % len]."""
    h, w, ch = samples.shape
    raw_rows = [samples[r].astype(">u2").tobytes() if depth == 16 else samples[r].astype(np.uint8).tobytes() for r in range(h)]
    bpp = ch * depth // 8
    out = bytearray()
    prev = bytes(len(raw_rows[0]))
    for r, row in enumerate(raw_rows):
        ft = (filters or [0])[r % len(filters or [0])]
        enc = bytearray(len(row))
        for i, x in enumerate(row):
            a = row[i - bpp] if i >= bpp else 0
            b = prev[i]
            c = prev[i - bpp] if i >= bpp else 0
            pred = [0, a, b, (a + b) >> 1, _paeth(a, b, c)][ft]
            enc[i] = (x - pred) & 0xff
        out += bytes([ft]) + enc
        prev = row
    z = zlib.compress(bytes(out), 6)
    cut = [len(z) * k // idat_split for k in range(idat_split + 1)]
    body = _chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, ctype, 0, 0, 0))
    if palette is not None:
        body += _chunk(b"PLTE", palette.astype(np.uint8).tobytes())
    body += _chunk(b"tEXt", b"Comment\0written by tests/test_png_ingest.py")
    for k in range(idat_split):
        body += _chunk(b"IDAT", z[cut[k]:cut[k + 1]])
    body += _chunk(b"IEND", b"")
    Path(path).write_bytes(b"\x89PNG\r\n\x1a\n" + body)


@pytest.mark.parametrize("ctype,channels", [(2, 3), (6, 4), (0, 1), (4, 2)])
def test_colour_types_and_all_row_filters(tmp_path, ctype, channels):
    rng = np.random.default_rng(ctype)
    w, h = 37, 23
    img = rng.integers(0, 256, size=(h, w, channels), dtype=np.uint8)
    img[5:9] = img[4]  # runs that the Up / Paeth predictors actually predict
    p = tmp_path / "t.png"
    write_png(p, img, ctype, filters=[0, 1, 2, 3, 4], idat_split=3)
    got = rtnw.load_png(p)
    want = img[:, :, :3] if channels >= 3 else np.repeat(img[:, :, :1], 3, axis=2)  # alpha dropped, grey expanded
    assert got.shape == (h, w, 3) and got.dtype == np.uint8 and np.array_equal(got, want)


def test_palette_and_sixteen_bit(tmp_path):
    rng = np.random.default_rng(7)
    pal = rng.integers(0, 256, size=(200, 3), dtype=np.uint8)
    idx = rng.integers(0, 200, size=(9, 31, 1), dtype=np.uint8)
    write_png(tmp_path / "p.png", idx, 3, palette=pal, filters=[0, 2])
    assert np.array_equal(rtnw.load_png(tmp_path / "p.png"), pal[idx[:, :, 0]])
    deep = rng.integers(0, 65536, size=(6, 11, 3), dtype=np.uint16)
    write_png(tmp_path / "d.png", deep, 2, depth=16, filters=[4, 1])
    assert np.array_equal(rtnw.load_png(tmp_path / "d.png"), (deep >> 8).astype(np.uint8))


def test_errors_are_reported_not_thrown(tmp_path):
    with pytest.raises(rtnw.RtnwError):
        rtnw.load_png(tmp_path / "missing.png")
    (tmp_path / "junk.png").write_bytes(b"P3\n1 1\n255\n0 0 0\n" * 8)
    with pytest.raises(rtnw.RtnwError):
        rtnw.load_png(tmp_path / "junk.png")
    img = np.zeros((4, 4, 3), dtype=np.uint8)
    write_png(tmp_path / "ok.png", img, 2)
    data = bytearray((tmp_path / "ok.png").read_bytes())
    (tmp_path / "cut.png").write_bytes(bytes(data[:60]))  # truncated inside IDAT
    with pytest.raises(rtnw.RtnwError):
        rtnw.load_png(tmp_path / "cut.png")
    with pytest.raises(rtnw.RtnwError):
        rtnw.HostScene(f"earth@{tmp_path / 'missing.png'}")


def test_earth_scene_takes_its_texture_from_the_file(tmp_path):
    """earth() (PSC/main.cpp:87-97) built from a PNG: the image pool of the flattened scene is the decoded file."""
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, size=(16, 32, 4), dtype=np.uint8)
    write_png(tmp_path / "e.png", img, 6, filters=[1, 4])
    hs = rtnw.HostScene(f"earth@{tmp_path / 'e.png'}")
    d = hs.desc
    tex = [d.textures[t] for t in range(d.n_textures) if d.textures[t].kind == 3]  # RTNW_TEX_IMAGE
    assert len(tex) == 1 and (tex[0].i1, tex[0].i2) == (32, 16)
    pool = np.ctypeslib.as_array(d.images, shape=(int(d.image_bytes),))
    assert np.array_equal(pool[tex[0].i0:tex[0].i0 + 32 * 16 * 3].reshape(16, 32, 3), img[:, :, :3])


REF_PNG = (Path(os.environ["RTNW_REFERENCE"]) / "Peter-Shirley-Project Code" / "cmake-build-debug" / "picture.png"
           if os.environ.get("RTNW_REFERENCE") else None)


@pytest.mark.skipif(REF_PNG is None or not REF_PNG.exists(), reason="RTNW_REFERENCE does not name a checkout of the reference project")
def test_reference_picture_png_decodes():
    """the file PSC/main.cpp:93 loads: decodes, has the IHDR size, and is an actual picture (not constant)"""
    w, h = struct.unpack(">II", REF_PNG.read_bytes()[16:24])
    got = rtnw.load_png(REF_PNG)
    assert got.shape == (h, w, 3) and got.std() > 5.0
