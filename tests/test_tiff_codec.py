"""CPU: the GeoTIFF block decoder's core (csrc/tiffcodec.cuh), which the device runs one warp per block, on the host
through hd_host_inflate / hd_host_tiff_lzw.  Deflate agrees with zlib.decompress byte for byte and rejects whatever zlib
rejects; LZW agrees with hd_host_lzw_decode (return value and bytes).  A hostile corpus (truncations, bit flips, broken
Huffman codes, bad headers and checksums) is rejected with a negative status and never writes past the capacity."""
import ctypes
import struct
import zlib

import numpy as np
import pytest
from PIL import Image

from hydrodem_b200 import _lib, geotiff

GUARD = 64


@pytest.fixture(scope="module")
def lib():
    return _lib.load()


def _call(fn, data, cap):
    """fn over data with an output of cap bytes followed by a guard band that must stay untouched."""
    src = np.frombuffer(bytes(data) + b"\0", dtype=np.uint8)          # never a null pointer, even for b""
    out = np.full(cap + GUARD, 0xA5, dtype=np.uint8)
    n = fn(ctypes.c_void_p(src.ctypes.data), len(data), ctypes.c_void_p(out.ctypes.data), cap)
    assert (out[cap:] == 0xA5).all(), "write past the capacity"
    return n, out[:max(n, 0)].tobytes()


def _zlib_or_none(data):
    try:
        return zlib.decompress(data)
    except zlib.error:
        return None


def _agrees_with_zlib(lib, data, cap=None):
    want = _zlib_or_none(data)
    if cap is None:
        cap = len(want) if want is not None else 4096
    n, got = _call(lib.hd_host_inflate, data, cap)
    if want is None:
        assert n < 0, "zlib rejects this stream"
    elif len(want) > cap:
        assert n == _lib.HD_ERR_WORKSPACE
    else:
        assert n == len(want) and got == want
    return want


def _dem_bytes(n, seed):
    rng = np.random.default_rng(seed)
    x = np.cumsum(rng.standard_normal(n // 2)) * 3 + rng.standard_normal(n // 2) * 0.5
    return np.round(x).astype("<i2").tobytes()[:n]


PAYLOADS = {
    "empty": b"",
    "one": b"\x07",
    "dem": _dem_bytes(120_000, 1),
    "noise": np.random.default_rng(2).integers(0, 256, 70_000, dtype=np.uint8).tobytes(),
    "run": b"\x00" * 100_000 + b"ab" * 3000,                        # distance 1 / 2, length 258
    "text": b"the quick brown fox jumps over the lazy dog " * 900,
}


@pytest.mark.parametrize("name", sorted(PAYLOADS))
@pytest.mark.parametrize("level", range(10))
def test_inflate_levels(lib, name, level):
    _agrees_with_zlib(lib, zlib.compress(PAYLOADS[name], level))


@pytest.mark.parametrize("strategy", ["Z_DEFAULT_STRATEGY", "Z_FILTERED", "Z_HUFFMAN_ONLY", "Z_RLE", "Z_FIXED"])
@pytest.mark.parametrize("wbits", range(9, 16))
def test_inflate_strategies_and_windows(lib, strategy, wbits):
    for name in ("dem", "run", "one", "empty"):
        c = zlib.compressobj(6, zlib.DEFLATED, wbits, 8, getattr(zlib, strategy))
        _agrees_with_zlib(lib, c.compress(PAYLOADS[name]) + c.flush())


def test_inflate_trailing_bytes_and_capacity(lib):
    data = zlib.compress(PAYLOADS["dem"], 6)
    _agrees_with_zlib(lib, data + b"trailing garbage")
    want = PAYLOADS["dem"]
    n, got = _call(lib.hd_host_inflate, data, len(want) + 100)           # more room than needed: the true length
    assert n == len(want) and got == want
    for cap in (0, 1, len(want) - 1):                                    # less: HD_ERR_WORKSPACE, nothing past cap
        n, _ = _call(lib.hd_host_inflate, data, cap)
        assert n == _lib.HD_ERR_WORKSPACE
    stored = zlib.compress(PAYLOADS["noise"][:5000], 0)
    assert _call(lib.hd_host_inflate, stored, 4000)[0] == _lib.HD_ERR_WORKSPACE
    assert lib.hd_host_inflate(None, 0, None, 0) == _lib.HD_ERR_NULL


def test_inflate_truncations(lib):
    for name, level in (("dem", 6), ("text", 9), ("noise", 0), ("run", 1)):
        data = zlib.compress(PAYLOADS[name][:20_000], level)
        for k in range(len(data)):
            if len(data) > 3000 and k % 7 and k < len(data) - 64:
                continue                                                 # every 7th cut, all of the last 64 bytes
            _agrees_with_zlib(lib, data[:k], cap=20_000)


def test_inflate_bit_flips(lib):
    rng = np.random.default_rng(7)
    for name, level, strategy in (("dem", 6, zlib.Z_DEFAULT_STRATEGY), ("text", 9, zlib.Z_FIXED),
                                  ("run", 1, zlib.Z_RLE), ("noise", 1, zlib.Z_HUFFMAN_ONLY)):
        c = zlib.compressobj(level, zlib.DEFLATED, 15, 8, strategy)
        data = bytearray(c.compress(PAYLOADS[name][:30_000]) + c.flush())
        for _ in range(300):
            bad = bytearray(data)
            for _ in range(int(rng.integers(1, 4))):
                bit = int(rng.integers(0, 8 * len(bad)))
                bad[bit // 8] ^= 1 << (bit % 8)
            _agrees_with_zlib(lib, bytes(bad), cap=30_000)


class _BitWriter:
    """LSB-first bit packer for hand-made Deflate blocks."""

    def __init__(self):
        self.bits = []

    def put(self, v, n):
        self.bits += [(v >> i) & 1 for i in range(n)]

    def huff(self, code, n):                                             # Huffman codes go most significant bit first
        self.bits += [(code >> (n - 1 - i)) & 1 for i in range(n)]

    def bytes(self):
        b = self.bits + [0] * (-len(self.bits) % 8)
        return bytes(sum(b[i + j] << j for j in range(8)) for i in range(0, len(b), 8))


def _zwrap(body, payload=b""):
    return b"\x78\x9c" + body + struct.pack(">I", zlib.adler32(payload))


def _dynamic_header(w, hlit, hdist, clens):
    w.put(1, 1)
    w.put(2, 2)
    w.put(hlit - 257, 5)
    w.put(hdist - 1, 5)
    w.put(len(clens) - 4, 4)
    for v in clens:
        w.put(v, 3)


def test_inflate_hand_made_corruption(lib):
    cases = {}
    # stored block with LEN / NLEN mismatch; and a correct one for contrast
    w = _BitWriter(); w.put(1, 1); w.put(0, 2)
    cases["stored_ok"] = _zwrap(w.bytes() + struct.pack("<HH", 3, 0xFFFC) + b"abc", b"abc")
    cases["stored_bad_nlen"] = _zwrap(w.bytes() + struct.pack("<HH", 3, 0xFFFD) + b"abc", b"abc")
    cases["block_type_3"] = _zwrap(bytes([0b111]))
    # fixed block: literal 'a' (0x30 + 0x61, 8 bits) then a distance of 2 at output length 1
    w = _BitWriter(); w.put(1, 1); w.put(1, 2); w.huff(0x30 + 0x61, 8); w.huff(1, 7); w.huff(1, 5); w.huff(0, 7)
    cases["distance_past_start"] = _zwrap(w.bytes(), b"aaaa")
    w = _BitWriter(); w.put(1, 1); w.put(1, 2); w.huff(0x30 + 0x61, 8); w.huff(1, 7); w.huff(30, 5)
    cases["distance_code_30"] = _zwrap(w.bytes())
    w = _BitWriter(); w.put(1, 1); w.put(1, 2); w.huff(0xC0 + 286 - 280, 8)
    cases["length_code_286"] = _zwrap(w.bytes())
    w = _BitWriter(); w.put(1, 1); w.put(1, 2); w.huff(0x30 + 0x61, 8); w.huff(0, 7)
    cases["fixed_ok"] = _zwrap(w.bytes(), b"a")
    # dynamic headers: code-length codes over-subscribed / incomplete / absent
    order = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15]
    for name, lens in (("codes_oversubscribed", {0: 1, 8: 1, 1: 1}), ("codes_incomplete", {0: 2, 8: 2, 1: 2}),
                       ("codes_none", {})):
        w = _BitWriter()
        _dynamic_header(w, 257, 1, [lens.get(s, 0) for s in order])
        cases[name] = _zwrap(w.bytes() + b"\0" * 64)
    # literal / length code over-subscribed: code-length code {8: '0', 1: '1'} (one bit each), then 257 lengths of 8 + 1
    w = _BitWriter()
    _dynamic_header(w, 257, 1, [{8: 1, 1: 1}.get(s, 0) for s in order])
    for _ in range(257):
        w.huff(0, 1)                                                     # length 8 for every literal / length symbol
    w.huff(1, 1)                                                         # one distance code of length 1
    cases["lit_oversubscribed"] = _zwrap(w.bytes() + b"\0" * 8)
    # repeat-previous (16) as the first code length
    w = _BitWriter()
    _dynamic_header(w, 257, 1, [{16: 1, 1: 1}.get(s, 0) for s in order])
    w.huff(0, 1); w.put(0, 2)
    cases["repeat_first"] = _zwrap(w.bytes() + b"\0" * 64)
    # header: bad FCHECK, FDICT, method 7, window 64 KB; bad Adler-32; no final block
    good = zlib.compress(b"hello hello hello", 9)
    cases["bad_fcheck"] = bytes([good[0], good[1] ^ 1]) + good[2:]
    cmf = 0x78
    flg = 0x20 | (31 - (cmf * 256 + 0x20) % 31) % 31
    cases["fdict"] = bytes([cmf, flg]) + b"\0\0\0\0" + good[2:]
    cmf = 0x77
    cases["method_7"] = bytes([cmf, (31 - (cmf * 256) % 31) % 31]) + good[2:]
    cmf = 0x88
    cases["window_64k"] = bytes([cmf, (31 - (cmf * 256) % 31) % 31]) + good[2:]
    cases["bad_adler"] = good[:-1] + bytes([good[-1] ^ 1])
    c = zlib.compressobj()
    cases["no_final_block"] = c.compress(b"abcabc" * 50) + c.flush(zlib.Z_SYNC_FLUSH)
    for name, data in cases.items():
        want = _agrees_with_zlib(lib, data, cap=4096 if _zlib_or_none(data) is None else None)
        assert (want is not None) == name.endswith("_ok"), name


# ---- LZW ---------------------------------------------------------------------------------------------------------------
def _lzw_strips(tmp_path, a, rows):
    p = tmp_path / "l.tif"
    Image.fromarray(a).save(p, format="TIFF", compression="tiff_lzw", tiffinfo={278: rows})
    info = geotiff.read_info(p)
    raw = p.read_bytes()
    return [raw[o:o + c] for o, c in zip(info.offsets, info.bytecounts)], rows * a.shape[1] * a.itemsize


def _lzw_agrees(lib, data, cap):
    want = _call(lib.hd_host_lzw_decode, data, cap)
    got = _call(lib.hd_host_tiff_lzw, data, cap)
    assert (got[0] < 0) == (want[0] < 0)
    if want[0] >= 0:
        assert got == want


@pytest.mark.parametrize("kind", ["smooth", "noise", "constant", "long"])
def test_lzw_core_equals_host_decoder(lib, tmp_path, kind):
    rng = np.random.default_rng(11)
    if kind == "smooth":
        yy, xx = np.mgrid[0:200, 0:700]
        a = np.round(100 + 20 * np.sin(xx / 40.0) + 15 * np.cos(yy / 55.0)).astype(np.uint16)
    elif kind == "noise":
        a = rng.integers(0, 65535, (150, 500), dtype=np.uint16)
    elif kind == "constant":
        a = np.full((300, 900), 7, dtype=np.uint16)
    else:
        a = np.repeat(rng.integers(0, 4, (1, 125000), dtype=np.uint8), 2, axis=0).reshape(250, 1000).astype(np.uint16)
    for rows in (1, 7, a.shape[0]):
        strips, cap = _lzw_strips(tmp_path, a, rows)
        for s in strips[:40]:
            for c in (cap, cap - 1, cap // 3, 0, cap + 50):               # exact, truncated and roomy outputs
                _lzw_agrees(lib, s, c)


def test_lzw_core_on_corrupt_streams(lib, tmp_path):
    rng = np.random.default_rng(3)
    yy, xx = np.mgrid[0:64, 0:300]
    a = np.round(50 + 20 * np.sin(xx / 9.0) + 9 * np.cos(yy / 7.0)).astype(np.uint16)
    strips, cap = _lzw_strips(tmp_path, a, 16)
    for s in strips:
        for k in range(0, len(s), 5):                                    # truncations: no EOI, short output
            _lzw_agrees(lib, s[:k], cap)
        for _ in range(200):
            bad = bytearray(s)
            bit = int(rng.integers(0, 8 * len(bad)))
            bad[bit // 8] ^= 1 << (bit % 8)
            _lzw_agrees(lib, bytes(bad), cap)
    for junk in (b"\x80\x3f\xff\xff\xff", rng.integers(0, 256, 4000, dtype=np.uint8).tobytes(), b"\xff" * 100):
        _lzw_agrees(lib, junk, 5000)
    assert lib.hd_host_tiff_lzw(None, 0, None, 0) == _lib.HD_ERR_NULL


def test_tiff_decode_argument_errors_need_no_gpu(lib):
    p = ctypes.c_void_p(1 << 20)
    ws = lib.hd_tiff_decode_workspace_bytes(10, 16, 100, _lib.I16)
    assert ws == 10 * 3200
    assert lib.hd_tiff_decode_workspace_bytes(10, 16, 100, _lib.C64) == 0
    assert lib.hd_tiff_decode_workspace_bytes(10, 1 << 20, 1 << 20, _lib.U8) == 0

    def call(**kw):
        a = dict(src=p, src_bytes=100, blocks=p, n=10, comp=8, pred=2, dt=_lib.I16, be=0, out=p, pitch=128, ny=100,
                 nx=100, bh=16, bw=100, status=p, ws=p, wsb=ws)
        a.update(kw)
        return lib.hd_tiff_decode(a["src"], a["src_bytes"], a["blocks"], a["n"], a["comp"], a["pred"], a["dt"], a["be"],
                                  a["out"], a["pitch"], a["ny"], a["nx"], a["bh"], a["bw"], a["status"], a["ws"], a["wsb"],
                                  None)
    assert call(out=None) == _lib.HD_ERR_NULL
    assert call(blocks=None) == _lib.HD_ERR_NULL
    assert call(comp=7) == _lib.HD_ERR_ARG
    assert call(pred=4) == _lib.HD_ERR_ARG
    assert call(pred=3) == _lib.HD_ERR_ARG                              # floating-point predictor on int16
    assert call(pred=2, dt=_lib.F32) == _lib.HD_ERR_ARG                 # horizontal predictor on floats
    assert call(dt=_lib.C64) == _lib.HD_ERR_ARG
    assert call(pitch=99) == _lib.HD_ERR_ARG
    assert call(n=-1) == _lib.HD_ERR_ARG
    assert call(wsb=ws - 1) == _lib.HD_ERR_WORKSPACE
    assert call(pitch=101) == _lib.HD_ERR_ALIGN
    assert call(out=ctypes.c_void_p((1 << 20) + 2)) == _lib.HD_ERR_ALIGN
