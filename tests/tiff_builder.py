"""Test-side writer of compressed single-band TIFFs (the package itself writes uncompressed files only): Deflate or TIFF LZW
strips and tiles, horizontal (2) and floating-point (3, TIFF TN3) predictors, either byte order, raw extra tags.  Used by
tests/test_gpu_tiff_decode.py and tools/geotiff_decode_time.py."""
import struct
import zlib

import numpy as np

_SAMPLE_FORMAT = {"u": 1, "i": 2, "f": 3}


def lzw_encode(data, eoi=True):
    """TIFF LZW as libtiff reads it: MSB-first codes, ClearCode first, 9..12 bits with the early change.  The code width
    of every emitted code is the width the decoder will read it with (its table lags the encoder's by one entry)."""
    out, acc, nacc = bytearray(), 0, 0

    def emit(code, width):
        nonlocal acc, nacc
        acc = (acc << width) | code
        nacc += width
        while nacc >= 8:
            out.append((acc >> (nacc - 8)) & 0xFF)
            nacc -= 8
        acc &= (1 << nacc) - 1

    table = {bytes([i]): i for i in range(256)}
    enc_next, dec_next, dec_bits, dec_old = 258, 258, 9, False

    def sent(code):                                     # the decoder's state after it has read `code`
        nonlocal dec_next, dec_bits, dec_old
        emit(code, dec_bits)
        if dec_old and dec_next < 4096:
            dec_next += 1
            if dec_next == (1 << dec_bits) - 1 and dec_bits < 12:
                dec_bits += 1
        dec_old = True

    emit(256, 9)
    w = b""
    for c in data:
        wc = w + bytes([c])
        if wc in table:
            w = wc
            continue
        sent(table[w])
        table[wc] = enc_next
        enc_next += 1
        w = bytes([c])
        if enc_next == 4094:                            # table full: start over
            emit(256, dec_bits)
            table = {bytes([i]): i for i in range(256)}
            enc_next, dec_next, dec_bits, dec_old = 258, 258, 9, False
    if w:
        sent(table[w])
    if eoi:
        emit(257, dec_bits)
    if nacc:
        out.append((acc << (8 - nacc)) & 0xFF)
    return bytes(out)


def predict(block, predictor, file_dtype):
    """The bytes of one block (rows x cols samples, host array) as stored before compression."""
    if predictor == 3:
        es = block.dtype.itemsize
        be = block.astype(">f" + str(es)).view(np.uint8).reshape(block.shape[0], block.shape[1], es)
        planes = np.ascontiguousarray(be.transpose(0, 2, 1)).reshape(block.shape[0], -1)     # most significant first
        d = planes.copy()
        d[:, 1:] = planes[:, 1:] - planes[:, :-1]
        return d.tobytes()
    t = block.astype(file_dtype.newbyteorder("="))
    if predictor == 2:
        t = t.copy()
        t[:, 1:] = t[:, 1:] - t[:, :-1]                                  # wraps modulo 2^bits
    return t.astype(file_dtype).tobytes()


def compress(raw, compression, level=6):
    return lzw_encode(raw) if compression == 5 else zlib.compress(raw, level)


def blocks_of(a, rows=None, tile=None):
    """(y0, x0, block array) in file order: strips of ``rows`` rows (the last one short) or ``tile`` = (th, tw) tiles
    zero-padded at the ragged edges."""
    ny, nx = a.shape
    if tile is None:
        rows = rows or ny
        return [(y, 0, a[y:y + rows]) for y in range(0, ny, rows)]
    th, tw = tile
    out = []
    for y in range(0, ny, th):
        for x in range(0, nx, tw):
            t = np.zeros((th, tw), dtype=a.dtype)
            part = a[y:y + th, x:x + tw]
            t[:part.shape[0], :part.shape[1]] = part
            out.append((y, x, t))
    return out


def build_tiff(blocks, tags, bo="<"):
    """A classic TIFF from compressed blocks + {tag: (type, values)} or {tag: (type, count, raw bytes)}; the offsets and
    byte counts tags are filled in here."""
    fmt = {3: "H", 4: "I", 12: "d"}
    data = b"".join(blocks)
    offs, pos = [], 8
    for b in blocks:
        offs.append(pos)
        pos += len(b)
    tiled = 322 in tags
    tags = dict(tags)
    tags[324 if tiled else 273] = (4, offs)
    tags[325 if tiled else 279] = (4, [len(b) for b in blocks])
    ifd_off = (8 + len(data) + 1) // 2 * 2
    extra_off = ifd_off + 2 + 12 * len(tags) + 4
    entries, extras = b"", b""
    for tag in sorted(tags):
        v = tags[tag]
        if len(v) == 3:
            typ, count, raw = v
        else:
            typ, vals = v
            count, raw = len(vals), struct.pack(bo + fmt[typ] * len(vals), *vals)
        if len(raw) <= 4:
            val = raw.ljust(4, b"\0")
        else:
            val = struct.pack(bo + "I", extra_off + len(extras))
            extras += raw + b"\0" * (len(raw) % 2)
        entries += struct.pack(bo + "HHI", tag, typ, count) + val
    head = (b"II" if bo == "<" else b"MM") + struct.pack(bo + "HI", 42, ifd_off)
    return (head + data + b"\0" * (ifd_off - 8 - len(data)) + struct.pack(bo + "H", len(tags)) + entries +
            struct.pack(bo + "I", 0) + extras)


def write(path, a, compression=8, predictor=1, bo="<", rows=None, tile=None, extra_tags=None, level=6, blocks=None):
    """Write ``a`` compressed.  ``extra_tags``: {tag: (type, count, raw little-endian bytes)} (georeference, nodata) --
    little-endian files only; ``blocks``: already compressed blocks to store instead of encoding ``a``."""
    dt = np.dtype(bo + a.dtype.str[1:])
    ny, nx = a.shape
    if blocks is None:
        blocks = [compress(predict(b, predictor, dt), compression, level) for _, _, b in blocks_of(a, rows, tile)]
    tags = {256: (4, [nx]), 257: (4, [ny]), 258: (3, [8 * dt.itemsize]), 259: (3, [compression]), 262: (3, [1]),
            277: (3, [1]), 284: (3, [1]), 317: (3, [predictor]), 339: (3, [_SAMPLE_FORMAT[dt.kind]])}
    if tile is None:
        tags[278] = (4, [rows or ny])
    else:
        tags[322], tags[323] = (4, [tile[1]]), (4, [tile[0]])
    if extra_tags:
        assert bo == "<"
        tags.update(extra_tags)
    with open(path, "wb") as f:
        f.write(build_tiff(blocks, tags, bo))
    return path
