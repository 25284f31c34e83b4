"""GeoTIFF ingest / egress for the callers of the chain (SURVEY.md section 8(f) rank 2).

The reference reads its rasters with ``gdal.Open(path).ReadAsArray()`` (image_srtm.py:125, :177;
image_hsheds.py:133, :202) and writes the result with ``utils_dem.array2raster`` (utils_dem.py:17-40: a float32 GTiff
whose geotransform and projection are copied from another raster).  GDAL is not part of this image, and once the
chain takes ~0.15 s for a 36000^2 mosaic the decode + host copies around it are the next cost.  This module is the
minimal replacement for exactly those two calls:

* ``read_array(path)``          == ``gdal.Open(path).ReadAsArray()`` for single-band rasters: classic TIFF and BigTIFF,
  either byte order, strips or tiles, uncompressed / Deflate / LZW, horizontal and floating-point predictors,
  8/16/32/64-bit samples (compressed blocks are decoded in parallel on the I/O threads).  An
  uncompressed striped file whose strips are contiguous (what GDAL and ``array2raster`` write) is ONE ``readinto``
  straight into a pinned host array -- the array the upload DMA reads from, no intermediate copy.
* ``read_to_device(path)``      the same file -> ``DeviceRaster``, row chunks read into two pinned staging buffers and
  uploaded on a copy stream while the next chunk is being read (int16 rasters cross PCIe as int16); Deflate and LZW
  files cross PCIe compressed and their blocks are decoded on the GPU (``hd_tiff_decode``, DESIGN §9d).
* ``array2raster(new, array, rasterfn)``  same signature and meaning as the reference's: float32, georeference tags
  (ModelPixelScale / ModelTiepoint / GeoKeyDirectory / GeoDoubleParams / GeoAsciiParams, i.e. geotransform + projection)
  copied from ``rasterfn``.  BigTIFF automatically above 4 GB.

JPEG, PackBits, ZSTD and multi-band rasters are not decoded: ``GeoTiffError`` says so (fail loudly).
"""
import struct
import zlib

import numpy as np

from .exceptions import HydroDEMException


class GeoTiffError(HydroDEMException):
    """The file is not a TIFF this module reads (says which feature is missing)."""

    def __init__(self, message):
        self.message = message
        super().__init__(message)

    def __str__(self):
        return self.message


# TIFF field types -> (struct code, size)
_TYPES = {1: ("B", 1), 2: ("c", 1), 3: ("H", 2), 4: ("I", 4), 5: ("II", 8), 6: ("b", 1), 7: ("B", 1), 8: ("h", 2),
          9: ("i", 4), 10: ("ii", 8), 11: ("f", 4), 12: ("d", 8), 16: ("Q", 8), 17: ("q", 8), 18: ("Q", 8)}
_NP_TYPES = {1: "u1", 7: "u1", 3: "u2", 4: "u4", 6: "i1", 8: "i2", 9: "i4", 11: "f4", 12: "f8", 16: "u8", 17: "i8", 18: "u8"}
GEO_TAGS = (33550, 33922, 34264, 34735, 34736, 34737)      # pixel scale, tiepoint, transformation, geo keys / doubles / ascii
GDAL_NODATA = 42113
_SAMPLE_DTYPES = {(1, 8): "u1", (1, 16): "u2", (1, 32): "u4", (1, 64): "u8", (2, 8): "i1", (2, 16): "i2", (2, 32): "i4",
                  (2, 64): "i8", (3, 32): "f4", (3, 64): "f8"}


class GeoTiffInfo:
    """Header of the first image of a TIFF file: geometry, sample type, data layout and the georeference tags as raw
    (type, count, bytes) triples so that ``array2raster`` can copy them bit for bit."""

    def __init__(self):
        self.byteorder = "<"
        self.big = False
        self.width = self.height = 0
        self.dtype = None
        self.compression = 1
        self.predictor = 1
        self.tiled = False
        self.block_w = self.block_h = 0            # strip = (width, rows_per_strip)
        self.offsets = self.bytecounts = None
        self.tags = {}                             # tag -> (type, count, raw bytes) of every tag (file byte order)
        self.nodata = None

    @property
    def shape(self):
        return self.height, self.width

    def geo_tags(self):
        return {t: self.tags[t] for t in GEO_TAGS if t in self.tags}

    def values(self, tag):
        """Decoded values of a tag (tuple; ASCII as str) or None."""
        if tag not in self.tags:
            return None
        typ, count, raw = self.tags[tag]
        if typ == 2:
            return raw.split(b"\0")[0].decode("latin-1")
        if typ in (5, 10):
            v = np.frombuffer(raw, dtype=self.byteorder + ("u4" if typ == 5 else "i4")).reshape(-1, 2)
            return tuple((int(a), int(b)) for a, b in v)
        return tuple(np.frombuffer(raw, dtype=self.byteorder + _NP_TYPES[typ]).tolist())

    def geotransform(self):
        """(origin_x, pixel_width, 0, origin_y, 0, pixel_height) like ``GetGeoTransform`` for north-up rasters
        (ModelPixelScale + ModelTiepoint), or None."""
        scale, tie = self.values(33550), self.values(33922)
        if not scale or not tie or len(tie) < 6:
            return None
        i, j, _, x, y, _ = tie[:6]
        return (x - i * scale[0], scale[0], 0.0, y + j * scale[1], 0.0, -scale[1])

    def geo_keys(self):
        """The GeoKeyDirectory (tag 34735) as {key id: value}: a SHORT, a float / tuple of floats from GeoDoubleParams
        (34736) or a str from GeoAsciiParams (34737, without the trailing '|').  {} when the file has no directory."""
        d = self.values(34735)
        if not d or len(d) < 4:
            return {}
        doubles, ascii_ = self.values(34736) or (), self.values(34737) or ""
        keys = {}
        for k in range(min(d[3], (len(d) - 4) // 4)):
            key, loc, count, off = d[4 + 4 * k:8 + 4 * k]
            if loc == 0:
                keys[key] = off
            elif loc == 34736:
                v = tuple(doubles[off:off + count])
                keys[key] = v[0] if count == 1 and v else v
            elif loc == 34737:
                keys[key] = ascii_[off:off + count].rstrip("|")
            elif loc == 34735:
                v = tuple(d[off:off + count])
                keys[key] = v[0] if count == 1 and v else v
        return keys


def read_info(path):
    """Parse the header and the first IFD of ``path``."""
    try:
        return _read_info(path)
    except struct.error:
        raise GeoTiffError(f"{path}: truncated or corrupt TIFF directory") from None


def _read_info(path):
    info = GeoTiffInfo()
    with open(path, "rb") as f:
        head = f.read(16)
        if len(head) < 8 or head[:2] not in (b"II", b"MM"):
            raise GeoTiffError(f"{path}: not a TIFF file")
        bo = info.byteorder = "<" if head[:2] == b"II" else ">"
        magic = struct.unpack(bo + "H", head[2:4])[0]
        if magic == 42:
            ifd = struct.unpack(bo + "I", head[4:8])[0]
            nfmt, efmt, esize, inline = "H", "HHI4s", 12, 4
        elif magic == 43:
            info.big = True
            ifd = struct.unpack(bo + "Q", head[8:16])[0]
            nfmt, efmt, esize, inline = "Q", "HHQ8s", 20, 8
        else:
            raise GeoTiffError(f"{path}: bad TIFF magic {magic}")
        f.seek(ifd)
        n = struct.unpack(bo + nfmt, f.read(struct.calcsize(nfmt)))[0]
        entries = f.read(n * esize)
        for k in range(n):
            tag, typ, count, val = struct.unpack(bo + efmt, entries[k * esize:(k + 1) * esize])
            if typ not in _TYPES:
                continue
            nbytes = _TYPES[typ][1] * count
            if nbytes <= inline:
                raw = val[:nbytes]
            else:
                off = struct.unpack(bo + ("Q" if info.big else "I"), val)[0]
                f.seek(off)
                raw = f.read(nbytes)
            info.tags[tag] = (typ, count, raw)

    def one(tag, default=None):
        v = info.values(tag)
        return default if not v else v[0]

    info.width, info.height = one(256), one(257)
    if not info.width or not info.height:
        raise GeoTiffError(f"{path}: no image dimensions")
    if one(277, 1) != 1:
        raise GeoTiffError(f"{path}: {one(277)} samples per pixel; single-band rasters only")
    key = (one(339, 1), one(258, 1))
    if key not in _SAMPLE_DTYPES:
        raise GeoTiffError(f"{path}: sample format {key[0]} with {key[1]} bits is not supported")
    info.dtype = np.dtype(info.byteorder + _SAMPLE_DTYPES[key])
    info.compression = one(259, 1)
    info.predictor = one(317, 1)
    if info.compression not in (1, 5, 8, 32946):
        raise GeoTiffError(f"{path}: compression {info.compression} is not decoded here (none, LZW and Deflate only)")
    if info.predictor not in (1, 2, 3):
        raise GeoTiffError(f"{path}: predictor {info.predictor} is not decoded here")
    if info.predictor == 3 and info.dtype.kind != "f":
        raise GeoTiffError(f"{path}: floating-point predictor on {info.dtype} samples")
    if 322 in info.tags:
        info.tiled = True
        info.block_w, info.block_h = one(322), one(323)
        info.offsets, info.bytecounts = info.values(324), info.values(325)
    else:
        info.block_w, info.block_h = info.width, min(one(278, info.height), info.height)
        info.offsets, info.bytecounts = info.values(273), info.values(279)
    if info.offsets is None or info.bytecounts is None:
        raise GeoTiffError(f"{path}: no strip / tile offsets")
    info.offsets = np.asarray(info.offsets, dtype=np.int64)
    info.bytecounts = np.asarray(info.bytecounts, dtype=np.int64)
    nd = info.values(GDAL_NODATA)
    if nd:
        try:
            info.nodata = float(nd)
        except ValueError:
            info.nodata = None
    return info


# ---- parallel file I/O: one read() copies page cache -> user memory at ~7 GB/s on one core; disjoint pread / pwrite
# calls from a few threads (the GIL is released inside the system call) scale with the cores -------------------------
_PIECE = 16 << 20


def _io_threads():
    import os
    local = int(os.environ.get("LOCAL_WORLD_SIZE", "1") or 1)
    return max(1, min(8, len(os.sched_getaffinity(0)) // max(local, 1)))


def _pool():
    global _POOL
    if _POOL is None:
        import concurrent.futures
        _POOL = concurrent.futures.ThreadPoolExecutor(max_workers=_io_threads(), thread_name_prefix="hydrodem-io")
    return _POOL


_POOL = None


def shutdown_pool():
    """Join the I/O threads (a process that is about to fork() should not carry idle pool threads)."""
    global _POOL
    if _POOL is not None:
        _POOL.shutdown(wait=True)
        _POOL = None


def _pread_into(fd, view, offset, path="file"):
    """Fill the byte view from ``offset`` of the file, in parallel pieces."""
    import os
    total = len(view)

    def piece(a):
        b = min(total, a + _PIECE)
        got = a
        while got < b:
            n = os.preadv(fd, [view[got:b]], offset + got)
            if n <= 0:
                raise GeoTiffError(f"{path}: truncated pixel data")
            got += n

    starts = range(0, total, _PIECE)
    if total <= _PIECE or _io_threads() == 1:
        for a in starts:
            piece(a)
    else:
        list(_pool().map(piece, starts))


def _contiguous(info):
    """True when the pixel data is one uncompressed block of rows in the file (what GDAL / array2raster write)."""
    if info.tiled or info.compression != 1 or info.predictor != 1:
        return False
    row = info.width * info.dtype.itemsize
    rows = np.minimum(info.block_h, info.height - np.arange(len(info.offsets)) * info.block_h)
    if len(info.offsets) != -(-info.height // info.block_h) or np.any(info.bytecounts < rows * row):
        return False
    return bool(np.all(info.offsets[1:] == info.offsets[:-1] + rows[:-1] * row))


def _host_array(shape, dtype, pinned):
    if pinned:
        try:
            import torch
            if torch.cuda.is_available():
                from . import device as dev
                return dev.pinned_empty(shape, dtype)
        except Exception:      # noqa: BLE001  (no torch / no driver: a plain array does)
            pass
    return np.empty(shape, dtype=dtype)


def _lzw(raw, nbytes):
    """TIFF LZW through the library's host decoder (hd_host_lzw_decode: C, no GPU involved)."""
    import ctypes
    from . import _lib
    out = np.empty(nbytes, dtype=np.uint8)
    src = np.frombuffer(raw, dtype=np.uint8)
    n = _lib.load().hd_host_lzw_decode(ctypes.c_void_p(src.ctypes.data), len(raw), ctypes.c_void_p(out.ctypes.data), nbytes)
    if n < 0:
        raise GeoTiffError("corrupt LZW stream")
    if n < nbytes:
        out[n:] = 0
    return out


def _decode_block(raw, info, rows, cols):
    es = info.dtype.itemsize
    if info.compression == 5:
        raw = _lzw(raw, rows * cols * es)
    elif info.compression != 1:
        raw = zlib.decompress(raw)
    if info.predictor == 3:
        # floating-point predictor (Adobe TIFF TN3): per row the bytes are grouped by significance (all most significant
        # bytes first) and then differenced byte-wise; undo both
        b = np.frombuffer(raw, dtype=np.uint8, count=rows * cols * es).reshape(rows, cols * es)
        b = np.cumsum(b, axis=1, dtype=np.uint8).reshape(rows, es, cols)
        return np.ascontiguousarray(b.transpose(0, 2, 1)).view(">f" + str(es)).reshape(rows, cols)
    a = np.frombuffer(raw, dtype=info.dtype, count=rows * cols).reshape(rows, cols)
    if info.predictor == 2:
        if info.dtype.kind == "f":
            raise GeoTiffError("horizontal predictor on floating-point samples")
        a = np.cumsum(a, axis=1, dtype=info.dtype.newbyteorder("="))       # wraps modulo 2^bits like the encoder
    return a


def read_array(path, pinned=True, info=None):
    """``gdal.Open(path).ReadAsArray()``: the first band as a C-contiguous (ny, nx) array in the file's sample type
    (native byte order).  ``pinned``: allocate the result in pinned host memory when a GPU is present."""
    info = info or read_info(path)
    native = info.dtype.newbyteorder("=")
    out = _host_array(info.shape, native, pinned)
    with open(path, "rb", buffering=0) as f:
        if _contiguous(info):
            _pread_into(f.fileno(), memoryview(out.reshape(-1).view(np.uint8)), int(info.offsets[0]), path)
            if info.dtype.byteorder == ">":
                out.byteswap(inplace=True)
            return out
        import os
        bw, bh = info.block_w, info.block_h
        across = -(-info.width // bw)
        fd = f.fileno()

        def block(k):                                           # blocks land in disjoint parts of `out`
            by, bx = (k // across, k % across) if info.tiled else (k, 0)
            y0, x0 = by * bh, bx * bw
            if y0 >= info.height:
                return
            raw = os.pread(fd, int(info.bytecounts[k]), int(info.offsets[k]))
            if len(raw) < int(info.bytecounts[k]):
                raise GeoTiffError(f"{path}: truncated pixel data")
            rows_in_block = bh if info.tiled else min(bh, info.height - y0)
            blk = _decode_block(raw, info, rows_in_block, bw)
            ys, xs = min(bh, info.height - y0), min(bw, info.width - x0)
            out[y0:y0 + ys, x0:x0 + xs] = blk[:ys, :xs]

        nblocks = len(info.offsets)
        if nblocks > 1 and _io_threads() > 1:
            list(_pool().map(block, range(nblocks)))             # zlib, the LZW decoder and pread release the GIL
        else:
            for k in range(nblocks):
                block(k)
    return out


def read_to_device(path, chunk_bytes=64 << 20):
    """The first band of ``path`` as a DeviceRaster in the file's sample type.  Contiguous uncompressed files are read in
    row chunks into two pinned staging buffers; chunk k uploads on a copy stream while chunk k+1 is read.  LZW and
    Deflate files cross PCIe compressed and are decoded on the device (``_read_compressed_to_device``, DESIGN §9d).
    Other layouts go through ``read_array`` (pinned) and one upload."""
    import ctypes
    import torch
    from . import _lib, device as dev
    dev.require_cuda()
    info = read_info(path)
    native = info.dtype.newbyteorder("=")
    swap = info.dtype.byteorder == ">" or (info.dtype.byteorder == "=" and not np.little_endian)
    if info.compression in (5, 8, 32946):
        return _read_compressed_to_device(path, info, chunk_bytes)
    if not _contiguous(info) or swap:
        return dev.upload(read_array(path, pinned=True, info=info))
    ny, nx = info.shape
    es = native.itemsize
    raster = dev.empty(ny, nx, dev.hd_dtype_of(native), native)
    rows = max(1, min(ny, chunk_bytes // (nx * es)))
    stage = [dev.pinned_empty((rows, nx), native) for _ in range(2)]
    events = [None, None]
    cur = torch.cuda.current_stream()
    copy = torch.cuda.Stream()
    copy.wait_stream(cur)
    lib = _lib.load()
    with open(path, "rb", buffering=0) as f:
        for k, y0 in enumerate(range(0, ny, rows)):
            n = min(rows, ny - y0)
            buf = stage[k & 1]
            if events[k & 1] is not None:
                events[k & 1].synchronize()                     # its previous upload has left the buffer
            view = memoryview(buf.reshape(-1).view(np.uint8))[:n * nx * es]
            _pread_into(f.fileno(), view, int(info.offsets[0]) + y0 * nx * es, path)
            sub = raster.sub(y0, y0 + n, 0, nx)
            _lib.check(lib.hd_memcpy2d_h2d(sub.ptr, sub.pitch * es, ctypes.c_void_p(buf.ctypes.data), nx * es, nx * es, n,
                                           ctypes.c_void_p(copy.cuda_stream)))
            events[k & 1] = torch.cuda.Event()
            events[k & 1].record(copy)
    cur.wait_stream(copy)
    raster.buf.record_stream(copy)
    for ev in events:
        if ev is not None:
            ev.synchronize()                                    # the staging buffers go out of scope
    return raster


_DECODE_CORRUPT, _DECODE_HOST = 1, 2                           # hd_tiff_decode's status words (0 = stored)


def _block_table(path, info):
    """(TIFF block index, file offset, byte count, y0, x0, rows) of every block inside the raster, as read_array walks
    them: strips hold min(block_h, height - y0) rows, tiles always block_h; blocks past the height are skipped."""
    n = len(info.offsets)
    k = np.arange(n, dtype=np.int64)
    across = -(-info.width // info.block_w)
    by, bx = (k // across, k % across) if info.tiled else (k, np.zeros_like(k))
    y0, x0 = by * info.block_h, bx * info.block_w
    keep = y0 < info.height
    if len(info.bytecounts) < n:
        raise GeoTiffError(f"{path}: fewer byte counts than blocks")
    rows = np.full(n, info.block_h, dtype=np.int64) if info.tiled else np.minimum(info.block_h, info.height - y0)
    tbl = np.stack([k, info.offsets, info.bytecounts[:n], y0, x0, rows], axis=1)[keep]
    empty = tbl[tbl[:, 2] <= 0]
    if len(empty):
        raise GeoTiffError(f"{path}: block {int(empty[0, 0])} has no data (sparse files are not read)")
    return tbl


def _read_compressed_to_device(path, info, chunk_bytes):
    """LZW / Deflate blocks -> DeviceRaster, bit for bit what ``dev.upload(read_array(path))`` gives.  The compressed
    bytes of a batch of blocks (about ``chunk_bytes``) are pread on the I/O threads into one of two pinned staging
    buffers and uploaded on a copy stream while the next batch is read; each batch is decoded on the current stream by
    ``hd_tiff_decode``.  The per-block status words are read once at the end: a corrupt block raises GeoTiffError
    naming it; a Deflate block that decodes to more than the block holds (legal: the surplus is ignored) is decoded
    again on the host by ``_decode_block`` and uploaded into its place."""
    import ctypes
    import os
    import torch
    from . import _lib, device as dev
    native = info.dtype.newbyteorder("=")
    hd = dev.hd_dtype_of(native)
    if info.predictor == 2 and info.dtype.kind == "f":
        raise GeoTiffError("horizontal predictor on floating-point samples")
    ny, nx = info.shape
    bh, bw, es = info.block_h, info.block_w, native.itemsize
    tbl = _block_table(path, info)
    with open(path, "rb", buffering=0) as f:
        fd = f.fileno()
        size = os.fstat(fd).st_size
        if len(tbl) and int((tbl[:, 1] + tbl[:, 2]).max()) > size:
            raise GeoTiffError(f"{path}: truncated pixel data")
        raster = dev.empty(ny, nx, hd, native)
        if not len(tbl):
            return raster
        # batches: consecutive blocks up to chunk_bytes compressed (and 4 * chunk_bytes decoded), at least one block
        slot = _lib.load().hd_tiff_decode_workspace_bytes(1, bh, bw, hd)
        if slot <= 0:
            raise GeoTiffError(f"{path}: blocks of {bh} x {bw} samples are too large")
        starts, comp, dec = [0], 0, 0
        for i, nb in enumerate(tbl[:, 2].tolist()):
            if i > starts[-1] and (comp + nb > chunk_bytes or dec + slot > 4 * chunk_bytes):
                starts.append(i)
                comp = dec = 0
            comp += nb
            dec += slot
        starts.append(len(tbl))
        src_off = np.zeros(len(tbl), dtype=np.int64)            # offset of each block inside its batch
        batch_bytes = []
        for a, b in zip(starts[:-1], starts[1:]):
            c = np.cumsum(tbl[a:b, 2])
            src_off[a:b] = c - tbl[a:b, 2]
            batch_bytes.append(int(c[-1]))
        max_blocks = max(b - a for a, b in zip(starts[:-1], starts[1:]))
        stage_bytes = max(batch_bytes)
        lib = _lib.load()
        device = dev.device()
        dtbl = torch.from_numpy(np.ascontiguousarray(np.stack([src_off, tbl[:, 2], tbl[:, 3], tbl[:, 4], tbl[:, 5]], 1))
                                ).to(device)
        status = torch.zeros(len(tbl), dtype=torch.int32, device=device)
        ws_bytes = lib.hd_tiff_decode_workspace_bytes(max_blocks, bh, bw, hd)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=device)
        host = [dev.pinned_empty((stage_bytes,), np.uint8) for _ in range(2)]
        dsrc = [torch.empty(stage_bytes, dtype=torch.uint8, device=device) for _ in range(2)]
        uploaded, decoded = [None, None], [None, None]
        cur = torch.cuda.current_stream()
        copy = torch.cuda.Stream()
        copy.wait_stream(cur)

        def read_batch(buf, a, b):
            def one(i):
                got = os.preadv(fd, [memoryview(buf)[src_off[i]:src_off[i] + tbl[i, 2]]], int(tbl[i, 1]))
                if got < tbl[i, 2]:
                    raise GeoTiffError(f"{path}: truncated pixel data")
            if b - a > 1 and _io_threads() > 1:
                list(_pool().map(one, range(a, b)))
            else:
                for i in range(a, b):
                    one(i)

        for j, (a, b) in enumerate(zip(starts[:-1], starts[1:])):
            s = j & 1
            if uploaded[s] is not None:
                uploaded[s].synchronize()                       # the upload of batch j - 2 has left host[s]
            read_batch(host[s], a, b)
            with torch.cuda.stream(copy):
                if decoded[s] is not None:
                    copy.wait_event(decoded[s])                 # batch j - 2 is decoded: dsrc[s] is free
                _lib.check(lib.hd_memcpy2d_h2d(ctypes.c_void_p(dsrc[s].data_ptr()), batch_bytes[j],
                                               ctypes.c_void_p(host[s].ctypes.data), batch_bytes[j], batch_bytes[j], 1,
                                               ctypes.c_void_p(copy.cuda_stream)))
                uploaded[s] = torch.cuda.Event()
                uploaded[s].record(copy)
            cur.wait_event(uploaded[s])
            _lib.check(lib.hd_tiff_decode(ctypes.c_void_p(dsrc[s].data_ptr()), batch_bytes[j],
                                          ctypes.c_void_p(dtbl[a].data_ptr()), b - a, info.compression, info.predictor,
                                          hd, int(info.dtype.byteorder == ">"), raster.ptr, raster.pitch, ny, nx, bh, bw,
                                          ctypes.c_void_p(status[a].data_ptr()), ctypes.c_void_p(ws.data_ptr()), ws_bytes,
                                          dev.stream_ptr()))
            decoded[s] = torch.cuda.Event()
            decoded[s].record(cur)
        for d in dsrc:
            d.record_stream(copy)
        st = status.cpu().numpy()                               # the one synchronisation of the decode
        for ev in uploaded:
            if ev is not None:
                ev.synchronize()                                # the staging buffers go out of scope
        bad = np.flatnonzero(st == _DECODE_CORRUPT)
        if len(bad):
            raise GeoTiffError(f"{path}: corrupt compressed block {int(tbl[bad[0], 0])}")
        for i in np.flatnonzero(st == _DECODE_HOST).tolist():
            k, off, nb, y0, x0, rows = (int(v) for v in tbl[i])
            try:
                blk = _decode_block(os.pread(fd, nb, off), info, rows, bw)
            except (zlib.error, ValueError) as e:
                raise GeoTiffError(f"{path}: corrupt compressed block {k} ({e})") from None
            ys, xs = min(bh, ny - y0), min(bw, nx - x0)
            host_blk = np.ascontiguousarray(blk[:ys, :xs], dtype=native)
            sub = raster.sub(y0, y0 + ys, x0, x0 + xs)
            _lib.check(lib.hd_memcpy2d_h2d(sub.ptr, sub.pitch * es, ctypes.c_void_p(host_blk.ctypes.data), xs * es,
                                           xs * es, ys, dev.stream_ptr()))
            _lib.check(lib.hd_stream_synchronize(dev.stream_ptr()))     # host_blk is pageable
    return raster


# ---- egress ----------------------------------------------------------------------------------------------------------
def _pack_entry(bo, big, tag, typ, count, raw, data_offset):
    """One IFD entry; returns (entry bytes, out-of-line bytes or b'')."""
    inline = 8 if big else 4
    if len(raw) <= inline:
        val, extra = raw.ljust(inline, b"\0"), b""
    else:
        val, extra = struct.pack(bo + ("Q" if big else "I"), data_offset), raw
    return struct.pack(bo + ("HHQ" if big else "HHI"), tag, typ, count) + val, extra


def write_geotiff(path, array, like=None, dtype=None, geo_tags=None, nodata=None, strip_bytes=1 << 20, bigtiff=None):
    """Write a single-band uncompressed striped little-endian (Big)TIFF.  ``like``: path or GeoTiffInfo whose
    georeference tags are copied; ``geo_tags``: explicit {tag: (type, count, raw little-endian bytes)} instead;
    ``bigtiff``: None = only when the file would exceed 4 GB."""
    if not isinstance(array, np.ndarray) or array.ndim != 2:
        raise GeoTiffError("write_geotiff expects a 2-D ndarray")
    dt = np.dtype(dtype if dtype is not None else array.dtype).newbyteorder("<")
    fmt = {v: k for k, v in _SAMPLE_DTYPES.items()}.get(dt.str[1:])
    if fmt is None:
        raise GeoTiffError(f"sample type {dt} cannot be written")
    ny, nx = array.shape
    tags = {}
    if like is not None:
        src = like if isinstance(like, GeoTiffInfo) else read_info(like)
        for t, (typ, count, raw) in src.geo_tags().items():
            if src.byteorder == ">" and _TYPES[typ][1] > 1 and typ != 2:       # re-encode little-endian
                raw = np.frombuffer(raw, dtype=">" + _NP_TYPES[typ]).astype("<" + _NP_TYPES[typ]).tobytes()
            tags[t] = (typ, count, raw)
    for t, v in (geo_tags or {}).items():
        tags[t] = v
    if nodata is not None:
        s = (str(int(nodata)) if float(nodata).is_integer() else repr(float(nodata))).encode() + b"\0"    # NaN: "nan"
        tags[GDAL_NODATA] = (2, len(s), s)
    row_bytes = nx * dt.itemsize
    rps = max(1, min(ny, strip_bytes // max(row_bytes, 1)))
    nstrips = -(-ny // rps)
    data_bytes = ny * row_bytes
    big = (data_bytes + 16 * nstrips + 4096 > 0xFFFF0000) if bigtiff is None else bool(bigtiff)
    bo = "<"
    head = 16 if big else 8
    data_off = (head + 15) // 16 * 16
    counts = np.minimum(rps, ny - np.arange(nstrips) * rps).astype(np.int64) * row_bytes
    offsets = data_off + np.concatenate([[0], np.cumsum(counts)[:-1]]).astype(np.int64)
    otype = 16 if big else 4
    ofmt = "<u8" if big else "<u4"
    base = {256: (4, 1, struct.pack("<I", nx)), 257: (4, 1, struct.pack("<I", ny)),
            258: (3, 1, struct.pack("<H", dt.itemsize * 8)), 259: (3, 1, struct.pack("<H", 1)),
            262: (3, 1, struct.pack("<H", 1)), 273: (otype, nstrips, offsets.astype(ofmt).tobytes()),
            277: (3, 1, struct.pack("<H", 1)), 278: (4, 1, struct.pack("<I", rps)),
            279: (otype, nstrips, counts.astype(ofmt).tobytes()), 284: (3, 1, struct.pack("<H", 1)),
            339: (3, 1, struct.pack("<H", fmt[0]))}
    base.update(tags)
    ifd_off = (data_off + data_bytes + 15) // 16 * 16
    n = len(base)
    esize, nsize, psize = (20, 8, 8) if big else (12, 2, 4)
    extra_off = ifd_off + nsize + n * esize + psize
    entries, extras = b"", b""
    for tag in sorted(base):
        typ, count, raw = base[tag]
        e, x = _pack_entry(bo, big, tag, typ, count, raw, extra_off + len(extras))
        entries += e
        if x:
            extras += x + b"\0" * (-len(x) % 2)                  # word alignment of out-of-line values
    with open(path, "wb") as f:
        if big:
            f.write(b"II" + struct.pack("<HHHQ", 43, 8, 0, ifd_off))
        else:
            f.write(b"II" + struct.pack("<HI", 42, ifd_off))
        f.write(b"\0" * (data_off - head))
        # Buffered writes to one file serialise on its inode lock, so the pieces are written in order by this thread;
        # what runs on the pool is their conversion to the output sample type (no full-size temporary: a window of
        # pieces at a time).
        step = max(1, _PIECE // max(row_bytes, 1))
        starts = list(range(0, ny, step))

        def convert(y0):
            return np.ascontiguousarray(array[y0:y0 + step], dtype=dt)

        if array.dtype == dt and array.flags.c_contiguous:
            f.write(memoryview(array.reshape(-1).view(np.uint8)))
        else:
            window = 2 * _io_threads()
            for w0 in range(0, len(starts), window):
                group = starts[w0:w0 + window]
                blocks = _pool().map(convert, group) if _io_threads() > 1 and len(group) > 1 else map(convert, group)
                for blk in blocks:
                    f.write(memoryview(blk.reshape(-1).view(np.uint8)))
        f.write(b"\0" * (ifd_off - data_off - data_bytes))
        f.write(struct.pack("<Q" if big else "<H", n) + entries + struct.pack("<Q" if big else "<I", 0) + extras)
    return path


def array2raster(new_rasterfn, array, rasterfn=None):
    """utils_dem.array2raster (utils_dem.py:17-40): ``array`` as a float32 GeoTIFF at ``new_rasterfn``, georeference
    (geotransform + projection = the GeoTIFF georeference tags) taken from the file ``rasterfn``."""
    write_geotiff(new_rasterfn, array, like=rasterfn, dtype=np.float32)


def process_geotiffs(srtm_tif, groves_tif, hsheds_tif, final_tif, rivers_tif=None, chain=None, envelope=None):
    """HydroDEMProcess.start between its reads and its write (hydro_dem_process.py:122-153): three (four) GeoTIFFs in,
    the conditioned DEM out as a float32 GeoTIFF georeferenced like the SRTM raster.  Returns the chain's host results
    (``final`` float64, ``filled``, ``d8``).

    ``envelope``: an ESRI shapefile of the area of interest, or a ``warp.Grid``.  The inputs (raw downloads, geographic
    WGS84 or EPSG:22184) are then first reprojected onto the envelope's EPSG:22184 90 m grid on the device
    (``warp.warp_to_device``, nearest neighbour: the reference's ``resample_and_cut`` step), go through the chain without
    leaving the device, and the DEM is written with that grid's georeference.  Each input may then also be a list of
    tile paths, mosaicked onto the grid as one virtual raster (``warp.warp_to_device``); without an envelope there is
    no grid to mosaic onto, and a list raises GeoTiffError."""
    from .pipeline import ConditioningChain
    chain = chain or ConditioningChain()
    if envelope is not None:
        return _process_on_grid(chain, srtm_tif, groves_tif, hsheds_tif, final_tif, rivers_tif, envelope)
    for name, p in (("srtm_tif", srtm_tif), ("groves_tif", groves_tif), ("hsheds_tif", hsheds_tif),
                    ("rivers_tif", rivers_tif)):
        if isinstance(p, (list, tuple)):
            raise GeoTiffError(f"{name}: a list of tiles needs an envelope (or a warp.Grid) to mosaic onto")
    srtm = read_array(srtm_tif)
    groves = read_array(groves_tif)
    hsheds = read_array(hsheds_tif)
    rivers = read_array(rivers_tif) if rivers_tif else None
    out = chain.apply_to_host(srtm, groves, hsheds, rivers)
    array2raster(final_tif, out["final"], srtm_tif)
    return out


def _process_on_grid(chain, srtm_tif, groves_tif, hsheds_tif, final_tif, rivers_tif, envelope):
    from . import warp
    from .pipeline import check_fill_status
    grid = warp.as_grid(envelope)
    paths = (srtm_tif, groves_tif, hsheds_tif) + ((rivers_tif,) if rivers_tif else ())
    rasters = [warp.warp_to_device(p, grid) for p in paths]
    res = chain.run_device(*rasters)
    out = {k: res.host(k) for k in ("final", "filled", "d8") if k in res.rasters}
    fill = res.info.get("fill")
    if fill is not None:
        check_fill_status(fill.status())
    write_geotiff(final_tif, out["final"], dtype=np.float32, geo_tags=grid.geo_tags())
    return out
