"""Row-band sharding of one large mosaic across the GPUs of a box (BASELINE.json configs[3] / [4]).

A mosaic of ``ny`` rows is cut into ``world`` contiguous row bands (one per rank / GPU; band starts are even so that
transforms which pack two rows keep the same pairs as on one GPU).  Everything here is built so that the sharded
result equals the single-GPU result BIT FOR BIT -- exact-class and tolerance-class stages alike:

* **Stencil stages** run the unchanged single-GPU stage code (``ConditioningChain._stage_*``) on the band EXTENDED by
  ``HALO`` rows of its neighbours.  The halo is exchanged ONCE per input (NCCL send / recv straight into the margin rows
  of a buffer that was allocated with them -- no per-stage copies); a stage with half-window h leaves h more rows at
  the cut edges invalid, and HALO = 24 covers the deepest dependency chain (closing 2 + 3 x quadratic 7 + 1 for the
  final 3x3 mean).  Every kernel's arithmetic for a cell is a fixed sequence of operations on that cell's window
  (csrc/quadratic.cu accumulates in double for exactly this reason), so cut positions cannot change a bit.
* **Fourier stage**: the row / column transforms of ``hd_fft2_forward_shift_abs`` / ``hd_fft2_masked_inverse_abs`` run
  on each rank's local rows through ``hd_fft_band_pass`` (the same row passes, same pairing), the four transposes
  become all-to-all exchanges (``fourier_exchanges``: the transposes store straight into the owning rank's memory,
  mapped through CUDA IPC; where the ranks cannot map each other's memory the transposed blocks travel as NCCL send /
  recv), the conjugate half of the spectrum is completed locally because each rank owns a set of spectrum rows closed
  under ky -> -ky ("K layout"), and the window-55 peak detector works on row slabs of the spectrum quarters with 61
  rows of context (|F| stays banded: no all-gather).
* **Sink-fill**: every rank relaxes [halo row | band | halo row] to its local fixed point, edge rows are exchanged, a
  small kernel lowers the halo rows and raises a DEVICE flag, the flags are all-reduced and the host reads one word
  per round.  The fixed point is unique, so the banded surface equals the single-GPU one; NaN restoration and D8 are
  one fused pass (``hd_pdfill_finish_d8``).

The communicator is abstract: ``DistComm`` (torch.distributed: NCCL on the GPU box, gloo in the CPU tests) or
``ThreadComm`` (ranks emulated as threads of one process on one device: the single-GPU parity tests).
"""
import ctypes
import threading
import typing

import numpy as np
import torch

from . import _lib, device as dev

HALO = 24               # rows of context every extended band carries (see module docstring)
MASK_HALO = 2 * 27 + 1 + 6     # MaskFourier: two hollow-mean passes (27 each), IsolatedPoints (1), Expand 13 (6)
LOAD_REAL, LOAD_C64, LOAD_MASKED, LOAD_HPAIR = 0, 1, 2, 3


class _Trace:
    """HD_BAND_TRACE=1: per-phase host and device times of the banded chain (tools/band_phases.py prints them)."""

    def __init__(self):
        import os
        self.on = bool(os.environ.get("HD_BAND_TRACE"))
        self.marks = []

    def mark(self, name):
        if self.on:
            import time
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.marks.append((name, time.perf_counter(), ev))

    def report(self):
        torch.cuda.synchronize()
        out = []
        for (n0, t0, e0), (n1, t1, e1) in zip(self.marks, self.marks[1:]):
            out.append((n1, (t1 - t0) * 1e3, e0.elapsed_time(e1)))
        self.marks = []
        return out


TRACE = _Trace()


def band_bounds(n, world, align=1):
    """Row range [r0, r1) of every rank; starts are multiples of ``align``; sizes differ by at most ``align``."""
    n, world, align = int(n), int(world), int(align)
    units = -(-n // align)
    base, rem = divmod(units, world)
    out, u = [], 0
    for k in range(world):
        c = base + (1 if k < rem else 0)
        out.append((min(n, u * align), min(n, (u + c) * align)))
        u += c
    return out


# ---- communicators -------------------------------------------------------------------------------------------------
class DistComm:
    """Point-to-point exchange over torch.distributed (NCCL on GPUs, gloo on CPU)."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist = dist
        self.group = group
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)

    def p2p(self, sends, recvs):
        """sends: [(contiguous tensor, dst rank)], recvs: [(contiguous tensor, src rank)].  Messages between one pair of
        ranks are matched in posting order.  One grouped batch: NCCL fuses it into a single kernel over NVLink, on its
        own stream."""
        dist = self.dist
        local = [t for t, d in sends if d == self.rank]
        ops = []
        for t, s in recvs:
            if s == self.rank:
                t.copy_(local.pop(0))
            else:
                ops.append(dist.P2POp(dist.irecv, t, s, self.group))
        for t, d in sends:
            if d != self.rank:
                ops.append(dist.P2POp(dist.isend, t, d, self.group))
        for w in dist.batch_isend_irecv(ops) if ops else []:
            w.wait()                            # NCCL: the current stream waits for the transfer, the host does not

    def allreduce_max_(self, t):
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX, group=self.group)
        return t

    same_process = False

    def gather_objects(self, obj):
        out = [None] * self.world
        self.dist.all_gather_object(out, obj, group=self.group)
        return out

    def device_barrier(self):
        """Stream-ordered barrier: kernels launched after it start only when every rank's earlier kernels are done."""
        if not hasattr(self, "_bar"):
            self._bar = torch.zeros(1, dtype=torch.int32,
                                    device="cuda" if self.dist.get_backend(self.group) == "nccl" else "cpu")
        self.dist.all_reduce(self._bar, group=self.group)


class ThreadComm:
    """Emulates ``world`` ranks as threads of one process (one GPU): the banded algorithms are tested against the
    single-GPU path without several devices.  ``ThreadComm.run(world, fn)`` starts fn(comm) per rank."""

    class _Shared:
        def __init__(self, world):
            self.world = world
            self.barrier = threading.Barrier(world)
            self.box = {}
            self.vals = [None] * world

    def __init__(self, shared, rank):
        self.shared, self.rank, self.world = shared, rank, shared.world

    def p2p(self, sends, recvs):
        sh = self.shared
        if torch.cuda.is_available():
            torch.cuda.synchronize()
        for t, d in sends:
            sh.box.setdefault((self.rank, d), []).append(t.clone())
        sh.barrier.wait()
        for t, s in recvs:
            src = sh.box[(s, self.rank)].pop(0)
            assert tuple(src.shape) == tuple(t.shape), (tuple(src.shape), tuple(t.shape))
            t.copy_(src)
        if torch.cuda.is_available():
            torch.cuda.synchronize()
        sh.barrier.wait()

    same_process = True

    def gather_objects(self, obj):
        sh = self.shared
        sh.vals[self.rank] = obj
        sh.barrier.wait()
        out = list(sh.vals)
        sh.barrier.wait()
        return out

    def device_barrier(self):
        if torch.cuda.is_available():
            torch.cuda.synchronize()
        self.shared.barrier.wait()

    def allreduce_max_(self, t):
        sh = self.shared
        if torch.cuda.is_available():
            torch.cuda.synchronize()
        sh.vals[self.rank] = t.clone()
        sh.barrier.wait()
        out = torch.stack(sh.vals).max(dim=0).values
        sh.barrier.wait()
        t.copy_(out)
        return t

    @staticmethod
    def run(world, fn):
        shared = ThreadComm._Shared(world)
        results, errors = [None] * world, []
        device = torch.cuda.current_device() if torch.cuda.is_available() else None

        def work(rank):
            try:
                if device is not None:
                    torch.cuda.set_device(device)
                results[rank] = fn(ThreadComm(shared, rank))
            except BaseException as exc:           # noqa: BLE001
                errors.append(exc)
                shared.barrier.abort()

        threads = [threading.Thread(target=work, args=(r,)) for r in range(world)]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]
        return results


# ---- row redistribution between two layouts ----------------------------------------------------------------------------
def _runs(src_ids, dst_ids):
    """Maximal runs that are contiguous in BOTH id lists: [(src_lo, dst_lo, length)], ordered by dst position."""
    src_ids, dst_ids = np.asarray(src_ids, dtype=np.int64), np.asarray(dst_ids, dtype=np.int64)
    if len(src_ids) == 0 or len(dst_ids) == 0:
        return []
    where = np.full(int(max(src_ids.max(), dst_ids.max())) + 2, -1, dtype=np.int64)
    where[src_ids] = np.arange(len(src_ids))
    p = where[dst_ids]                                   # source position of every wanted row, -1 = held elsewhere
    k = np.nonzero(p >= 0)[0]
    if len(k) == 0:
        return []
    brk = np.nonzero((np.diff(k) != 1) | (np.diff(p[k]) != 1))[0] + 1
    starts = np.concatenate([[0], brk])
    ends = np.concatenate([brk, [len(k)]])
    return [(int(p[k[a]]), int(k[a]), int(b - a)) for a, b in zip(starts, ends)]


_PLAN_CACHE = {}


def redistribute_rows(comm, src, src_ids, dst_ids, dst, key=None):
    """Move rows between two layouts of the same global row set.  src / dst: 2-D tensors (local rows x cols, a row is
    contiguous); src_ids[r] / dst_ids[r]: the global row ids rank r holds / wants, in local order (the same lists on
    every rank).  A global row may be wanted by several ranks (halos) but is held by exactly one.  ``key``: caches the
    message plan (the layouts of a mosaic shape do not change from step to step)."""
    me = comm.rank
    plan = _PLAN_CACHE.get((key, me, comm.world)) if key is not None else None
    if plan is None:
        plan = ([(s0, ln, j) for j in range(comm.world) for s0, _, ln in _runs(src_ids[me], dst_ids[j])],
                [(d0, ln, i) for i in range(comm.world) for _, d0, ln in _runs(src_ids[i], dst_ids[me])])
        if key is not None:
            _PLAN_CACHE[(key, me, comm.world)] = plan
    comm.p2p([(src[s0:s0 + ln], j) for s0, ln, j in plan[0]], [(dst[d0:d0 + ln], i) for d0, ln, i in plan[1]])
    return dst


def _cview(t):
    """complex64 tensor -> float32 view with a trailing dimension of 2 (what the communicators move)."""
    return torch.view_as_real(t) if t.is_complex() else t


# ---- geometry of the sharded Fourier stage (host only) --------------------------------------------------------------------
def k_layouts(ny, world):
    """Per rank: spectrum rows ky in [a, b) plus their mirrors ("K layout", hd_klayout_*): dict(a, b, rows, nlo, nhi, hlo,
    ky = the ky of every local row)."""
    lib = _lib.load()
    out = []
    for a, b in band_bounds(ny // 2 + 1, world, 1):
        n = int(lib.hd_klayout_rows(a, b, ny))
        nlo = b - a
        nhi = n - nlo
        hlo = int(lib.hd_klayout_ky(a, b, ny, nlo)) if nhi else 0
        out.append(dict(a=a, b=b, rows=n, nlo=nlo, nhi=nhi, hlo=hlo,
                        ky=np.concatenate([np.arange(a, b), np.arange(hlo, hlo + nhi)]).astype(np.int64)))
    return out


class Exchange(typing.NamedTuple):
    """One pass of the sharded Fourier stage: every rank transforms its local rows and transposes the result T (one row
    per frequency / pixel of the transformed axis, one column per local row); T then changes hands.
      ranges[j]   row ranges of T that rank j holds, concatenated in this order in its buffer ``dest``
      colsegs[i]  [(local row0, column0, length)]: where rank i's local rows land along the ``cols`` columns of ``dest``;
                  they cover rank i's rows 0 .. n_i - 1 of the pass, so they also say how many rows it transforms"""
    ranges: list
    colsegs: list
    dest: str
    cols: int


def fourier_exchanges(ny, nx, bounds):
    """The K layouts and the four exchanges {"F1", "F2", "I1", "I2"} of DetectApplyFourier on row bands ``bounds``."""
    W = len(bounds)
    nh = nx // 2 + 1
    odd = bool((ny & 1) and (nx & 1))
    CB, XB = band_bounds(nh, W, 1), band_bounds(nx, W, 2)
    KL = k_layouts(ny, W)

    def spans(bb):                                       # rank i's rows land at the columns of its own band bb[i]
        return [[(0, a, b - a)] for a, b in bb]

    return KL, {
        # forward along x (two real rows per transform, half spectrum kept): my columns of the half spectrum, all y
        "F1": Exchange([[c] for c in CB], spans(bounds), "at", ny),
        # forward along y into the K layout: rank j gets rows ky in [a_j, b_j) and their mirrors
        "F2": Exchange([[(k["a"], k["b"]), (k["hlo"], k["hlo"] + k["nhi"])] for k in KL], spans(CB), "half", nh),
        # inverse along x of (1 - mask) * F on my spectrum rows (the Hermitian, odd x odd, path needs only ky <= ny/2;
        # hd_conj_mirror_fill writes the other columns): my x columns, all ky
        "I1": Exchange([[x] for x in XB],
                       [[(0, k["a"], k["nlo"])] + ([(k["nlo"], k["hlo"], k["nhi"])] if k["nhi"] and not odd else [])
                        for k in KL], "bt", ny),
        # inverse along y, real output (two columns per transform on the Hermitian path): my rows, all x
        "I2": Exchange([[r] for r in bounds], spans(XB), "dem", nx),
    }


# ---- peer memory: persistent exchange buffers every rank can store into ---------------------------------------------------
class PeerBuffers:
    """Named device buffers of this rank, living in ONE allocation that the other ranks have mapped (CUDA IPC; ranks that
    are threads of one process simply share the pointers).  ``ptr(rank, name)`` is valid in this process's kernels."""

    def __init__(self, comm, sizes):
        lib = _lib.load()
        self.comm = comm
        self.offsets, total = {}, 0
        for name, nbytes in sizes.items():
            self.offsets[name] = total
            total += (int(nbytes) + 255) // 256 * 256
        self.arena = torch.empty(max(total, 256), dtype=torch.uint8, device=dev.device())
        base = self.arena.data_ptr()
        self.ok = True
        if comm.same_process:
            infos = comm.gather_objects((base, self.offsets))
            self.bases = [b for b, _ in infos]
        else:
            # every rank runs the same sequence of collectives whatever fails locally; `ok` is agreed on at the end
            handle = ctypes.create_string_buffer(64)
            off = ctypes.c_int64(0)
            mine = None
            if lib.hd_ipc_export(ctypes.c_void_p(base), handle, ctypes.byref(off)) == _lib.HD_OK:
                mine = (handle.raw, off.value, self.offsets)
            infos = comm.gather_objects(mine if mine is not None else (None, 0, self.offsets))
            self.bases, self._opened = [], []
            good = mine is not None and all(i[0] is not None for i in infos)
            for j, (raw, off_j, _) in enumerate(infos):
                if j == comm.rank or not good:
                    self.bases.append(base)
                    continue
                p = ctypes.c_void_p()
                if lib.hd_ipc_import(ctypes.create_string_buffer(raw, 64), ctypes.byref(p)) != _lib.HD_OK:
                    good = False
                    self.bases.append(base)
                    continue
                self._opened.append(p)
                self.bases.append(p.value + off_j)
            self.ok = all(comm.gather_objects(bool(good)))
        self.peer_offsets = [info[-1] for info in infos]

    def ptr(self, rank, name):
        return self.bases[rank] + self.peer_offsets[rank][name]

    def view(self, name, rows, cols, dtype):
        """This rank's buffer ``name`` as a dense DeviceRaster."""
        tdt = {_lib.C64: torch.complex64, _lib.F32: torch.float32, _lib.U8: torch.uint8}[dtype]
        n = int(rows) * int(cols) * torch.empty(0, dtype=tdt).element_size()
        o = self.offsets[name]
        t = self.arena[o:o + max(n, 0)].view(tdt).view(int(rows), int(cols)) if rows and cols else \
            torch.empty((1, int(cols)), dtype=tdt, device=self.arena.device)
        return dev.DeviceRaster(t, rows, cols, dtype)

    def close(self):
        lib = _lib.load()
        for p in getattr(self, "_opened", []):
            lib.hd_ipc_close(p)
        self._opened = []


# ---- one rank's view of the mosaic --------------------------------------------------------------------------------------
class ExtRaster:
    """A band with its halo margins: ``raster`` has up + rows + down rows; rows [up, up + rows) are owned."""

    def __init__(self, raster, up, rows, down):
        self.raster, self.up, self.rows, self.down = raster, up, rows, down

    def owned(self):
        r = self.raster
        return r.sub(self.up, self.up + self.rows, 0, r.nx)

    def with_halo(self, h):
        """View of the owned rows plus h halo rows (fewer at the ends of the mosaic)."""
        r = self.raster
        u, d = min(h, self.up), min(h, self.down)
        return r.sub(self.up - u, self.up + self.rows + d, 0, r.nx), u, d


class Band:
    """One rank's view of the mosaic."""

    def __init__(self, comm, ny, nx, halo=HALO):
        self.comm, self.ny, self.nx, self.halo = comm, int(ny), int(nx), int(halo)
        # band starts are multiples of 8: even (two rows share one transform on the device) and aligned with the 8x8 blocks
        # of the sink-fill's coarse level (a block never straddles a cut)
        self.bounds = band_bounds(ny, comm.world, 8)
        self.r0, self.r1 = self.bounds[comm.rank]
        if comm.world > 1 and min(b - a for a, b in self.bounds) < self.halo:
            # the same test on every rank (it only depends on ny and world): nobody enters a collective alone
            raise ValueError(f"{ny} rows over {comm.world} ranks leave bands thinner than the {self.halo}-row halo")
        import os
        self.fill_overlap = max(8, int(os.environ.get("HD_FILL_OVERLAP", "64")) // 8 * 8)
        from .pipeline import narrow_final_default
        self.narrow_final = narrow_final_default()                       # apply_to_host: final DEM down as int16
        if comm.world > 1 and min(b - a for a, b in self.bounds) < 2 * self.fill_overlap:
            self.fill_overlap = max(8, min(b - a for a, b in self.bounds) // 16 * 8)
        self.up, self.down = self._margins(comm.rank)
        self.fill_rounds = None

    def _margins(self, rank):
        """Halo rows above / below the band of ``rank`` (none at the ends of the mosaic)."""
        return (self.halo if rank > 0 else 0), (self.halo if rank < self.comm.world - 1 else 0)

    @property
    def rows(self):
        return self.r1 - self.r0

    def take(self, mosaic):
        """This rank's rows of a host mosaic (tests / loaders)."""
        return np.ascontiguousarray(mosaic[self.r0:self.r1])

    # -- halo plumbing ------------------------------------------------------------------------------------------------
    def alloc_ext(self, dtype, ref_dtype=None):
        """Uninitialised extended raster [halo | band | halo] (no halo at the ends of the mosaic)."""
        r = dev.empty(self.up + self.rows + self.down, self.nx, dtype, ref_dtype)
        return ExtRaster(r, self.up, self.rows, self.down)

    def exchange_halo(self, ext, h=None):
        """Fill the margin rows of ``ext`` with the neighbours' edge rows: sends / receives whole pitched rows straight
        from / into the buffer (a row range of a pitched raster is contiguous)."""
        h = self.halo if h is None else int(h)
        buf, up, rows = ext.raster.buf, ext.up, ext.rows
        y0 = ext.raster._y0
        sends, recvs = [], []
        if ext.up:
            sends.append((buf[y0 + up:y0 + up + h], self.comm.rank - 1))
            recvs.append((buf[y0 + up - h:y0 + up], self.comm.rank - 1))
        if ext.down:
            sends.append((buf[y0 + up + rows - h:y0 + up + rows], self.comm.rank + 1))
            recvs.append((buf[y0 + up + rows:y0 + up + rows + h], self.comm.rank + 1))
        self.comm.p2p([(_cview(t), d) for t, d in sends], [(_cview(t), s) for t, s in recvs])
        return ext

    def extended(self, raster):
        """Extended copy of a band raster (inputs: done once per input, not per stage) with the halo exchanged."""
        ext = self.alloc_ext(raster.dtype, raster.ref_dtype)
        ext.owned().tensor().copy_(raster.tensor())
        return self.exchange_halo(ext)

    def apply(self, filt, raster, h):
        """Run a single-GPU filter (anything with ``run_device``) on the band with an h-row halo; returns the band's
        rows of the result."""
        ext = self.extended(raster)
        view, u, _ = ext.with_halo(h)
        out = filt.run_device(view)
        return out.sub(u, u + self.rows, 0, raster.nx)

    # -- the Fourier stage ------------------------------------------------------------------------------------------------
    def _dense(self, rows, cols, dtype):
        tdt = {_lib.C64: torch.complex64, _lib.F32: torch.float32, _lib.U8: torch.uint8}[dtype]
        return dev.DeviceRaster(torch.empty((max(int(rows), 1), int(cols)), dtype=tdt, device=dev.device()), rows, cols, dtype)

    def _fourier_setup(self):
        """The K layouts and exchanges of the Fourier stage, and its persistent exchange buffers in peer-mapped memory
        (``self._peers``; once per Band).  No peers: the ranks could not map each other's memory (or HD_BAND_DIRECT=0)
        -- the exchanges then go through NCCL send / recv."""
        if not hasattr(self, "_fourier"):
            import os
            self._fourier = fourier_exchanges(self.ny, self.nx, self.bounds)
            self._peers = None
            if self.comm.world > 1 and os.environ.get("HD_BAND_DIRECT", "1") != "0":
                sizes = {}
                for ex in self._fourier[1].values():
                    rows, pitch, _, itemsize = self._buffer_shape(ex, self.comm.rank)
                    sizes[ex.dest] = rows * pitch * itemsize
                peers = PeerBuffers(self.comm, sizes)
                if peers.ok:
                    self._peers = peers
        return self._fourier

    def _buffer_shape(self, ex, rank):
        """Buffer ``ex.dest`` of ``rank``: (rows, pitch in elements, first row the exchange writes, bytes per element).
        "dem" is the stripe-free DEM with the band's halo margins (the layout of ``alloc_ext``); the others are dense."""
        rows = sum(b - a for a, b in ex.ranges[rank])
        if ex.dest != "dem":
            return rows, ex.cols, 0, 8
        up, down = self._margins(rank)
        return up + rows + down, int(_lib.load().hd_pitch_elems(self.nx, _lib.F32)), up, 4

    def _buffer(self, ex):
        """This rank's buffer ``ex.dest`` (a view of the peer arena, else a new allocation; an ExtRaster for "dem") and,
        when the ranks store into each other's memory, every rank's (address of the first written row, pitch)."""
        rows, pitch, _, _ = self._buffer_shape(ex, self.comm.rank)
        dtype = _lib.F32 if ex.dest == "dem" else _lib.C64
        peers, targets = self._peers, None
        if peers is None:
            buf = self._dense(rows, pitch, dtype)
        else:
            buf = peers.view(ex.dest, rows, pitch, dtype)
            targets = []
            for j in range(self.comm.world):
                _, pitch_j, first_j, itemsize = self._buffer_shape(ex, j)
                targets.append((peers.ptr(j, ex.dest) + first_j * pitch_j * itemsize, pitch_j))
        buf = buf.sub(0, rows, 0, ex.cols)
        if ex.dest == "dem":
            buf = ExtRaster(buf.with_ref(np.float64), self.up, self.rows, self.down)
        return buf, targets

    def _exchange(self, plan, axis, load, src, ex, keep_cols=0, mask=None, shift_cols=0, inverse=0, real_out=0):
        """One pass of the sharded Fourier stage: the row transforms of this rank's rows of ``src`` (hd_fft_band_pass,
        ``load`` and the keywords as there), then exchange ``ex`` of the transposed result.  Returns the buffer
        ``ex.dest``.  With peer-mapped buffers the transpose stores every element straight into the memory of the rank
        that owns it (hd_fft_band_pass_scatter) and a device barrier follows ("all stores landed"); otherwise the
        transposed block goes out by send / recv and the blocks received are put in place.  Every rank takes part in
        the barrier / the send / recv, with or without rows of its own."""
        lib = _lib.load()
        comm, W, me = self.comm, self.comm.world, self.comm.rank
        n = self.nx if axis == 0 else self.ny
        nrows = [max((l0 + ln for l0, _, ln in segs), default=0) for segs in ex.colsegs]
        out, targets = self._buffer(ex)
        mp, mpitch = (mask.ptr, mask.pitch) if mask is not None else (None, 0)

        def band_pass(fn, *out_args):                  # out_args: (out_t, out_t pitch) or (hd_scatter*,)
            nbytes = int(lib.hd_fft_band_workspace_bytes(nrows[me], n))
            work = dev.scratch(nbytes)
            _lib.check(fn(plan, axis, load, src.ptr, src.pitch, nrows[me], mp, mpitch, int(shift_cols), int(inverse),
                          int(real_out), *out_args, int(keep_cols), ctypes.c_void_p(work.data_ptr()), nbytes,
                          dev.stream_ptr()))

        if targets is not None:
            # segment = a row range of T in one rank's buffer, at its offset in that rank's concatenation
            sc = _lib.Scatter()
            for j, (ptr, pitch) in enumerate(targets):
                off = 0
                for a, b in ex.ranges[j]:
                    if b > a:
                        sc.seg[sc.nseg] = _lib.ScatterSeg(a, b, ptr, pitch, off)
                        sc.nseg += 1
                    off += b - a
            for l0, c0, ln in ex.colsegs[me]:
                sc.col_local0[sc.ncolseg], sc.col_dst0[sc.ncolseg], sc.col_len[sc.ncolseg] = l0, c0, ln
                sc.ncolseg += 1
            if nrows[me]:
                band_pass(lib.hd_fft_band_pass_scatter, ctypes.byref(sc))
            comm.device_barrier()
            return out
        region = out.owned() if isinstance(out, ExtRaster) else out
        sends = []
        if nrows[me]:
            t = self._dense(keep_cols or n, nrows[me], region.dtype)
            band_pass(lib.hd_fft_band_pass, t.ptr, t.pitch)
            tt = t.tensor()
            sends = [(_cview(tt[a:b]), j) for j in range(W) for a, b in ex.ranges[j] if b > a]
        to = region.tensor()
        recvs, places = [], []
        for i in range(W):
            off = 0
            for a, b in ex.ranges[me]:
                if b > a and nrows[i]:
                    buf = torch.empty((b - a, nrows[i]), dtype=to.dtype, device=to.device)
                    recvs.append((_cview(buf), i))
                    places.append((buf, off, i))
                off += b - a
        comm.p2p(sends, recvs)
        for buf, off, i in places:
            for l0, c0, ln in ex.colsegs[i]:
                to[off:off + buf.shape[0], c0:c0 + ln].copy_(buf[:, l0:l0 + ln])
        return out

    def detect_apply_fourier(self, srtm):
        """DetectApplyFourier (custom_filters.py:1053-1101) on a banded mosaic.  ``srtm``: F32 device raster of this
        rank's rows.  Returns an ExtRaster (F32 storage, float64 reference dtype) whose owned rows hold the stripe-free
        DEM -- bit-identical to ``DetectApplyFourier().run_device`` on the whole mosaic; its halo rows are NOT filled."""
        from .filters import custom_filters as cf
        lib = _lib.load()
        comm, W, me = self.comm, self.comm.world, self.comm.rank
        ny, nx = self.ny, self.nx
        nh = nx // 2 + 1
        odd = bool((ny & 1) and (nx & 1))
        KL, ex = self._fourier_setup()
        kl = KL[me]
        plan = dev.fft_plan(ny, nx)
        src = dev.convert(srtm, _lib.F32)

        TRACE.mark("daf:start")
        if self._peers is not None:
            comm.device_barrier()          # destinations free: no rank still reads its buffers of the last call
        at = self._exchange(plan, 0, LOAD_REAL, src, ex["F1"], keep_cols=nh)
        TRACE.mark("F1 rows + T1")
        half = self._exchange(plan, 1, LOAD_C64, at, ex["F2"])
        del at
        TRACE.mark("F2 cols + T2")
        # conjugate half, column shift, |F|  (FourierInitial, custom_filters.py:859-877)
        nk = kl["rows"]
        fshift = self._dense(nk, nx, _lib.C64)
        fabs = self._dense(nk, nx, _lib.F32)
        _lib.check(lib.hd_hermitian_complete(half.ptr, half.pitch, fshift.ptr, fshift.pitch, fabs.ptr, fabs.pitch, kl["a"],
                                             kl["b"], ny, nx, dev.stream_ptr()))
        del half
        TRACE.mark("hermitian complete")

        # ---- peak detector on row slabs of the two upper quarters (FourierProcessQuarters, :880-1050) -------------
        my, y_odd, mx, x_odd = ny // 2, ny & 1, nx // 2, nx & 1
        m = cf.FOURIER_MARGIN
        qh, qw = my - m, mx - m
        cf.check_window((qh, qw), cf.BLANKS_WINDOW)
        shifted = [(k["ky"] + ny // 2) % ny for k in KL]            # shifted row id of every local K row, per rank
        # a rank's slab = the quarter rows it already owns (its mirror rows are a contiguous range of the upper half):
        # only the 61 rows of context on either side have to travel
        SL = []
        for sh in shifted:
            q = np.sort(sh[sh < qh])
            SL.append((int(q[0]), int(q[-1]) + 1) if len(q) and q[-1] - q[0] + 1 == len(q) else None)
        if any(x is None for x in SL) or sorted(SL) != sorted(set(SL)) or sum(b - a for a, b in SL) != qh \
                or min(b - a for a, b in SL) < 16:
            SL = band_bounds(qh, W, 1)
            if min(b - a for a, b in SL) < 16:                       # tiny quarters: one rank runs the detector
                SL = [(0, qh)] + [(qh, qh)] * (W - 1)
        ctx = [(max(0, a - MASK_HALO), min(qh, b + MASK_HALO)) if b > a else (0, 0) for a, b in SL]
        slab_ids = [np.arange(lo, hi) for lo, hi in ctx]
        s0, s1 = SL[me]
        lo, hi = ctx[me]
        masks = []
        slab = self._dense(hi - lo, nx, _lib.F32)
        redistribute_rows(comm, fabs.tensor(), shifted, slab_ids, slab.tensor()[:hi - lo], key=("fabs", ny, nx))
        TRACE.mark("fabs to slabs")
        x0 = mx + m + x_odd
        for (xa, xb) in ((0, qw), (x0, nx)):
            own = self._dense(s1 - s0, qw, _lib.U8)
            if hi > lo:
                q = dev.empty(hi - lo, qw, _lib.F32)
                dev.elementwise(_lib.OP_COPY, slab.sub(0, hi - lo, xa, xb), None, q)
                mk = dev.convert(cf.MaskFourier().run_device(q), _lib.U8)
                own.tensor().copy_(mk.tensor()[s0 - lo:s1 - lo])
            masks.append(own)
        del slab
        TRACE.mark("peak detector")
        # the quarter-mask rows each rank's K rows look at (point mirror for the lower half, :1002-1027)
        need = []
        for sh in shifted:
            top = sh < my
            by = np.where(top, sh, sh - my - y_odd)
            qy = np.where(top, by, my - 1 - by)
            ok = (by >= 0) & (qy >= 0) & (qy < qh)
            need.append((int(qy[ok].min()), int(qy[ok].max()) + 1) if ok.any() else (0, 0))
        own_ids = [np.arange(a, b) for a, b in SL]
        need_ids = [np.arange(a, b) for a, b in need]
        q0, q1 = need[me]
        loc = []
        for own in masks:
            mloc = self._dense(q1 - q0, qw, _lib.U8)
            redistribute_rows(comm, own.tensor()[:s1 - s0], own_ids, need_ids, mloc.tensor()[:q1 - q0], key=("qmask", ny, nx))
            loc.append(mloc)
        mask = self._dense(nk, nx, _lib.U8)
        _lib.check(lib.hd_fourier_mask_assemble_rows(loc[0].ptr, loc[0].pitch, loc[1].ptr, loc[1].pitch, q0, q1 - q0,
                                                     mask.ptr, mask.pitch, nk, kl["a"], kl["b"], ny, nx, m,
                                                     dev.stream_ptr()))
        self._last_mask = (mask, kl)
        TRACE.mark("mask back + assemble")

        # ---- inverse: along x (1 - mask) * F, then along y with real output ----------------------------------------
        bt = self._exchange(plan, 0, LOAD_MASKED, fshift, ex["I1"], mask=mask, shift_cols=nx // 2, inverse=1)
        del fshift
        TRACE.mark("I1 rows + T3")
        if odd:
            _lib.check(lib.hd_conj_mirror_fill(bt.ptr, bt.pitch, bt.ny, ny, dev.stream_ptr()))
        dem = self._exchange(plan, 1, LOAD_HPAIR if odd else LOAD_C64, bt, ex["I2"], inverse=1, real_out=1)
        del bt
        TRACE.mark("I2 cols + T4")
        return dem

    # -- the whole chain on row bands (BASELINE.json configs[4]: one mosaic over the GPUs of a box) --------------------
    def conditioning_chain(self, srtm, groves_class, hsheds, groves_iterations=3, with_hydrology=True, keep_complete=False,
                           ready=None, on_ready=None):
        """HydroDEMProcess.start (hydro_dem_process.py:122-153) on this rank's rows of a mosaic.  Inputs: device rasters
        of the band's rows (F32, U8 0/1, F32), or ExtRaster objects whose owned rows are already in place (groves,
        hsheds: saves the input copy).  Returns {"final", "dem_complete", "filled", "d8"} for the band's rows -- every
        one of them bit-identical to the single-GPU ConditioningChain on the whole mosaic."""
        from .pipeline import ConditioningChain
        chain = ConditioningChain(groves_iterations=groves_iterations, with_hydrology=False, keep_complete=keep_complete)
        TRACE.mark("chain:start")
        g_ext = groves_class if isinstance(groves_class, ExtRaster) else self.extended(dev.convert(groves_class, _lib.U8))
        h_ext = hsheds if isinstance(hsheds, ExtRaster) else self.extended(hsheds)
        cur = torch.cuda.current_stream()

        def input_halo(name, ext, given):
            if ready and ready.get(name) is not None:
                cur.wait_event(ready[name])               # its upload ran underneath the stages before
            if given is ext:
                self.exchange_halo(ext)

        if ready is None:
            input_halo("groves", g_ext, groves_class)
            input_halo("hsheds", h_ext, hsheds)
            TRACE.mark("input halos")
        elif ready.get("srtm") is not None:
            cur.wait_event(ready["srtm"])
        dem = self.detect_apply_fourier(srtm)                                        # image_srtm.py:125-126
        st = {"fourier": dem.raster}
        if ready is not None:
            input_halo("hsheds", h_ext, hsheds)
        chain._stage_lagoons(st, h_ext.raster)                                       # LagoonsDetection: HydroSHEDS only
        TRACE.mark("lagoons")
        if ready is not None:
            input_halo("groves", g_ext, groves_class)
        self.exchange_halo(dem)
        TRACE.mark("dem halo")
        chain._stage_groves(st, g_ext.raster)                                        # image_srtm.py:177-199
        TRACE.mark("groves")
        chain._stage_final(st, None)                                                 # final terms ... :149
        TRACE.mark("combine")
        own = lambda r: r.sub(self.up, self.up + self.rows, 0, self.nx)              # noqa: E731
        out = {"final": own(st["final"])}
        if on_ready:
            on_ready("final", out["final"])
        if keep_complete:
            out["dem_complete"] = own(st["dem_complete"])
        if with_hydrology:
            out["filled"], out["d8"] = self.sinkfill(ExtRaster(st["final32"], self.up, self.rows, self.down))
            TRACE.mark("sink-fill + D8")
            if on_ready:
                on_ready("filled", out["filled"])
                on_ready("d8", out["d8"])
        return out

    # -- sink-fill + D8 -----------------------------------------------------------------------------------------------------
    def sinkfill(self, z, max_rounds=10000):
        """Banded Planchon-Darboux fixed point + D8 (bit-identical to the single-GPU result).  ``z``: F32 device raster
        of the band's rows, or an ExtRaster whose owned rows hold them (its margin rows are overwritten)."""
        lib = _lib.load()
        comm = self.comm
        # The bands OVERLAP by FILL_OVERLAP rows on either side of a cut (an alternating Schwarz iteration converges in far
        # fewer rounds with overlap: a drainage path has to wander that many rows across a cut before it costs another
        # round).  The outermost row of the extended band is the boundary row received from the neighbour; the rows in
        # between are relaxed by both ranks and agree at the fixed point.
        ov = self.fill_overlap if comm.world > 1 else 1
        src = z.owned() if isinstance(z, ExtRaster) else dev.convert(z, _lib.F32)
        up, down = (ov if comm.rank > 0 else 0), (ov if comm.rank < comm.world - 1 else 0)
        zx = ExtRaster(dev.empty(up + self.rows + down, self.nx, _lib.F32, np.float32), up, self.rows, down)
        zx.owned().tensor().copy_(src.tensor())
        z = zx
        self.exchange_halo(z, ov)
        zv, n_up, n_down = z.with_halo(ov)
        rows, nx = self.rows, self.nx
        w = dev.empty(zv.ny, nx, _lib.F32, np.float32)
        d8 = dev.empty(zv.ny, nx, _lib.U8, np.uint8)
        nbytes = lib.hd_pdfill_workspace_bytes(zv.ny, nx)
        work = dev.scratch(nbytes)
        wp = ctypes.c_void_p(work.data_ptr())
        flags = (2 if n_up else 0) | (4 if n_down else 0)          # halo rows are not raster frame
        lowered = torch.zeros(1, dtype=torch.int32, device=dev.device())
        tw = w.tensor()
        recv_up = torch.empty(nx, dtype=torch.float32, device=dev.device()) if n_up else None
        recv_down = torch.empty(nx, dtype=torch.float32, device=dev.device()) if n_down else None
        rounds = 0
        TRACE.mark("fill: overlap exchange")
        # global multigrid start: pool my band, all-gather the coarse DEM, fill the whole coarse mosaic on every rank
        nyc, nxc = -(-self.ny // 8), -(-nx // 8)
        cp = (nxc + 31) // 32 * 32
        zc_g = torch.empty((nyc, cp), dtype=torch.float32, device=dev.device())
        wc_g = torch.empty((nyc, cp), dtype=torch.float32, device=dev.device())
        cb = [(a // 8, -(-b // 8)) for a, b in self.bounds]
        c0, c1 = cb[comm.rank]
        scratch = torch.zeros(((c1 - c0) // 64 + 2) * (nxc // 64 + 2), dtype=torch.int32, device=dev.device())
        own = z.owned()
        _lib.check(lib.hd_fill_pool_band(own.ptr, own.pitch, rows, nx, ctypes.c_void_p(zc_g[c0].data_ptr()),
                                         ctypes.c_void_p(wc_g[c0].data_ptr()), cp, flags,
                                         ctypes.c_void_p(scratch.data_ptr()), dev.stream_ptr()))
        for g in (zc_g, wc_g):
            comm.p2p([(g[c0:c1], j) for j in range(comm.world) if j != comm.rank],
                     [(g[a:b], i) for i, (a, b) in enumerate(cb) if i != comm.rank])
        cbytes = lib.hd_pdfill_workspace_bytes(nyc, nxc)
        cwork = dev.scratch(cbytes)
        _lib.check(lib.hd_pdfill_coarse(ctypes.c_void_p(zc_g.data_ptr()), ctypes.c_void_p(wc_g.data_ptr()), cp, nyc, nxc,
                                        ctypes.c_void_p(cwork.data_ptr()), cbytes, dev.stream_ptr()))
        TRACE.mark("fill: global coarse level")
        while True:
            if rounds == 0:
                _lib.check(lib.hd_pdfill_band_start(zv.ptr, zv.pitch, w.ptr, w.pitch, zv.ny, nx, wp, nbytes, flags,
                                                    ctypes.c_void_p(wc_g.data_ptr()), cp, self.r0 - n_up, dev.stream_ptr()))
            else:
                _lib.check(lib.hd_pdfill_band(zv.ptr, zv.pitch, w.ptr, w.pitch, zv.ny, nx, wp, nbytes, flags, None,
                                              dev.stream_ptr()))
            rounds += 1
            if comm.world == 1:
                break
            lowered.zero_()
            sends, recvs = [], []
            if n_up:                                               # my first / last OWNED rows go to the neighbours' halo rows
                sends.append((tw[2 * n_up - 1, :nx], comm.rank - 1))      # = the neighbour's last (boundary) row
                recvs.append((recv_up, comm.rank - 1))
            if n_down:
                sends.append((tw[n_up + rows - n_down, :nx], comm.rank + 1))   # = the neighbour's first (boundary) row
                recvs.append((recv_down, comm.rank + 1))
            comm.p2p(sends, recvs)
            lp = ctypes.c_void_p(lowered.data_ptr())
            if n_up:
                _lib.check(lib.hd_halo_min_flag(w.ptr, ctypes.c_void_p(recv_up.data_ptr()), nx, lp, dev.stream_ptr()))
            if n_down:
                last = w.sub(zv.ny - 1, zv.ny, 0, nx)
                _lib.check(lib.hd_halo_min_flag(last.ptr, ctypes.c_void_p(recv_down.data_ptr()), nx, lp, dev.stream_ptr()))
            comm.allreduce_max_(lowered)
            TRACE.mark(f"fill: round {rounds}")
            if int(lowered.item()) == 0:                           # the one host read of the round
                break
            if rounds >= max_rounds:
                raise dev.DeviceError("banded sink-fill did not converge")
        self.fill_rounds = rounds
        # at the fixed point a halo row equals the neighbour's owned row, so D8 needs no further exchange; NaN
        # restoration and the flow directions are one fused pass
        _lib.check(lib.hd_pdfill_finish_d8(zv.ptr, zv.pitch, w.ptr, w.pitch, d8.ptr, d8.pitch, zv.ny, nx, wp,
                                           dev.stream_ptr()))
        self._fill_work = work
        return w.sub(n_up, n_up + rows, 0, nx), d8.sub(n_up, n_up + rows, 0, nx)

    def fill_status(self):
        """Sticky status word of the last sinkfill on this rank (0 = fixed point reached)."""
        st = ctypes.c_int(-1)
        _lib.check(_lib.load().hd_pdfill_status(ctypes.c_void_p(self._fill_work.data_ptr()), ctypes.byref(st),
                                                dev.stream_ptr()))
        return st.value

    # -- host API: one rank's rows in, one rank's rows out --------------------------------------------------------------
    def apply_to_host(self, srtm_rows, groves_rows, hsheds_rows):
        """The banded chain through host buffers: this rank's rows of the three input mosaics (ndarrays: float32,
        uint8 / bool, float32; pinned memory is copied asynchronously) -> {"final" float64, "filled" float32, "d8" uint8}
        ndarrays of the same rows.  What bench.py's e2e measures at N > 1."""
        from .pipeline import copy_streams, overlapped_to_host
        for a in (srtm_rows, groves_rows, hsheds_rows):
            if not isinstance(a, np.ndarray):
                from .exceptions import NumpyArrayExpectedError
                raise NumpyArrayExpectedError(a)
            if a.shape != (self.rows, self.nx):
                raise ValueError(f"expected this rank's rows {(self.rows, self.nx)}, got {a.shape}")
        # the SRTM rows go up first, HydroSHEDS + groves follow underneath the Fourier stage, straight into the owned rows
        # of their extended rasters, and the final DEM travels down while the sink-fill rounds run
        g_ext, h_ext = self.alloc_ext(_lib.U8, np.uint8), self.alloc_ext(_lib.F32, np.float32)
        g = np.ascontiguousarray(groves_rows)
        inputs = [("srtm", np.ascontiguousarray(srtm_rows, dtype=np.float32), None),
                  ("hsheds", np.ascontiguousarray(hsheds_rows, dtype=np.float32), h_ext.owned()),
                  ("groves", g.view(np.uint8) if g.dtype == np.bool_ else g.astype(np.uint8, copy=False), g_ext.owned())]

        def run(rasters, ready, on_ready):
            self.conditioning_chain(rasters["srtm"], g_ext, h_ext, ready=ready, on_ready=on_ready)
            return self.fill_status

        out, self.last_transfer_bytes = overlapped_to_host(copy_streams(self), inputs, run, self.narrow_final)
        return out
