// NEW stages N2 / N3 -- sink-fill and D8 flow direction.  Neither exists in the reference (SURVEY.md 0.3):
// parity is against this repo's own oracle (oracle/hydrology.py, oracle/c/hydro_oracle.c), "parity unpinned".
//
// Sink-fill: fixed point of Planchon & Darboux (2001) with eps = 0 and 8-connectivity,
//     W = z on the raster frame, NaN cells are outlets (-inf while iterating, NaN in the result),
//     W(c) = max(z(c), min_{n in N8} W(n))  wherever that lowers W(c).
// The fixed point is unique (it is the minimax path elevation to an outlet), so any update order -- including
// the racy, in-place one used here -- converges to the same bits: the result does not depend on the
// schedule, the tile size or the number of GPUs.
//
// Kernels (DESIGN.md section 5):
//   fill_async_kernel   the default on one GPU and per band: persistent CTAs pull 64x64 tiles from a device-side FIFO,
//                       relax each to its local fixed point (check pass + four simultaneous marching sweeps) and poke
//                       exactly the neighbours whose cells can still be lowered;
//   fill_pool_kernel /  multigrid start: block maxima give coarse DEMs whose fill is an upper bound of the fine fill, so
//   fill_refine_kernel  every level starts from the level above instead of +inf (same result, no raster-crossing wave);
//   d8_kernel           flow directions of the filled surface (fill_finish_d8_kernel: the same decision, d8_code, fused
//                       with the fill's last pass).
//
// Algorithmic HBM traffic: 4 B (z) + 4 B (W) read + 4 B (W) written per cell of a visited tile.
#include <cstdio>
#include <cstdlib>

#include "common.cuh"
#include "tile_common.cuh"

namespace {

constexpr int FT = 64;                    // tile edge
constexpr int CB = 8;                     // block edge between two levels of the multigrid start of the fill (4: no fewer fine visits, one more level of latency)
constexpr int FNT = 256;
constexpr int WS_STRIDE = FT + 3;         // 67: odd stride -> row marches are bank-conflict free

__global__ void __launch_bounds__(256) fill_init_kernel(const float* __restrict__ z, int64_t z_pitch, float* __restrict__ w,
                                                        int64_t w_pitch, int64_t ny, int64_t nx, int top_is_halo = 0,
                                                        int bottom_is_halo = 0, int* __restrict__ tile_has_nodata = nullptr,
                                                        int tiles_x = 0, int* __restrict__ seen = nullptr,
                                                        const float* __restrict__ wc = nullptr, int64_t c_pitch = 0,
                                                        int64_t wc_y0 = 0)
{
    // seen[0] = 1: z holds a nodata cell, seen[1] = 1: z holds a -0.0 (what fill_finish_kernel has to rewrite)
    const int64_t nxq = (nx + 3) / 4;                                            // four consecutive cells per thread
    for (CellIter it(nxq); it.y < ny; it.next()) {
        const int64_t y = it.y, x0 = 4 * it.x;
        float v4[4], r4[4];
        gload4(z + y * z_pitch + x0, x0, nx, v4);
        // interior cells start from the coarse-level fill of their block (an upper bound of the answer, see
        // fill_pool_kernel) instead of +inf; a quad never straddles two blocks (CB is a multiple of 4)
        // (wc_y0: row of the coarse raster's frame of reference that local row 0 corresponds to -- a band of a mosaic
        // looks up the GLOBAL coarse fill)
        const float start = wc ? __ldg(wc + ((y + wc_y0) / CB) * c_pitch + x0 / CB) : __int_as_float(0x7f800000);
        const bool yframe = (y == 0 && !top_is_halo) || (y == ny - 1 && !bottom_is_halo);
        bool nodata = false, negzero = false;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int64_t x = x0 + j;
            const float v = v4[j];
            float r = start;                                                     // +inf (or the coarse bound) inside
            if (v != v) {
                r = __int_as_float(0xff800000);                                  // nodata: outlet at -inf
                nodata |= x < nx;
            }
            else if (yframe || x == 0 || x == nx - 1)
                r = v;                                                           // frame: W = z (a band's halo rows are not frame)
            negzero |= __float_as_uint(v) == 0x80000000u;                        // (cells past the row end read +0)
            r4[j] = r;
        }
        if (nodata) {                                                            // benign races: every writer stores 1
            if (tile_has_nodata) tile_has_nodata[(y / FT) * tiles_x + (x0 / FT)] = 1;
            if (seen) seen[0] = 1;
        }
        if (negzero && seen) seen[1] = 1;
        store4<float>(w, w_pitch, y, x0, nx, r4);
    }
}

__global__ void __launch_bounds__(256) fill_finish_kernel(const float* __restrict__ z, int64_t z_pitch,
                                                          float* __restrict__ w, int64_t w_pitch, int64_t ny, int64_t nx,
                                                          const int* __restrict__ seen = nullptr,
                                                          const int* __restrict__ status = nullptr,
                                                          const int* __restrict__ pending = nullptr)
{
    // Every zero of the result is +0.0: the racy update order decides which signed zero of z a cell takes first (a
    // candidate that only differs in the sign of zero never replaces it), so the sign is rewritten here.  W only ever
    // holds values of z and +-inf, so without a -0.0 in z (seen[1], fill_init_kernel) there is none to rewrite.
    const bool nodata = !seen || seen[0], negzero = !seen || seen[1];
    if (nodata || negzero) {
        for (CellIter it(nx); it.y < ny; it.next()) {
            const int64_t y = (int64_t)it.y, x = (int64_t)it.x;
            float* p = w + y * w_pitch + x;
            if (nodata) {
                const float v = z[y * z_pitch + x];
                if (v != v) { *p = v; continue; }                                // nodata stays nodata
            }
            if (negzero && __float_as_uint(*p) == 0x80000000u) *p = 0.f;
        }
    }
    // a fill that stalled must not pass for a result: poison the first cell (see STATUS_OFF) -- after the pass above,
    // in which this same thread handled that cell
    if (blockIdx.x == 0 && threadIdx.x == 0 && ((status && *status != 0) || (pending && *pending != 0)))
        w[0] = __int_as_float(0x7fc00000);
}

// ---- asynchronous worklist ----------------------------------------------------------------------------------------------
// A level-synchronous schedule needs one launch per "ring" of tiles the fill wave crosses (39 sweeps on a 3601^2 tile)
// and visits every active tile once per sweep.  Here a persistent grid of co-resident CTAs pulls tiles from a device-side
// FIFO: a tile that changed pushes exactly the neighbours whose halo it changed, so the wave advances as fast as single
// tiles finish and nothing waits for a grid-wide barrier.  Because the fixed point is unique, the (racy) order in which
// tiles are processed cannot change the result.
//   queue  : ring of tile ids; producers reserve a slot with atomicAdd(tail), consumers take tickets with
//            atomicAdd(head) and wait for "their" slot; `queued[tile]` de-duplicates; `pending` = tiles queued or in
//            flight, 0 means the global fixed point is reached.
//   memory : W is read with ld.global.cg (L2, never a stale L1 line) and written with plain stores followed by
//            __threadfence() before the neighbour is published.
//
// Memory-ordering argument of the poke / ticket protocol (compute-sanitizer is closed on the measurement pool, so the
// argument is written down here and the kernel is stress-tested against the CPU priority-flood oracle instead:
// tests/test_gpu_new_stages.py::test_fill_worklist_stress):
//   1. Single writer.  A tile's W cells are stored only by the CTA that holds the tile in state T_RUNNING; the state
//      moves IDLE -> QUEUED (poker, atomicCAS) -> RUNNING (the ticket holder, atomicExch) -> IDLE / QUEUED (the same CTA,
//      atomicCAS).  A poke that finds RUNNING turns it into DIRTY and the running CTA re-queues the tile itself, so two
//      CTAs never relax the same tile concurrently and a lowered W can never be overwritten by a stale higher value.
//   2. Publication.  The writer stores W, executes __threadfence() (release at device scope), and only then pokes the
//      neighbour (atomicCAS on its state + atomicAdd on `tail` + volatile store of the slot).  The consumer obtains the
//      tile id from the slot (volatile load in a spin loop), performs atomicExch(state, RUNNING) + __threadfence()
//      (acquire) and loads W with ld.global.cg.  Slot store -> slot load is the synchronises-with edge; the fences on
//      either side order the W stores before it and the W loads after it, so a visit triggered by a poke sees at least
//      the values that caused the poke.  (Seeing NEWER values is harmless: W only decreases towards the fixed point.)
//   3. Halo reads race by design.  A tile reads its neighbours' edge cells while they may be running.  Every value ever
//      stored in W is an upper bound of the fixed point and a candidate max(z, min(neighbours)) computed from upper bounds
//      is again an upper bound, so a stale read can only delay a lowering, never produce a wrong one; and a neighbour that
//      lowers an edge cell afterwards pokes this tile (test in step "decide which neighbours have to look again" re-reads
//      the halo cell from L2 before deciding), so no lowering is lost.  32-bit aligned stores / loads are single-copy
//      atomic, and the 16-byte vector stores are four of them: a torn read mixes old and new upper bounds.
//   4. Termination.  `pending` counts tiles queued or running: incremented before a tile id becomes visible in a slot,
//      decremented (after a __threadfence) only when the visit's own pokes have been issued.  It can therefore reach 0
//      only when no tile is queued, running or about to be poked, i.e. at the global fixed point; waiting CTAs leave when
//      they read pending <= 0.  A CTA that waits longer than SPIN_LIMIT sets the sticky status word (FILL_STALLED): the
//      finish pass poisons W[0][0] and hd_pdfill_status reports it -- a stalled fill cannot pass silently.
//   5. Ring capacity.  A slot is written only after its previous occupant was consumed: at most ntiles entries are
//      outstanding (one per tile: QUEUED is exclusive), the ring has ntiles + 8192 slots, consumers reset a slot to
//      SLOT_EMPTY before using the id, and tickets (`head`) can run ahead of `tail` by at most the number of CTAs.
struct FillCtl {
    int head, tail, pending, error;
    unsigned long long visits, changed_visits, iterations;
    int qcap, seen[2], pad_;          // seen: fill_init_kernel found a nodata cell / a -0.0 in z
    unsigned long long cycles[6];     // per-phase SM cycles of thread 0, summed over visits (HD_FILL_TRACE)
};
constexpr int SLOT_EMPTY = -1;
constexpr int SPIN_LIMIT = 1 << 22;
// Sticky status word of a fill, at byte STATUS_OFF of the workspace (inside the 256 bytes reserved for the finest level's
// control block, cleared once per fill: hd_pdfill, hd_pdfill_d8, hd_pdfill_coarse, hd_pdfill_band_start): set by ANY
// level whose worklist stalled (a waiting CTA ran out of patience: preemption, MPS, a debugger) or whose in-tile
// iteration hit its cap.  The finish kernels poison W[0][0] with NaN when it is set, and hd_pdfill_status reads it
// back: a fill that did not reach the fixed point can never pass silently, with or without statistics, inside or
// outside a CUDA graph.
constexpr int STATUS_OFF = 192;
enum { FILL_STALLED = 1, FILL_ITER_CAP = 2, FILL_PENDING = 4 };
// per-tile state: a tile is never processed by two CTAs at once (a second writer could overwrite a lower W with a
// higher one); a tile that is poked while running is marked dirty and re-queued by its own worker when it finishes
enum { T_IDLE = 0, T_QUEUED = 1, T_RUNNING = 2, T_DIRTY = 3 };

__device__ __forceinline__ void fill_push(FillCtl* ctl, int* slots, int qcap, int tile)
{
    atomicAdd(&ctl->pending, 1);
    const int t = atomicAdd(&ctl->tail, 1);
    *(volatile int*)(slots + (t % qcap)) = tile;
}
__device__ __forceinline__ void fill_poke(FillCtl* ctl, int* slots, int qcap, int* state, int tile)
{
    for (;;) {
        const int st = atomicCAS(&state[tile], T_IDLE, T_QUEUED);
        if (st == T_IDLE) { fill_push(ctl, slots, qcap, tile); return; }
        if (st == T_QUEUED || st == T_DIRTY) return;
        if (atomicCAS(&state[tile], T_RUNNING, T_DIRTY) == T_RUNNING) return;     // else the state moved: retry
    }
}

__global__ void __launch_bounds__(256) fill_seed_kernel(int tiles_x, int tiles_y, int64_t ny, FillCtl* ctl,
                                                        int* __restrict__ slots, int* __restrict__ queued, int edge_rows_only)
{
    // A tile is seeded when it touches the raster frame or contains a nodata cell (fill_init_kernel left a 1 in
    // queued[tile] for those).  Continuing a banded fill, only tiles that hold a refreshed halo row, or read it as
    // their own halo (the row next to it), can change.
    const int ntiles = tiles_x * tiles_y;
    for (int tile = blockIdx.x * blockDim.x + threadIdx.x; tile < ntiles; tile += gridDim.x * blockDim.x) {
        const int ty = tile / tiles_x, tx = tile % tiles_x;
        bool seed;
        if (edge_rows_only < 0)
            seed = true;                                           // multigrid start: every tile has cells to lower
        else if (edge_rows_only)
            seed = ((edge_rows_only & 2) && ty == 0) || ((edge_rows_only & 4) && ty >= (int)((ny - 2) / FT));
        else
            seed = ty == 0 || tx == 0 || ty == tiles_y - 1 || tx == tiles_x - 1 || queued[tile] != 0;
        queued[tile] = seed ? T_QUEUED : T_IDLE;
        if (seed) fill_push(ctl, slots, ctl->qcap, tile);
    }
}

// ---- coarse level of the fill -------------------------------------------------------------------------------------
// z_c(block) = max of the block's cells.  Every cell of a block can reach every other cell of it without exceeding
// z_c, blocks that touch are 8-connected at cell level, so the fill of the coarse DEM is an UPPER BOUND of the fill of
// the fine DEM on each block.  A block that holds an outlet (a frame cell or a nodata cell) is an outlet of the coarse
// problem at level z_c.  Starting the fine iteration from that bound instead of +inf changes nothing in the result
// (the fixed point is unique) but removes the long dependency chain of the tile wave: the global drainage structure
// is solved on 1/64 of the cells, the fine level only relaxes locally and all its tiles are busy from the start.
// w_in (levels >= 1): the finer level's own start -- a finite value marks an outlet cell of that level.
__global__ void __launch_bounds__(256) fill_pool_kernel(const float* __restrict__ z, int64_t z_pitch, int64_t ny, int64_t nx,
                                                        float* __restrict__ zc, float* __restrict__ wc, int64_t c_pitch,
                                                        int64_t nyc, int64_t nxc, int* __restrict__ tile_flags, int tiles_x_c,
                                                        const float* __restrict__ w_in, int top_is_halo, int bottom_is_halo)
{
    for (CellIter it(nxc); it.y < nyc; it.next()) {
        const int64_t by = it.y, bx = it.x, y0 = by * CB, x0 = bx * CB;
        float m = __int_as_float(0xff800000);
        bool has_nan = false, any_valid = false;
        for (int dy = 0; dy < CB && y0 + dy < ny; ++dy) {
            const float* row = z + (y0 + dy) * z_pitch + x0;
#pragma unroll
            for (int q = 0; q < CB; q += 4) {
                float v[4], wv[4] = {0.f, 0.f, 0.f, 0.f};
                gload4(row + q, x0 + q, nx, v);
                if (w_in) gload4(w_in + (y0 + dy) * z_pitch + x0 + q, x0 + q, nx, wv);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    if (x0 + q + j >= nx) continue;
                    if (v[j] != v[j]) has_nan = true;
                    else { m = fmaxf(m, v[j]); any_valid = true; }
                    if (w_in && wv[j] != __int_as_float(0x7f800000)) has_nan = true;      // an outlet of the finer level
                }
            }
        }
        // (the first / last row of a band that continues on another GPU is a halo row, not raster frame)
        const bool frame = (y0 == 0 && !top_is_halo) || x0 == 0 || (y0 + CB >= ny && !bottom_is_halo) || x0 + CB >= nx;
        const bool seed = has_nan || frame;
        zc[by * c_pitch + bx] = any_valid ? m : __int_as_float(0x7fc00000);
        wc[by * c_pitch + bx] = !any_valid ? __int_as_float(0xff800000) : (seed ? m : __int_as_float(0x7f800000));
        if (seed) tile_flags[(by / FT) * tiles_x_c + bx / FT] = 1;        // benign race: every writer stores 1
    }
}

// non-outlet cells of a coarse level start from the (solved) next coarser level instead of +inf
__global__ void __launch_bounds__(256) fill_refine_kernel(float* __restrict__ w, int64_t pitch, int64_t ny, int64_t nx,
                                                          const float* __restrict__ wc, int64_t c_pitch)
{
    for (CellIter it(nx); it.y < ny; it.next()) {
        float* p = w + it.y * pitch + it.x;
        if (*p == __int_as_float(0x7f800000)) *p = __ldg(wc + (it.y / CB) * c_pitch + it.x / CB);
    }
}

__global__ void fill_ctl_init_kernel(FillCtl* ctl, int qcap) { ctl->qcap = qcap; }

// three-input min (FMNMX3 on sm_100); like fminf it returns the non-NaN operand(s)
__device__ __forceinline__ float fmin3(float a, float b, float c)
{
    float d;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

__device__ __forceinline__ float fmax3(float a, float b, float c)
{
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

// One marching sweep of a 64-thread group through the tile: F = shared-memory step along the march, L = step to the
// neighbouring thread's line.  A cell is relaxed against the three cells behind it and its two lateral neighbours
// (the opposite group covers the three ahead; the check pass covers all eight).  Per step: three reads of the next
// row, the thread's own previous result in a register and the two diagonal cells behind from the neighbouring lanes
// by shuffle -- they were updated one step ago, so a level runs diagonally through the tile in a single sweep and no
// step waits for a shared-memory store to come back.
// One relaxation of every cell of the tile, no dependency chain: warp w takes tile rows 8w..8w+7, a lane two columns,
// sliding a three-row window down its strip.
__device__ __forceinline__ bool fill_check(float* __restrict__ ws, const float* __restrict__ zs, int warp, int lane32)
{
    bool changed = false;
#pragma unroll
    for (int h = 0; h < 2; ++h) {
        float* wp = ws + (8 * warp) * WS_STRIDE + lane32 + 32 * h + 1;         // box row above the strip
        const float* zp = zs + (8 * warp + 1) * WS_STRIDE + lane32 + 32 * h + 1;
        float am = wp[-1], a0 = wp[0], ap = wp[1];
        float cm = wp[WS_STRIDE - 1], c0 = wp[WS_STRIDE], cp = wp[WS_STRIDE + 1];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float bm = wp[(i + 2) * WS_STRIDE - 1], b0 = wp[(i + 2) * WS_STRIDE], bp = wp[(i + 2) * WS_STRIDE + 1];
            const float m = fminf(fmin3(am, a0, ap), fmin3(bm, b0, bp));
            const float cand = fmaxf(zp[i * WS_STRIDE], fmin3(cm, cp, m));
            if (cand < c0) { wp[(i + 1) * WS_STRIDE] = cand; c0 = cand; changed = true; }
            am = cm; a0 = c0; ap = cp;
            cm = bm; c0 = b0; cp = bp;
        }
    }
    return changed;
}

template <int F, int L>
__device__ __forceinline__ void fill_march(float* __restrict__ ws, const float* __restrict__ zs, int p0)
{
    float* wp = ws + p0;
    const float* zp = zs + p0;
    float bm = wp[-F - L], b0 = wp[-F], bp = wp[-F + L];
    float cm = wp[-L], own = wp[0], cp = wp[L];
    float zc = zp[0];
#pragma unroll 1
    for (int kk = 0; kk < FT; kk += 8) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            // the next step's current row, read before this step's store (all offsets are immediates)
            const float fm = wp[(j + 1) * F - L], f0 = wp[(j + 1) * F], fp = wp[(j + 1) * F + L];
            const float zn = zp[(j + 1) * F];
            const float cand = fmaxf(zc, fmin3(cm, cp, fmin3(bm, b0, bp)));     // fmin / fmax skip NaN operands
            if (cand < own) { wp[j * F] = cand; own = cand; }                   // only ever lowers W
            // the diagonal cells behind the next step: the neighbouring lanes' results of this step.  The end lanes of
            // a warp get their own value back (no information, no harm)
            bm = __shfl_up_sync(0xffffffffu, own, 1);
            bp = __shfl_down_sync(0xffffffffu, own, 1);
            b0 = own; cm = fm; own = f0; cp = fp; zc = zn;
        }
        wp += 8 * F;
        zp += 8 * F;
    }
}

__global__ void __launch_bounds__(FNT, 4) fill_async_kernel(const float* __restrict__ z, int64_t z_pitch, float* __restrict__ w,
                                                         int64_t w_pitch, int64_t ny, int64_t nx, int tiles_x, int tiles_y,
                                                         FillCtl* ctl, int* slots, int* queued, int* status)
{
    // This kernel does not use TMA: W must be read L2-coherently (ld.global.cg) while other CTAs update it, and both
    // boxes have to land in a padded (conflict-free) layout that a dense TMA box cannot produce.
    // Shared memory: three (FT+2) x WS_STRIDE boxes with a one-cell halo and the same indexing -- z, W as loaded, W.
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ int s_tile;
    __shared__ unsigned s_edges;
    constexpr int BOX = (FT + 2) * WS_STRIDE;
    float* zs = reinterpret_cast<float*>(smem);
    float* wold = zs + BOX;
    float* ws = wold + BOX;
    const int qcap = ctl->qcap;
    const int group = threadIdx.x >> 6, lane64 = threadIdx.x & 63, lane32 = threadIdx.x & 31;
    const float qnan = __int_as_float(0x7fc00000);
    const bool zvec_ok = ((z_pitch & 3) == 0) && ((((uintptr_t)z) & 15) == 0);
    const bool wvec_ok = ((w_pitch & 3) == 0) && ((((uintptr_t)w) & 15) == 0);
    // Thread 32 takes the tickets: it waits for the next tile while warp 0 is still publishing the previous one.
    auto take_ticket = [&]() {
        const long long t0 = clock64();
        int tile = -1;
        const int my = atomicAdd(&ctl->head, 1);
        volatile int* slot = slots + (my % qcap);
        for (int spin = 0;; ++spin) {
            const int v = *slot;
            if (v != SLOT_EMPTY) { *slot = SLOT_EMPTY; tile = v; break; }
            if (*(volatile int*)&ctl->pending <= 0 || *(volatile int*)&ctl->error) break;
            if (spin > SPIN_LIMIT) { atomicExch(&ctl->error, 1); atomicOr(status, FILL_STALLED); break; }
            __nanosleep(100);
        }
        if (tile >= 0) { atomicExch(&queued[tile], T_RUNNING); __threadfence(); }
        s_tile = tile;
        atomicAdd(&ctl->cycles[0], (unsigned long long)(clock64() - t0));
    };
    if (threadIdx.x == 0) s_edges = 0u;
    if (threadIdx.x == 32) take_ticket();
    for (;;) {
        long long tc1 = 0, tc2 = 0, tc3 = 0, tc4 = 0;
        __syncthreads();
        const int tile = s_tile;
        if (tile < 0) return;
        if (threadIdx.x == 0) tc1 = clock64();
        const int ty0 = (tile / tiles_x) * FT, tx0 = (tile % tiles_x) * FT;

        // ---- load z and W boxes: all global loads of a thread are issued before the first shared store ---------------
        // items 0..1055: row r = item / 16 of the box, aligned quad k = item % 16 of the 64 tile columns
        // items 1056..1187: the two halo columns.  Outside the raster: W = NaN (ignored by fmin), z = 0.
        {
            float4 zq[5], wq[5];
#pragma unroll
            for (int j = 0; j < 5; ++j) {
                const int item = threadIdx.x + j * FNT;
                zq[j] = make_float4(0.f, 0.f, 0.f, 0.f);
                wq[j] = make_float4(qnan, qnan, qnan, qnan);
                if (item < 1056) {
                    const int r = item >> 4, k = item & 15;
                    const int64_t y = (int64_t)ty0 - 1 + r, x = (int64_t)tx0 + 4 * k;
                    if (y >= 0 && y < ny) {
                        const float* pz = z + y * z_pitch + x;
                        const float* pw = w + y * w_pitch + x;
                        if (x + 3 < nx && zvec_ok && wvec_ok) {
                            zq[j] = __ldg(reinterpret_cast<const float4*>(pz));
                            wq[j] = __ldcg(reinterpret_cast<const float4*>(pw));
                        } else {
                            if (x < nx) { zq[j].x = __ldg(pz); wq[j].x = __ldcg(pw); }
                            if (x + 1 < nx) { zq[j].y = __ldg(pz + 1); wq[j].y = __ldcg(pw + 1); }
                            if (x + 2 < nx) { zq[j].z = __ldg(pz + 2); wq[j].z = __ldcg(pw + 2); }
                            if (x + 3 < nx) { zq[j].w = __ldg(pz + 3); wq[j].w = __ldcg(pw + 3); }
                        }
                    }
                } else if (item < 1056 + 2 * (FT + 2)) {
                    const int h = item - 1056, r = h >> 1;
                    const int64_t y = (int64_t)ty0 - 1 + r, x = (h & 1) ? (int64_t)tx0 + FT : (int64_t)tx0 - 1;
                    if (y >= 0 && y < ny && x >= 0 && x < nx) {
                        zq[j].x = __ldg(z + y * z_pitch + x);
                        wq[j].x = __ldcg(w + y * w_pitch + x);
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < 5; ++j) {
                const int item = threadIdx.x + j * FNT;
                if (item < 1056) {
                    const int o = (item >> 4) * WS_STRIDE + 1 + 4 * (item & 15);
                    zs[o] = zq[j].x; zs[o + 1] = zq[j].y; zs[o + 2] = zq[j].z; zs[o + 3] = zq[j].w;
                    ws[o] = wq[j].x; ws[o + 1] = wq[j].y; ws[o + 2] = wq[j].z; ws[o + 3] = wq[j].w;
                    wold[o] = wq[j].x; wold[o + 1] = wq[j].y; wold[o + 2] = wq[j].z; wold[o + 3] = wq[j].w;
                } else if (item < 1056 + 2 * (FT + 2)) {
                    const int h = item - 1056;
                    const int o = (h >> 1) * WS_STRIDE + ((h & 1) ? FT + 1 : 0);
                    zs[o] = zq[j].x; ws[o] = wq[j].x; wold[o] = wq[j].x;
                }
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) tc2 = clock64();

        // ---- relax to the local fixed point ------------------------------------------------------------------------
        // A marching iteration (four groups going down / up / right / left simultaneously) carries a level across the
        // whole tile but costs 64 dependent steps; the check pass relaxes every cell once with no dependency chain at
        // 1/6 of the instructions.  The visit starts with a check (almost half of all visits find nothing to lower and
        // end right there) and every marching iteration is followed by one: a check that stores nothing has read a
        // static tile, i.e. verified the local fixed point.
        bool tile_changed = false;
        int iters = 0;
        const int warp = threadIdx.x >> 5;
        while (__syncthreads_or(fill_check(ws, zs, warp, lane32))) {
            tile_changed = true;
            if (group == 0)      fill_march<WS_STRIDE, 1>(ws, zs, 1 * WS_STRIDE + lane64 + 1);
            else if (group == 1) fill_march<-WS_STRIDE, 1>(ws, zs, FT * WS_STRIDE + lane64 + 1);
            else if (group == 2) fill_march<1, WS_STRIDE>(ws, zs, (lane64 + 1) * WS_STRIDE + 1);
            else                 fill_march<-1, WS_STRIDE>(ws, zs, (lane64 + 1) * WS_STRIDE + FT);
            ++iters;
            __syncthreads();
            if (iters > 4096) {                          // (unreachable on real terrain; never silently)
                if (threadIdx.x == 0) atomicOr(status, FILL_ITER_CAP);
                break;
            }
        }
        if (threadIdx.x == 0) { atomicAdd(&ctl->iterations, (unsigned long long)iters); tc3 = clock64(); }

        // ---- write the lowered cells back; decide which neighbours have to look again ------------------------------------
        if (tile_changed) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int item = threadIdx.x + j * FNT;                  // quad k of tile row r
                const int r = item >> 4, k = item & 15;
                const int o = (r + 1) * WS_STRIDE + 1 + 4 * k;
                const float n0 = ws[o], n1 = ws[o + 1], n2 = ws[o + 2], n3 = ws[o + 3];
                const bool any = n0 != wold[o] || n1 != wold[o + 1] || n2 != wold[o + 2] || n3 != wold[o + 3];
                const int64_t y = (int64_t)ty0 + r, x = (int64_t)tx0 + 4 * k;
                if (any && y < ny) {                                     // (NaN cells lie outside the raster: never changed)
                    float* pw = w + y * w_pitch + x;
                    if (x + 3 < nx && wvec_ok) {
                        *reinterpret_cast<float4*>(pw) = make_float4(n0, n1, n2, n3);
                    } else {
                        if (x < nx) pw[0] = n0;
                        if (x + 1 < nx) pw[1] = n1;
                        if (x + 2 < nx) pw[2] = n2;
                        if (x + 3 < nx) pw[3] = n3;
                    }
                }
            }
            // One thread per cell of the tile's outer ring.  A neighbouring tile is poked only if a lowered ring cell can
            // still lower one of ITS cells h: max(z(h), new value) < W(h), with z(h) and W(h) from the halo as loaded
            // (W only ever decreases, so a stale W(h) errs on the safe side).  This test is exact: it drops the "poke
            // back" to the tile the level came from and every poke that z(h) would absorb.    bit = (dy+1)*3 + (dx+1)
            unsigned edges = 0u;
            if (threadIdx.x < 4 * FT - 4) {
                const int t = threadIdx.x;
                int r, c;
                if (t < FT) { r = 0; c = t; }
                else if (t < 2 * FT) { r = FT - 1; c = t - FT; }
                else if (t < 3 * FT - 2) { r = t - 2 * FT + 1; c = 0; }
                else { r = t - (3 * FT - 2) + 1; c = FT - 1; }
                const int o = (r + 1) * WS_STRIDE + c + 1;
                const float nv = ws[o];
                if (nv < wold[o]) {
#pragma unroll
                    for (int a = -1; a <= 1; ++a)
#pragma unroll
                        for (int b = -1; b <= 1; ++b) {
                            const int rr = r + a, cc = c + b;
                            const int dy = rr < 0 ? -1 : (rr >= FT ? 1 : 0), dx = cc < 0 ? -1 : (cc >= FT ? 1 : 0);
                            if (dy | dx) {
                                const int oh = o + a * WS_STRIDE + b;
                                const float lim = fmaxf(zs[oh], nv);
                                if (lim < ws[oh]) {                             // halo W outside the raster is NaN: false
                                    // the neighbour may have lowered h since this tile was loaded: look again
                                    const float fresh = __ldcg(w + ((int64_t)ty0 + rr) * w_pitch + (int64_t)tx0 + cc);
                                    if (lim < fresh) edges |= 1u << ((dy + 1) * 3 + (dx + 1));
                                }
                            }
                        }
                }
            }
            edges = __reduce_or_sync(0xffffffffu, edges);
            if (edges && lane32 == 0) atomicOr(&s_edges, edges);
            __threadfence();                                   // W stores visible device-wide before neighbours are published
        }
        __syncthreads();
        if (threadIdx.x == 0) tc4 = clock64();
        // ---- publish (warp 0) while thread 32 already fetches the next tile ---------------------------------------------
        // lanes 0..8 poke one neighbour each, lane 9 moves the tile's own state; `pending` drops last, after a fence, so it
        // can never read 0 while a poke of this visit is still on its way
        if (threadIdx.x < 32) {
            const unsigned edges = s_edges;
            const int k = threadIdx.x;
            if (k < 9 && ((edges >> k) & 1u)) {
                const int tyy = tile / tiles_x + k / 3 - 1, txx = tile % tiles_x + k % 3 - 1;
                if (tyy >= 0 && tyy < tiles_y && txx >= 0 && txx < tiles_x)
                    fill_poke(ctl, slots, qcap, queued, tyy * tiles_x + txx);
            } else if (k == 9) {
                if (atomicCAS(&queued[tile], T_RUNNING, T_IDLE) != T_RUNNING) {     // poked while running: go again
                    atomicExch(&queued[tile], T_QUEUED);
                    fill_push(ctl, slots, qcap, tile);
                }
            }
            __syncwarp();
            if (k == 0) {
                s_edges = 0u;
                atomicAdd(&ctl->visits, 1ull);
                if (tile_changed) atomicAdd(&ctl->changed_visits, 1ull);
                __threadfence();
                atomicSub(&ctl->pending, 1);
                const long long tc5 = clock64();
                atomicAdd(&ctl->cycles[1], (unsigned long long)(tc2 - tc1));
                atomicAdd(&ctl->cycles[2], (unsigned long long)(tc3 - tc2));
                atomicAdd(&ctl->cycles[3], (unsigned long long)(tc4 - tc3));
                atomicAdd(&ctl->cycles[4], (unsigned long long)(tc5 - tc4));
            }
        } else if (threadIdx.x == 32) {
            take_ticket();
        }
    }
}

// ---- D8 ------------------------------------------------------------------------------------------------------
// ESRI codes E=1 SE=2 S=4 SW=8 W=16 NW=32 N=64 NE=128; steepest positive drop, diagonal drops scaled by
// 0.70710678f in float32; ties keep the first in that order; frame cells, NaN centres, no drop -> 0.
// The code of cell j of a quad from its window: three rows of (left neighbour, aligned quad, right neighbour).
__device__ __forceinline__ uint8_t d8_code(const float (&win)[3][6], int j)
{
    const float c = win[1][j + 1];
    // E, SE, S, SW, W, NW, N, NE; diagonal drops scaled in float32
    const float d0 = __fsub_rn(c, win[1][j + 2]), d1 = __fmul_rn(__fsub_rn(c, win[2][j + 2]), 0.70710678f);
    const float d2 = __fsub_rn(c, win[2][j + 1]), d3 = __fmul_rn(__fsub_rn(c, win[2][j]), 0.70710678f);
    const float d4 = __fsub_rn(c, win[1][j]), d5 = __fmul_rn(__fsub_rn(c, win[0][j]), 0.70710678f);
    const float d6 = __fsub_rn(c, win[0][j + 1]), d7 = __fmul_rn(__fsub_rn(c, win[0][j + 2]), 0.70710678f);
    // "first strictly larger drop wins" == the FIRST direction that attains the maximum, if it is positive
    // (three-input max: 4 instructions; NaN drops are skipped by max and never compare equal)
    const float best = fmax3(fmax3(d0, d1, d2), fmax3(d3, d4, d5), fmax3(d6, d7, 0.f));
    unsigned code = 0u;
    code = d7 == best ? 128u : code;
    code = d6 == best ? 64u : code;
    code = d5 == best ? 32u : code;
    code = d4 == best ? 16u : code;
    code = d3 == best ? 8u : code;
    code = d2 == best ? 4u : code;
    code = d1 == best ? 2u : code;
    code = d0 == best ? 1u : code;
    return best > 0.f ? (uint8_t)code : (uint8_t)0;
}

__global__ void __launch_bounds__(256) d8_kernel(const float* __restrict__ w, int64_t w_pitch, uint8_t* __restrict__ out,
                                                 int64_t out_pitch, int64_t ny, int64_t nx)
{
    // four consecutive cells per thread: three rows of (left neighbour, aligned quad, right neighbour)
    const int64_t nxq = (nx + 3) / 4;
    for (CellIter it(nxq); it.y < ny; it.next()) {
        const int64_t y = it.y, x0 = 4 * it.x;
        uint8_t codes[4] = {0, 0, 0, 0};
        if (y > 0 && y < ny - 1) {
            float win[3][6];
#pragma unroll
            for (int dy = 0; dy < 3; ++dy) {
                const float* p = w + (y + dy - 1) * w_pitch + x0;
                float q[4];
                gload4(p, x0, nx, q);
                win[dy][0] = x0 > 0 ? __ldg(p - 1) : 0.f;
                win[dy][1] = q[0]; win[dy][2] = q[1]; win[dy][3] = q[2]; win[dy][4] = q[3];
                win[dy][5] = x0 + 4 < nx ? __ldg(p + 4) : 0.f;
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int64_t x = x0 + j;
                if (x == 0 || x >= nx - 1) continue;
                codes[j] = d8_code(win, j);
            }
        }
        store4v<uint8_t>(out, out_pitch, y, x0, nx, codes);
    }
}


// Last pass of the fill FUSED with the D8 pass: nodata cells (outlets at -inf while iterating) get their NaN back and
// every cell's flow direction is written in the same sweep over W -- 4 B read + 1 B written per cell, W is not read
// a second time by a separate D8 launch.  A fill that stalled (status word set, see FILL_*) poisons W[0][0] and the
// first code with NaN / 255 so that it cannot pass for a result.
// W = -inf does not make a cell nodata: a cell whose own z is -inf keeps -inf when it drains to an outlet at -inf.
// Only a window that holds a -inf reads z, and only at its -inf cells.
__global__ void __launch_bounds__(256) fill_finish_d8_kernel(const float* __restrict__ z, int64_t z_pitch,
                                                             float* __restrict__ w, int64_t w_pitch, uint8_t* __restrict__ out,
                                                             int64_t out_pitch, int64_t ny, int64_t nx,
                                                             const FillCtl* __restrict__ ctl, const int* __restrict__ status)
{
    const float ninf = __int_as_float(0xff800000), qnan = __int_as_float(0x7fc00000);
    const bool bad = (status && *status != 0) || (ctl && ctl->pending != 0);
    const int64_t nxq = (nx + 3) / 4;
    for (CellIter it(nxq); it.y < ny; it.next()) {
        const int64_t y = it.y, x0 = 4 * it.x;
        float win[3][6];
#pragma unroll
        for (int dy = 0; dy < 3; ++dy) {
            const int64_t yy = y + dy - 1;
            if (yy < 0 || yy >= ny) {
#pragma unroll
                for (int j = 0; j < 6; ++j) win[dy][j] = 0.f;
                continue;
            }
            const float* p = w + yy * w_pitch + x0;
            float q[4];
            if (x0 + 3 < nx && ((reinterpret_cast<uintptr_t>(p) & 15) == 0)) {
                const float4 v = __ldcg(reinterpret_cast<const float4*>(p));       // (neighbours may be rewriting -inf as NaN)
                q[0] = v.x; q[1] = v.y; q[2] = v.z; q[3] = v.w;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) q[j] = (x0 + j < nx) ? __ldcg(p + j) : 0.f;
            }
            win[dy][0] = x0 > 0 ? __ldcg(p - 1) : 0.f;
            win[dy][1] = q[0]; win[dy][2] = q[1]; win[dy][3] = q[2]; win[dy][4] = q[3];
            win[dy][5] = x0 + 4 < nx ? __ldcg(p + 4) : 0.f;
        }
        // nodata cells are -inf here: only a window that holds a -inf needs the NaN conversion (and the restore below)
        float lowest = win[0][0];
#pragma unroll
        for (int dy = 0; dy < 3; ++dy)
#pragma unroll
            for (int j = 0; j < 6; j += 2) lowest = fmin3(lowest, win[dy][j], win[dy][j + 1]);
        const bool has_nodata = lowest == ninf;
        if (has_nodata) {
#pragma unroll
            for (int dy = 0; dy < 3; ++dy) {
                const int64_t yy = y + dy - 1;                           // (cells outside the raster hold 0, never -inf)
                const float* p = z + yy * z_pitch + x0;
                if (win[dy][1] == ninf || win[dy][2] == ninf || win[dy][3] == ninf || win[dy][4] == ninf) {
                    float zq[4];
                    gload4(p, x0, nx, zq);
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (win[dy][j + 1] == ninf && zq[j] != zq[j]) win[dy][j + 1] = qnan;
                }
                if (win[dy][0] == ninf && __ldg(p - 1) != __ldg(p - 1)) win[dy][0] = qnan;
                if (win[dy][5] == ninf && __ldg(p + 4) != __ldg(p + 4)) win[dy][5] = qnan;
            }
        }
        uint8_t codes[4] = {0, 0, 0, 0};
        bool restore = false;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int64_t x = x0 + j;
            const float c = win[1][j + 1];
            // nodata cells get NaN back; every zero becomes +0.0 (see fill_finish_kernel).  No D8 decision depends on the
            // sign of a zero: a drop between two zeros is a zero, never positive
            restore |= ((has_nodata && c != c) || __float_as_uint(c) == 0x80000000u) && x < nx;
            if (y == 0 || y >= ny - 1 || x == 0 || x >= nx - 1) continue;
            codes[j] = d8_code(win, j);
        }
        if (restore) {                                                    // rare: rewrite the quad's nodata cells and -0.0
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float c = win[1][j + 1];
                if (x0 + j < nx && (c != c || __float_as_uint(c) == 0x80000000u)) w[y * w_pitch + x0 + j] = c != c ? qnan : 0.f;
            }
        }
        if (bad && y == 0 && x0 == 0) { w[0] = qnan; codes[0] = 255; }
        store4v<uint8_t>(out, out_pitch, y, x0, nx, codes);
    }
}

// halo row of a band after an exchange: W = min(W, received); *lowered |= 1 when any cell went down (the banded fill
// needs another round).  -inf (nodata) and NaN never count.
__global__ void __launch_bounds__(256) halo_min_kernel(float* __restrict__ w, const float* __restrict__ recv, int64_t nx,
                                                       int* __restrict__ lowered)
{
    bool any = false;
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < nx; x += (int64_t)gridDim.x * blockDim.x) {
        const float r = recv[x], c = w[x];
        if (r < c) { w[x] = r; any = true; }
    }
    if (__syncthreads_or(any) && threadIdx.x == 0) atomicExch(lowered, 1);
}

int stream_grid(int64_t total)
{
    const int64_t b = (total + 255) / 256, cap = (int64_t)hd_num_sms() * 16;
    return (int)(b < cap ? b : cap);
}

}  // namespace


// flags: 1 = W already initialised (continue a banded fill), 2 / 4 = the top / bottom raster row is a halo row of a
// neighbouring band (not frame); finish = restore NaN at nodata cells afterwards
struct FillOpts {
    bool preinit = false;         // W and the per-tile flags are already set up (coarse level)
    bool seed_all = false;        // every tile starts queued (fine level of the multigrid start)
    const float* wc = nullptr;    // coarse-level fill used as the starting W of interior cells
    int64_t c_pitch = 0;
    int64_t wc_y0 = 0;            // local row 0 = row wc_y0 of the raster the coarse level was pooled from
    int* status = nullptr;        // sticky status word of the whole fill (root workspace + STATUS_OFF)
};

static int launch_finish_d8(const void* z, int64_t z_pitch, void* w, int64_t w_pitch, void* d8, int64_t d8_pitch, int64_t ny,
                            int64_t nx, const void* workspace, cudaStream_t s)
{
    const FillCtl* ctl = (const FillCtl*)workspace;
    const int* status = workspace ? (const int*)((const char*)workspace + STATUS_OFF) : nullptr;
    hd_prof_begin("fill_finish_d8_kernel", s);
    fill_finish_d8_kernel<<<stream_grid(ny * ((nx + 3) / 4)), 256, 0, s>>>((const float*)z, z_pitch, (float*)w, w_pitch, (uint8_t*)d8,
                                                                          d8_pitch, ny, nx, ctl, status);
    HD_LAUNCH_CHECK(); hd_count_launch();
    return HD_OK;
}

static int pdfill_async(const void* z, int64_t z_pitch, void* w, int64_t w_pitch, int64_t ny, int64_t nx, void* workspace,
                        int* visits_out, cudaStream_t s, int flags = 0, bool finish = true, FillOpts opt = FillOpts())
{
    if (!opt.status) opt.status = (int*)((char*)workspace + STATUS_OFF);
    const int tiles_x = hd_cdiv(nx, FT), tiles_y = hd_cdiv(ny, FT), ntiles = tiles_x * tiles_y;
    FillCtl* ctl = (FillCtl*)workspace;
    const int qcap = ntiles + 8192;
    int* slots = (int*)((char*)workspace + 256);
    int* queued = slots + qcap;
    const size_t smem = 3 * (size_t)(FT + 2) * WS_STRIDE * 4;
    HD_CUDA_OK(cudaFuncSetAttribute(fill_async_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    HD_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fill_async_kernel, FNT, smem));
    if (const char* e = getenv("HD_FILL_CTAS_PER_SM")) {      // experiments: fewer co-resident CTAs, less MIO contention
        const int v = atoi(e);
        if (v >= 1 && v < per_sm) per_sm = v;
    }
    int grid = hd_num_sms() * (per_sm < 1 ? 1 : per_sm);       // every CTA must be co-resident: they wait on each other
    if (grid > ntiles) grid = ntiles;
    // (no host-to-device copy of a stack object here: the whole call must be capturable in a CUDA graph)
    HD_CUDA_OK(cudaMemsetAsync(ctl, 0, sizeof(FillCtl), s));
    HD_CUDA_OK(cudaMemsetAsync(slots, 0xff, (size_t)qcap * sizeof(int), s));        // SLOT_EMPTY = -1
    if (!opt.preinit) HD_CUDA_OK(cudaMemsetAsync(queued, 0, (size_t)ntiles * sizeof(int), s));
    fill_ctl_init_kernel<<<1, 1, 0, s>>>(ctl, qcap);
    HD_LAUNCH_CHECK();
    if (!(flags & 1) && !opt.preinit) {
        hd_prof_begin("fill_init_kernel", s);
        fill_init_kernel<<<stream_grid(ny * ((nx + 3) / 4)), 256, 0, s>>>((const float*)z, z_pitch, (float*)w, w_pitch, ny, nx, flags & 2,
                                                             flags & 4, queued, tiles_x, ctl->seen, opt.wc, opt.c_pitch,
                                                             opt.wc_y0);
        HD_LAUNCH_CHECK(); hd_count_launch();
    }
    hd_prof_begin("fill_seed_kernel", s);
    fill_seed_kernel<<<hd_cdiv(ntiles, 256) < 1184 ? hd_cdiv(ntiles, 256) : 1184, 256, 0, s>>>(
        tiles_x, tiles_y, ny, ctl, slots, queued, opt.seed_all ? -1 : ((flags & 1) ? (flags & 6) : 0));
    HD_LAUNCH_CHECK(); hd_count_launch();
    hd_prof_begin("fill_async_kernel", s);
    fill_async_kernel<<<grid, FNT, smem, s>>>((const float*)z, z_pitch, (float*)w, w_pitch, ny, nx, tiles_x, tiles_y, ctl,
                                              slots, queued, opt.status);
    HD_LAUNCH_CHECK(); hd_count_launch();
    if (finish) {
        hd_prof_begin("fill_finish_kernel", s);
        fill_finish_kernel<<<stream_grid(ny * nx), 256, 0, s>>>((const float*)z, z_pitch, (float*)w, w_pitch, ny, nx,
                                                               (flags & 1) ? nullptr : ctl->seen, opt.status,
                                                               &ctl->pending);
        HD_LAUNCH_CHECK(); hd_count_launch();
    }
    if (!visits_out && !getenv("HD_FILL_TRACE")) return HD_OK;      // fully asynchronous when nobody asks for statistics
    static thread_local FillCtl* h_ctl = nullptr;          // per calling thread: concurrent fills never share it
    if (!h_ctl) HD_CUDA_OK(cudaHostAlloc((void**)&h_ctl, sizeof(FillCtl), cudaHostAllocDefault));
    HD_CUDA_OK(cudaMemcpyAsync(h_ctl, ctl, sizeof(FillCtl), cudaMemcpyDeviceToHost, s));
    HD_CUDA_OK(cudaStreamSynchronize(s));
    if (getenv("HD_FILL_TRACE"))
        fprintf(stderr, "pdfill async: %llu tile visits (%llu changed, %llu in-tile iterations) over %d tiles, grid %d\n",
                h_ctl->visits, h_ctl->changed_visits, h_ctl->iterations, ntiles, grid);
    if (getenv("HD_FILL_TRACE") && h_ctl->visits)
        fprintf(stderr, "  cycles per visit: wait %.0f  load %.0f  iterate %.0f  writeback %.0f  publish %.0f\n",
                (double)h_ctl->cycles[0] / h_ctl->visits, (double)h_ctl->cycles[1] / h_ctl->visits,
                (double)h_ctl->cycles[2] / h_ctl->visits, (double)h_ctl->cycles[3] / h_ctl->visits,
                (double)h_ctl->cycles[4] / h_ctl->visits);
    if (visits_out) *visits_out = (int)h_ctl->visits;
    if (h_ctl->error || h_ctl->pending != 0) return HD_ERR_UNSUPPORTED;    // worklist stalled (should not happen)
    return HD_OK;
}

static int64_t fill_level_bytes(int64_t ny, int64_t nx)
{
    const int64_t ntiles = (int64_t)hd_cdiv(ny, FT) * hd_cdiv(nx, FT);
    // what pdfill_async lays out: control block, FIFO ring (ntiles + slack slots), per-tile states
    const int64_t b = 256 + (2 * ntiles + 8192) * (int64_t)sizeof(int);
    return (b + 255) / 256 * 256;
}
static int64_t coarse_pitch(int64_t nxc) { return (nxc + 31) / 32 * 32; }
constexpr int MAX_LEVELS = 8;
// coarse levels exist while the next one still has a few tiles
static bool level_worth_it(int64_t nyc, int64_t nxc) { return (int64_t)hd_cdiv(nyc, FT) * hd_cdiv(nxc, FT) >= 4; }

extern "C" int64_t hd_pdfill_workspace_bytes(int64_t ny, int64_t nx)
{
    // fine level control block, then per coarse level: control block + that level's z and W rasters
    int64_t total = fill_level_bytes(ny, nx);
    for (int l = 1; l < MAX_LEVELS; ++l) {
        const int64_t nyc = hd_cdiv(ny, CB), nxc = hd_cdiv(nx, CB);
        if (!level_worth_it(nyc, nxc)) break;
        total += fill_level_bytes(nyc, nxc) + 2 * nyc * coarse_pitch(nxc) * (int64_t)sizeof(float);
        ny = nyc; nx = nxc;
    }
    return total;
}

// Multigrid start (see fill_pool_kernel): the coarse levels below a raster, by block maxima, laid out in its workspace
// after its own control block; the coarsest level is filled from scratch, every finer one from the level above it.
// The first level pools z: its outlet marks come from the frame and the NaN cells, plus those of `marks` when given
// (a coarse raster whose W carries its own outlet marks, same pitch as z).  *first = the finest coarse level, whose w
// is nullptr when the raster is too small for one.
struct FillLevel { int64_t ny, nx, pitch; float* z; float* w; char* ctl; };

static int fill_coarse_levels(const float* z, const float* marks, int64_t pitch, int64_t ny, int64_t nx, void* workspace,
                              cudaStream_t s, FillLevel* first)
{
    FillLevel lv[MAX_LEVELS];
    int nlev = 0;
    char* cur = (char*)workspace + fill_level_bytes(ny, nx);
    // downward: block maxima + outlet marks of every level
    for (int l = 1; l < MAX_LEVELS; ++l) {
        const int64_t nyc = hd_cdiv(ny, CB), nxc = hd_cdiv(nx, CB);
        if (!level_worth_it(nyc, nxc)) break;
        FillLevel& L = lv[nlev++];
        L.ny = nyc; L.nx = nxc; L.pitch = coarse_pitch(nxc);
        L.ctl = cur;
        L.z = (float*)(cur + fill_level_bytes(nyc, nxc));
        L.w = L.z + nyc * L.pitch;
        cur = (char*)(L.w + nyc * L.pitch);
        const int tiles_x_c = hd_cdiv(nxc, FT), ntiles_c = tiles_x_c * hd_cdiv(nyc, FT);
        int* queued_c = (int*)(L.ctl + 256) + (ntiles_c + 8192);
        HD_CUDA_OK(cudaMemsetAsync(queued_c, 0, (size_t)ntiles_c * sizeof(int), s));
        hd_prof_begin("fill_pool_kernel", s);
        fill_pool_kernel<<<stream_grid(nyc * nxc), 256, 0, s>>>(z, pitch, ny, nx, L.z, L.w, L.pitch, nyc, nxc, queued_c,
                                                                tiles_x_c, marks, 0, 0);
        HD_LAUNCH_CHECK(); hd_count_launch();
        z = L.z; marks = L.w; pitch = L.pitch; ny = nyc; nx = nxc;
    }
    // upward: coarsest level from scratch, every finer one from the level above
    for (int l = nlev - 1; l >= 0; --l) {
        const FillLevel& L = lv[l];
        FillOpts o;
        o.preinit = true;
        o.status = (int*)((char*)workspace + STATUS_OFF);
        if (l < nlev - 1) {
            hd_prof_begin("fill_refine_kernel", s);
            fill_refine_kernel<<<stream_grid(L.ny * L.nx), 256, 0, s>>>(L.w, L.pitch, L.ny, L.nx, lv[l + 1].w, lv[l + 1].pitch);
            HD_LAUNCH_CHECK(); hd_count_launch();
            o.seed_all = true;
        }
        if (int e = pdfill_async(L.z, L.pitch, L.w, L.pitch, L.ny, L.nx, L.ctl, nullptr, s, 0, false, o)) return e;
    }
    *first = nlev ? lv[0] : FillLevel{};
    return HD_OK;
}

// Fill of one whole raster: the fine level starts from the fill of the coarse levels.
static int pdfill_multilevel(const void* z, int64_t z_pitch, void* w, int64_t w_pitch, int64_t ny, int64_t nx, void* workspace,
                             int* visits_out, cudaStream_t s, bool finish)
{
    FillLevel first;
    if (int e = fill_coarse_levels((const float*)z, nullptr, z_pitch, ny, nx, workspace, s, &first)) return e;
    FillOpts fine;
    if (first.w) {
        fine.seed_all = true;
        fine.wc = first.w;
        fine.c_pitch = first.pitch;
    }
    return pdfill_async(z, z_pitch, w, w_pitch, ny, nx, workspace, visits_out, s, 0, finish, fine);
}

extern "C" int hd_pdfill(const void* z, int64_t z_pitch, void* w, int64_t w_pitch, int64_t ny, int64_t nx, void* workspace,
                         int64_t workspace_bytes, int* visits_out, void* stream)
{
    if (!z || !w || !workspace) return HD_ERR_NULL;
    if (ny < 1 || nx < 1 || z_pitch < nx || w_pitch < nx) return HD_ERR_ARG;
    if (workspace_bytes < hd_pdfill_workspace_bytes(ny, nx)) return HD_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    HD_CUDA_OK(cudaMemsetAsync((char*)workspace + STATUS_OFF, 0, sizeof(int), s));
    return pdfill_multilevel(z, z_pitch, w, w_pitch, ny, nx, workspace, visits_out, s, true);
}

// Next round of a banded fill, after a halo exchange: W holds the previous round's result (the first round is
// hd_pdfill_band_start), only the tile rows next to the halo rows are re-seeded.
extern "C" int hd_pdfill_band(const void* z, int64_t z_pitch, void* w, int64_t w_pitch, int64_t ny, int64_t nx,
                              void* workspace, int64_t workspace_bytes, int flags, int* visits_out, void* stream)
{
    if (!z || !w || !workspace) return HD_ERR_NULL;
    if (ny < 1 || nx < 1 || z_pitch < nx || w_pitch < nx || (flags & ~6)) return HD_ERR_ARG;
    if (workspace_bytes < hd_pdfill_workspace_bytes(ny, nx)) return HD_ERR_WORKSPACE;
    return pdfill_async(z, z_pitch, w, w_pitch, ny, nx, workspace, visits_out, (cudaStream_t)stream, flags | 1, false);
}

extern "C" int hd_d8(const void* w, int64_t w_pitch, void* out, int64_t out_pitch, int64_t ny, int64_t nx, void* stream)
{
    if (!w || !out) return HD_ERR_NULL;
    if (ny < 1 || nx < 1 || w_pitch < nx || out_pitch < nx) return HD_ERR_ARG;
    hd_prof_begin("d8_kernel", (cudaStream_t)stream);
    d8_kernel<<<stream_grid(ny * ((nx + 3) / 4)), 256, 0, (cudaStream_t)stream>>>((const float*)w, w_pitch, (uint8_t*)out, out_pitch, ny,
                                                                    nx);
    HD_LAUNCH_CHECK(); hd_count_launch();
    return HD_OK;
}

// hd_pdfill + hd_d8 in one call: the fill, then ONE pass that restores NaN at the nodata cells and writes the flow
// directions (fill_finish_d8_kernel).  Fully asynchronous, capturable in a CUDA graph.
extern "C" int hd_pdfill_d8(const void* z, int64_t z_pitch, void* w, int64_t w_pitch, void* d8, int64_t d8_pitch, int64_t ny,
                            int64_t nx, void* workspace, int64_t workspace_bytes, int* visits_out, void* stream)
{
    if (!z || !w || !d8 || !workspace) return HD_ERR_NULL;
    if (ny < 1 || nx < 1 || z_pitch < nx || w_pitch < nx || d8_pitch < nx) return HD_ERR_ARG;
    if (workspace_bytes < hd_pdfill_workspace_bytes(ny, nx)) return HD_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    HD_CUDA_OK(cudaMemsetAsync((char*)workspace + STATUS_OFF, 0, sizeof(int), s));
    if (int e = pdfill_multilevel(z, z_pitch, w, w_pitch, ny, nx, workspace, visits_out, s, false)) return e;
    return launch_finish_d8(z, z_pitch, w, w_pitch, d8, d8_pitch, ny, nx, workspace, s);
}

// The fused last pass on its own (row-band fill: after the last round and the final halo refresh).
extern "C" int hd_pdfill_finish_d8(const void* z, int64_t z_pitch, void* w, int64_t w_pitch, void* d8, int64_t d8_pitch,
                                   int64_t ny, int64_t nx, const void* workspace, void* stream)
{
    if (!z || !w || !d8) return HD_ERR_NULL;
    if (ny < 1 || nx < 1 || z_pitch < nx || w_pitch < nx || d8_pitch < nx) return HD_ERR_ARG;
    return launch_finish_d8(z, z_pitch, w, w_pitch, d8, d8_pitch, ny, nx, workspace, (cudaStream_t)stream);
}

// Sticky status of the last fill that used this workspace (synchronises the stream): 0 = reached the fixed point.
extern "C" int hd_pdfill_status(const void* workspace, int* status_out, void* stream)
{
    if (!workspace || !status_out) return HD_ERR_NULL;
    static thread_local int* h_word = nullptr;
    if (!h_word) HD_CUDA_OK(cudaHostAlloc((void**)&h_word, 2 * sizeof(int), cudaHostAllocDefault));
    cudaStream_t s = (cudaStream_t)stream;
    HD_CUDA_OK(cudaMemcpyAsync(h_word, (const char*)workspace + STATUS_OFF, sizeof(int), cudaMemcpyDeviceToHost, s));
    HD_CUDA_OK(cudaMemcpyAsync(h_word + 1, &((const FillCtl*)workspace)->pending, sizeof(int), cudaMemcpyDeviceToHost, s));
    HD_CUDA_OK(cudaStreamSynchronize(s));
    *status_out = h_word[0] | (h_word[1] != 0 ? FILL_PENDING : 0);
    return HD_OK;
}

// Row-band fill, after a halo exchange: w_halo = min(w_halo, received row); *lowered (device int) is set to 1 when a
// cell went down.  No host synchronisation: the ranks all-reduce the device flags and read ONE word per round.
extern "C" int hd_halo_min_flag(void* w_halo, const void* received, int64_t nx, int* lowered, void* stream)
{
    if (!w_halo || !received || !lowered) return HD_ERR_NULL;
    if (nx < 1) return HD_ERR_ARG;
    hd_prof_begin("halo_min_kernel", (cudaStream_t)stream);
    halo_min_kernel<<<(int)((nx + 255) / 256 < 64 ? (nx + 255) / 256 : 64), 256, 0, (cudaStream_t)stream>>>(
        (float*)w_halo, (const float*)received, nx, lowered);
    HD_LAUNCH_CHECK(); hd_count_launch();
    return HD_OK;
}

// ---- row-band fill with a GLOBAL multigrid start ---------------------------------------------------------------------
// A band that starts from its own coarse levels solves the drainage structure with the cut rows closed: every later
// round then has to carry corrections from the cut deep into the band, one dependent tile hop after the other (7 rounds
// of ~2 ms on a 36000^2 mosaic over 8 GPUs).  Instead the ranks pool their bands (hd_fill_pool_band), all-gather the
// coarse DEM (1/64 of the cells), every rank fills the WHOLE coarse mosaic (hd_pdfill_coarse: cheap, redundant) and each
// band starts from that global upper bound (hd_pdfill_band_start): the rounds that follow only repair cells next to the
// cuts.  The fixed point is unique, so the result is the same surface, bit for bit.

// Block maxima + outlet marks of a band whose first row is a multiple of 8 in mosaic coordinates.  flags 2 / 4: the top /
// bottom edge of the band is an interior cut, not mosaic frame.  zc, wc: (ceil(ny / 8) x ceil(nx / 8)), pitch c_pitch.
extern "C" int hd_fill_pool_band(const void* z, int64_t z_pitch, int64_t ny, int64_t nx, void* zc, void* wc, int64_t c_pitch,
                                 int flags, void* tile_flags_scratch, void* stream)
{
    if (!z || !zc || !wc || !tile_flags_scratch) return HD_ERR_NULL;
    const int64_t nyc = hd_cdiv(ny, CB), nxc = hd_cdiv(nx, CB);
    if (ny < 1 || nx < 1 || z_pitch < nx || c_pitch < nxc || (flags & ~6)) return HD_ERR_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    hd_prof_begin("fill_pool_kernel", s);
    fill_pool_kernel<<<stream_grid(nyc * nxc), 256, 0, s>>>((const float*)z, z_pitch, ny, nx, (float*)zc, (float*)wc, c_pitch, nyc,
                                                            nxc, (int*)tile_flags_scratch, hd_cdiv(nxc, FT), nullptr, flags & 2,
                                                            flags & 4);
    HD_LAUNCH_CHECK(); hd_count_launch();
    return HD_OK;
}

// Fill of a coarse DEM whose W already carries the outlet marks (finite = outlet at that level, +inf elsewhere), with
// its own multigrid start.  Workspace: hd_pdfill_workspace_bytes(nyc, nxc).
extern "C" int hd_pdfill_coarse(const void* zc, void* wc, int64_t c_pitch, int64_t nyc, int64_t nxc, void* workspace,
                                int64_t workspace_bytes, void* stream)
{
    if (!zc || !wc || !workspace) return HD_ERR_NULL;
    if (nyc < 1 || nxc < 1 || c_pitch < nxc) return HD_ERR_ARG;
    if (workspace_bytes < hd_pdfill_workspace_bytes(nyc, nxc)) return HD_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    HD_CUDA_OK(cudaMemsetAsync((char*)workspace + STATUS_OFF, 0, sizeof(int), s));
    FillLevel first;
    if (int e = fill_coarse_levels((const float*)zc, (const float*)wc, c_pitch, nyc, nxc, workspace, s, &first)) return e;
    if (first.w) {
        hd_prof_begin("fill_refine_kernel", s);
        fill_refine_kernel<<<stream_grid(nyc * nxc), 256, 0, s>>>((float*)wc, c_pitch, nyc, nxc, first.w, first.pitch);
        HD_LAUNCH_CHECK(); hd_count_launch();
    }
    FillOpts top;
    top.preinit = true;
    top.seed_all = true;
    return pdfill_async(zc, c_pitch, wc, c_pitch, nyc, nxc, workspace, nullptr, s, 0, false, top);
}

// First round of a band ([halo row | band | halo row], flags as hd_pdfill_band) from the filled GLOBAL coarse mosaic:
// wc_global (pitch c_pitch) covers the whole mosaic, y_origin = mosaic row of the raster's row 0.
extern "C" int hd_pdfill_band_start(const void* z, int64_t z_pitch, void* w, int64_t w_pitch, int64_t ny, int64_t nx,
                                    void* workspace, int64_t workspace_bytes, int flags, const void* wc_global,
                                    int64_t c_pitch, int64_t y_origin, void* stream)
{
    if (!z || !w || !workspace || !wc_global) return HD_ERR_NULL;
    if (ny < 1 || nx < 1 || z_pitch < nx || w_pitch < nx || (flags & ~6) || y_origin < 0) return HD_ERR_ARG;
    if (workspace_bytes < hd_pdfill_workspace_bytes(ny, nx)) return HD_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    HD_CUDA_OK(cudaMemsetAsync((char*)workspace + STATUS_OFF, 0, sizeof(int), s));
    FillOpts fine;
    fine.status = (int*)((char*)workspace + STATUS_OFF);
    fine.seed_all = true;
    fine.wc = (const float*)wc_global;
    fine.c_pitch = c_pitch;
    fine.wc_y0 = y_origin;
    return pdfill_async(z, z_pitch, w, w_pitch, ny, nx, workspace, nullptr, s, flags, false, fine);
}
