// rrt_split.cuh -- the split render pipeline: trace / media / fold as three kernels over a sample pool in HBM.
//
// Why.  A media sample (reference src/raymarcher.cu:67-115) does not feed back into the trajectory: the densities are
// taken at the pre-step position, the redshift at the post-step velocity, and the result only enters
// `I += e (1 - s) T; T *= s`.  In the fused render_kernel a ray that stays in the disk plane is nevertheless ONE
// dependency chain of 2000 x (RK4 step + disk density + dust density): 17 ms on an empty GPU, 60-70 ms when its SM
// sub-partition is shared six ways -- the tail of every frame and the whole single-frame latency of a band-parallel
// frame on 8 GPUs (profiles/r2_tile_timeline_*.txt).
//
// What.  Per frame, on one stream, in passes that each fit the pool:
//   trace_kernel_p the tracing loop of render_kernel_p (two rays per thread in packed f32x2 registers, FMAD contract; the
//   / trace_kernel scalar trace_ray otherwise), in kMediaEmit mode: an in-zone step stores its sample (32 B: q, v, r, zones)
//                  instead of evaluating it.  A ray that stored nothing is finished on the spot; a ray with samples leaves its
//                  exit state behind them and its tile is queued.  The longest chain is now the trajectory alone.  With no
//                  media code in the tracer the packed step pays off (the fused packed kernel lost its gain to per-half
//                  media calls) and the burst idea extends into the step-size zones (zone bursts, trace_kernel_p).
//   media_kernel   evaluates the queued tiles' samples 128 at a time, every lane busy, with the SAME out-of-line functions
//                  the fused kernel calls (disk_density / dust_base / dust_strands / media_final), the expensive dust
//                  strands compacted once more through shared memory, and overwrites each sample with (e.rgb, s).
//   fold_kernel    one warp per queued group of 32 rays: every lane folds its ray's samples in step order,
//                  `I += e (1 - s) T; T *= s` with the fused kernel's own operations, then background, effects, store.
//   sweep_kernel   the fused code for whatever the enqueued passes left (normally nothing).
// Every ray is traced, sampled and folded by the same arithmetic in the same order as in render_kernel: frames, planes
// and counters are bit-identical (tests/test_gpu_split.py).
//
// Pool layout (one pool per stream in flight, HBM; `slot` = 32 bytes, `row` = 32 slots, one per lane).
//   A tracing warp owns a stream of rows, cut into chunks of `chunk_rows` rows which it takes from the pool with one
//   atomic each (a chunk is used up by successive tiles; the next tile continues in the current chunk).  Lane l's k-th
//   sample of a tile goes to slot l of the tile's k-th row (row 2 k + hf for the two rays of a packed thread) -- so
//   storing a sample needs NO communication between lanes and no allocation: a counter, an address, one 256-bit store.
//   The chunks a tile can possibly reach are taken BEFORE it is traced (see Emitter: nothing atomic may sit in the ray
//   loop; the first forms of this pipeline, which allocated per step or per chunk inside the loop, paid for it with a
//   5-15 ms tail -- profiles/r2_split_history.md).  Rows are as long as the tile's busiest lane needs; slots of lanes with
//   fewer samples stay unused (never written, never read).  A lane that stored samples puts its ray's exit state behind
//   its last one; a lane that stored none finishes its ray on the spot.
//   sample = {q.xyz, v.xyz, r, tag}, tag = zones | zone_index << 2;  after media_kernel the first 16 bytes are
//            {e.r, e.g, e.b, s}, s = -1 for a sample that did not pass the 0.001 density gate (:71) -- or, for a capture
//            (rrt_capture_render), the same 16 bytes are written to a separate array `results[slot]` and the sample stays;
//   state  = {p.xyz, v.xyz, steps | end << 28, 0}, stored by each lane behind its own last sample.
//   A queued group of 32 rays is described by a TileDesc (chunk bases, first row, row stride, samples per lane);
//   media_kernel takes its work as (group, first sample) items of kMediaBatch samples, so a disk-plane tile (64 000 samples)
//   is spread over 500 warps.
// A pass ends when the pool is used up: a warp that cannot take its next tile's worst-case rows puts the tile on the pass's
// redo list and stops; the next pass traces it.  Whatever is left after the last pass the host enqueued is rendered by
// sweep_kernel, so the frame is complete for any pool size and any guess of the pass count.
#pragma once

namespace rrtk {
constexpr int kDescChunks = 40;   // chunks one tile's rows can span: ((1 or 2) * (max_steps + 1) + 1) / chunk_rows + 2 must fit
struct PassCtrl {
    unsigned cursor;          // slots handed out to warps so far (chunk granularity; may overshoot capacity)
    unsigned full;            // an allocation failed: stop taking tiles
    unsigned pend_count;      // tiles queued for media + fold
    unsigned work_count;      // media work items
    unsigned media_ticket, fold_ticket, redo_ticket;
    unsigned redo_out_count;  // tiles given up in this pass
};
struct TileDesc {
    unsigned tile;                    // tile index (8x4 tiles, or 16x4 tiles for the packed tracer)
    unsigned row0;                    // row of this ray group's first sample inside chunk[0]
    unsigned stride_kind;             // row stride between a lane's consecutive samples (1, or 2 for the halves of a packed
                                      // tile, whose rows interleave) | kind << 8: 0 an 8x4 tile, 1 / 2 the even / odd pixels
                                      // of a 16x4 tile (trace_kernel_p)
    unsigned total;                   // samples of the group
    unsigned chunk[kDescChunks];      // slot index of each chunk the tile's rows live in
    unsigned short n[32];             // samples per lane; lane l's exit state sits behind its last sample (its n-th row)
};
struct WorkItem {
    unsigned desc, first;             // TileDesc index, first sample (in lane-major order) of this batch
};
struct SplitArgs {
    uint4* slots;             // 2 x uint4 per slot
    unsigned capacity;        // slots
    unsigned high_water;      // stop taking tiles beyond this cursor (unused since chunks are taken before a tile is traced: 2^32 - 1)
    unsigned chunk_rows;      // power of two
    unsigned chunk_shift;     // log2(chunk_rows)
    PassCtrl* pc;             // this pass
    const PassCtrl* pc_prev;  // previous pass (its redo list is this pass's first work), or null
    const unsigned* redo_in;
    unsigned* redo_out;
    unsigned redo_cap;
    TileDesc* desc;           // one per queued tile
    WorkItem* work;
    unsigned work_cap;
    unsigned* stats;          // [0] split passes that took tiles, [1] tiles rendered by sweep_kernel, [2] tiles taken by the split passes
    unsigned pass;
    unsigned tile16;          // tickets and redo lists count 16x4 tiles (the packed tracer) instead of 8x4 tiles
    uint4* results;           // media_kernel<true> / fold_kernel<true>: {e.rgb, s} per slot, indexed like `slots` (rrt_capture)
};
// The tracers are indexed [lens][spin != 0]; lens: the ray source of the LENS template argument (kRaysPinhole, kRaysLens,
// kRaysPano).  Media and fold read only samples and planes and serve every source.
struct SplitKernels {
    void (*trace[kRaySources][2])(const FrameArgs, const SplitArgs, const LensArgs);
    void (*trace_packed[kRaySources][2])(const FrameArgs, const SplitArgs, const LensArgs);   // two rays per thread (FMAD contract only, else null)
    void (*media)(const FrameArgs, const SplitArgs);
    void (*fold)(const FrameArgs, const SplitArgs);
    void (*sweep[kRaySources][2])(const FrameArgs, const SplitArgs, const LensArgs);
    void (*media_results)(const FrameArgs, const SplitArgs);   // media_kernel<true>: the samples stay, results go to S.results
    void (*fold_results)(const FrameArgs, const SplitArgs);    // fold_kernel<true>: reads them from there
};
const SplitKernels* rrt_split_kernels_strict();
const SplitKernels* rrt_split_kernels_fmad();
}  // namespace rrtk

using rrtk::PassCtrl;
using rrtk::SplitArgs;
using rrtk::TileDesc;
using rrtk::WorkItem;
using rrtk::kDescChunks;

namespace {

constexpr unsigned kNone = 0xffffffffu;   // "no chunk" / allocation failure / "no tile"
constexpr int kMediaBlock = 128;          // media_kernel CTA
constexpr int kMediaBatch = 128;          // samples per media work item

// pixel of a lane in a tile (the centre-outwards tile order of render_kernel)
struct TilePix {
    int x, y, ly;
    bool valid;
};
__device__ __forceinline__ TilePix tile_pixel(const FrameArgs& A, unsigned tile, int lane) {
    const int ntx = (A.w + kRTileW - 1) / kRTileW;
    const int nty = (A.local_rows + kRTileH - 1) / kRTileH;
    const int tx = (int)(tile % (unsigned)ntx), k = (int)(tile / (unsigned)ntx);
    const int ty = centre_out_row(k, nty);
    TilePix t;
    t.x = tx * kRTileW + (lane & (kRTileW - 1));
    t.ly = ty * kRTileH + lane / kRTileW;
    t.y = band_row(A, t.ly);
    t.valid = t.x < A.w && t.ly < A.local_rows && t.y < A.h;
    return t;
}
__device__ __forceinline__ unsigned num_tiles(const FrameArgs& A) {
    return (unsigned)(((A.w + kRTileW - 1) / kRTileW) * ((A.local_rows + kRTileH - 1) / kRTileH));
}

// the same for the packed tracer's 16x4 tiles: thread (lane & 7, lane >> 3) owns pixels (2 lx + hf, ly), hf = 0, 1
constexpr int kTile16W = 16, kTile16H = 4;
__device__ __forceinline__ TilePix tile_pixel16(const FrameArgs& A, unsigned tile, int lane, int hf) {
    const int ntx = (A.w + kTile16W - 1) / kTile16W;
    const int nty = (A.local_rows + kTile16H - 1) / kTile16H;
    const int tx = (int)(tile % (unsigned)ntx), k = (int)(tile / (unsigned)ntx);
    const int ty = centre_out_row(k, nty);
    TilePix t;
    t.x = tx * kTile16W + 2 * (lane & 7) + hf;
    t.ly = ty * kTile16H + (lane >> 3);
    t.y = band_row(A, t.ly);
    t.valid = t.x < A.w && t.ly < A.local_rows && t.y < A.h;
    return t;
}
__device__ __forceinline__ unsigned num_tiles16(const FrameArgs& A) {
    return (unsigned)(((A.w + kTile16W - 1) / kTile16W) * ((A.local_rows + kTile16H - 1) / kTile16H));
}

// Next tile of a pass (lane 0 decides, everyone gets it): the previous pass's redo list first, then fresh tickets.
// `may_stop` lets a split pass end early (pool used up).
__device__ __forceinline__ unsigned next_tile(const FrameArgs& A, const SplitArgs& S, unsigned ntiles, bool may_stop) {
    unsigned tile = kNone;
    if ((threadIdx.x & 31) == 0) {
        bool stop = false;
        if (may_stop) {
            const volatile PassCtrl* pc = S.pc;
            stop = pc->full != 0u || pc->cursor > S.high_water;
        }
        if (!stop) {
            const unsigned n_redo = S.pc_prev ? S.pc_prev->redo_out_count : 0u;
            if (n_redo) {
                const unsigned t = atomicAdd(&S.pc->redo_ticket, 1u);
                if (t < n_redo && t < S.redo_cap) tile = S.redo_in[t];
            }
            if (tile == kNone) {
                const unsigned t = atomicAdd(A.ticket, 1u);
                if (t < ntiles) tile = t;
            }
        }
    }
    return __shfl_sync(0xffffffffu, tile, 0);
}

// ---- emitter: the sample rows of one tracing warp -----------------------------------------------------------------
// Shared memory per warp: tab[j] = slot index of the j-th chunk the CURRENT tile's rows can touch; tab[0] is the chunk the
// warp was in when the tile began.  Chunks a tile did not reach stay in the table for the next tile.
// A slot is one 32-byte sector: it is written with ONE 256-bit store (sm_100: STG.256) instead of two halves.
__device__ __forceinline__ void pool_put(uint4* slots, unsigned slot, uint4 a, uint4 b) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(slots + 2ull * slot), "r"(a.x), "r"(a.y), "r"(a.z),
                 "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w)
                 : "memory");
}
// A chunk for the calling lane's table entry (kNone: the pool is exhausted).  Only called between tiles.
__device__ __forceinline__ unsigned claim_chunk(const SplitArgs& S) {
    if (*(volatile unsigned*)&S.pc->full) return kNone;
    const unsigned chunk_slots = S.chunk_rows * 32u;
    const unsigned nb = atomicAdd(&S.pc->cursor, chunk_slots);
    if (nb > S.capacity || S.capacity - nb < chunk_slots) {
        atomicExch(&S.pc->full, 1u);
        return kNone;
    }
    return nb;
}
// NOTHING in here may contain an atomic, a warp-synchronous intrinsic or a call to code that does: with one of those in
// trace_ray's loop nvcc gives the loop a weaker convergence barrier (BSSY instead of BSSY.RELIABLE), the lanes of a tile
// drift apart, vacuum bursts run with half the lanes and a disk-plane tile takes 4x longer (measured: tools/r2_gpu21/27/30.sh,
// profiles/r2_split_history.md).  So every chunk a tile can possibly touch is taken BEFORE the tile is traced
// (trace_kernel) and storing a sample is pure arithmetic plus one table look-up per chunk_rows samples.
struct Emitter {
    const SplitArgs& S;
    const unsigned* tab;
    unsigned row0;      // first row of the current tile inside tab[0] (warp-uniform)
    unsigned count;     // samples this lane has stored for the current tile
    unsigned cur;       // slot of this lane in its next row
    unsigned left;      // rows left in the chunk `cur` points into (0: look the next row's chunk up first)
    float isco, disk_out;

    __device__ __forceinline__ Emitter(const SplitArgs& s, const unsigned* t, const Consts& C)
        : S(s), tab(t), row0(0u), count(0u), cur(0u), left(0u), isco(C.isco), disk_out(C.disk_out) {}

    // slot of lane `lane` in row `row` of the current tile (rows counted from the tile's first)
    __device__ __forceinline__ unsigned row_slot(unsigned row, unsigned lane, unsigned& rows_left) const {
        const unsigned pos = row0 + row, off = pos & (S.chunk_rows - 1u);
        rows_left = S.chunk_rows - off;
        return tab[pos >> S.chunk_shift] + off * 32u + lane;
    }
    // one in-zone sample (trace_ray, kMediaEmit)
    __device__ __forceinline__ void emit(V3 q, V3 v, float r, int zone_index, unsigned z) {
        // Outside the ring ISCO <= R <= DISK_OUT both density functions return 0 before anything else
        // (densities.h:21-22, 70-71): such a sample cannot pass the gate of raymarcher.cu:71 and is not stored.
        const float R = sqrtf(rrt::ring_r2(q));
        if (R < isco || R > disk_out) return;
        if (left == 0u) cur = row_slot(count, threadIdx.x & 31u, left);
        pool_put(S.slots, cur, make_uint4(__float_as_uint(q.x), __float_as_uint(q.y), __float_as_uint(q.z), __float_as_uint(v.x)),
                 make_uint4(__float_as_uint(v.y), __float_as_uint(v.z), __float_as_uint(r), z | ((unsigned)zone_index << 2)));
        cur += 32u;
        --left;
        ++count;
    }
};

struct TileCounters {
    unsigned long long steps = 0, disk = 0, dust = 0, dense = 0;
    unsigned cap = 0, esc = 0, exh = 0, touch = 0;
    __device__ __forceinline__ void flush(unsigned long long* counters) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            steps += __shfl_xor_sync(0xffffffffu, steps, o);
            disk += __shfl_xor_sync(0xffffffffu, disk, o);
            dust += __shfl_xor_sync(0xffffffffu, dust, o);
            dense += __shfl_xor_sync(0xffffffffu, dense, o);
            cap += __shfl_xor_sync(0xffffffffu, cap, o);
            esc += __shfl_xor_sync(0xffffffffu, esc, o);
            exh += __shfl_xor_sync(0xffffffffu, exh, o);
            touch += __shfl_xor_sync(0xffffffffu, touch, o);
        }
        if ((threadIdx.x & 31) == 0 && counters) {
            if (steps) atomicAdd(counters + 0, steps);
            if (disk) atomicAdd(counters + 1, disk);
            if (dust) atomicAdd(counters + 2, dust);
            if (dense) atomicAdd(counters + 3, dense);
            if (cap) atomicAdd(counters + 4, (unsigned long long)cap);
            if (esc) atomicAdd(counters + 5, (unsigned long long)esc);
            if (exh) atomicAdd(counters + 6, (unsigned long long)exh);
            if (touch) atomicAdd(counters + 7, (unsigned long long)touch);
        }
    }
};

// Queues one group of 32 rays (an 8x4 tile, or one half of a packed 16x4 tile) for media_kernel and fold_kernel: its
// descriptor and its media work items.  Called by the whole warp; `count` = samples of this lane's ray.
__device__ __forceinline__ void queue_group(const SplitArgs& S, const unsigned* tab, unsigned tile, unsigned row0, unsigned stride, unsigned kind,
                                            unsigned count, int lane) {
    const unsigned total = __reduce_add_sync(0xffffffffu, count);
    const unsigned n_items = (total + kMediaBatch - 1) / kMediaBatch;
    unsigned di = 0u, wi = 0u;
    if (lane == 0) {
        di = atomicAdd(&S.pc->pend_count, 1u);
        wi = atomicAdd(&S.pc->work_count, n_items);
    }
    di = __shfl_sync(0xffffffffu, di, 0);
    wi = __shfl_sync(0xffffffffu, wi, 0);
    TileDesc* d = S.desc + di;
    if (lane == 0) { d->tile = tile; d->row0 = row0; d->stride_kind = stride | (kind << 8); d->total = total; }
    d->n[lane] = (unsigned short)count;
    for (int j = lane; j < kDescChunks; j += 32) d->chunk[j] = tab[j];
    for (unsigned i = (unsigned)lane; i < n_items; i += 32u)
        if (wi + i < S.work_cap) S.work[wi + i] = WorkItem{di, i * kMediaBatch};
}
// The next tile continues `used` rows further on: drop the chunks that are used up, keep the rest of the stock.
__device__ __forceinline__ void advance_rows(const SplitArgs& S, unsigned* tab, unsigned& row_next, unsigned used, int lane) {
    const unsigned pos = row_next + used, jn = pos >> S.chunk_shift;
    unsigned keep[(kDescChunks + 31) / 32];
#pragma unroll
    for (int k = 0; k < (kDescChunks + 31) / 32; ++k) {
        const unsigned j = (unsigned)(k * 32 + lane) + jn;
        keep[k] = j < (unsigned)kDescChunks ? tab[j] : kNone;
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < (kDescChunks + 31) / 32; ++k)
        if (k * 32 + lane < kDescChunks) tab[k * 32 + lane] = keep[k];
    row_next = pos & (S.chunk_rows - 1u);
    __syncwarp();
}
// Before a tile is traced: every chunk its rows can reach (`rows` of them from row_next on) is taken.  False: pool used up.
__device__ __forceinline__ bool stock_chunks(const SplitArgs& S, unsigned* tab, unsigned row_next, unsigned rows, int lane) {
    const unsigned last = (row_next + rows) >> S.chunk_shift;
    bool ok = true;
    for (unsigned j = (unsigned)lane; j <= last && j < (unsigned)kDescChunks; j += 32u)
        if (tab[j] == kNone) {
            const unsigned nb = claim_chunk(S);
            if (nb == kNone) ok = false; else tab[j] = nb;
        }
    __syncwarp();
    return __all_sync(0xffffffffu, ok);
}
__device__ __forceinline__ void redo_later(const SplitArgs& S, unsigned tile, int lane) {
    if (lane == 0) {
        const unsigned i = atomicAdd(&S.pc->redo_out_count, 1u);
        if (i < S.redo_cap) S.redo_out[i] = tile;
    }
}

// ---- pass kernel 1: trajectories ------------------------------------------------------------------------------------
template <bool SPIN, int LENS>
__global__ void __launch_bounds__(kRenderBlock, kMinBlocks) trace_kernel(const __grid_constant__ FrameArgs A,
                                                                              const __grid_constant__ SplitArgs S,
                                                                              const __grid_constant__ LensArgs L) {
    __shared__ unsigned chunk_tab[kRenderBlock / 32][kDescChunks];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned* tab = chunk_tab[warp];
    for (int j = lane; j < kDescChunks; j += 32) tab[j] = kNone;
    __syncwarp();
    const unsigned ntiles = num_tiles(A);
    TileCounters cnt;
    Emitter em(S, tab, A.C);
    unsigned taken = 0;
    unsigned row_next = 0;   // first free row inside tab[0] (warp-uniform)

    for (;;) {
        const unsigned tile = next_tile(A, S, ntiles, true);
        if (tile == kNone) break;
        ++taken;
        // every chunk this tile's rows can reach (max_steps sample rows + one for the exit states) is taken now
        if (!stock_chunks(S, tab, row_next, (unsigned)A.C.max_steps + 1u, lane)) {
            redo_later(S, tile, lane);   // the pool is used up: the next pass (or the sweep) takes this tile
            continue;                    // (next_tile sees the full pool and ends the pass for this warp)
        }
        const TilePix px = tile_pixel(A, tile, lane);
        RayResult R;
        R.steps = 0; R.n_disk = R.n_dust = R.n_dense = 0;
        R.captured = R.touched = R.exhausted = false;
        R.p = R.v = mk(0.f, 0.f, 0.f);
        R.T = 1.0f; R.I[0] = R.I[1] = R.I[2] = 0.f;
        R.uvx = R.uvy = 0.f;
        em.row0 = row_next;
        em.count = 0u;
        em.left = 0u;
#ifdef RRT_WITH_TILE_LOG
        unsigned long long t_begin = 0;
        if (A.tile_log) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_begin));
#endif
        if (px.valid) trace_ray<SPIN, kMediaEmit, LENS>(A, L, px.x, px.y, R, em);
        __syncwarp();
#ifdef RRT_WITH_TILE_LOG   // profiling build only (rrt_debug_tile_log): when did this warp trace which tile
        if (A.tile_log) {
            const int most = __reduce_max_sync(0xffffffffu, R.steps);
            if (lane == 0 && tile < A.tile_log_cap) {
                unsigned long long t_end;
                unsigned smid;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_end));
                asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
                unsigned long long* e = A.tile_log + 4ull * tile;
                const int ntx = (A.w + kRTileW - 1) / kRTileW;
                e[0] = t_begin; e[1] = t_end; e[2] = ((unsigned long long)(px.ly / kRTileH) << 32) | (unsigned)(tile % (unsigned)ntx);
                e[3] = ((unsigned long long)smid << 32) | (unsigned)most;
            }
        }
#endif
        const unsigned n_rows = __reduce_max_sync(0xffffffffu, em.count);
        const unsigned end = (R.captured ? kEndCaptured : 0u) | (R.exhausted ? kEndExhausted : 0u);
        if (em.count == 0u) {   // nothing stored: this ray is finished here
            if (px.valid) finish_ray_inl(A, px.x, px.y, px.ly, R.uvx, R.uvy, 0.f, 0.f, 0.f, R.T, R.p, R.v, R.steps, end);
        } else {                // the exit state goes behind the ray's samples; fold_kernel finishes it
            unsigned rows_left;
            pool_put(S.slots, em.row_slot(em.count, (unsigned)lane, rows_left),
                     make_uint4(__float_as_uint(R.p.x), __float_as_uint(R.p.y), __float_as_uint(R.p.z), __float_as_uint(R.v.x)),
                     make_uint4(__float_as_uint(R.v.y), __float_as_uint(R.v.z), (unsigned)R.steps | (end << 28), 0u));
        }
        if (n_rows != 0u) {     // the tile is queued for media + fold
            queue_group(S, tab, tile, em.row0, 1u, 0u, em.count, lane);
            advance_rows(S, tab, row_next, n_rows + 1u, lane);
        }
        if (px.valid) {
            cnt.steps += (unsigned)R.steps;
            cnt.disk += R.n_disk; cnt.dust += R.n_dust;
            cnt.cap += R.captured; cnt.exh += R.exhausted; cnt.esc += (!R.captured && !R.exhausted);
        }
    }
    if (lane == 0 && taken) {
        atomicMax(S.stats + 0, S.pass + 1u);
        atomicAdd(S.stats + 2, taken);
    }
    cnt.flush(A.counters);
}

#if RRT_FMAD
// ---- pass kernel 1, packed: trajectories with two rays per thread (rrt_packed.cuh) ------------------------------------------
// The tracing loop of render_kernel_p (16x4-pixel tiles, thread (lx, ly) owns pixels (2 lx, ly) and (2 lx + 1, ly) as the halves
// of f32x2 registers, warp-uniform vacuum bursts, checked iterations per half) with the media sample of an in-zone step
// stored instead of evaluated.  The packed step is ~6 % faster than the scalar one on the FMA pipe (profiles/r2_rf_model.md) and
// the fused packed kernel lost that to its per-half media calls; here there are none.  The rows of the two halves interleave
// (half hf's k-th sample row is row 2 k + hf of the tile), each half is queued as its own group of 32 rays.
struct Emitter2 {
    const SplitArgs& S;
    const unsigned* tab;
    unsigned row0;
    unsigned count[2];
    float isco, disk_out;
    __device__ __forceinline__ Emitter2(const SplitArgs& s, const unsigned* t, const Consts& C)
        : S(s), tab(t), row0(0u), isco(C.isco), disk_out(C.disk_out) { count[0] = count[1] = 0u; }
    __device__ __forceinline__ unsigned slot(int hf, unsigned k, unsigned lane) const {
        const unsigned pos = row0 + 2u * k + (unsigned)hf;
        return tab[pos >> S.chunk_shift] + (pos & (S.chunk_rows - 1u)) * 32u + lane;
    }
    __device__ __forceinline__ void emit(int hf, V3 q, V3 v, float r, int zone_index, unsigned z) {
        const float R = sqrtf(rrt::ring_r2(q));   // see Emitter::emit
        if (R < isco || R > disk_out) return;
        pool_put(S.slots, slot(hf, count[hf], threadIdx.x & 31u),
                 make_uint4(__float_as_uint(q.x), __float_as_uint(q.y), __float_as_uint(q.z), __float_as_uint(v.x)),
                 make_uint4(__float_as_uint(v.y), __float_as_uint(v.z), __float_as_uint(r), z | ((unsigned)zone_index << 2)));
        ++count[hf];
    }
};

template <bool SPIN, int LENS>
__global__ void __launch_bounds__(32, kPackedMinBlocks) trace_kernel_p(const __grid_constant__ FrameArgs A, const __grid_constant__ SplitArgs S,
                                                                          const __grid_constant__ LensArgs L) {
    using rrtp::F2;
    using rrtp::V3x2;
    __shared__ unsigned chunk_tab[kDescChunks];
    const Consts& C = A.C;
    const int lane = threadIdx.x & 31;
    unsigned* tab = chunk_tab;
    for (int j = lane; j < kDescChunks; j += 32) tab[j] = kNone;
    __syncwarp();
    const unsigned ntiles = num_tiles16(A);
    const int max_steps = C.max_steps;
    const bool want_disk = (C.flags & RRT_FLAG_DISK) != 0, want_dust = (C.flags & RRT_FLAG_DUST) != 0;
    const float zone_rmax = fmaxf(18.0f, fmaxf(C.disk_zone_r, C.dust_zone_r));
    const V3 cam_p = mk(A.cam.pos[0], A.cam.pos[1], A.cam.pos[2]);
    const bool fast_ok = (LENS == kRaysLens ? L.near != 0 : rrt::dot3(cam_p, cam_p) < 1.0e8f) && C.acc_rmin < C.horizon_r && C.horizon_r >= 1e-3f;
    const float redo_below = fast_ok ? C.acc_rmin : __int_as_float(0x7f800000);
    const V3 park_p = mk(0.0f, 100.0f, 0.0f), park_v = mk(0.0f, 0.0f, 0.0f);   // inert state of a finished half, see render_kernel_p
    const float burst_min = fmaxf(zone_rmax, fmaxf(C.horizon_r, redo_below));
    const float burst_margin = 1.25f * (float)kBurst * C.h[0];
    const float burst_lo = burst_min + burst_margin, burst_hi = 250.0f - burst_margin;
    // Zone bursts: the same idea inside the two step-size zones that matter -- near the hole (r < 18, step h[1]) and in the
    // disk zone (r >= 18, |y| < DISK_H * 5, r < DISK_OUT + 5, step h[2]); reference raymarcher.cu:56-62.  While every ray of
    // the warp sits well inside SOME zone (each its own: vacuum counts), kBurst steps are taken with each ray's zone step
    // and none of the per-step zone logic; each step still stores its media sample (the zone flags of a sample do not
    // influence the trajectory).  Afterwards the burst is validated -- every pre-step state of a ray must have been in the
    // zone its step came from, at or above the horizon radius (:47), and every pre-step and stage radius at or above
    // redo_below (the branch-free domain); in the disk zone also at most 250 (the escape test, :120, which the near-hole
    // zone's r < 18 already rules out) -- and rolled back otherwise (the samples it stored are overwritten).  None of these
    // thresholds is ordered against 18 or 250 in general (a hole with event_horizon > 17.8 puts the horizon inside the disk
    // zone, disk_out > 245 puts the escape sphere inside it, and without fast_ok redo_below is infinite), so each zone's
    // window and validation take all of them.
    const float zb_floor = fmaxf(C.horizon_r, redo_below);
    const float disk_floor = fmaxf(18.0f, zb_floor);
    const float zb_m1 = 1.25f * (float)kBurst * C.h[1], zb_m2 = 1.25f * (float)kBurst * C.h[2];
    const float near_lo = zb_floor + zb_m1, near_hi = 18.0f - zb_m1;
    const float disk_lo = disk_floor + zb_m2, disk_hi = fminf(C.disk_zone_r, 250.0f) - zb_m2, disk_y = C.disk_zone_y - zb_m2;
    const float kInf = __int_as_float(0x7f800000);
    auto zone_for_burst = [&](float r, float ay) -> int {
        if (r >= burst_lo && r <= burst_hi) return 0;
        if (r >= near_lo && r <= near_hi) return 1;
        if (r >= disk_lo && r <= disk_hi && ay < disk_y) return 2;
        return -1;
    };
    auto burst_was_valid = [&](int m, float mn, float mx, float my) -> bool {
        if (m == 0) return mn >= burst_min && mx <= 250.0f;                      // no zone, no medium, no escape test to miss
        if (m == 1) return mn >= zb_floor && mx < 18.0f;                         // :56
        return mn >= disk_floor && mx < C.disk_zone_r && mx <= 250.0f && my < C.disk_zone_y;   // :57 and not :56
    };
    TileCounters cnt;
    Emitter2 em(S, tab, C);
    unsigned taken = 0, row_next = 0;

    for (;;) {
        const unsigned tile = next_tile(A, S, ntiles, true);
        if (tile == kNone) break;
        ++taken;
        if (!stock_chunks(S, tab, row_next, 2u * ((unsigned)max_steps + 1u) + 1u, lane)) {
            redo_later(S, tile, lane);
            continue;
        }
        const TilePix px0 = tile_pixel16(A, tile, lane, 0), px1 = tile_pixel16(A, tile, lane, 1);
        const int x0 = px0.x, y = px0.y, ly = px0.ly;
        bool alive[2] = {px0.valid, px1.valid};
        em.row0 = row_next;
        em.count[0] = em.count[1] = 0u;
        if (alive[0] || alive[1]) {
            V3x2 P, V;
            {
                // the two halves are neighbouring pixels: with kRaysLens each starts from its own camera, with kRaysPano
                // each takes its own column
                const rrt_camera &camA = ray_camera<LENS>(A, L, x0, y), &camB = ray_camera<LENS>(A, L, x0 + 1, y);
                const V3 vA = alive[0] ? ray_dir_src<LENS>(A, L, camA, x0, y) : park_v, vB = alive[1] ? ray_dir_src<LENS>(A, L, camB, x0 + 1, y) : park_v;
                const V3 pA = alive[0] ? (LENS == kRaysLens ? cam_pos(camA) : cam_p) : park_p, pB = alive[1] ? (LENS == kRaysLens ? cam_pos(camB) : cam_p) : park_p;
                P.x = rrtp::pk(pA.x, pB.x); P.y = rrtp::pk(pA.y, pB.y); P.z = rrtp::pk(pA.z, pB.z);
                V.x = rrtp::pk(vA.x, vB.x); V.y = rrtp::pk(vA.y, vB.y); V.z = rrtp::pk(vA.z, vB.z);
            }
            unsigned n_disk = 0, n_dust = 0;
            // retire one half: a ray without samples is finished here, one with samples leaves its exit state behind them
            auto retire = [&](int hf, int steps, unsigned end) {
                const V3 p = rrtp::half_of(P, hf), v = rrtp::half_of(V, hf);
                if (em.count[hf] == 0u) {
                    finish_ray(A, x0 + hf, y, ly, 0.f, 0.f, 0.f, (end & kEndCaptured) ? 0.0f : 1.0f, p, v, steps, end);
                } else {
                    pool_put(S.slots, em.slot(hf, em.count[hf], (unsigned)lane),
                             make_uint4(__float_as_uint(p.x), __float_as_uint(p.y), __float_as_uint(p.z), __float_as_uint(v.x)),
                             make_uint4(__float_as_uint(v.y), __float_as_uint(v.z), (unsigned)steps | (end << 28), 0u));
                }
                cnt.steps += (unsigned)steps;
                cnt.cap += (end & kEndCaptured) ? 1u : 0u;
                cnt.exh += (end & kEndExhausted) ? 1u : 0u;
                cnt.esc += (end & (kEndCaptured | kEndExhausted)) ? 0u : 1u;
                alive[hf] = false;
                rrtp::set_half(P, hf, park_p);
                rrtp::set_half(V, hf, park_v);
            };

            int it = 0;
            int burst_after = 0, zburst_after = 0;
            F2 R2 = rrtp::norm2_loop_2(P);
            F2 R = rrtp::sqrt2(R2);                                                              // :44
            for (;;) {
                // ---- phase 1: unchecked vacuum bursts, warp-uniform (see render_kernel_p / trace_ray) ------------------
                {
                    const unsigned in_loop = __activemask();
                    const F2 H = rrtp::bc(C.h[0]), HH = rrtp::bc(C.hh[0]), H6 = rrtp::bc(C.h6[0]);
#pragma unroll 1
                    for (;;) {
                        float r0, r1;
                        rrtp::upk(R, r0, r1);
                        const bool ok = fminf(r0, r1) >= burst_lo && fmaxf(r0, r1) <= burst_hi && it >= burst_after && it + kBurst < max_steps;
                        if (!(ok && __activemask() == in_loop)) break;
                        const V3x2 Ps = P, Vs = V;
                        const F2 R2s = R2, Rs = R;
                        float mn = fminf(r0, r1), mx = fmaxf(r0, r1);
#pragma unroll 1
                        for (int kb = 0; kb < kBurst; ++kb) {
                            float ma, mb;
                            rrtp::rk4_step2<SPIN>(C, P, V, H, HH, H6, R2, R, ma, mb);            // :64
                            R2 = rrtp::norm2_loop_2(P);
                            R = rrtp::sqrt2(R2);
                            rrtp::upk(R, r0, r1);
                            mn = fminf(mn, fminf(fminf(ma, mb), fminf(r0, r1)));
                            mx = fmaxf(mx, fmaxf(r0, r1));
                        }
                        if (mn >= burst_min && mx <= 250.0f) { it += kBurst; continue; }
                        P = Ps; V = Vs; R2 = R2s; R = Rs;
                        burst_after = it + kBurst;
                        break;
                    }
                    // ---- phase 1b: zone bursts, one zone per ray --------------------------------------------------------------
#pragma unroll 1
                    for (;;) {
                        float r0, r1, y0, y1;
                        rrtp::upk(R, r0, r1);
                        rrtp::upk(P.y, y0, y1);
                        // the zone each ray is well inside of: 0 vacuum, 1 near the hole, 2 disk zone, -1 none (a parked half: vacuum)
                        const int m0 = !alive[0] ? 0 : zone_for_burst(r0, fabsf(y0)), m1 = !alive[1] ? 0 : zone_for_burst(r1, fabsf(y1));
                        const bool ok = it >= zburst_after && it + kBurst < max_steps && m0 >= 0 && m1 >= 0;
                        if (!(ok && __activemask() == in_loop)) break;
                        const F2 ZH = rrtp::pk(C.h[m0], C.h[m1]), ZHH = rrtp::pk(C.hh[m0], C.hh[m1]), ZH6 = rrtp::pk(C.h6[m0], C.h6[m1]);
                        const V3x2 Ps = P, Vs = V;
                        const F2 R2s = R2, Rs = R;
                        const unsigned c0s = em.count[0], c1s = em.count[1];
                        unsigned bd = 0, bu = 0;
                        float mn0 = kInf, mx0 = 0.0f, my0 = 0.0f, mn1 = kInf, mx1 = 0.0f, my1 = 0.0f;
#pragma unroll 1
                        for (int kb = 0; kb < kBurst; ++kb) {
                            const V3x2 Q = P;
                            float q0, q1, yy0, yy1, ma, mb;
                            rrtp::upk(R, q0, q1);             // pre-step radii
                            rrtp::upk(P.y, yy0, yy1);
                            yy0 = fabsf(yy0); yy1 = fabsf(yy1);
                            rrtp::rk4_step2<SPIN>(C, P, V, ZH, ZHH, ZH6, R2, R, ma, mb);         // :64
                            R2 = rrtp::norm2_loop_2(P);
                            R = rrtp::sqrt2(R2);
                            mn0 = fminf(mn0, fminf(q0, ma)); mx0 = fmaxf(mx0, q0); my0 = fmaxf(my0, yy0);
                            mn1 = fminf(mn1, fminf(q1, mb)); mx1 = fmaxf(mx1, q1); my1 = fmaxf(my1, yy1);
                            if (alive[0] && q0 < zone_rmax) {
                                const unsigned z = (yy0 < C.disk_zone_y && q0 < C.disk_zone_r && want_disk ? 1u : 0u) |
                                                   (yy0 < C.dust_zone_y && q0 < C.dust_zone_r && want_dust ? 2u : 0u);      // :57-58, :67
                                if (z) { bd += z & 1u; bu += z >> 1; em.emit(0, rrtp::half_of(Q, 0), rrtp::half_of(V, 0), q0, m0, z); }
                            }
                            if (alive[1] && q1 < zone_rmax) {
                                const unsigned z = (yy1 < C.disk_zone_y && q1 < C.disk_zone_r && want_disk ? 1u : 0u) |
                                                   (yy1 < C.dust_zone_y && q1 < C.dust_zone_r && want_dust ? 2u : 0u);
                                if (z) { bd += z & 1u; bu += z >> 1; em.emit(1, rrtp::half_of(Q, 1), rrtp::half_of(V, 1), q1, m1, z); }
                            }
                        }
                        // every pre-step state of a ray in the zone its step size came from (:56-62), above the horizon (:47), short
                        // of the escape test (:120) and in the branch-free domain; `mn` also holds the stage radii
                        const bool good = (!alive[0] || burst_was_valid(m0, mn0, mx0, my0)) && (!alive[1] || burst_was_valid(m1, mn1, mx1, my1));
                        if (good) { it += kBurst; n_disk += bd; n_dust += bu; continue; }
                        P = Ps; V = Vs; R2 = R2s; R = Rs;
                        em.count[0] = c0s; em.count[1] = c1s;
                        zburst_after = it + kBurst;
                        break;
                    }
                }
                // ---- phase 2: checked iterations ----------------------------------------------------------------------
                bool rewind = false;
#pragma unroll 1
                while (it < max_steps) {                                                         // :41
                    float r[2];
                    rrtp::upk(R, r[0], r[1]);
                    bool parked = false;
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf)
                        if (alive[hf] && r[hf] < C.horizon_r) {                                  // :47-51
                            retire(hf, it, kEndCaptured);
                            parked = true;
                        }
                    if (!(alive[0] || alive[1])) break;
                    if (parked) {
                        R2 = rrtp::norm2_loop_2(P);
                        R = rrtp::sqrt2(R2);
                        rrtp::upk(R, r[0], r[1]);
                    }
                    float h[2], h6[2];
                    unsigned zones[2];
                    int zidx[2];
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf) {
                        h[hf] = C.h[0];
                        h6[hf] = C.h6[0];
                        zones[hf] = 0u;
                        zidx[hf] = 0;
                        if (r[hf] < zone_rmax) {
                            const float py = rrtp::half_of(P.y, hf);
                            const bool near_bh = r[hf] < 18.0f;                                  // :56
                            const bool disk_zone = fabsf(py) < C.disk_zone_y && r[hf] < C.disk_zone_r;   // :57
                            const bool dust_zone = fabsf(py) < C.dust_zone_y && r[hf] < C.dust_zone_r;   // :58
                            const int zi = near_bh ? 1 : (disk_zone ? 2 : (dust_zone ? 3 : 0));  // :60-62
                            h[hf] = C.h[zi];
                            h6[hf] = C.h6[zi];
                            zidx[hf] = zi;
                            zones[hf] = (disk_zone && want_disk ? 1u : 0u) | (dust_zone && want_dust ? 2u : 0u);   // :67
                        }
                    }
                    const F2 H = rrtp::pk(h[0], h[1]), H6 = rrtp::pk(h6[0], h6[1]);
                    const F2 HH = rrtp::mul2(H, rrtp::bc(0.5f));   // exact (power of two)
                    const V3x2 Q = P, Vin = V;         // pre-step state: media and the escape test use Q (:68-69, :120)
                    float rmin[2];
                    rrtp::rk4_step2<SPIN>(C, P, V, H, HH, H6, R2, R, rmin[0], rmin[1]);          // :64
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf)
                        if (alive[hf] && !(rmin[hf] >= redo_below)) {   // general-domain redo, see trace_ray
                            const PV sres = rk4_step_general<SPIN>(C, rrtp::half_of(Q, hf), rrtp::half_of(Vin, hf), h[hf], h[hf] * 0.5f, h6[hf]);
                            rrtp::set_half(P, hf, sres.p);
                            rrtp::set_half(V, hf, sres.v);
                        }
                    ++it;
                    const F2 R2n = rrtp::norm2_loop_2(P);
                    const F2 Rn = rrtp::sqrt2(R2n);
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf)
                        if (alive[hf] && zones[hf]) {                                            // :67
                            n_disk += zones[hf] & 1u;
                            n_dust += zones[hf] >> 1;
                            em.emit(hf, rrtp::half_of(Q, hf), rrtp::half_of(V, hf), r[hf], zidx[hf], zones[hf]);
                        }
                    bool gone = false;
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf)
                        if (alive[hf] && r[hf] > 250.0f && rrt::dot3(rrtp::half_of(Q, hf), rrtp::half_of(V, hf)) > 0.0f) {   // :120
                            retire(hf, it, 0u);
                            gone = true;
                        }
                    if (!(alive[0] || alive[1])) break;
                    if (gone) {
                        R2 = rrtp::norm2_loop_2(P);
                        R = rrtp::sqrt2(R2);
                    } else {
                        R2 = R2n;
                        R = Rn;
                    }
                    {
                        const unsigned in_loop = __activemask();
                        float r0, r1;
                        rrtp::upk(R, r0, r1);
                        if (fminf(r0, r1) >= burst_lo && fmaxf(r0, r1) <= burst_hi && it >= burst_after && it + kBurst < max_steps &&
                            __activemask() == in_loop) { rewind = true; break; }
                        float y0, y1;
                        rrtp::upk(P.y, y0, y1);
                        if (it >= zburst_after && it + kBurst < max_steps && (!alive[0] || zone_for_burst(r0, fabsf(y0)) >= 0) &&
                            (!alive[1] || zone_for_burst(r1, fabsf(y1)) >= 0) && __activemask() == in_loop) { rewind = true; break; }
                    }
                }
                if (!rewind) break;
            }
#pragma unroll
            for (int hf = 0; hf < 2; ++hf)
                if (alive[hf]) retire(hf, it, kEndExhausted);  // the loop ran out (:41)
            cnt.disk += n_disk; cnt.dust += n_dust;
        }
        __syncwarp();
        // queue the halves that stored samples; the rows of the two halves interleave
        const unsigned most = __reduce_max_sync(0xffffffffu, max(em.count[0], em.count[1]));
        if (most != 0u) {
#pragma unroll
            for (int hf = 0; hf < 2; ++hf)
                if (__any_sync(0xffffffffu, em.count[hf] != 0u)) queue_group(S, tab, tile, em.row0 + (unsigned)hf, 2u, 1u + (unsigned)hf, em.count[hf], lane);
            advance_rows(S, tab, row_next, 2u * (most + 1u), lane);
        }
    }
    if (lane == 0 && taken) {
        atomicMax(S.stats + 0, S.pass + 1u);
        atomicAdd(S.stats + 2, taken);
    }
    cnt.flush(A.counters);
}
#endif  // RRT_FMAD

// slot of (lane, k-th sample) of a queued tile, given the tile's chunk table
__device__ __forceinline__ unsigned desc_slot(const SplitArgs& S, const unsigned* chunk, unsigned row0, unsigned stride, unsigned k, unsigned lane) {
    const unsigned pos = row0 + k * stride;
    return chunk[pos >> S.chunk_shift] + (pos & (S.chunk_rows - 1u)) * 32u + lane;
}

// ---- pass kernel 2: the samples ---------------------------------------------------------------------------------------
// One warp per work item = kMediaBatch consecutive samples of one queued tile, in lane-major order (all of lane 0's
// samples, then lane 1's ...; neighbours in that order are consecutive steps of one ray, i.e. nearly the same work).
// Stage 1 evaluates, lane per sample, the disk density and the dust envelope.  The dust strands -- 19 value-noise
// evaluations, needed only where the envelope survived its 0.001 cut (densities.h:84) -- are collected over the whole
// batch and evaluated 32 at a time.  Stage 3 is media_final for every sample.
// RESULTS = false overwrites the first 16 bytes of each sample with {e.rgb, s}; RESULTS = true (rrt_capture_render) writes
// them to S.results[slot] instead and leaves the sample as it is, so the same samples can be evaluated again at another time.
__device__ __forceinline__ void pool_get(const uint4* slots, unsigned slot, uint4& a, uint4& b) {   // one 256-bit load
    asm volatile("ld.global.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w)
                 : "l"(slots + 2ull * slot));
}
template <bool RESULTS>
__global__ void __launch_bounds__(kMediaBlock, 4) media_kernel(const __grid_constant__ FrameArgs A, const __grid_constant__ SplitArgs S) {
    __shared__ float s_dd[kMediaBlock / 32][kMediaBatch];
    __shared__ float s_dc[kMediaBlock / 32][kMediaBatch];      // dust envelope, then dust density
    __shared__ unsigned s_slot[kMediaBlock / 32][kMediaBatch];
    __shared__ uint4 s_a[kMediaBlock / 32][kMediaBatch];       // the batch's samples: {q.xyz, v.x}
    __shared__ uint4 s_b[kMediaBlock / 32][kMediaBatch];       //                      {v.y, v.z, r, tag}
    __shared__ unsigned short s_list[kMediaBlock / 32][kMediaBatch];
    __shared__ unsigned s_chunk[kMediaBlock / 32][kDescChunks];
    __shared__ unsigned s_pref[kMediaBlock / 32][33];
    const Consts& C = A.C;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned n_work = min(S.pc->work_count, S.work_cap);
    float* dd_w = s_dd[warp];
    float* dc_w = s_dc[warp];
    unsigned* slot_w = s_slot[warp];
    uint4* a_w = s_a[warp];
    uint4* b_w = s_b[warp];
    unsigned short* list = s_list[warp];
    unsigned* chunk = s_chunk[warp];
    unsigned* pref = s_pref[warp];
    for (;;) {
        unsigned t = 0;
        if (lane == 0) t = atomicAdd(&S.pc->media_ticket, 1u);
        t = __shfl_sync(0xffffffffu, t, 0);
        if (t >= n_work) break;
        const WorkItem w = S.work[t];
        const TileDesc* d = S.desc + w.desc;
        // samples per lane -> exclusive prefix: sample index -> (lane, k)
        unsigned incl = d->n[lane];
        const unsigned row0 = d->row0, total = d->total, stride = d->stride_kind & 0xffu;
        for (int j = lane; j < kDescChunks; j += 32) chunk[j] = d->chunk[j];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned up = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += up;
        }
        pref[lane + 1] = incl;
        if (lane == 0) pref[0] = 0u;
        __syncwarp();
        // fetch: the whole batch's samples into shared memory, all loads of a lane in flight together
        {
            unsigned slot[kMediaBatch / 32];
            uint4 a[kMediaBatch / 32], b[kMediaBatch / 32];
#pragma unroll
            for (int k = 0; k < kMediaBatch / 32; ++k) {
                const unsigned sidx = w.first + (unsigned)k * 32u + (unsigned)lane;
                slot[k] = kNone;
                a[k] = b[k] = make_uint4(0u, 0u, 0u, 0u);
                if (sidx < total) {
                    unsigned lo = 0u, hi = 32u;   // largest l with pref[l] <= sidx
#pragma unroll
                    for (int bb = 0; bb < 5; ++bb) {
                        const unsigned mid = (lo + hi) >> 1;
                        if (pref[mid] <= sidx) lo = mid; else hi = mid;
                    }
                    slot[k] = desc_slot(S, chunk, row0, stride, sidx - pref[lo], lo);
                    pool_get(S.slots, slot[k], a[k], b[k]);
                }
            }
#pragma unroll
            for (int k = 0; k < kMediaBatch / 32; ++k) {
                const unsigned i = (unsigned)k * 32u + (unsigned)lane;
                slot_w[i] = slot[k];
                a_w[i] = a[k];
                b_w[i] = b[k];
            }
        }
        __syncwarp();
        unsigned n_list = 0;
        // stage 1
#pragma unroll 1
        for (int k = 0; k < kMediaBatch / 32; ++k) {
            const unsigned i = (unsigned)k * 32u + (unsigned)lane;
            const uint4 a = a_w[i];
            const unsigned tag = b_w[i].w;   // 0 for the lanes behind the group's last sample
            float dd = 0.0f, base_d = 0.0f;
            const V3 q = mk(__uint_as_float(a.x), __uint_as_float(a.y), __uint_as_float(a.z));
            if (tag & 1u) dd = rrt::disk_density_gated(C, q, A.time);                         // :68 (0 where the gate of :71 cannot pass)
            if (tag & 2u) base_d = rrt::dust_base(C, q);                                      // :69, densities.h:70-84
            dd_w[i] = dd;
            dc_w[i] = 0.0f;
            const bool strands = base_d != 0.0f;
            const unsigned m = __ballot_sync(0xffffffffu, strands);
            if (strands) {
                list[n_list + (unsigned)__popc(m & ((1u << lane) - 1u))] = (unsigned short)i;
                dc_w[i] = base_d;
            }
            n_list += (unsigned)__popc(m);
        }
        __syncwarp();
        // stage 2: dust strands of the survivors, 32 at a time
#pragma unroll 1
        for (unsigned j0 = 0; j0 < n_list; j0 += 32u) {
            const unsigned j = j0 + (unsigned)lane;
            if (j < n_list) {
                const unsigned i = list[j];
                const uint4 a = a_w[i];
                const V3 q = mk(__uint_as_float(a.x), __uint_as_float(a.y), __uint_as_float(a.z));
                dc_w[i] = rrt::dust_strands(C, q, A.time, dc_w[i]);
            }
        }
        __syncwarp();
        // stage 3: emission colour and step transmittance
#pragma unroll 1
        for (int k = 0; k < kMediaBatch / 32; ++k) {
            const unsigned i = (unsigned)k * 32u + (unsigned)lane, slot = slot_w[i];
            if (slot != kNone) {
                const uint4 a = a_w[i], b = b_w[i];
                const V3 q = mk(__uint_as_float(a.x), __uint_as_float(a.y), __uint_as_float(a.z));
                const V3 v = mk(__uint_as_float(a.w), __uint_as_float(b.x), __uint_as_float(b.y));
                const MediaOut m = media_final(C, q, v, __uint_as_float(b.z), C.h[(b.w >> 2) & 3u], dd_w[i], dc_w[i]);
                const uint4 e = make_uint4(__float_as_uint(m.er), __float_as_uint(m.eg), __float_as_uint(m.eb),
                                           __float_as_uint(m.dense ? m.s : -1.0f));
                if (RESULTS) S.results[slot] = e;
                else S.slots[2ull * slot] = e;
            }
        }
        __syncwarp();
    }
}

// ---- pass kernel 3: fold + finish, one warp per queued tile ----------------------------------------------------------
// RESULTS: read each sample's {e.rgb, s} from S.results (media_kernel<true>) instead of from the sample's slot.
template <bool RESULTS>
__global__ void __launch_bounds__(128) fold_kernel(const __grid_constant__ FrameArgs A, const __grid_constant__ SplitArgs S) {
    __shared__ unsigned s_chunk[4][kDescChunks];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned* chunk = s_chunk[warp];
    const unsigned n_pend = S.pc->pend_count;
    TileCounters cnt;
    for (;;) {
        unsigned t = 0;
        if (lane == 0) t = atomicAdd(&S.pc->fold_ticket, 1u);
        t = __shfl_sync(0xffffffffu, t, 0);
        if (t >= n_pend) break;
        const TileDesc* d = S.desc + t;
        __syncwarp();
        for (int j = lane; j < kDescChunks; j += 32) chunk[j] = d->chunk[j];
        __syncwarp();
        const unsigned row0 = d->row0, n = d->n[lane], stride = d->stride_kind & 0xffu, kind = d->stride_kind >> 8;
        const TilePix px = kind == 0u ? tile_pixel(A, d->tile, lane) : tile_pixel16(A, d->tile, lane, (int)kind - 1);
        // a lane without samples finished its ray in the trace kernel; the others left their exit state behind their samples
        uint4 sa = make_uint4(0u, 0u, 0u, 0u), sb = sa;
        if (n) {
            const unsigned st = desc_slot(S, chunk, row0, stride, n, (unsigned)lane);
            sa = S.slots[2ull * st];
            sb = S.slots[2ull * st + 1];
        }
        const V3 p = mk(__uint_as_float(sa.x), __uint_as_float(sa.y), __uint_as_float(sa.z));
        const V3 v = mk(__uint_as_float(sa.w), __uint_as_float(sb.x), __uint_as_float(sb.y));
        const int steps = (int)(sb.z & 0x0fffffffu);
        unsigned end = sb.z >> 28;
        float Ir = 0.f, Ig = 0.f, Ib = 0.f, T = 1.0f;
        unsigned n_dense = 0;
        // every lane walks its own samples; the addresses do not depend on the data, so four loads are in flight at a time
        for (unsigned k0 = 0; k0 < n; k0 += 4u) {
            uint4 e[4];
#pragma unroll
            for (int u = 0; u < 4; ++u)
                e[u] = k0 + u < n ? (RESULTS ? S.results[desc_slot(S, chunk, row0, stride, k0 + u, (unsigned)lane)]
                                             : S.slots[2ull * desc_slot(S, chunk, row0, stride, k0 + u, (unsigned)lane)])
                                  : make_uint4(0u, 0u, 0u, 0xbf800000u);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const float s = __uint_as_float(e[u].w);
                if (s != -1.0f) {                                                             // :71
                    ++n_dense;
                    const float wgt = rrt::mul(rrt::sub(1.0f, s), T);                         // :109
                    Ir = rrt::mad(__uint_as_float(e[u].x), wgt, Ir);                          // :111-113
                    Ig = rrt::mad(__uint_as_float(e[u].y), wgt, Ig);
                    Ib = rrt::mad(__uint_as_float(e[u].z), wgt, Ib);
                    T = rrt::mul(T, s);                                                       // :115
                }
            }
        }
        if (n_dense) end |= kEndTouched;
        if (end & kEndCaptured) T = 0.0f;                                                     // :49
        if (px.valid && n) {
            float uvx, uvy;
            pixel_uv(A, px.x, px.y, uvx, uvy);
            finish_ray_inl(A, px.x, px.y, px.ly, uvx, uvy, Ir, Ig, Ib, T, p, v, steps, end);
            cnt.dense += n_dense;
            cnt.touch += n_dense ? 1u : 0u;
        }
    }
    cnt.flush(A.counters);
}

// ---- after the last pass: whatever the split passes left, with the fused code ------------------------------------------
template <bool SPIN, int LENS>
__global__ void __launch_bounds__(kRenderBlock, LENS != kRaysPinhole ? kMinBlocksMediaLens : kMinBlocksMedia)
    sweep_kernel(const __grid_constant__ FrameArgs A, const __grid_constant__ SplitArgs S, const __grid_constant__ LensArgs L) {
    const int lane = threadIdx.x & 31;
    const unsigned ntiles = num_tiles(A);
    TileCounters cnt;
    unsigned taken = 0;
    const int ntx16 = (A.w + kTile16W - 1) / kTile16W, ntx8 = (A.w + kRTileW - 1) / kRTileW;
    for (;;) {
        const unsigned ticket = next_tile(A, S, S.tile16 ? num_tiles16(A) : ntiles, false);
        if (ticket == kNone) break;
        ++taken;
        for (int sub = 0; sub < (S.tile16 ? 2 : 1); ++sub) {
            unsigned tile = ticket;
            if (S.tile16) {   // a 16x4 tile of the packed tracer = the 8x4 tiles (2 tx, ty) and (2 tx + 1, ty), same row order
                const int tx8 = 2 * (int)(ticket % (unsigned)ntx16) + sub;
                if (tx8 >= ntx8) continue;
                tile = (ticket / (unsigned)ntx16) * (unsigned)ntx8 + (unsigned)tx8;
            }
            const TilePix px = tile_pixel(A, tile, lane);
            if (!px.valid) continue;
            RayResult R;
            NoEmit no_emit;
            trace_ray<SPIN, kMediaInline, LENS>(A, L, px.x, px.y, R, no_emit);
            finish_ray_inl(A, px.x, px.y, px.ly, R.uvx, R.uvy, R.I[0], R.I[1], R.I[2], R.T, R.p, R.v, R.steps,
                           (R.captured ? kEndCaptured : 0u) | (R.touched ? kEndTouched : 0u) | (R.exhausted ? kEndExhausted : 0u));
            cnt.steps += (unsigned)R.steps;
            cnt.disk += R.n_disk; cnt.dust += R.n_dust; cnt.dense += R.n_dense;
            cnt.cap += R.captured; cnt.exh += R.exhausted; cnt.esc += (!R.captured && !R.exhausted); cnt.touch += R.touched;
        }
    }
    if (lane == 0 && taken) atomicAdd(S.stats + 1, taken);
    if (blockIdx.x == 0 && threadIdx.x == 0) { S.stats[3] = S.pass; S.stats[4] = S.tile16 ? num_tiles16(A) : ntiles; }   // what the host enqueued, for its next guess
    cnt.flush(A.counters);
}

const rrtk::SplitKernels kSplitKernels = {
    {{trace_kernel<false, 0>, trace_kernel<true, 0>}, {trace_kernel<false, 1>, trace_kernel<true, 1>}, {trace_kernel<false, 2>, trace_kernel<true, 2>}},
#if RRT_FMAD
    {{trace_kernel_p<false, 0>, trace_kernel_p<true, 0>}, {trace_kernel_p<false, 1>, trace_kernel_p<true, 1>},
     {trace_kernel_p<false, 2>, trace_kernel_p<true, 2>}},
#else
    {{nullptr, nullptr}, {nullptr, nullptr}, {nullptr, nullptr}},
#endif
    media_kernel<false>, fold_kernel<false>,
    {{sweep_kernel<false, 0>, sweep_kernel<true, 0>}, {sweep_kernel<false, 1>, sweep_kernel<true, 1>}, {sweep_kernel<false, 2>, sweep_kernel<true, 2>}},
    media_kernel<true>, fold_kernel<true>,
};
}  // namespace

namespace rrtk {
#if RRT_FMAD
const SplitKernels* rrt_split_kernels_fmad() { return &kSplitKernels; }
#else
const SplitKernels* rrt_split_kernels_strict() { return &kSplitKernels; }
#endif
}  // namespace rrtk
