// Pieces shared by the translation units that hold kernels (kernels.cu: binning + forward, kernels_bwd.cu: adjoint):
// device environment, warp-level adjoint scatter, owner decoding, edge-tile descriptors, and the host-side helpers that
// bracket launches (phase timers, stream fork / join).  Compiling the forward and adjoint kernels separately halves the
// build time (the instances are many: channel capacity x texture x perspective x error mode).
#pragma once

#include <cuda_runtime.h>

#include "../../include/deodr_b200.h"
#include "phases.h"
#include "tma.cuh"
#include "workspace.h"

using namespace deodr;

// ------------------------------------------------------------------------------------------------ device Env

struct DevEnv {
    static __device__ __forceinline__ int atomic_add(int *p, int v) { return atomicAdd(p, v); }
    static __device__ __forceinline__ void atomic_add(float *p, float v) { atomicAdd(p, v); }
    static __device__ __forceinline__ void atomic_add(double *p, double v) { atomicAdd(p, v); }
    static __device__ __forceinline__ void atomic_or(int *p, int v) { atomicOr(p, v); }
    static __device__ __forceinline__ int shared_inc(int *p) { return atomicAdd(p, 1); }  // p in shared memory
};

// Interior adjoint of one pixel per lane with a warp-level reduce-by-owner before the scatter: the lanes of a warp that
// share the adjoint owner (neighbouring pixels of a large triangle) first sum their vertex gradients with a tree of
// shuffles over the group (__match_any_sync gives the groups), then ONE lane per group issues the atomics.  Measured on
// the 1M-triangle scene: float-atomic throughput was 38 of k_interior_bwd's 67 us.  Must be called by all 32 lanes.
template <int MAXC>
static __device__ __forceinline__ void interior_adjoint_warp(const SceneView &s, int x, int y, bool has,
                                                             const PixelState<MAXC> &p, const float *g,
                                                             const DeodrGrads &grads, float *depths_b = nullptr) {
    const int lane = (int)(threadIdx.x & 31), C = s.nb_colors;
    TriAttr t;
    VertexGrads<MAXC> acc;
    zero_vertex_grads<MAXC>(s, &acc);
    float dz[3] = {0.0f, 0.0f, 0.0f};  // depths_b (perspective_correct only)
    t.textured = false;
    if (has) {
        tri_attr(s, p.bown & TRI_INDEX_MASK, &t);
        pixel_adjoint<MAXC, DevEnv>(s, t, x, y, g, &acc, grads.texture_b, dz);
    }
    const int key = has ? (p.bown & TRI_INDEX_MASK) : -1 - lane;  // idle lanes: groups of one
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    const int rank = __popc(peers & ((1u << lane) - 1u)), size = __popc(peers);
    const int max_size = __reduce_max_sync(0xffffffffu, size);
    const bool any_textured = __any_sync(0xffffffffu, has && t.textured);
    const bool any_plain = __any_sync(0xffffffffu, has && !t.textured);
    for (int stride = 1; stride < max_size; stride <<= 1) {
        // tree over the members of a group: member `rank` (a multiple of 2*stride) takes member rank + stride
        const bool take = (rank & (2 * stride - 1)) == 0 && rank + stride < size;
        const int src = take ? (int)__fns(peers, 0, rank + stride + 1) : lane;
#define DEODR_TAKE(field)                                                  \
        {                                                                      \
            const float other = __shfl_sync(0xffffffffu, (field), src);        \
            if (take) (field) += other;                                        \
        }
#pragma unroll
        for (int i = 0; i < 3; i++) {
            DEODR_TAKE(acc.ij[i][0]);
            DEODR_TAKE(acc.ij[i][1]);
        }
        if (s.perspective_correct) {
#pragma unroll
            for (int i = 0; i < 3; i++) DEODR_TAKE(dz[i]);
        }
        if (any_textured) {
#pragma unroll
            for (int i = 0; i < 3; i++) {
                DEODR_TAKE(acc.uv[i][0]);
                DEODR_TAKE(acc.uv[i][1]);
                DEODR_TAKE(acc.shade[i]);
            }
        }
        if (any_plain) {
#pragma unroll
            for (int i = 0; i < 3; i++)
#pragma unroll
                for (int c = 0; c < MAXC; c++)
                    if (c < C) DEODR_TAKE(acc.attr[i][c]);
        }
#undef DEODR_TAKE
    }
    if (has && rank == 0)
        flush_vertex_grads<MAXC, AtomicEmit<DevEnv>>(s, t, acc, grads.ij_b, grads.colors_b, grads.uv_b, grads.shade_b,
                                                     AtomicEmit<DevEnv>(), dz, depths_b);
}

// The <1> and <3> instances are only launched for exactly 1 / 3 colour channels: telling the compiler turns every
// `for (c < nb_colors)` loop of the inlined shading code into straight-line code (the <4> and <16> instances keep the
// run-time channel count: 2 or 4, 5..16).
template <int MAXC, bool TEX = true>
static __device__ __forceinline__ void fix_channel_count(SceneView &s) {
    if (MAXC == 1 || MAXC == 3) s.nb_colors = MAXC;
    // TEX = false instances are launched for scenes without a textured triangle (the plan remembers; a textured
    // triangle met by k_bin raises OVF_TEXTURE): nulling the texture pointer of the kernel's copy of the scene folds
    // every texture branch (tri_attr / edge_hit test it)
    if (!TEX) s.texture = nullptr;
}

static_assert(sizeof(SceneView) == sizeof(DeodrSceneView), "SceneView must mirror DeodrSceneView");

struct TieTable {
    int *pairs;     // (own, bown) per tie pixel
    int *counter;   // number of entries requested so far (one slot per pixel is reserved: never overflows)
    int capacity;
};


// decodes an owner code into (forward owner, adjoint owner); -1 = background
static __device__ __forceinline__ void decode_owner(int code, const TieTable &ties, int *own, int *bown) {
    if (code <= -2) {
        *own = ties.pairs[2 * (-2 - code)];
        *bown = ties.pairs[2 * (-2 - code) + 1];
    } else {
        *own = *bown = code;
    }
}

// Block b of a kernel that walks a two-ended tile list of capacity n with `heavy` crowded tiles at its front.
static __device__ __forceinline__ int two_ended_at(const int *list, int n, int heavy, int b) {
    return b < heavy ? list[b] : list[n - 1 - (b - heavy)];
}

#ifndef DEODR_EDGE_MIN_CTAS
#define DEODR_EDGE_MIN_CTAS 3  // 85 registers: edge_bwd 62.9 us vs 68 us at 64, 77 us at 51 (measured, c5)
#endif
static_assert(EDGE_ROWS == TS, "the span cache shared by k_edge_fwd and k_raster_bwd holds whole tiles");

// What the edge kernels need to find their tiles: the two-ended list (crowded tiles first) and its device-side sizes.
struct EdgeTiles {
    const int *list;
    int num_tiles;          // capacity of the list = tiles of the image
    const int *scal;        // SC_HEAVY_TILES / SC_LIGHT_TILES / SC_OVERFLOW
    TileSegments seg;       // edge references per tile
    const int *refs;        // ordered far to near
    const EdgeRec *recs;
};

// ---------------------------------------------------------------------------- TMA (bulk async copy) + mbarrier

static __device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

static __device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

static __device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

// global -> shared bulk copy (SASS: UBLKCP), completion signalled on `bar` as transaction bytes.
// dst, src 16-byte aligned, bytes a multiple of 16.
static __device__ __forceinline__ void bulk_load(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

static __device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LAB_DONE;\n"
        "bra LAB_WAIT;\n"
        "LAB_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}


// Tensor maps over a view's framebuffers, for the kernels that move whole 16x16 tiles with the TMA engine; `ok` is false
// when a buffer does not qualify (pitch / alignment / more than 4 channels): the kernels then use plain loads / stores.
struct FrameMaps {
    TileMap image;    // [H, W*C] fp32: forward output (stored) / image_b (loaded)
    TileMap owner;    // [H, W] int32
    TileMap z;        // [H, W] fp64
    int ok;
};

// ------------------------------------------------------------------------------------------------- host side

// RAII bracket: records a (start, stop) event pair around a group of launches when timing is enabled
struct PhaseTimer {
    DeodrWorkspace *ws;
    cudaStream_t st;
    int slot;
    PhaseTimer(DeodrWorkspace *w, int phase, cudaStream_t s) : ws(w), st(s), slot(-1) {
        if (ws->ev_used < (int)ws->ev_start.size()) {
            slot = ws->ev_used++;
            ws->ev_phase[slot] = phase;
            cudaEventRecord(ws->ev_start[slot], st);
        }
    }
    ~PhaseTimer() {
        if (slot >= 0) cudaEventRecord(ws->ev_stop[slot], st);
    }
};

static inline int grid_for(size_t n, int block) { return (int)((n + block - 1) / block); }
static inline int at_least_one(int n) { return n > 0 ? n : 1; }

// Fork: auxiliary stream i of the lane continues from the current point of the lane's main stream; join: the main
// stream waits for it.  Independent kernel chains then overlap (tails of one fill with CTAs of the other; no gaps).
static inline cudaStream_t fork_stream(DeodrWorkspace *ws, Lane &lane, int i, bool *first) {
    if (!ws->overlap) return lane.main;
    if (*first) { cudaEventRecord(lane.ev_fork, lane.main); *first = false; }
    cudaStreamWaitEvent(lane.aux[i], lane.ev_fork, 0);
    return lane.aux[i];
}
static inline void join_stream(DeodrWorkspace *ws, Lane &lane, int i) {
    if (!ws->overlap) return;
    cudaEventRecord(lane.ev_join[i], lane.aux[i]);
    cudaStreamWaitEvent(lane.main, lane.ev_join[i], 0);
}

static TieTable tie_table(const ViewSlot *v) { return TieTable{v->tie_pairs.as<int>(), v->scal + SC_TIES, v->tie_capacity}; }

static EdgeTiles edge_tiles_of(const ViewSlot *v) {
    return EdgeTiles{v->edge_tiles.as<int>(), v->num_tiles, v->scal, {v->edge_offset.as<int>(), v->edge_cursor},
                     v->edge_refs.as<int>(), v->edge_recs.as<EdgeRec>()};
}


// kernels_bwd.cu: enqueues the adjoint pass of one view on the lane's streams
// rows of one edge's fp64 accumulators in the adjoint of view s (edge_acc_stride / edge_acc_stride_persp)
int deodr_edge_acc_stride(const SceneView &s);
// (depths_b: [V] fp32 of the view or NULL; only the perspective-correct instances write it)
void deodr_launch_backward(DeodrWorkspace *ws, ViewSlot *v, Lane &lane, const SceneView &s, const DeodrViewIO &io,
                           double sigma, int flags, const DeodrGrads &g, float *depths_b);
