// deodr_b200: the adjoint pass (replaces renderScene_B, DR.h:2903-3135) - kernels + their launch sequence.
//   k_raster_bwd + k_finalize_edges       (aux)  edge tiles: replay, reverse sweep, per-edge plane adjoints
//   k_interior_bwd                        (aux)  pixels of large triangles elsewhere
//   k_small_tri_bwd                              triangle-parallel adjoint of the small triangles
// Everything strides over device-side counts left by the forward pass of the same view slot (kernels.cu); a forward
// that overflowed its plan makes these kernels return at once (nothing is accumulated).  The perspective-correct
// instances (PERSP) run the same phases with pixel_adjoint_persp and the edge layout of edge_acc_stride_persp.
#include <cstdlib>
#include <cstring>

#include "kernels_common.cuh"

// antialiase_error adjoint, pixels outside every edge band: image_b = -2 (obs - image) err_b (DR.h:3054-3060), consumed
// unchanged by the interior adjoint kernels.
__global__ void k_error_image_b(const float *image, const float *obs, const float *err_b, float *image_b, size_t pixels,
                                int C, const int *scal) {
    if (scal[SC_OVERFLOW]) return;
    const size_t n = pixels * C;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        image_b[i] = (float)(-2.0 * ((double)obs[i] - (double)image[i]) * (double)err_b[i / C]);
}

// Adjoint of the tiles that have silhouette edges: fp64 forward replay of the tile's ordered edges, reverse sweep with
// un-blend (DR.h:1738), per-edge plane adjoints as fp64 moments, then the interior adjoint of all the tile's pixels with
// what is left of their colour adjoint.  ERR: the antialiase_error variant (DR.h:2296-2336, 2542-2576); compat = the
// reference's dropped row term reproduced (phase_edge_adjoint_error).
// (register budgets are pinned: the allocator's own choice moved 64 -> 80 on an unrelated signature change)
// PERSP: perspective_correct as a compile-time constant (instances with ERR = false only; depths_b is written by them).
template <int MAXC, bool TEX, bool ERR, bool PERSP>
__global__ void __launch_bounds__(EDGE_NT, DEODR_EDGE_MIN_CTAS) k_raster_bwd(SceneView s, double sigma, TileDiv tiles_x, EdgeTiles et,
                                                   const uint32_t *span_cache, TieTable ties,
                                                   const double *z_buffer,
                                                   const int *owner, const float *image_b, const float *obs,
                                                   const float *err_b, int compat, DeodrGrads grads,
                                                   double *edge_acc, const __grid_constant__ FrameMaps maps,
                                                   float *depths_b) {
    static_assert(!(ERR && PERSP), "antialiase_error has no perspective-correct adjoint");
    if (et.scal[SC_OVERFLOW]) return;
    fix_channel_count<MAXC, TEX>(s);
    s.perspective_correct = PERSP ? 1 : 0;  // folds the branches
    __shared__ TileShared sh;
    // the tile's image_b / owner / z-buffer blocks arrive as three TMA tile loads (UTMALDG) issued by one thread
    __shared__ alignas(128) float t_img[MAXC <= 4 ? NT * MAXC : 4];
    __shared__ alignas(128) int t_own[NT];
    __shared__ alignas(128) double t_z[NT];
    __shared__ alignas(8) uint64_t tile_bar;
    const int tid = threadIdx.x;
    const bool tma_tiles = MAXC <= 4 && maps.ok;
    if (tma_tiles) {
        if (tid == 0) mbar_init(&tile_bar, 1);
        __syncthreads();
    }
    const int heavy = et.scal[SC_HEAVY_TILES], total = heavy + et.scal[SC_LIGHT_TILES];
    if ((int)blockIdx.x >= total) return;  // one CTA per entry of the list (launched for the plan's capacity)
    {
        const int tile_id = two_ended_at(et.list, et.num_tiles, heavy, blockIdx.x);
        const Tile tile = tile_of(tile_id, tiles_x);
        const int c = tid % TS, r = tid / TS;
        const int x = tile.x0 + c, y = tile.y0 + r;
        const bool inside = x < s.width && y < s.height;
        const size_t idx = inside ? (size_t)y * s.width + x : 0;
        const int n_edge = segment_size(et.seg, tile_id);

        PixelState<MAXC> p;
        AdjointState<MAXC> a;
        ErrorAdjointState<MAXC> ea;
        a.has_colour = false;
        ea.has = false;
        ea.g = 0.0;
        p.z = __longlong_as_double(0x7ff0000000000000LL);
        p.own = p.bown = -1;
        if (tma_tiles) {
            if (tid == 0) {
                mbar_expect_tx(&tile_bar, (uint32_t)(NT * (s.nb_colors * sizeof(float) + sizeof(int) + sizeof(double))));
                tma_load_tile(t_img, &maps.image, tile.x0 * s.nb_colors, tile.y0, &tile_bar);
                tma_load_tile(t_own, &maps.owner, tile.x0, tile.y0, &tile_bar);
                tma_load_tile(t_z, &maps.z, tile.x0, tile.y0, &tile_bar);
            }
            mbar_wait(&tile_bar, 0);
            if (inside) {
                p.z = t_z[tid];
                decode_owner(t_own[tid], ties, &p.own, &p.bown);
                for (int k = 0; k < s.nb_colors; k++) a.g[k] = t_img[tid * s.nb_colors + k];
            }
        } else if (inside) {
            p.z = z_buffer[idx];
            decode_owner(owner[idx], ties, &p.own, &p.bown);
            for (int k = 0; k < s.nb_colors; k++) a.g[k] = image_b[idx * s.nb_colors + k];
        }
        if (ERR && inside) ea.g = (double)err_b[idx];
        const float *obs_px = ERR ? obs + idx * s.nb_colors : nullptr;

        {
            const int edge_base = et.seg.offset[tile_id];
            const bool single = n_edge <= EDGE_CHUNK;
            auto load_spans = [&](int base, int m) {  // (all loads of a pass before its stores, see phase_edge_setup)
                const uint32_t *src = span_cache + (size_t)(edge_base + base) * TS;
                for (int first = tid; first < m * TS; first += 4 * EDGE_NT) {
                    uint32_t v[4];
#pragma unroll
                    for (int j = 0; j < 4; j++)
                        if (first + j * EDGE_NT < m * TS) v[j] = __ldg(src + first + j * EDGE_NT);
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const int item = first + j * EDGE_NT;
                        if (item < m * TS) sh.edge.span[item / TS][item % TS] = v[j];
                    }
                }
            };
            auto adjoint = [&](int m) {
                if (!inside) return;
                if (ERR) {
                    if (ea.has)
                        phase_edge_adjoint_error<MAXC, DevEnv>(s, x, y, r, m, &sh, p, obs_px, &ea, edge_acc,
                                                               grads.texture_b, compat != 0);
                } else if (a.has_colour) {
                    phase_edge_adjoint<MAXC, DevEnv>(s, x, y, r, m, &sh, p, &a, edge_acc, grads.texture_b);
                }
            };
            // pass A: forward replay (far to near) to obtain the final colour / residual in fp64
            for (int base = 0; base < n_edge; base += EDGE_CHUNK) {
                const int m = min(EDGE_CHUNK, n_edge - base);
                phase_edge_setup(tid, EDGE_NT, m, et.refs + edge_base + base, et.recs, &sh);
                load_spans(base, m);  // computed by the forward pass (k_edge_fwd)
                __syncthreads();
                if (inside) {
                    if (ERR) phase_edge_replay_error<MAXC>(s, x, y, r, m, &sh, p, obs_px, &ea);
                    else phase_edge_replay<MAXC>(s, x, y, r, m, &sh, p, &a);
                }
                if (single) adjoint(m);
                __syncthreads();
            }
            // pass B: reverse sweep (near to far), chunks in reverse order
            if (!single) {
                const int last = ((n_edge - 1) / EDGE_CHUNK) * EDGE_CHUNK;
                for (int base = last; base >= 0; base -= EDGE_CHUNK) {
                    const int m = min(EDGE_CHUNK, n_edge - base);
                    phase_edge_setup(tid, EDGE_NT, m, et.refs + edge_base + base, et.recs, &sh);
                    load_spans(base, m);
                    __syncthreads();
                    adjoint(m);
                    __syncthreads();
                }
            }
        }
        // a pixel overdrawn by edges in error mode: its colour adjoint comes from what is left of the residual's
        if (ERR && inside && ea.has) residual_adjoint<MAXC>(s, ea.col, obs_px, ea.g, a.g);
        interior_adjoint_warp<MAXC>(s, x, y, inside && p.bown >= 0, p, a.g, grads, depths_b);
    }
}

// Interior adjoint of the pixels owned by LARGE triangles in the tiles without silhouette edges: no shared memory, no
// z-buffer read; the gradients are summed per owner inside each warp before the scatter (interior_adjoint_warp).
template <int MAXC, bool TEX, bool PERSP>
#ifndef DEODR_INTERIOR_MIN_CTAS
#define DEODR_INTERIOR_MIN_CTAS 3  // 85 registers: 39.2 us vs 40.3 us at 64 and 47.6 us at 51 (measured, c5)
#endif
__global__ void __launch_bounds__(NT, DEODR_INTERIOR_MIN_CTAS) k_interior_bwd(SceneView s, TileDiv tiles_x, const int *large_tiles,
                                                     const int *scal, const int *edge_cursor, TieTable ties,
                                                     const int *owner, const float *image_b, DeodrGrads grads,
                                                     float *depths_b) {
    if (scal[SC_OVERFLOW]) return;
    fix_channel_count<MAXC, TEX>(s);
    s.perspective_correct = PERSP ? 1 : 0;  // folds the branches
    const int tid = threadIdx.x, total = scal[SC_LARGE_TILES];
    for (int b = blockIdx.x; b < total; b += gridDim.x) {  // one CTA per tile with large triangles binned
        const int tile_id = large_tiles[b];
        if (edge_cursor && edge_cursor[tile_id] > 0) continue;  // handled by k_raster_bwd
        const Tile tile = tile_of(tile_id, tiles_x);
        const int x = tile.x0 + tid % TS, y = tile.y0 + tid / TS;
        const bool inside = x < s.width && y < s.height;
        PixelState<MAXC> p;
        p.z = 0.0;  // only read by the perspective-correct forward path (the adjoint recomputes the pixel's depth)
        p.own = p.bown = -1;
        float g[MAXC];
        if (inside) {
            const size_t idx = (size_t)y * s.width + x;
            decode_owner(owner[idx], ties, &p.own, &p.bown);
            if (p.bown >= 0 && (p.bown & SMALL_FLAG)) p.bown = -1;  // taken by k_small_tri_bwd (triangle-parallel)
            if (p.bown >= 0)
                for (int k = 0; k < s.nb_colors; k++) g[k] = image_b[idx * s.nb_colors + k];
        }
        interior_adjoint_warp<MAXC>(s, x, y, inside && p.bown >= 0, p, g, grads, depths_b);
    }
}

// Triangle-parallel interior adjoint of the small triangles (one thread per entry of the compacted small list).
template <int MAXC, bool TEX, bool PERSP>
#ifndef DEODR_SMALL_MIN_CTAS
#define DEODR_SMALL_MIN_CTAS 8
#endif
__global__ void __launch_bounds__(128, DEODR_SMALL_MIN_CTAS) k_small_tri_bwd(SceneView s, int tiles_x, const int *small_ids, const int *scal,
                                                       const int *edge_cursor, TieTable ties, const int *owner,
                                                       const float *image_b, DeodrGrads grads, float *depths_b) {
    if (scal[SC_OVERFLOW]) return;
    fix_channel_count<MAXC, TEX>(s);
    s.perspective_correct = PERSP ? 1 : 0;  // folds the branches
    // one thread per entry (no stride loop: its registers cost this kernel its occupancy); the launch covers the exact
    // count when the forward's verdict has been read, every triangle otherwise
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= scal[SC_SMALL]) return;
    small_triangle_adjoint<MAXC, DevEnv>(s, small_ids[i], tiles_x, edge_cursor, owner, ties.pairs, image_b, grads.ij_b,
                                         grads.colors_b, grads.uv_b, grads.shade_b, grads.texture_b, depths_b);
}

// Record-parallel interior adjoint of the small triangles (small_record_adjoint, phases.h; opt-in, see launch_bwd for the
// measurements that keep the triangle-parallel form the default): one CTA per tile without
// silhouette edges, one thread per pre-masked record of the tile's list (written by the binning pass for the z pass:
// consecutive threads read consecutive 64-byte records).  The tile's owner codes and colour adjoints arrive in shared
// memory as two TMA tile loads (UTMALDG.2D; cooperative loads when the buffers do not qualify): a record tests its 3-4
// covered pixels there instead of reading the 33 pixels of its triangle's bounding box from the owner map.
struct SharedTileFetch {
    const int *own;
    const float *img;
    int C;
    __device__ __forceinline__ int owner(int px) const { return own[px]; }
    __device__ __forceinline__ float g(int px, int q) const { return img[px * C + q]; }
};

template <int MAXC, bool TEX>
__global__ void __launch_bounds__(128, DEODR_SMALL_MIN_CTAS) k_small_rec_bwd(SceneView s, TileDiv tiles_x, TileSegments seg, const PreRec *recs,
                                                       const int *scal, const int *edge_cursor, TieTable ties,
                                                       const int *owner, const float *image_b, DeodrGrads grads,
                                                       const __grid_constant__ FrameMaps maps) {
    if (scal[SC_OVERFLOW]) return;
    fix_channel_count<MAXC, TEX>(s);
    s.perspective_correct = 0;  // perspective-correct views take k_small_tri_bwd (launch_bwd): folds the branches
    const int tile_id = blockIdx.x, tid = threadIdx.x;
    const int n = segment_size(seg, tile_id);
    if (n == 0) return;
    if (edge_cursor && edge_cursor[tile_id] > 0) return;  // every pixel of that tile belongs to k_raster_bwd
    const Tile tile = tile_of(tile_id, tiles_x);
    const PreRec *list = recs + seg.offset[tile_id];
    if constexpr (MAXC <= 4) {
        __shared__ alignas(128) float t_img[NT * MAXC];
        __shared__ alignas(128) int t_own[NT];
        __shared__ alignas(8) uint64_t bar;
        if (maps.ok) {
            if (tid == 0) mbar_init(&bar, 1);
            __syncthreads();
            if (tid == 0) {
                mbar_expect_tx(&bar, (uint32_t)(NT * (s.nb_colors * sizeof(float) + sizeof(int))));
                tma_load_tile(t_img, &maps.image, tile.x0 * s.nb_colors, tile.y0, &bar);
                tma_load_tile(t_own, &maps.owner, tile.x0, tile.y0, &bar);  // (outside the image: zeros, no record's code)
            }
            mbar_wait(&bar, 0);
        } else {
            for (int px = tid; px < NT; px += blockDim.x) {
                const int x = tile.x0 + (px & (TS - 1)), y = tile.y0 + (px >> 4);
                const bool inside = x < s.width && y < s.height;
                const size_t idx = inside ? (size_t)y * s.width + x : 0;
                t_own[px] = inside ? owner[idx] : -1;
                for (int q = 0; q < s.nb_colors; q++) t_img[px * s.nb_colors + q] = inside ? image_b[idx * s.nb_colors + q] : 0.0f;
            }
            __syncthreads();
        }
        const SharedTileFetch fetch{t_own, t_img, s.nb_colors};
        for (int i = tid; i < n; i += blockDim.x)
            small_record_adjoint<MAXC, DevEnv>(s, list[i], tile, fetch, ties.pairs, grads.ij_b, grads.colors_b, grads.uv_b,
                                               grads.shade_b, grads.texture_b);
    } else {
        const GlobalTileFetch fetch{owner, image_b, tile, s.width, s.height, s.nb_colors};
        for (int i = tid; i < n; i += blockDim.x)
            small_record_adjoint<MAXC, DevEnv>(s, list[i], tile, fetch, ties.pairs, grads.ij_b, grads.colors_b, grads.uv_b,
                                               grads.shade_b, grads.texture_b);
    }
}

template <bool PERSP>
__global__ void k_finalize_edges(SceneView s, EdgeList edges, const int *scal, double sigma, const double *edge_acc,
                                 DeodrGrads grads, float *depths_b) {
    if (scal[SC_OVERFLOW]) return;
    s.perspective_correct = PERSP ? 1 : 0;
    const int stride = PERSP ? edge_acc_stride_persp(s.nb_colors) : edge_acc_stride(s.nb_colors);
    const int n = min(*edges.count, edges.capacity);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        finalize_edge<DevEnv>(s, edges.ids[i], sigma, edge_acc + (size_t)i * stride, grads.ij_b, grads.colors_b,
                              grads.uv_b, grads.shade_b, depths_b);
}

// Rows of the per-edge accumulators of a view (the perspective-correct instances use their own layout).
int deodr_edge_acc_stride(const SceneView &s) {
    return s.perspective_correct ? edge_acc_stride_persp(s.nb_colors) : edge_acc_stride(s.nb_colors);
}

template <int MAXC, bool PERSP>
static void launch_bwd(DeodrWorkspace *ws, ViewSlot *v, Lane &lane, const SceneView &s, const DeodrViewIO &io,
                       double sigma, int flags, const DeodrGrads &g, float *depths_b) {
    // Three independent chains (disjoint pixel sets, all accumulate with atomics): edge tiles (longest tail: launched
    // first so that its CTAs are dispatched first), tiles with large triangles, small triangles.
    cudaStream_t st = lane.main;
    bool first = true;
    const FwdPlan &plan = v->plan;
    const bool tex = plan.tex != 0;
    const bool err_mode = (flags & DEODR_B200_ANTIALIASE_ERROR) != 0;
    const int compat = (flags & DEODR_B200_ERROR_ADJOINT_COMPLETE) ? 0 : 1;
    const int C = s.nb_colors;
    const bool edges = plan.cap_edges > 0;
    const TileDiv div = make_tile_div(v->tiles_x);
    const TieTable ties = tie_table(v);
    const int *edge_cursor = edges ? v->edge_cursor : nullptr;
    const float *image_b = io.image_b;
    if (err_mode) {  // colour adjoint of the pixels outside the edge bands, before the three chains fork
        const size_t pixels = (size_t)s.height * s.width;
        k_error_image_b<<<grid_for(pixels * C, 256) < 4096 ? grid_for(pixels * C, 256) : 4096, 256, 0, st>>>(
            io.image, io.obs, io.err_buffer_b, v->error_image_b.as<float>(), pixels, C, v->scal);
        image_b = v->error_image_b.as<float>();
        ws->launches++;
    }
    // tensor maps of the tile-shaped reads of the adjoint (image_b / owner / z-buffer blocks): k_raster_bwd, k_small_rec_bwd
    FrameMaps maps;
    memset(&maps, 0, sizeof(maps));
    static const bool tma_allowed = !(getenv("DEODR_B200_TMA_TILES") && atoi(getenv("DEODR_B200_TMA_TILES")) == 0);
    maps.ok = tma_allowed && C <= 4 &&
              encode_tile_map(&maps.image, image_b, 4, true, s.height, s.width * C, TS, TS * C) &&
              encode_tile_map(&maps.owner, io.owner, 4, false, s.height, s.width, TS, TS) &&
              encode_tile_map(&maps.z, io.z_buffer, 8, false, s.height, s.width, TS, TS);
    if (edges) {
        cudaStream_t se = fork_stream(ws, lane, 1, &first);
        cudaMemsetAsync(v->edge_acc.ptr, 0, (size_t)plan.cap_edges * deodr_edge_acc_stride(s) * sizeof(double), se);
        const EdgeTiles et = edge_tiles_of(v);
        const int grid = at_least_one(v->hints_exact && !ws->capturing_internally ? plan.hint_edge_tiles : plan.cap_edge_tiles);
        {
            PhaseTimer timer(ws, DEODR_B200_PH_EDGE_BWD, se);
#define DEODR_RASTER_BWD(X, R) k_raster_bwd<MAXC, X, R, PERSP && !R><<<grid, EDGE_NT, 0, se>>>(s, sigma, div, et, v->edge_spans.as<uint32_t>(), ties, io.z_buffer, io.owner, image_b, io.obs, io.err_buffer_b, compat, g, v->edge_acc.as<double>(), maps, depths_b)
            if (PERSP) { if (tex) DEODR_RASTER_BWD(true, false); else DEODR_RASTER_BWD(false, false); }  // (no ERR)
            else if (tex) { if (err_mode) DEODR_RASTER_BWD(true, true); else DEODR_RASTER_BWD(true, false); }
            else     { if (err_mode) DEODR_RASTER_BWD(false, true); else DEODR_RASTER_BWD(false, false); }
#undef DEODR_RASTER_BWD
        }
        {
            PhaseTimer timer(ws, DEODR_B200_PH_EDGE_FINALIZE, se);
            const EdgeList el{v->scal + SC_EDGES, v->edge_ids.as<int>(), v->edge_keys.as<uint64_t>(), plan.cap_edges};
            k_finalize_edges<PERSP><<<at_least_one(grid_for(plan.hint_edges, 128)), 128, 0, se>>>(
                s, el, v->scal, sigma, v->edge_acc.as<double>(), g, depths_b);
        }
        ws->launches += 2;
    }
    const bool large = plan.cap_large > 0 && plan.hint_large_tiles > 0;
    if (large) {  // pixels owned by large triangles, tiles without silhouette edges
        cudaStream_t sl = fork_stream(ws, lane, 2, &first);
        PhaseTimer timer(ws, DEODR_B200_PH_INTERIOR_BWD, sl);
        const int grid = at_least_one(plan.hint_large_tiles < v->num_tiles ? plan.hint_large_tiles : v->num_tiles);
        (tex ? k_interior_bwd<MAXC, true, PERSP> : k_interior_bwd<MAXC, false, PERSP>)<<<grid, NT, 0, sl>>>(
            s, div, v->large_tiles.as<int>(), v->scal, edge_cursor, ties, io.owner, image_b, g, depths_b);
        ws->launches++;
    }
    {
        PhaseTimer timer(ws, DEODR_B200_PH_SMALL_BWD, st);
        // Triangle-parallel (default) or record-parallel (DEODR_B200_SMALL_ADJOINT=record) adjoint of the small triangles.
        // Measured, same session: 1M-triangle scene 0.324 ms per step (triangle) vs 0.331 (record: as long itself - the
        // vertex gathers and the fifteen atomics per thread are what it costs, not the bounding-box reads, and 1.7x
        // more threads pay them - and k_interior_bwd beside it slows from 61 to 73 us); 16 renders of 200k triangles at
        // 512^2: 0.723 vs 0.695 ms; 1M textured triangles: 0.621 vs 0.632 ms.
        // Perspective-correct views always take the triangle-parallel form (k_small_rec_bwd has no PERSP instance).
        if (!ws->small_by_record || PERSP) {  // (read from the environment when the workspace is created)
            const int entries = v->hints_exact && !ws->capturing_internally ? plan.hint_small : s.nb_triangles;
            (tex ? k_small_tri_bwd<MAXC, true, PERSP> : k_small_tri_bwd<MAXC, false, PERSP>)<<<at_least_one(grid_for(entries, 128)), 128, 0, st>>>(
                s, v->tiles_x, v->small_ids.as<int>(), v->scal, edge_cursor, ties, io.owner, image_b, g, depths_b);
        } else {
            const TileSegments seg{v->small_offset.as<int>(), v->small_cursor};
            (tex ? k_small_rec_bwd<MAXC, true> : k_small_rec_bwd<MAXC, false>)<<<v->num_tiles, 128, 0, st>>>(
                s, div, seg, v->small_recs.as<PreRec>(), v->scal, edge_cursor, ties, io.owner, image_b, g, maps);
        }
        ws->launches++;
    }
    if (edges) join_stream(ws, lane, 1);
    if (large) join_stream(ws, lane, 2);
}


template <bool PERSP>
static void launch_bwd_channels(DeodrWorkspace *ws, ViewSlot *v, Lane &lane, const SceneView &s, const DeodrViewIO &io,
                                double sigma, int flags, const DeodrGrads &g, float *depths_b) {
    const int C = s.nb_colors;
    if (C == 1) launch_bwd<1, PERSP>(ws, v, lane, s, io, sigma, flags, g, depths_b);
    else if (C == 3) launch_bwd<3, PERSP>(ws, v, lane, s, io, sigma, flags, g, depths_b);
    else if (C <= 4) launch_bwd<4, PERSP>(ws, v, lane, s, io, sigma, flags, g, depths_b);
    else launch_bwd<16, PERSP>(ws, v, lane, s, io, sigma, flags, g, depths_b);
}

void deodr_launch_backward(DeodrWorkspace *ws, ViewSlot *v, Lane &lane, const SceneView &s, const DeodrViewIO &io,
                           double sigma, int flags, const DeodrGrads &g, float *depths_b) {
    if (s.perspective_correct) launch_bwd_channels<true>(ws, v, lane, s, io, sigma, flags, g, depths_b);
    else launch_bwd_channels<false>(ws, v, lane, s, io, sigma, flags, g, depths_b);
}
