// deodr_b200: sm_100a kernels + device-level C-ABI (include/deodr_b200.h) of the differentiable rasteriser.
//
// One forward pass of one view (DESIGN.md section 4), nothing in it waits for the host:
//   memset                                       scalars + segment cursors of the view's slot
//   k_bin            1 thread / triangle         ONE gather per triangle: classify (DR.h:2751-2779), append silhouette
//                                                edges, pre-masked 64-byte records of the small triangles / tile
//                                                references of the large ones, into segments reserved by the PLAN
//   k_bin_edges      1 warp / edge        (aux)  band stencil record (DR.h:1366-1460), slot -> tiles of the band
//   k_sort_tile_edges 1 CTA / tile        (aux)  far-to-near order (DR.h:2781) inside every tile, list of edge tiles
//   k_publish                             (aux)  verdict word + counts -> pinned host memory (read by the host AFTER
//                                                the whole pass has been enqueued)
//   k_tile_z         1 CTA / 16x16 tile          TMA bulk copies of the tile's records (two-deep pipeline), exact z test,
//                                                owner ids, colour of the owner (+ residual / G-buffer weights), TMA
//                                                tile store of the colours
//   k_shade          1 thread / pixel            the colour pass on its own, when the colours arrive after the z pass
//   k_edge_fwd       1 CTA / edge tile           ordered silhouette-edge overdraw (DR.h:2839-2899)
// and one adjoint pass:
//   k_raster_bwd + k_finalize_edges       (aux)  edge tiles: replay, reverse sweep, per-edge plane adjoints
//   k_interior_bwd                        (aux)  pixels of large triangles elsewhere
//   k_small_tri_bwd                              triangle-parallel adjoint of the small triangles (k_small_rec_bwd: its
//                                                record-parallel form, opt-in)
// A forward can also be enqueued in two calls (binning | everything else: DEODR_B200_FORWARD_GEOMETRY / _RESUME).
// The plan (segment capacities) comes from a count-only pass (k_bin<true> + k_scan_tiles) run once per shape and
// again whenever a pass reports that a list outgrew it.
//
// There is no CPU fallback: every entry point fails with DEODR_B200_ECUDA if no device is usable.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <limits>
#include <new>
#include <vector>

#include "kernels_common.cuh"

// ------------------------------------------------------------------------------------------------- kernels

// The binning pass (COUNT_ONLY = false) / the count pass that builds a plan (COUNT_ONLY = true): one thread per triangle.
#ifndef DEODR_BIN_MIN_CTAS
#define DEODR_BIN_MIN_CTAS 8  // 61 registers, no spills (the 176-byte frame is the two tile-column mask arrays)
#endif
template <bool COUNT_ONLY>
__global__ void __launch_bounds__(128, DEODR_BIN_MIN_CTAS) k_bin(SceneView s, double sigma, int tiles_x, TriBins bins,
                                                                int *scal, int *small_ids, EdgeList edges,
                                                                int *edge_tile_count, int plan_tex) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= s.nb_triangles) return;
    if (scal[SC_BAD_INDEX]) return;  // out-of-range face indices found by k_check_scene: touch nothing
    // does the scene hold ANY textured triangle?  Scenes without one run kernel instances compiled without the
    // texture paths (fewer registers, no local memory); the plan remembers the answer of the pass it was built from
    if (s.textured[k] && s.shaded[k]) {
        if (*(volatile int *)(scal + SC_TEXTURED) == 0) atomicOr(scal + SC_TEXTURED, 1);
        if (!COUNT_ONLY && !plan_tex && (*(volatile int *)(scal + SC_OVERFLOW) & OVF_TEXTURE) == 0)
            atomicOr(scal + SC_OVERFLOW, OVF_TEXTURE);
    }
    bin_triangle<DevEnv, COUNT_ONLY>(s, k, sigma, tiles_x, bins, scal + SC_SMALL, small_ids, edges, edge_tile_count);
}

// Plan building: exclusive scans of the per-tile counts of the count pass, each count first padded with slack
// (c + c/4 + SEG_SLACK) so that the segments survive the drift of an optimisation loop: blockIdx 0 small triangles
// (records), 1 large triangles (references), 2 silhouette edges (references).  1024 threads per CTA; offsets[n] and
// scal[] receive the grand totals; the number of non-empty tiles (launch hints) rides in the high word of the scan.
struct ScanJob {
    const int *count[3];
    int *offset[3];
    int total_slot[3];
    int nonempty_slot[3];  // scal[] slot receiving the number of tiles with count > 0 (-1: not wanted)
};
constexpr int SEG_SLACK = 4;

// Each thread owns SCAN_IPT consecutive tiles, so 16384 tiles take ONE block scan instead of sixteen; counts and
// offsets pass through a padded shared-memory stage so that every global access stays coalesced (the kernel runs on
// three SMs only: 16 uncoalesced wavefronts per load instruction would be its whole duration).
constexpr int SCAN_IPT = 16;
constexpr int SCAN_TILE = 1024 * SCAN_IPT;
constexpr int SCAN_SMEM = (SCAN_TILE + SCAN_TILE / 32) * (int)sizeof(int);
static __device__ __forceinline__ int scan_slot(int i) { return i + (i >> 5); }  // conflict-free for stride-16 readers
__global__ void __launch_bounds__(1024) k_scan_tiles(ScanJob job, int n, int *scal, int *host_totals, int seq) {
    extern __shared__ int stage[];
    __shared__ unsigned long long warp_sums[32];
    const int *count = job.count[blockIdx.x];
    int *offset = job.offset[blockIdx.x];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned long long carry = 0;
    for (int base = 0; base < n; base += SCAN_TILE) {
        {
            // all sixteen loads first (the compiler cannot move a generic-pointer load above a shared-memory store on
            // its own: interleaved they would cost sixteen serial memory round trips)
            int in[SCAN_IPT];
#pragma unroll
            for (int k = 0; k < SCAN_IPT; k++) in[k] = base + k * 1024 + tid < n ? __ldg(count + base + k * 1024 + tid) : -1;
#pragma unroll
            for (int k = 0; k < SCAN_IPT; k++) stage[scan_slot(k * 1024 + tid)] = in[k];
        }
        __syncthreads();
        const int first = tid * SCAN_IPT;
        unsigned long long c[SCAN_IPT];  // low word: padded capacity of the tile, high word: 1 if it is not empty
        unsigned long long v = 0;
#pragma unroll
        for (int k = 0; k < SCAN_IPT; k++) {
            // (bit 30 of a count: "the tile is touched by a triangle of the pixel-parallel adjoint", set by the count
            // pass for record-path triangles that are not small: it only feeds the non-empty tally, a launch hint)
            const int flagged = stage[scan_slot(first + k)];
            const int raw = flagged < 0 ? -1 : (flagged & 0x3fffffff);
            c[k] = raw < 0 ? 0ull
                           : (unsigned long long)(unsigned)(raw + (raw >> 2) + SEG_SLACK) | ((unsigned long long)(flagged > 0) << 32);
            v += c[k];
        }
        unsigned long long incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_sums[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            unsigned long long w = warp_sums[lane];
            for (int o = 1; o < 32; o <<= 1) {
                unsigned long long t = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += t;
            }
            warp_sums[lane] = w;
        }
        __syncthreads();
        unsigned long long run = carry + (warp ? warp_sums[warp - 1] : 0ull) + incl - v;
#pragma unroll
        for (int k = 0; k < SCAN_IPT; k++) {
            stage[scan_slot(first + k)] = (int)(unsigned)run;
            run += c[k];
        }
        carry += warp_sums[31];
        __syncthreads();
        {
            int outv[SCAN_IPT];
#pragma unroll
            for (int k = 0; k < SCAN_IPT; k++) outv[k] = stage[scan_slot(k * 1024 + tid)];
#pragma unroll
            for (int k = 0; k < SCAN_IPT; k++)
                if (base + k * 1024 + tid < n) offset[base + k * 1024 + tid] = outv[k];
        }
        __syncthreads();
    }
    if (tid == 0) {
        offset[n] = (int)(unsigned)carry;
        scal[job.total_slot[blockIdx.x]] = (int)(unsigned)carry;
        if (job.nonempty_slot[blockIdx.x] >= 0) scal[job.nonempty_slot[blockIdx.x]] = (int)(carry >> 32);
        // The last CTA to finish publishes the scalars straight into the host's (pinned, device-visible) buffer and
        // raises a sequence flag the host is polling: no copy engine, no stream synchronisation.
        __threadfence();
        const int ticket = atomicAdd(&scal[SC_TICKET], 1);
        if (host_totals && ticket == (int)gridDim.x - 1) {
            __threadfence();
            for (int i = 0; i < SC_WORDS; i++) host_totals[i] = ((volatile int *)scal)[i];
            __threadfence_system();
            ((volatile int *)host_totals)[SC_WORDS] = seq;
        }
    }
}

// One WARP per appended silhouette edge (stride loop over the device-side count): stencil record + tile lists.  Every
// lane computes the edge's record (same instructions, one merged store) and then takes its share of the tiles of the
// band, so that the returning atomics of the segment appends - 10 to 30 per edge, a serial chain of L2 round trips when
// one thread walks them - are issued side by side.  The scenes this matters for are the small ones, where this kernel
// sits on the forward's critical path (1k-triangle scene at 640x480: 32 us with one thread per edge).
__global__ void __launch_bounds__(128) k_bin_edges(SceneView s, double sigma, int tiles_x, EdgeList edges, EdgeBins bins,
                                                   EdgeRec *recs, const int *scal) {
    if (scal[SC_OVERFLOW]) return;
    const int n = min(*edges.count, edges.capacity);
    const int lane = threadIdx.x & 31, warps = (gridDim.x * blockDim.x) >> 5;
    for (int slot = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; slot < n; slot += warps) {
        double V[2][2];
        edge_record(s, edges.ids[slot], slot, edges.keys[slot], sigma, &recs[slot], V);
        const TileBox b = edge_tile_box(V, sigma, s.width, s.height);
        if (b.tx0 > b.tx1) continue;
        const int bw = b.tx1 - b.tx0 + 1, count = bw * (b.ty1 - b.ty0 + 1);
        for (int j = lane; j < count; j += 32) bin_edge_tile<DevEnv>(slot, (b.ty0 + j / bw) * tiles_x + b.tx0 + j % bw, bins);
    }
}

// Orders the edge list of every tile that has one far to near (tile_edge_position, phases.h) and moves the tile to the
// two-ended list the edge kernels walk: tiles with more than one chunk of edges at the front (they set those kernels'
// duration and must start first), the others from the back.  One CTA per entry of the arrival-order list k_bin_edges
// built; (key, id) pairs are staged in shared memory 256 at a time.
constexpr int SORT_CHUNK = 256;
__global__ void __launch_bounds__(128) k_sort_tile_edges(TileSegments seg, int num_tiles, const int *refs_in,
                                                         int *refs_out, const EdgeRec *recs, const int *tiles_raw,
                                                         int *edge_tiles, int *scal) {
    if (scal[SC_OVERFLOW]) return;
    __shared__ unsigned long long sk[SORT_CHUNK];
    __shared__ int si[SORT_CHUNK];
    if ((int)blockIdx.x >= scal[SC_EDGE_TILES]) return;
    const int tile = tiles_raw[blockIdx.x];
    const int n = segment_size(seg, tile), base = seg.offset[tile];
    if (threadIdx.x == 0) {
        if (n > EDGE_CHUNK) edge_tiles[atomicAdd(scal + SC_HEAVY_TILES, 1)] = tile;
        else edge_tiles[num_tiles - 1 - atomicAdd(scal + SC_LIGHT_TILES, 1)] = tile;
    }
    for (int i0 = 0; i0 < n; i0 += blockDim.x) {
        const int i = i0 + threadIdx.x;
        int ref = 0, id = 0, pos = 0;
        unsigned long long key = 0;
        if (i < n) {
            ref = refs_in[base + i];
            key = recs[ref].key;
            id = recs[ref].id;
        }
        for (int c0 = 0; c0 < n; c0 += SORT_CHUNK) {
            const int m = min(SORT_CHUNK, n - c0);
            __syncthreads();
            for (int j = threadIdx.x; j < m; j += blockDim.x) {
                const EdgeRec &o = recs[refs_in[base + c0 + j]];
                sk[j] = o.key;
                si[j] = o.id;
            }
            __syncthreads();
            if (i < n)
                for (int j = 0; j < m; j++) pos += (int)(sk[j] < key || (sk[j] == key && si[j] < id));
        }
        if (i < n) refs_out[base + pos] = ref;
    }
}

// Verdict + counts of the binning kernels -> pinned host memory + sequence flag (one warp).
__global__ void k_publish(const int *scal, int *host_totals, int seq) {
    const int lane = threadIdx.x;
    if (lane < SC_WORDS) host_totals[lane] = ((const volatile int *)scal)[lane];
    __threadfence_system();
    __syncwarp();
    if (lane == 0) ((volatile int *)host_totals)[SC_WORDS] = seq;
}

// Forward, kernel 1 of 3 - z-buffer, owner ids and (fused) colours, one 16x16 tile per CTA.
// Small triangles: the tile's pre-masked records are pulled into shared memory by bulk copies (cp.async.bulk +
// mbarrier, SASS UBLKCP) 128 at a time through a two-deep pipeline - chunks c and c+1 are in flight when the tile
// starts, chunk c+2 is issued as soon as chunk c has been consumed, so a crowded tile (the 1M-triangle scene has 400
// tiles with more than 256 records, the 200k-triangle 512^2 views average 280) pays the copy latency once; two threads
// per record scatter its index into per-pixel candidate lists; each pixel then z-tests its own candidates exactly.
// Large triangles: stencil per triangle -> coverage masks (8 threads each) -> mask test.
// One tile per CTA, scheduled by the hardware: measured faster than persistent CTAs with a static stride (168 us vs
// 199 us x4 / 300 us x2 per SM on the 1M-triangle scene, round 2) - the tiles are very uneven.
#ifndef DEODR_TILEZ_MIN_CTAS
#define DEODR_TILEZ_MIN_CTAS 6  // measured on the 1M-triangle scene (fused instance): 117 us at 4, 103 us at 5, 94 us at 6
#endif
// PERSP: perspective_correct as a compile-time constant (the 1/z division and its registers leave the common instance).
// FUSE: the colour of every pixel is computed in this kernel's epilogue (the owner stays in registers: no owner map
// re-read, no second launch); MAXC / TEX as in k_shade.  The unfused instance <1, PERSP, false, false> + k_shade is
// what a forward uses when the colours arrive late (colours-ready event: the z pass then overlaps the all-reduce).
template <int MAXC, bool PERSP, bool TEX, bool FUSE>
__global__ void __launch_bounds__(NT, DEODR_TILEZ_MIN_CTAS) k_tile_z(SceneView s, TileDiv tiles_x, int num_tiles, TriBins bins, TieTable ties,
                                                  double *z_buffer, int *owner, int *face_id, int *scal,
                                                  int *large_tiles, float *image, const float *obs, float *err,
                                                  float *bary, const __grid_constant__ TileMap image_map, int tma_store) {
    // a list outgrew the plan: the pass is void (the host re-plans and re-runs).  OVF_EDGE_REFS is left out: it is
    // raised by k_bin_edges, which runs beside this kernel, and the early return must be uniform across the CTA
    if (scal[SC_OVERFLOW] & ~OVF_EDGE_REFS) return;
    s.perspective_correct = PERSP ? 1 : 0;
    // (only the triangle part of the tile kernels' working set: shared memory is what bounds this kernel's CTAs per SM)
    __shared__ alignas(16) unsigned char sh_raw[sizeof(TileShared::TriPart)];
    TileShared &sh = *reinterpret_cast<TileShared *>(sh_raw);
    __shared__ alignas(16) PreRec pre[2][PRE_CHUNK];
    __shared__ alignas(8) uint64_t bar[2];
    // fused shading, up to 4 channels: the tile's colours are staged here and leave as ONE TMA tile store (UTMASTG)
    // instead of C four-byte stores per pixel at a 4C-byte stride
    __shared__ alignas(128) float stage[FUSE && MAXC <= 4 ? NT * MAXC : 4];
    const int tid = threadIdx.x;
    const int tile_id = blockIdx.x;
    if (tile_id >= num_tiles) return;
    // the tile's four list words are fetched by every thread at once (broadcast loads, ONE memory round trip)
    const int c_small = bins.small.cursor[tile_id];
    const int c_large = bins.large.cursor[tile_id];
    const int o_begin = bins.small.offset[tile_id];
    const int o_end = bins.small.offset[tile_id + 1];
    const Tile tile = tile_of(tile_id, tiles_x);
    const int x = tile.x0 + tid % TS, y = tile.y0 + tid / TS;
    const bool inside = x < s.width && y < s.height;
    // Tiles nothing was binned into (most of the image around a mesh: half of the tiles of the 1M-triangle scene) take a
    // short cut: background written straight away, no barrier, no copy pipeline.
    if ((c_small | c_large) == 0) {
        if (!inside) return;
        const size_t idx = (size_t)y * s.width + x;
        z_buffer[idx] = __longlong_as_double(0x7ff0000000000000LL);
        owner[idx] = -1;
        if (face_id) face_id[idx] = -1;
        if (FUSE) {
            SceneView sc = s;
            fix_channel_count<MAXC, TEX>(sc);
            PixelState<MAXC> q;
            q.own = q.bown = -1;
            q.z = 0.0;
            phase_shade<MAXC>(sc, x, y, &q);
            for (int k = 0; k < sc.nb_colors; k++) image[idx * sc.nb_colors + k] = q.col[k];
            if (err) err[idx] = (float)pixel_residual<MAXC>(sc, q.col, obs + idx * sc.nb_colors);
            if (bary) { bary[3 * idx] = 0.0f; bary[3 * idx + 1] = 0.0f; bary[3 * idx + 2] = 0.0f; }
        }
        return;
    }
    const int n_small = min(c_small, o_end - o_begin);
    const PreRec *list = bins.small_recs + o_begin;
    const int n_chunks = (n_small + PRE_CHUNK - 1) / PRE_CHUNK;
    sh.tri.pix_cnt[tid] = 0;
    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
    }
    auto issue = [&](int chunk) {  // thread 0: start the copy of records [chunk * PRE_CHUNK, ...) into buffer chunk & 1
        const int m = min(PRE_CHUNK, n_small - chunk * PRE_CHUNK);
        mbar_expect_tx(&bar[chunk & 1], (uint32_t)(m * sizeof(PreRec)));
        bulk_load(pre[chunk & 1], list + chunk * PRE_CHUNK, (uint32_t)(m * sizeof(PreRec)), &bar[chunk & 1]);
    };
    __syncthreads();  // barriers initialised, candidate counters cleared
    if (tid == 0) {
        if (n_chunks > 0) issue(0);
        if (n_chunks > 1) issue(1);
    }
    PixelState<1> p;
    p.z = __longlong_as_double(0x7ff0000000000000LL);
    p.own = -1;
    p.bown = -1;
    uint32_t parity0 = 0, parity1 = 0;
    for (int chunk = 0; chunk < n_chunks; chunk++) {
        const int b = chunk & 1;
        const int m = min(PRE_CHUNK, n_small - chunk * PRE_CHUNK);
        if (b == 0) { mbar_wait(&bar[0], parity0); parity0 ^= 1u; }
        else        { mbar_wait(&bar[1], parity1); parity1 ^= 1u; }
        phase_pre_scatter<DevEnv>(tid, m, pre[b], &sh);
        __syncthreads();
        phase_pix_test<1>(s, tid, m, tile, pre[b], &sh, &p);  // (pixels outside the image have no candidates)
        if (chunk + 1 < n_chunks) {
            // every pixel is done with buffer b and with its candidate list: the next chunk may be scattered, and the
            // chunk after it may land in buffer b while that one is tested
            __syncthreads();
            if (tid == 0 && chunk + 2 < n_chunks) issue(chunk + 2);
        }
        // (after the last chunk: the large-triangle phases use other fields of sh, the epilogue ends with a barrier)
    }
    // large triangles: by index, stencil set-up and row spans computed here, one thread per triangle
    const int n_large = min(c_large, bins.large.offset[tile_id + 1] - bins.large.offset[tile_id]);
    if (n_large > 0) {
        const int *large = bins.large_refs + bins.large.offset[tile_id];
        for (int base = 0; base < n_large; base += LARGE_CHUNK) {
            const int m = min(LARGE_CHUNK, n_large - base);
            if (base > 0) __syncthreads();  // the previous chunk's stencils / masks have been consumed
            phase_tri_setup(s, tid, m, large + base, &sh);
            __syncthreads();
            phase_tri_masks(s, tid, m, tile, &sh);
            __syncthreads();
            if (inside) phase_tri_test<1>(s, tid, m, tile, &sh, &p);
        }
    }
    if (inside) {
        const size_t idx = (size_t)y * s.width + x;
        z_buffer[idx] = p.z;
        int code = p.bown;
        if (p.own != p.bown) {  // exact z tie between distinct triangles: keep both ids in the side table
            int slot = atomicAdd(ties.counter, 1);
            if (slot < ties.capacity) {
                ties.pairs[2 * slot] = p.own;
                ties.pairs[2 * slot + 1] = p.bown;
                code = -2 - slot;
            }
        }
        owner[idx] = code;
        if (face_id) face_id[idx] = p.own >= 0 ? (p.own & TRI_INDEX_MASK) : -1;
        if (FUSE) {
            SceneView sc = s;
            fix_channel_count<MAXC, TEX>(sc);
            PixelState<MAXC> q;
            q.own = p.own;
            q.bown = p.bown;
            q.z = PERSP && p.own >= 0 ? p.z : 0.0;
            float w[3];
            phase_shade<MAXC>(sc, x, y, &q, bary ? w : nullptr);
            if (MAXC <= 4 && tma_store) {
                for (int k = 0; k < sc.nb_colors; k++) stage[tid * sc.nb_colors + k] = q.col[k];
            } else {
                for (int k = 0; k < sc.nb_colors; k++) image[idx * sc.nb_colors + k] = q.col[k];
            }
            if (err) err[idx] = (float)pixel_residual<MAXC>(sc, q.col, obs + idx * sc.nb_colors);
            if (bary) { bary[3 * idx] = w[0]; bary[3 * idx + 1] = w[1]; bary[3 * idx + 2] = w[2]; }
        }
    }
    // the adjoint's pixel-parallel kernel walks the tiles where a pixel is owned by a triangle that the
    // triangle-parallel adjoint does not take (medium and large triangles)
    const bool other = inside && p.bown >= 0 && !(p.bown & SMALL_FLAG);
    if (FUSE && MAXC <= 4 && tma_store) fence_proxy_async();  // this thread's staged colours -> visible to the TMA engine
    const bool listed = __syncthreads_or(other);
    if (tid == 0) {
        if (listed) large_tiles[atomicAdd(scal + SC_LARGE_TILES, 1)] = tile_id;
        if (FUSE && MAXC <= 4 && tma_store) {
            // rows / columns of the box that stick out of the image are clipped by the hardware
            tma_store_tile(&image_map, tile.x0 * s.nb_colors, tile.y0, stage);
            tma_store_wait_read();  // the staging buffer must outlive the copy engine's read
        }
    }
}

// Forward, kernel 2 of 3 - colour of every pixel from its owner (one thread per pixel, tile-shaped blocks for
// locality of the vertex gathers).  Reads owner (and z with perspective_correct), writes image; optionally the
// squared residual against `obs` (antialiase_error mode, DR.h:2824-2837) and the owner's interpolation weights.
template <int MAXC, bool PERSP, bool TEX>
#ifndef DEODR_SHADE_MIN_CTAS
#define DEODR_SHADE_MIN_CTAS 6  // 40 registers: measured 55.5 us vs 58.6 us at 48 (5 CTAs / SM) and 67 us at 56
#endif
__global__ void __launch_bounds__(NT, DEODR_SHADE_MIN_CTAS) k_shade(SceneView s, TileDiv tiles_x, TieTable ties, const int *owner,
                                              const double *z_buffer, float *image, const float *obs, float *err,
                                              float *bary, const int *scal) {
    if (scal[SC_OVERFLOW] & ~OVF_EDGE_REFS) return;  // (see k_tile_z)
    fix_channel_count<MAXC, TEX>(s);
    s.perspective_correct = PERSP ? 1 : 0;
    const Tile tile = tile_of(blockIdx.x, tiles_x);
    const int x = tile.x0 + threadIdx.x % TS, y = tile.y0 + threadIdx.x / TS;
    if (x >= s.width || y >= s.height) return;
    const size_t idx = (size_t)y * s.width + x;
    PixelState<MAXC> p;
    decode_owner(owner[idx], ties, &p.own, &p.bown);
    p.z = s.perspective_correct && p.own >= 0 ? z_buffer[idx] : 0.0;
    if (bary) {
        float w[3];
        phase_shade<MAXC>(s, x, y, &p, w);
        bary[3 * idx] = w[0];
        bary[3 * idx + 1] = w[1];
        bary[3 * idx + 2] = w[2];
    } else {
        phase_shade<MAXC>(s, x, y, &p);
    }
    for (int k = 0; k < s.nb_colors; k++) image[idx * s.nb_colors + k] = p.col[k];
    if (err) err[idx] = (float)pixel_residual<MAXC>(s, p.col, obs + idx * s.nb_colors);
}

// Forward, kernel 3 of 3 - ordered silhouette-edge overdraw on the tiles that have edges (DR.h:2839-2899).
// One CTA per tile (stride loop over the device-side list), the tiles with more than one chunk of edges first: the few
// crowded tiles set the kernel's duration.  Per chunk of <= 64 edges: records copied to shared memory, (edge, row) x
// spans computed (and saved for the adjoint pass), then every pixel blends the edges of its own 64-bit hit mask in
// far-to-near order.  ERR: antialiase_error mode - the edges overdraw the squared residual instead of the colours
// (DR.h:2186-2187, 2467-2468); the image keeps its aliased edges.
template <int MAXC, bool PERSP, bool TEX, bool ERR>
__global__ void __launch_bounds__(EDGE_NT, DEODR_EDGE_MIN_CTAS) k_edge_fwd(SceneView s, double sigma, TileDiv tiles_x, EdgeTiles et,
                                                      uint32_t *span_cache, const double *z_buffer, float *image,
                                                      const float *obs, float *err_buffer) {
    if (et.scal[SC_OVERFLOW]) return;
    fix_channel_count<MAXC, TEX>(s);
    s.perspective_correct = PERSP ? 1 : 0;
    __shared__ TileShared sh;
    const int tid = threadIdx.x;
    const int heavy = et.scal[SC_HEAVY_TILES], total = heavy + et.scal[SC_LIGHT_TILES];
    // one CTA per entry of the list (the launch covers the plan's capacity; k_bin_edges raises OVF_EDGE_TILES beyond it)
    if ((int)blockIdx.x >= total) return;
    {
        const int tile_id = two_ended_at(et.list, et.num_tiles, heavy, blockIdx.x);
        const int n_edge = segment_size(et.seg, tile_id);
        const Tile tile = tile_of(tile_id, tiles_x);
        const int r = tid / TS;
        const int x = tile.x0 + tid % TS, y = tile.y0 + r;
        const bool inside = x < s.width && y < s.height;
        const size_t idx = inside ? (size_t)y * s.width + x : 0;
        PixelState<MAXC> p;
        float err = 0.0f;
        p.z = 0.0;
        p.own = p.bown = -1;
        if (inside) {
            p.z = z_buffer[idx];
            if (ERR) err = err_buffer[idx];
            else
                for (int k = 0; k < s.nb_colors; k++) p.col[k] = image[idx * s.nb_colors + k];
        }
        const int edge_base = et.seg.offset[tile_id];
        for (int base = 0; base < n_edge; base += EDGE_CHUNK) {
            const int m = min(EDGE_CHUNK, n_edge - base);
            phase_edge_setup(tid, EDGE_NT, m, et.refs + edge_base + base, et.recs, &sh);
            __syncthreads();
            phase_edge_spans(s, tid, EDGE_NT, m, tile, 0, EDGE_ROWS, &sh);
            __syncthreads();
            // the backward pass reuses the spans (same scene, same sigma): 64 bytes per (tile, edge), coalesced
            for (int item = tid; item < m * TS; item += EDGE_NT)
                span_cache[(size_t)(edge_base + base) * TS + item] = sh.edge.span[item / TS][item % TS];
            if (inside) {
                if (ERR) phase_edge_blend_error<MAXC>(s, x, y, r, m, &sh, p.z, obs + idx * s.nb_colors, &err);
                else phase_edge_blend<MAXC>(s, x, y, r, m, &sh, &p);
            }
            __syncthreads();
        }
        if (inside) {
            if (ERR) err_buffer[idx] = err;
            else
                for (int k = 0; k < s.nb_colors; k++) image[idx * s.nb_colors + k] = p.col[k];
        }
    }
}

__global__ void k_check_scene(SceneView s, int *bad) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 3 * s.nb_triangles) return;
    if (s.faces[i] >= (uint32_t)s.nb_vertices) atomicOr(bad, 1);
    if (s.faces_uv[i] >= (uint32_t)s.nb_uv) atomicOr(bad, 2);
}

// ------------------------------------------------------------------------------------------------- host side

char *deodr_error_buffer() {
    static thread_local char buffer[512] = "";
    return buffer;
}

static int sm_count_cached = 0;

static bool stream_is_capturing(cudaStream_t st) {
    cudaStreamCaptureStatus status = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &status) != cudaSuccess) { cudaGetLastError(); return false; }
    return status != cudaStreamCaptureStatusNone;
}

// persp_adjoint: the caller is the entry point that has the perspective-correct adjoint (deodr_b200_render_b_views_depths)
static int validate_view(const DeodrSceneView *v, bool backward, bool persp_adjoint = false) {
    if (!v) return set_error(DEODR_B200_EINVAL, "scene == NULL");
    // zero-sized arrays may legitimately come with a null data pointer
    const bool tris = v->nb_triangles > 0, verts = v->nb_vertices > 0;
    if (tris && !v->faces) return set_error(DEODR_B200_EINVAL, "scene.faces == NULL");
    if (tris && !v->faces_uv) return set_error(DEODR_B200_EINVAL, "scene.faces_uv == NULL");
    if (verts && !v->depths) return set_error(DEODR_B200_EINVAL, "scene.depths == NULL");
    if (v->nb_uv > 0 && !v->uv) return set_error(DEODR_B200_EINVAL, "scene.uv == NULL");
    if (verts && !v->ij) return set_error(DEODR_B200_EINVAL, "scene.ij == NULL");
    if (verts && !v->shade) return set_error(DEODR_B200_EINVAL, "scene.shade == NULL");
    if (verts && !v->colors) return set_error(DEODR_B200_EINVAL, "scene.colors == NULL");
    if (tris && !v->edgeflags) return set_error(DEODR_B200_EINVAL, "scene.edgeflags == NULL");
    if (tris && !v->textured) return set_error(DEODR_B200_EINVAL, "scene.textured == NULL");
    if (tris && !v->shaded) return set_error(DEODR_B200_EINVAL, "scene.shaded == NULL");
    if (v->texture_height > 0 && v->texture_width > 0 && !v->texture)
        return set_error(DEODR_B200_EINVAL, "scene.texture == NULL");
    if (!v->background_image && !v->background_color)
        return set_error(DEODR_B200_EINVAL, "scene.background == NULL and scene.background_color == NULL");
    if (v->height <= 0 || v->width <= 0 || v->height > 32767 || v->width > 32767)
        return set_error(DEODR_B200_EINVAL, "image sides must be in [1, 32767] (short loop counters, DR.h:925)");
    if (v->nb_colors < 1 || v->nb_colors > 16)
        return set_error(DEODR_B200_EUNSUPPORTED, "nb_colors must be in [1, 16]");
    if (v->nb_triangles < 0 || v->nb_vertices < 0 || v->nb_uv < 0)
        return set_error(DEODR_B200_EINVAL, "negative size");
    if (backward) {
        if (!v->backface_culling)
            return set_error(DEODR_B200_EUNSUPPORTED,
                             "You have to use backface_culling true if you ant to compute gradients");
        if (v->perspective_correct && !persp_adjoint)
            return set_error(DEODR_B200_EUNSUPPORTED,
                             "backward gradient propagation not supported yet with perspective_correct=True");
    }
    return DEODR_B200_OK;
}

// ---- view slots ------------------------------------------------------------------------------------------------

static void free_slot(ViewSlot *v) {
    if (!v) return;
    DevBuf *bufs[] = {&v->zeroed, &v->small_offset, &v->large_offset, &v->edge_offset, &v->small_recs, &v->large_refs,
                      &v->small_ids, &v->large_tiles, &v->edge_tiles, &v->edge_tiles_raw, &v->edge_ids, &v->edge_keys, &v->edge_recs,
                      &v->edge_refs_tmp, &v->edge_refs, &v->edge_spans, &v->edge_acc, &v->tie_pairs, &v->error_image_b};
    for (DevBuf *b : bufs) b->release();
    if (v->host_totals) cudaFreeHost(v->host_totals);
    delete v;
}

static int get_slot(DeodrWorkspace *ws, int index, ViewSlot **out) {
    if (index < 0 || index >= 65536) return set_error(DEODR_B200_EINVAL, "bad view index");
    while ((int)ws->slots.size() <= index) ws->slots.push_back(nullptr);
    if (!ws->slots[index]) {
        ViewSlot *v = new (std::nothrow) ViewSlot();
        if (!v) return set_error(DEODR_B200_ENOMEM, "out of host memory");
        memset(&v->fwd_scene, 0, sizeof(v->fwd_scene));
        memset(&v->fwd_io, 0, sizeof(v->fwd_io));
        if (cudaMallocHost(&v->host_totals, (SC_WORDS + 8) * sizeof(int)) != cudaSuccess) {
            delete v;
            return set_error(DEODR_B200_ECUDA, "cudaMallocHost failed");
        }
        memset(v->host_totals, 0, (SC_WORDS + 8) * sizeof(int));
        ws->slots[index] = v;
    }
    *out = ws->slots[index];
    return DEODR_B200_OK;
}

// Buffers whose size follows from the shape alone; invalidates the plan when the shape differs from the plan's.
static int prepare_slot(DeodrWorkspace *ws, ViewSlot *v, const SceneView &s, double sigma) {
    const int tiles_x = (s.width + TS - 1) / TS, tiles_y = (s.height + TS - 1) / TS, nt = tiles_x * tiles_y;
    FwdPlan &plan = v->plan;
    if (plan.valid && (plan.T != s.nb_triangles || plan.H != s.height || plan.W != s.width ||
                       plan.edges_possible != (sigma > 0)))
        plan.valid = false;
    v->tiles_x = tiles_x;
    v->tiles_y = tiles_y;
    v->num_tiles = nt;
    const size_t T = (size_t)s.nb_triangles;
    int rc = 0;
    rc |= v->zeroed.ensure((SC_WORDS + 3 * (size_t)nt) * sizeof(int), &ws->bytes);
    rc |= v->small_offset.ensure(((size_t)nt + 1) * sizeof(int), &ws->bytes);
    rc |= v->large_offset.ensure(((size_t)nt + 1) * sizeof(int), &ws->bytes);
    rc |= v->edge_offset.ensure(((size_t)nt + 1) * sizeof(int), &ws->bytes);
    rc |= v->large_tiles.ensure(((size_t)nt + 1) * sizeof(int), &ws->bytes);
    rc |= v->edge_tiles.ensure(((size_t)nt + 1) * sizeof(int), &ws->bytes);
    rc |= v->small_ids.ensure((T + 4) * sizeof(int), &ws->bytes);
    // one (own, bown) slot per pixel: the exact-tie table can never overflow
    const size_t pixels = (size_t)s.height * s.width;
    if ((size_t)v->tie_capacity < pixels) {
        rc |= v->tie_pairs.ensure(2 * pixels * sizeof(int), &ws->bytes);
        if (!rc) v->tie_capacity = (int)pixels;
    }
    if (rc) return DEODR_B200_ECUDA;
    v->scal = v->zeroed.as<int>();
    v->small_cursor = v->scal + SC_WORDS;
    v->large_cursor = v->small_cursor + nt;
    v->edge_cursor = v->large_cursor + nt;
    return DEODR_B200_OK;
}

// Waits for the sequence flag a kernel raises in the slot's pinned totals (k_scan_tiles / k_publish); polls the stream
// every few microseconds as a safety net (flag lost / launch failed).
static int wait_totals(ViewSlot *v, cudaStream_t st) {
    volatile int *flag = v->host_totals + SC_WORDS;
    for (unsigned spins = 1; *flag != v->totals_seq; spins++) {
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
        if ((spins & 0xfffu) == 0) {
            const cudaError_t q = cudaStreamQuery(st);
            if (q == cudaSuccess) {
                if (*flag != v->totals_seq) {  // not expected; fall back to an explicit copy
                    CUDA_TRY(cudaMemcpyAsync(v->host_totals, v->scal, SC_WORDS * sizeof(int), cudaMemcpyDeviceToHost, st));
                    CUDA_TRY(cudaStreamSynchronize(st));
                }
                break;
            }
            if (q != cudaErrorNotReady) return set_error(DEODR_B200_ECUDA, "forward pass failed: %s", cudaGetErrorString(q));
        }
    }
    __atomic_thread_fence(__ATOMIC_ACQUIRE);
    return DEODR_B200_OK;
}

// The handshake of the pinned totals: the HOST clears the flag before it launches the kernels of a pass, the publishing
// kernel raises it to 1.  (A constant instead of a per-pass sequence number: the launch is then identical from pass to
// pass, which is what lets the library replay it from a captured graph.)
static int next_seq(ViewSlot *v) {
    v->totals_seq = 1;
    ((volatile int *)v->host_totals)[SC_WORDS] = 0;
    __atomic_thread_fence(__ATOMIC_SEQ_CST);
    return 1;
}

static int bad_index_error(const ViewSlot *v) {
    if (v->host_totals[SC_BAD_INDEX] & 1)
        return set_error(DEODR_B200_EINVAL, "scene.faces value greater than scene.nb_vertices");
    if (v->host_totals[SC_BAD_INDEX] & 2)
        return set_error(DEODR_B200_EINVAL, "scene.faces_uv value greater than scene.nb_uv");
    return DEODR_B200_OK;
}

#ifndef DEODR_SMALL_TEXTURED_MIN_TRIANGLES
#define DEODR_SMALL_TEXTURED_MIN_TRIANGLES 262144  // measured: 50k-triangle scene 0.287 -> 0.204 ms without, 1M-triangle scene 0.600 vs 0.651 ms with
#endif
// Height limit of the record path for triangles that are not small: RECORD_ROWS once the binning pass has enough
// threads to fill the chip (a few resident warps per SM sub-partition), 0 below (DEODR_B200_RECORD_ROWS overrides).
static int record_rows_for(int nb_triangles) {
    static const int forced = getenv("DEODR_B200_RECORD_ROWS") ? atoi(getenv("DEODR_B200_RECORD_ROWS")) : -1;
    if (forced >= 0) return forced < RECORD_ROWS ? forced : RECORD_ROWS;
    return nb_triangles >= 32768 ? RECORD_ROWS : 0;
}

// May textured triangles be "small" (triangle-parallel adjoint, TriBins::small_textured)?  One thread then walks up to
// 64 pixels of dependent texture fetches + twelve texel atomics each: it needs several hundred thousand triangles in
// flight to hide that latency.  Below, textured triangles are owned through the pixel-parallel adjoint (measured on
// the 50k-triangle textured scene, see DESIGN.md).  DEODR_B200_SMALL_TEXTURED = 0 / 1 overrides.
static int small_textured_for(int nb_triangles) {
    static const int forced = getenv("DEODR_B200_SMALL_TEXTURED") ? atoi(getenv("DEODR_B200_SMALL_TEXTURED")) : -1;
    if (forced >= 0) return forced != 0;
    return nb_triangles >= DEODR_SMALL_TEXTURED_MIN_TRIANGLES;
}

// Plan building: count pass + scans + ONE read-back, then the list buffers are (re)allocated.
static int build_plan(DeodrWorkspace *ws, ViewSlot *v, const SceneView &s, double sigma, cudaStream_t st,
                      bool check_indices) {
    PhaseTimer timer(ws, DEODR_B200_PH_PLAN, st);
    FwdPlan &plan = v->plan;
    plan.valid = false;
    const int T = s.nb_triangles, nt = v->num_tiles;
    CUDA_TRY(cudaMemsetAsync(v->scal, 0, (SC_WORDS + 3 * (size_t)nt) * sizeof(int), st));
    if (T > 0) {
        if (check_indices) {
            k_check_scene<<<grid_for(3 * (size_t)T, 256), 256, 0, st>>>(s, v->scal + SC_BAD_INDEX);
            ws->launches++;
        }
        TriBins bins{{nullptr, v->small_cursor}, nullptr, {nullptr, v->large_cursor}, nullptr, v->scal + SC_OVERFLOW,
                     record_rows_for(T), small_textured_for(T)};
        EdgeList edges{v->scal + SC_EDGES, nullptr, nullptr, 0};
        k_bin<true><<<grid_for(T, 128), 128, 0, st>>>(s, sigma, v->tiles_x, bins, v->scal, nullptr, edges,
                                                     v->edge_cursor, 1);
        ws->launches++;
    }
    ScanJob job{{v->small_cursor, v->large_cursor, v->edge_cursor},
                {v->small_offset.as<int>(), v->large_offset.as<int>(), v->edge_offset.as<int>()},
                {SC_TOTAL_SMALL, SC_TOTAL_LARGE, SC_TOTAL_EDGE_REFS},
                {-1, SC_PLAN_LARGE_TILES, SC_PLAN_EDGE_TILES}};
    k_scan_tiles<<<3, 1024, SCAN_SMEM, st>>>(job, nt, v->scal, v->host_totals, next_seq(v));
    ws->launches++;
    CUDA_TRY(cudaGetLastError());
    if (int rc = wait_totals(v, st)) return rc;
    if (check_indices)
        if (int rc = bad_index_error(v)) return rc;
    const int *tot = v->host_totals;
    const int E = tot[SC_EDGES];
    plan.T = T; plan.H = s.height; plan.W = s.width;
    plan.edges_possible = sigma > 0;
    plan.cap_small = tot[SC_TOTAL_SMALL];
    plan.cap_large = tot[SC_TOTAL_LARGE];
    plan.cap_edges = E > 0 ? E + E / 4 + 64 : 0;
    plan.cap_edge_refs = E > 0 ? tot[SC_TOTAL_EDGE_REFS] : 0;
    plan.tex = tot[SC_TEXTURED] != 0;
    plan.hint_small = T;
    plan.hint_edges = E;
    plan.cap_edge_tiles = E > 0 ? std::min(nt, tot[SC_PLAN_EDGE_TILES] + tot[SC_PLAN_EDGE_TILES] / 4 + 8) : 0;
    plan.hint_edge_tiles = plan.cap_edge_tiles;
    plan.hint_large_tiles = tot[SC_PLAN_LARGE_TILES] + tot[SC_PLAN_LARGE_TILES] / 4 + 8;
    int rc = 0;
    rc |= v->small_recs.ensure(((size_t)plan.cap_small + 1) * sizeof(PreRec), &ws->bytes);
    rc |= v->large_refs.ensure(((size_t)plan.cap_large + 4) * sizeof(int), &ws->bytes);
    if (plan.cap_edges > 0) {
        rc |= v->edge_ids.ensure(((size_t)plan.cap_edges + 4) * sizeof(int), &ws->bytes);
        rc |= v->edge_keys.ensure(((size_t)plan.cap_edges + 4) * sizeof(uint64_t), &ws->bytes);
        rc |= v->edge_recs.ensure(((size_t)plan.cap_edges + 1) * sizeof(EdgeRec), &ws->bytes);
        rc |= v->edge_refs_tmp.ensure(((size_t)plan.cap_edge_refs + 4) * sizeof(int), &ws->bytes);
        rc |= v->edge_refs.ensure(((size_t)plan.cap_edge_refs + 4) * sizeof(int), &ws->bytes);
        rc |= v->edge_spans.ensure(((size_t)plan.cap_edge_refs + 4) * TS * sizeof(uint32_t), &ws->bytes);
        rc |= v->edge_tiles_raw.ensure(((size_t)plan.cap_edge_tiles + 4) * sizeof(int), &ws->bytes);
    }
    if (rc) return DEODR_B200_ECUDA;
    plan.valid = true;
    ws->replans++;
    return DEODR_B200_OK;
}

// `stage`: 0 = z pass (shading fused when possible), colour pass if unfused, edge overdraw; 1 = the UNFUSED z pass only
// (the geometry half of a forward in two calls); 2 = what follows it (colour pass + edge overdraw).
template <int MAXC>
static void launch_raster_fwd(DeodrWorkspace *ws, ViewSlot *v, Lane &lane, const SceneView &s, const DeodrViewIO &io,
                              double sigma, bool err_mode, bool edge_chain, const TriBins &bins, int stage = 0) {
    cudaStream_t st = lane.main;
    const bool tex = v->plan.tex != 0;
    const TileDiv div = make_tile_div(v->tiles_x);
    const TieTable ties = tie_table(v);
    // shading fused into the z pass unless the colours arrive late (see k_tile_z) or DEODR_B200_FUSE_SHADE=0 (A/B)
    static const bool fuse_allowed = !(getenv("DEODR_B200_FUSE_SHADE") && atoi(getenv("DEODR_B200_FUSE_SHADE")) == 0);
    // DEODR_B200_LATE_COLORS=shade: with a colours-ready event keep the colour pass apart so that the z pass too overlaps
    // the caller's communication (default: stay fused and wait in front of the z pass - the binning pass alone, 75 us on
    // the 1M-triangle scene, hides an all-reduce of the colour gradient, and fusion is worth 24 us every step)
    static const bool late_shade = getenv("DEODR_B200_LATE_COLORS") && !strcmp(getenv("DEODR_B200_LATE_COLORS"), "shade");
    const bool fuse = stage == 0 && fuse_allowed && !(ws->colors_ready && late_shade);
    // (inside a capture - the library's own or the caller's - the wait becomes an EXTERNAL event wait node: every replay
    // waits for whatever the caller has recorded on the event by the time the replay gets there)
    const unsigned wait_flags = (ws->capturing_internally || stream_is_capturing(st)) ? cudaEventWaitExternal : 0;
    if (fuse && ws->colors_ready) cudaStreamWaitEvent(st, ws->colors_ready, wait_flags);
    if (stage != 2) {
        PhaseTimer timer(ws, DEODR_B200_PH_TILE_Z, st);
        const int grid = v->num_tiles;  // one CTA per tile (see k_tile_z)
        const float *obs = err_mode ? io.obs : nullptr;
        float *err = err_mode ? io.err_buffer : nullptr;
        TileMap image_map;
        memset(&image_map, 0, sizeof(image_map));
        static const bool tma_allowed = !(getenv("DEODR_B200_TMA_TILES") && atoi(getenv("DEODR_B200_TMA_TILES")) == 0);
        const int tma_store = fuse && tma_allowed && s.nb_colors <= 4 &&
                              encode_tile_map(&image_map, io.image, 4, true, s.height, s.width * s.nb_colors, TS, TS * s.nb_colors);
#define DEODR_TILE_Z(C_, P, X, F) k_tile_z<C_, P, X, F><<<grid, NT, 0, st>>>(s, div, v->num_tiles, bins, ties, io.z_buffer, io.owner, io.face_id, v->scal, v->large_tiles.as<int>(), io.image, obs, err, io.barycentric, image_map, tma_store)
        if (!fuse) {
            if (s.perspective_correct) DEODR_TILE_Z(1, true, false, false); else DEODR_TILE_Z(1, false, false, false);
        } else if (s.perspective_correct) {
            if (tex) DEODR_TILE_Z(MAXC, true, true, true); else DEODR_TILE_Z(MAXC, true, false, true);
        } else {
            if (tex) DEODR_TILE_Z(MAXC, false, true, true); else DEODR_TILE_Z(MAXC, false, false, true);
        }
#undef DEODR_TILE_Z
        ws->launches++;
    }
    if (stage == 1) return;
    if (!fuse) {
        if (ws->colors_ready) cudaStreamWaitEvent(st, ws->colors_ready, wait_flags);  // first reader of the colours here
        PhaseTimer timer(ws, DEODR_B200_PH_SHADE, st);
        (s.perspective_correct ? (tex ? k_shade<MAXC, true, true> : k_shade<MAXC, true, false>)
                               : (tex ? k_shade<MAXC, false, true> : k_shade<MAXC, false, false>))<<<v->num_tiles, NT, 0, st>>>(
            s, div, ties, io.owner, io.z_buffer, io.image, err_mode ? io.obs : nullptr, err_mode ? io.err_buffer : nullptr,
            io.barycentric, v->scal);
        ws->launches++;
    }
    if (edge_chain) {
        join_stream(ws, lane, 0);  // the edge lists are ready
        PhaseTimer timer(ws, DEODR_B200_PH_EDGE_FWD, st);
        const EdgeTiles et = edge_tiles_of(v);
        const int grid = at_least_one(v->plan.cap_edge_tiles);
        uint32_t *spans = v->edge_spans.as<uint32_t>();
#define DEODR_EDGE_FWD(P, X, R) k_edge_fwd<MAXC, P, X, R><<<grid, EDGE_NT, 0, st>>>(s, sigma, div, et, spans, io.z_buffer, io.image, io.obs, io.err_buffer)
        const int sel = (s.perspective_correct ? 4 : 0) | (tex ? 2 : 0) | (err_mode ? 1 : 0);
        switch (sel) {
            case 0: DEODR_EDGE_FWD(false, false, false); break;
            case 1: DEODR_EDGE_FWD(false, false, true); break;
            case 2: DEODR_EDGE_FWD(false, true, false); break;
            case 3: DEODR_EDGE_FWD(false, true, true); break;
            case 4: DEODR_EDGE_FWD(true, false, false); break;
            case 5: DEODR_EDGE_FWD(true, false, true); break;
            case 6: DEODR_EDGE_FWD(true, true, false); break;
            default: DEODR_EDGE_FWD(true, true, true); break;
        }
#undef DEODR_EDGE_FWD
        ws->launches++;
    }
}

// Enqueues one forward pass of the view on the lane's streams, against the slot's plan; nothing here waits.
// `part`: 0 = the whole pass; 1 = its head only (list reset, index check, binning: DEODR_B200_FORWARD_GEOMETRY);
// 2 = everything after the head (DEODR_B200_FORWARD_RESUME).
static int enqueue_forward(DeodrWorkspace *ws, ViewSlot *v, Lane &lane, const SceneView &s, const DeodrViewIO &io,
                           double sigma, int flags, bool check_indices, int part = 0) {
    cudaStream_t st = lane.main;
    const FwdPlan &plan = v->plan;
    const int T = s.nb_triangles, nt = v->num_tiles;
    const bool err_mode = (flags & DEODR_B200_ANTIALIASE_ERROR) != 0;
    TriBins bins{{v->small_offset.as<int>(), v->small_cursor}, v->small_recs.as<PreRec>(),
                 {v->large_offset.as<int>(), v->large_cursor}, v->large_refs.as<int>(), v->scal + SC_OVERFLOW,
                 record_rows_for(T), small_textured_for(T)};
    EdgeList edges{v->scal + SC_EDGES, v->edge_ids.as<int>(), v->edge_keys.as<uint64_t>(), plan.cap_edges};
    const bool edge_chain = plan.cap_edges > 0;
    if (part != 2) {
        PhaseTimer timer(ws, DEODR_B200_PH_BIN, st);
        CUDA_TRY(cudaMemsetAsync(v->scal, 0, (SC_WORDS + 3 * (size_t)nt) * sizeof(int), st));
        if (T > 0) {
            if (check_indices) {  // checkSceneValid (DR.h:2703-2714) on the device, before any index is dereferenced
                k_check_scene<<<grid_for(3 * (size_t)T, 256), 256, 0, st>>>(s, v->scal + SC_BAD_INDEX);
                ws->launches++;
            }
            k_bin<false><<<grid_for(T, 128), 128, 0, st>>>(s, sigma, v->tiles_x, bins, v->scal, v->small_ids.as<int>(),
                                                          edges, nullptr, plan.tex);
            ws->launches++;
        }
    }
    // A forward in two calls: the head is the binning pass (75 us on the 1M-triangle scene, enough to hide a 6 MB
    // all-reduce on NVLink) and the second call runs the fused z pass.  DEODR_B200_GEOMETRY_Z=1 moves the z pass -
    // unfused: it reads no colour either - into the head as well: 150+ us to hide a slower collective behind, at the
    // price of the separate colour pass.  Measured on 2 GPUs (1M triangles, 2048^2): 0.352 ms per step without, 0.361 -
    // 0.389 ms with; one GPU, no collective: 0.312 ms.
    static const bool geometry_z = getenv("DEODR_B200_GEOMETRY_Z") && atoi(getenv("DEODR_B200_GEOMETRY_Z")) != 0;
    const int C = s.nb_colors;
    const int stage = part == 0 || !geometry_z ? 0 : part;
#define DEODR_RASTER_FWD(STAGE)                                                                            \
    do {                                                                                                   \
        if (C == 1) launch_raster_fwd<1>(ws, v, lane, s, io, sigma, err_mode, edge_chain, bins, STAGE);     \
        else if (C == 3) launch_raster_fwd<3>(ws, v, lane, s, io, sigma, err_mode, edge_chain, bins, STAGE); \
        else if (C <= 4) launch_raster_fwd<4>(ws, v, lane, s, io, sigma, err_mode, edge_chain, bins, STAGE); \
        else launch_raster_fwd<16>(ws, v, lane, s, io, sigma, err_mode, edge_chain, bins, STAGE);           \
    } while (0)
    if (part == 1) {
        if (geometry_z) DEODR_RASTER_FWD(1);
        CUDA_TRY(cudaGetLastError());
        return DEODR_B200_OK;
    }
    // ---- side chain (aux stream 0): silhouette-edge records + tile lists + their order, then the verdict goes to
    // the host; it overlaps the z pass and the shading and is joined before k_edge_fwd
    bool first_fork = true;
    cudaStream_t se = fork_stream(ws, lane, 0, &first_fork);
    if (edge_chain) {
        if (ws->colors_ready)  // the edge records hold end-point colours (external wait node inside a capture)
            cudaStreamWaitEvent(se, ws->colors_ready,
                                (ws->capturing_internally || stream_is_capturing(st)) ? cudaEventWaitExternal : 0);
        const EdgeBins ebins{{v->edge_offset.as<int>(), v->edge_cursor}, v->edge_refs_tmp.as<int>(), v->scal + SC_OVERFLOW,
                             v->edge_tiles_raw.as<int>(), v->scal + SC_EDGE_TILES, plan.cap_edge_tiles};
        {
            PhaseTimer timer(ws, DEODR_B200_PH_EDGE_BIN, se);
            k_bin_edges<<<at_least_one(grid_for(32 * (size_t)plan.hint_edges, 128)), 128, 0, se>>>(s, sigma, v->tiles_x, edges, ebins,
                                                                                      v->edge_recs.as<EdgeRec>(), v->scal);
        }
        {
            PhaseTimer timer(ws, DEODR_B200_PH_EDGE_TILE_SORT, se);
            k_sort_tile_edges<<<at_least_one(plan.cap_edge_tiles), 128, 0, se>>>(
                ebins.seg, nt, v->edge_refs_tmp.as<int>(), v->edge_refs.as<int>(), v->edge_recs.as<EdgeRec>(),
                v->edge_tiles_raw.as<int>(), v->edge_tiles.as<int>(), v->scal);
        }
        ws->launches += 2;
    }
    k_publish<<<1, 32, 0, se>>>(v->scal, v->host_totals, next_seq(v));
    ws->launches++;
    v->pending = true;
    v->hints_exact = false;
    if (!ws->overlap || !edge_chain) {
        // (serial mode: everything is on the main stream already; without an edge chain the main chain does not
        // depend on the aux stream, but the lane must still be joined for stream capture / ordering of the next pass)
    }
    // ---- main chain: z pass, shading, (join) edge overdraw
    DEODR_RASTER_FWD(stage);
#undef DEODR_RASTER_FWD
    if (!edge_chain) join_stream(ws, lane, 0);
    CUDA_TRY(cudaGetLastError());
    return DEODR_B200_OK;
}

// Reads the verdict of the slot's pending pass (waits for its flag) and folds the counts into the plan's hints.
// *overflow: the pass is void.
static int read_verdict(DeodrWorkspace *ws, ViewSlot *v, cudaStream_t st, bool *overflow) {
    *overflow = false;
    if (!v->pending) return DEODR_B200_OK;
    if (int rc = wait_totals(v, st)) return rc;
    v->pending = false;
    const int *tot = v->host_totals;
    FwdPlan &plan = v->plan;
    if (tot[SC_OVERFLOW]) {
        *overflow = true;
        plan.valid = false;
        v->fwd_valid = 0;
        return DEODR_B200_OK;
    }
    plan.hint_small = tot[SC_SMALL];
    plan.hint_edges = tot[SC_EDGES];
    plan.hint_edge_tiles = tot[SC_HEAVY_TILES] + tot[SC_LIGHT_TILES];
    v->hints_exact = true;  // the adjoint of this pass can be launched for exactly these counts
    if (plan.tex && !tot[SC_TEXTURED]) plan.tex = 0;  // next pass: instances without the texture paths
    (void)ws;
    return DEODR_B200_OK;
}

struct ViewCall {
    SceneView s;
    DeodrViewIO io;
};

static int check_forward_args(const DeodrSceneView *scene, const DeodrViewIO *io, double sigma, int flags) {
    if (int rc = validate_view(scene, false)) return rc;
    if (!io) return set_error(DEODR_B200_EINVAL, "io == NULL");
    if (!io->image) return set_error(DEODR_B200_EINVAL, "image_ptr is NULL");
    if (!io->z_buffer) return set_error(DEODR_B200_EINVAL, "z_buffer_ptr is NULL");
    if (!io->owner) return set_error(DEODR_B200_EINVAL, "owner is NULL");
    if (!(sigma >= 0)) return set_error(DEODR_B200_EINVAL, "sigma must be >= 0");
    if (flags & DEODR_B200_ANTIALIASE_ERROR) {
        if (!io->obs) return set_error(DEODR_B200_EINVAL, "obs_ptr is NULL");
        if (!io->err_buffer) return set_error(DEODR_B200_EINVAL, "err_buffer_ptr is NULL");
    }
    return DEODR_B200_OK;
}

// Lanes of a multi-view call: lane 0 is the caller's stream, lanes > 0 are forked from it / joined to it.
static void open_lanes(DeodrWorkspace *ws, cudaStream_t st, int used) {
    ws->lanes[0].main = st;
    if (used <= 1) return;
    cudaEventRecord(ws->lanes[0].ev_begin, st);
    for (int l = 1; l < used; l++) cudaStreamWaitEvent(ws->lanes[l].main, ws->lanes[0].ev_begin, 0);
}
static void close_lanes(DeodrWorkspace *ws, cudaStream_t st, int used) {
    for (int l = 1; l < used; l++) {
        cudaEventRecord(ws->lanes[l].ev_end, ws->lanes[l].main);
        cudaStreamWaitEvent(st, ws->lanes[l].ev_end, 0);
    }
}
static int lanes_for(const DeodrWorkspace *ws, int n_views) {
    if (!ws->overlap || n_views <= 1) return 1;
    return n_views < ws->num_lanes ? n_views : ws->num_lanes;
}

// ---- captured launch sequences (GraphCache, workspace.h) -----------------------------------------------------------

struct KeyWriter {
    std::vector<unsigned char> bytes;
    template <class T>
    void put(const T &v) {
        const unsigned char *p = reinterpret_cast<const unsigned char *>(&v);
        bytes.insert(bytes.end(), p, p + sizeof(T));
    }
};

// what a slot contributes to a key: its plan and the buffers the launches point into (a re-plan may move them)
static void put_slot(KeyWriter *k, const ViewSlot *v) {
    const FwdPlan &p = v->plan;
    k->put(p.T); k->put(p.H); k->put(p.W); k->put(p.cap_small); k->put(p.cap_large); k->put(p.cap_edges);
    k->put(p.cap_edge_refs); k->put(p.cap_edge_tiles); k->put(p.tex); k->put(p.hint_large_tiles);
    const void *ptrs[] = {v->zeroed.ptr, v->small_offset.ptr, v->small_recs.ptr, v->large_refs.ptr, v->small_ids.ptr,
                          v->edge_ids.ptr, v->edge_recs.ptr, v->edge_refs.ptr, v->edge_refs_tmp.ptr, v->edge_spans.ptr,
                          v->edge_acc.ptr, v->tie_pairs.ptr, v->error_image_b.ptr, v->edge_tiles_raw.ptr,
                          v->large_tiles.ptr, v->edge_tiles.ptr, v->host_totals};
    for (const void *q : ptrs) k->put(q);
}

static bool is_default_stream(cudaStream_t st) { return st == nullptr || st == cudaStreamLegacy; }

static bool graphs_usable(const DeodrWorkspace *ws, cudaStream_t st, bool capturing) {
    // not inside the caller's own capture, not while the per-kernel events of the timing API are switched on (they would
    // have to live inside the graph); the per-thread default stream is left alone
    return ws->graphs && !capturing && st != cudaStreamPerThread && ws->ev_start.empty() && ws->overlap;
}

// The legacy default stream cannot be captured: work submitted on it runs on the workspace's proxy stream instead,
// ordered after everything already in the default stream and before everything submitted to it afterwards.
static cudaStream_t hop_in(DeodrWorkspace *ws, cudaStream_t st) {
    if (!is_default_stream(st)) return st;
    cudaEventRecord(ws->proxy_in, st);
    cudaStreamWaitEvent(ws->proxy, ws->proxy_in, 0);
    return ws->proxy;
}
static void hop_out(DeodrWorkspace *ws, cudaStream_t st) {
    if (!is_default_stream(st)) return;
    cudaEventRecord(ws->proxy_out, ws->proxy);
    cudaStreamWaitEvent(st, ws->proxy_out, 0);
}

// Runs `enqueue` (which launches on `st` and on streams forked from it) either directly or through the cache: replay when
// the key is the one the graph was captured for, capture + instantiate otherwise.  A failed capture switches the cache off.
template <class Enqueue>
static int launch_cached(DeodrWorkspace *ws, GraphCache *cache, const KeyWriter &key, cudaStream_t st, Enqueue enqueue) {
    if (cache->exec && cache->key == key.bytes) {
        cache->misses = 0;
        ws->launches += cache->launches;
        CUDA_TRY(cudaGraphLaunch(cache->exec, st));
        return DEODR_B200_OK;
    }
    if (++cache->misses > 8) {  // the caller's arguments change every call: capturing every time would cost more than it saves
        cache->drop();
        return enqueue();
    }
    cache->drop();
    if (cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
        cudaGetLastError();
        ws->graphs = false;
        return enqueue();
    }
    ws->capturing_internally = true;
    const int64_t before = ws->launches;
    const int rc = enqueue();
    ws->capturing_internally = false;
    cudaGraph_t graph = nullptr;
    const cudaError_t end = cudaStreamEndCapture(st, &graph);
    if (rc != DEODR_B200_OK || end != cudaSuccess || !graph) {
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        ws->graphs = false;
        ws->launches = before;
        if (rc != DEODR_B200_OK) return rc;
        return enqueue();  // nothing ran during the failed capture: run it now, kernel by kernel
    }
    cudaGraphExec_t exec = nullptr;
    const cudaError_t inst = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (inst != cudaSuccess || !exec) {
        cudaGetLastError();
        ws->graphs = false;
        ws->launches = before;
        return enqueue();
    }
    cache->exec = exec;
    cache->key = key.bytes;
    cache->launches = (int)(ws->launches - before);
    CUDA_TRY(cudaGraphLaunch(exec, st));
    return DEODR_B200_OK;
}

static int render_views_impl(DeodrWorkspace *ws, int n_views, const DeodrSceneView *views, const DeodrViewIO *io,
                             double sigma, int flags, void *stream, bool check_indices) {
    if (!ws) return set_error(DEODR_B200_EINVAL, "ws == NULL");
    if (n_views < 0 || (n_views > 0 && (!views || !io))) return set_error(DEODR_B200_EINVAL, "bad view list");
    for (int i = 0; i < n_views; i++)
        if (int rc = check_forward_args(&views[i], &io[i], sigma, flags)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ws->device));
    const bool capturing = stream_is_capturing(st);
    const bool deferred = ws->deferred || capturing;
    // a pass in two calls: 1 = head only, 2 = the rest of the pass whose head the previous call enqueued
    const int part = (flags & DEODR_B200_FORWARD_GEOMETRY) ? 1 : (flags & DEODR_B200_FORWARD_RESUME) ? 2 : 0;
    if ((flags & DEODR_B200_FORWARD_GEOMETRY) && (flags & DEODR_B200_FORWARD_RESUME))
        return set_error(DEODR_B200_EINVAL, "FORWARD_GEOMETRY and FORWARD_RESUME are two calls, not one");
    flags &= ~(DEODR_B200_FORWARD_GEOMETRY | DEODR_B200_FORWARD_RESUME);
    std::vector<ViewSlot *> slots(n_views);
    std::vector<SceneView> scenes(n_views);
    // ---- plans first (a plan needs the device: not possible while capturing)
    for (int i = 0; i < n_views; i++) {
        if (int rc = get_slot(ws, i, &slots[i])) return rc;
        memcpy(&scenes[i], &views[i], sizeof(SceneView));
        ViewSlot *v = slots[i];
        if (v->pending && !capturing) {  // deferred mode: an unread verdict of an earlier pass
            bool overflow;
            if (int rc = read_verdict(ws, v, st, &overflow)) return rc;
        }
        v->fwd_valid = 0;
        const bool same_shape = v->plan.valid && v->plan.T == scenes[i].nb_triangles && v->plan.H == scenes[i].height &&
                                v->plan.W == scenes[i].width && v->plan.edges_possible == (sigma > 0);
        if (part == 2) {  // the head has filled the lists of THIS plan: nothing may be rebuilt in between
            if (!v->head_enqueued || !same_shape)
                return set_error(DEODR_B200_EINVAL, "FORWARD_RESUME must follow FORWARD_GEOMETRY of the same views");
            continue;
        }
        v->head_enqueued = false;
        if (!capturing) {
            if (int rc = prepare_slot(ws, v, scenes[i], sigma)) return rc;
        } else if (!v->plan.valid || v->plan.T != scenes[i].nb_triangles || v->plan.H != scenes[i].height ||
                   v->plan.W != scenes[i].width || v->plan.edges_possible != (sigma > 0)) {
            return set_error(DEODR_B200_EINVAL,
                             "stream capture needs a plan: run the same views once outside the capture first");
        }
        if (!v->plan.valid)
            if (int rc = build_plan(ws, v, scenes[i], sigma, st, check_indices)) return rc;
    }
    // ---- enqueue every view, round-robin over the lanes (directly, or as the replay of the captured sequence)
    const int used = lanes_for(ws, n_views);
    const cudaStream_t caller_stream = st;
    auto enqueue_all = [&]() -> int {
        open_lanes(ws, st, used);
        for (int i = 0; i < n_views; i++)
            if (int rc = enqueue_forward(ws, slots[i], ws->lanes[i % used], scenes[i], io[i], sigma, flags, check_indices, part))
                return rc;
        close_lanes(ws, st, used);
        return DEODR_B200_OK;
    };
    if (part == 1) {  // head only: no verdict yet, no forward state for the adjoint yet, the colours-ready event is kept
        if (int rc = enqueue_all()) return rc;
        for (int i = 0; i < n_views; i++) slots[i]->head_enqueued = true;
        return DEODR_B200_OK;
    }
    for (int i = 0; i < n_views; i++) slots[i]->head_enqueued = false;
    if (part == 0 && graphs_usable(ws, st, capturing)) {
        const cudaStream_t caller = st;
        st = hop_in(ws, caller);
        KeyWriter key;
        key.put(n_views); key.put(sigma); key.put(flags); key.put(check_indices); key.put(ws->colors_ready);
        key.put(ws->overlap); key.put(used);
        for (int i = 0; i < n_views; i++) {
            key.put(views[i]);
            key.put(io[i]);
            put_slot(&key, slots[i]);
        }
        for (int i = 0; i < n_views; i++) next_seq(slots[i]);  // (clears the pinned flags: must happen for a replay too)
        const int rc = launch_cached(ws, &ws->fwd_graph, key, st, enqueue_all);
        hop_out(ws, caller);
        if (rc) return rc;
        for (int i = 0; i < n_views; i++) { slots[i]->pending = true; slots[i]->hints_exact = false; }
    } else {
        if (int rc = enqueue_all()) return rc;
    }
    for (int i = 0; i < n_views; i++) {
        ViewSlot *v = slots[i];
        v->generation = ++ws->generation_counter;
        v->sigma = sigma;
        v->fwd_C = scenes[i].nb_colors;
        v->fwd_flags = flags;
        v->fwd_scene = views[i];
        v->fwd_io = io[i];
        v->fwd_check_indices = check_indices;
        v->fwd_valid = 1;
    }
    ws->colors_ready = nullptr;  // one-shot
    if (deferred) return DEODR_B200_OK;
    // ---- verdicts: every pass is already queued, the device does not wait for this
    for (int i = 0; i < n_views; i++) {
        ViewSlot *v = slots[i];
        bool overflow = false;
        if (int rc = read_verdict(ws, v, st, &overflow)) return rc;
        if (check_indices)
            if (int rc = bad_index_error(v)) { v->fwd_valid = 0; return rc; }
        if (!overflow) continue;
        // the lists outgrew the plan (the kernels of that pass returned at once): new plan, same pass again
        if (int rc = build_plan(ws, v, scenes[i], sigma, st, check_indices)) return rc;
        ws->lanes[0].main = st;
        if (int rc = enqueue_forward(ws, v, ws->lanes[0], scenes[i], io[i], sigma, flags, check_indices)) return rc;
        if (int rc = read_verdict(ws, v, st, &overflow)) return rc;
        if (overflow) return set_error(DEODR_B200_ECUDA, "forward pass overflowed a freshly built plan (internal error)");
        v->fwd_valid = 1;
        if (st != caller_stream) hop_out(ws, caller_stream);  // the re-run went to the proxy stream too
    }
    return DEODR_B200_OK;
}

// depths_b: per-view [V] fp32 device pointers (or NULL entries) of deodr_b200_render_b_views_depths; NULL for the entry
// points without the perspective-correct adjoint.
static int render_b_views_impl(DeodrWorkspace *ws, int n_views, const DeodrSceneView *views, const DeodrViewIO *io,
                               const DeodrGrads *grads, float *const *depths_b, bool persp_adjoint, double sigma,
                               int flags, void *stream) {
    if (!ws) return set_error(DEODR_B200_EINVAL, "ws == NULL");
    if (n_views < 0 || (n_views > 0 && (!views || !io || !grads))) return set_error(DEODR_B200_EINVAL, "bad view list");
    const bool err_mode = (flags & DEODR_B200_ANTIALIASE_ERROR) != 0;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ws->device));
    const bool capturing = stream_is_capturing(st);
    for (int i = 0; i < n_views; i++) {
        if (int rc = validate_view(&views[i], true, persp_adjoint)) return rc;
        if (err_mode && views[i].perspective_correct)
            return set_error(DEODR_B200_EUNSUPPORTED,
                             "antialiase_error has no adjoint with perspective_correct=True");
        const DeodrViewIO &o = io[i];
        if (!o.z_buffer || !o.owner) return set_error(DEODR_B200_EINVAL, "z_buffer / owner is NULL");
        if (err_mode) {
            if (!o.err_buffer_b) return set_error(DEODR_B200_EINVAL, "err_buffer_b_ptr is NULL");
            if (!o.obs) return set_error(DEODR_B200_EINVAL, "obs_ptr is NULL");
            if (!o.image) return set_error(DEODR_B200_EINVAL, "image_ptr is NULL");
        } else if (!o.image_b) {
            return set_error(DEODR_B200_EINVAL, "image_b_ptr is NULL");
        }
        const DeodrGrads &g = grads[i];
        if ((views[i].nb_vertices > 0 && (!g.ij_b || !g.colors_b || !g.shade_b)) || (views[i].nb_uv > 0 && !g.uv_b))
            return set_error(DEODR_B200_EINVAL, "ij_b / colors_b / uv_b / shade_b must be provided");
        if (i >= (int)ws->slots.size() || !ws->slots[i])
            return set_error(DEODR_B200_EINVAL, "render_b must follow render on the same workspace, scene and sigma");
        const ViewSlot *v = ws->slots[i];
        if (!v->fwd_valid || v->sigma != sigma || v->plan.T != views[i].nb_triangles || v->plan.H != views[i].height ||
            v->plan.W != views[i].width || v->fwd_C != views[i].nb_colors || v->fwd_io.z_buffer != o.z_buffer ||
            v->fwd_io.owner != o.owner || ((v->fwd_flags ^ flags) & DEODR_B200_ANTIALIASE_ERROR))
            return set_error(DEODR_B200_EINVAL,
                             "render_b must follow render on the same workspace slot, scene, sigma, mode and "
                             "z_buffer / owner arrays");
    }
    if (err_mode && !capturing)
        for (int i = 0; i < n_views; i++) {
            ViewSlot *v = ws->slots[i];
            const size_t need = (size_t)views[i].height * views[i].width * views[i].nb_colors * sizeof(float);
            if (v->error_image_b.ensure(need, &ws->bytes)) return DEODR_B200_ECUDA;
        }
    for (int i = 0; i < n_views; i++) {  // accumulators (not while capturing: a warm-up pass has sized them)
        ViewSlot *v = ws->slots[i];
        if (v->plan.cap_edges > 0) {
            SceneView sv;
            memcpy(&sv, &views[i], sizeof(sv));
            const size_t need = (size_t)v->plan.cap_edges * deodr_edge_acc_stride(sv) * sizeof(double);
            if (need > v->edge_acc.bytes) {
                if (capturing) return set_error(DEODR_B200_EINVAL, "stream capture needs a warm-up pass outside the capture");
                if (v->edge_acc.ensure(need, &ws->bytes)) return DEODR_B200_ECUDA;
            }
        }
    }
    const int used = lanes_for(ws, n_views);
    auto enqueue_all = [&]() -> int {
        open_lanes(ws, st, used);
        for (int i = 0; i < n_views; i++) {
            SceneView s;
            memcpy(&s, &views[i], sizeof(s));
            deodr_launch_backward(ws, ws->slots[i], ws->lanes[i % used], s, io[i], sigma, flags, grads[i],
                                  depths_b ? depths_b[i] : nullptr);
        }
        close_lanes(ws, st, used);
        CUDA_TRY(cudaGetLastError());
        return DEODR_B200_OK;
    };
    if (graphs_usable(ws, st, capturing)) {
        const cudaStream_t caller = st;
        st = hop_in(ws, caller);
        KeyWriter key;
        key.put(n_views); key.put(sigma); key.put(flags); key.put(ws->overlap); key.put(used);
        for (int i = 0; i < n_views; i++) {
            key.put(views[i]);
            key.put(io[i]);
            key.put(grads[i]);
            key.put(depths_b ? depths_b[i] : nullptr);
            put_slot(&key, ws->slots[i]);
        }
        const int rc = launch_cached(ws, &ws->bwd_graph, key, st, enqueue_all);
        hop_out(ws, caller);
        return rc;
    }
    return enqueue_all();
}

extern "C" {

const char *deodr_b200_last_error(void) { return deodr_error_buffer(); }
const char *deodr_b200_version(void) { return "deodr_b200 0.2 (sm_100a)"; }

const char *deodr_b200_phase_name(int phase) {
    static const char *names[] = {"plan",     "edge_bin",      "bin",          "edge_tile_sort", "tile_z",       "shade",
                                  "edge_fwd", "small_tri_bwd", "interior_bwd", "edge_bwd",       "edge_finalize"};
    return phase >= 0 && phase < DEODR_B200_PH_COUNT ? names[phase] : "?";
}

int deodr_b200_timing_enable(DeodrWorkspace *ws, int max_records) {
    if (!ws) return set_error(DEODR_B200_EINVAL, "ws == NULL");
    CUDA_TRY(cudaSetDevice(ws->device));
    for (cudaEvent_t e : ws->ev_start) cudaEventDestroy(e);
    for (cudaEvent_t e : ws->ev_stop) cudaEventDestroy(e);
    ws->ev_start.clear();
    ws->ev_stop.clear();
    ws->ev_phase.clear();
    ws->ev_used = 0;
    for (int i = 0; i < max_records; i++) {
        cudaEvent_t a, b;
        CUDA_TRY(cudaEventCreate(&a));
        CUDA_TRY(cudaEventCreate(&b));
        ws->ev_start.push_back(a);
        ws->ev_stop.push_back(b);
        ws->ev_phase.push_back(0);
    }
    return DEODR_B200_OK;
}

int deodr_b200_timing_collect(DeodrWorkspace *ws, int32_t *phase, float *ms, int capacity) {
    if (!ws || !phase || !ms) return -1;
    int n = ws->ev_used < capacity ? ws->ev_used : capacity;
    for (int i = 0; i < n; i++) {
        if (cudaEventSynchronize(ws->ev_stop[i]) != cudaSuccess) return -1;
        float t = 0;
        if (cudaEventElapsedTime(&t, ws->ev_start[i], ws->ev_stop[i]) != cudaSuccess) return -1;
        phase[i] = ws->ev_phase[i];
        ms[i] = t;
    }
    if (getenv("DEODR_B200_TRACE_GAPS")) {  // development aid: idle time between consecutive timed phases
        double gap[DEODR_B200_PH_COUNT] = {0};
        int cnt[DEODR_B200_PH_COUNT] = {0};
        for (int i = 1; i < n; i++) {
            float t = 0;
            if (cudaEventElapsedTime(&t, ws->ev_stop[i - 1], ws->ev_start[i]) != cudaSuccess) continue;
            gap[ws->ev_phase[i]] += t;
            cnt[ws->ev_phase[i]]++;
        }
        for (int k = 0; k < DEODR_B200_PH_COUNT; k++)
            if (cnt[k]) fprintf(stderr, "[deodr_b200] gap before %-14s %.1f us\n", deodr_b200_phase_name(k), 1e3 * gap[k] / cnt[k]);
    }
    ws->ev_used = 0;
    return n;
}

int deodr_b200_workspace_create(DeodrWorkspace **out, int device) {
    if (!out) return set_error(DEODR_B200_EINVAL, "ws == NULL");
    int count = 0;
    cudaError_t err = cudaGetDeviceCount(&count);
    if (err != cudaSuccess || count == 0)
        return set_error(DEODR_B200_ECUDA, "no CUDA device available (%s): deodr_b200 has no CPU fallback",
                         cudaGetErrorString(err));
    if (device < 0 || device >= count) return set_error(DEODR_B200_EINVAL, "bad device index");
    CUDA_TRY(cudaSetDevice(device));
    DeodrWorkspace *ws = new (std::nothrow) DeodrWorkspace();
    if (!ws) return set_error(DEODR_B200_ENOMEM, "out of host memory");
    ws->device = device;
    CUDA_TRY(cudaMallocHost(&ws->host_scratch, 32 * sizeof(int)));
    memset(ws->host_scratch, 0, 32 * sizeof(int));
    CUDA_TRY(cudaFuncSetAttribute(k_scan_tiles, cudaFuncAttributeMaxDynamicSharedMemorySize, SCAN_SMEM));
    ws->overlap = !(getenv("DEODR_B200_SERIAL") && atoi(getenv("DEODR_B200_SERIAL")));
    // opt-in (DEODR_B200_GRAPHS=1): measured neutral at N = 1 (two replays + the verdict read between them against the
    // gaps of a dozen launches) and the default-stream hop it needs serialises with a communication stream at N > 1
    ws->graphs = getenv("DEODR_B200_GRAPHS") && atoi(getenv("DEODR_B200_GRAPHS")) != 0;
    ws->small_by_record = getenv("DEODR_B200_SMALL_ADJOINT") && !strcmp(getenv("DEODR_B200_SMALL_ADJOINT"), "record");
    if (const char *e = getenv("DEODR_B200_LANES")) ws->num_lanes = atoi(e) < 1 ? 1 : (atoi(e) > MAX_LANES ? MAX_LANES : atoi(e));
    int prio_low = 0, prio_high = 0;
    CUDA_TRY(cudaDeviceGetStreamPriorityRange(&prio_low, &prio_high));
    for (int l = 0; l < MAX_LANES; l++) {
        Lane &lane = ws->lanes[l];
        if (l > 0) CUDA_TRY(cudaStreamCreateWithFlags(&lane.main, cudaStreamNonBlocking));
        for (int i = 0; i < LANE_AUX; i++) {
            // the forward's side chain is short and the main chain waits for it at the join: its CTAs go first
            CUDA_TRY(cudaStreamCreateWithPriority(&lane.aux[i], cudaStreamNonBlocking, i == 0 ? prio_high : prio_low));
            CUDA_TRY(cudaEventCreateWithFlags(&lane.ev_join[i], cudaEventDisableTiming));
        }
        CUDA_TRY(cudaEventCreateWithFlags(&lane.ev_fork, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&lane.ev_begin, cudaEventDisableTiming));
        CUDA_TRY(cudaEventCreateWithFlags(&lane.ev_end, cudaEventDisableTiming));
    }
    CUDA_TRY(cudaStreamCreateWithFlags(&ws->proxy, cudaStreamNonBlocking));
    CUDA_TRY(cudaEventCreateWithFlags(&ws->proxy_in, cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&ws->proxy_out, cudaEventDisableTiming));
    if (ws->scalars.ensure(8 * sizeof(int), &ws->bytes)) return DEODR_B200_ECUDA;
    if (!sm_count_cached) cudaDeviceGetAttribute(&sm_count_cached, cudaDevAttrMultiProcessorCount, device);
    *out = ws;
    return DEODR_B200_OK;
}

void deodr_b200_workspace_destroy(DeodrWorkspace *ws) {
    if (!ws) return;
    cudaSetDevice(ws->device);
    cudaDeviceSynchronize();
    ws->fwd_graph.drop();
    ws->bwd_graph.drop();
    if (ws->proxy) cudaStreamDestroy(ws->proxy);
    if (ws->proxy_in) cudaEventDestroy(ws->proxy_in);
    if (ws->proxy_out) cudaEventDestroy(ws->proxy_out);
    for (ViewSlot *v : ws->slots) free_slot(v);
    DevBuf *bufs[] = {&ws->scalars, &ws->h_faces, &ws->h_faces_uv, &ws->h_ij, &ws->h_depths, &ws->h_uv,
                      &ws->h_colors, &ws->h_shade, &ws->h_edgeflags, &ws->h_textured, &ws->h_shaded, &ws->h_texture,
                      &ws->h_background, &ws->h_image, &ws->h_z, &ws->h_owner, &ws->h_image_b,
                      &ws->h_grads, &ws->h_obs, &ws->h_err, &ws->h_err_b};
    for (DevBuf *b : bufs) b->release();
    deodr_host_path_destroy(ws);
    if (ws->host_scratch) cudaFreeHost(ws->host_scratch);
    for (cudaEvent_t e : ws->ev_start) cudaEventDestroy(e);
    for (cudaEvent_t e : ws->ev_stop) cudaEventDestroy(e);
    for (int l = 0; l < MAX_LANES; l++) {
        Lane &lane = ws->lanes[l];
        if (l > 0 && lane.main) cudaStreamDestroy(lane.main);
        for (int i = 0; i < LANE_AUX; i++) {
            if (lane.aux[i]) cudaStreamDestroy(lane.aux[i]);
            if (lane.ev_join[i]) cudaEventDestroy(lane.ev_join[i]);
        }
        if (lane.ev_fork) cudaEventDestroy(lane.ev_fork);
        if (lane.ev_begin) cudaEventDestroy(lane.ev_begin);
        if (lane.ev_end) cudaEventDestroy(lane.ev_end);
    }
    delete ws;
}

int64_t deodr_b200_workspace_bytes(const DeodrWorkspace *ws) { return ws ? ws->bytes : 0; }
int64_t deodr_b200_workspace_launches(const DeodrWorkspace *ws) { return ws ? ws->launches : 0; }

int deodr_b200_workspace_set_deferred(DeodrWorkspace *ws, int on) {
    if (!ws) return set_error(DEODR_B200_EINVAL, "ws == NULL");
    ws->deferred = on != 0;
    return DEODR_B200_OK;
}

int deodr_b200_workspace_status(DeodrWorkspace *ws) {
    if (!ws) return set_error(DEODR_B200_EINVAL, "ws == NULL");
    CUDA_TRY(cudaSetDevice(ws->device));
    CUDA_TRY(cudaDeviceSynchronize());  // every pass enqueued so far has published its verdict after this
    int overflowed = 0;
    for (ViewSlot *v : ws->slots) {
        if (!v) continue;
        // a captured graph re-publishes with the sequence number it was captured with, so the flag cannot tell a new
        // verdict from an old one: after the synchronisation the pinned words ARE the verdict of the slot's last pass
        __atomic_thread_fence(__ATOMIC_ACQUIRE);
        v->pending = false;
        if (((volatile int *)v->host_totals)[SC_OVERFLOW]) {
            v->host_totals[SC_OVERFLOW] = 0;
            v->plan.valid = false;
            v->fwd_valid = 0;
            overflowed++;
        }
    }
    if (overflowed)
        return set_error(DEODR_B200_EREPLAN,
                         "a forward pass overflowed the lists its plan had reserved: its results are void, the plan has "
                         "been dropped - run the pass again (outside a stream capture) to rebuild it");
    return DEODR_B200_OK;
}

int deodr_b200_workspace_set_colors_ready(DeodrWorkspace *ws, void *event) {
    if (!ws) return set_error(DEODR_B200_EINVAL, "ws == NULL");
    ws->colors_ready = (cudaEvent_t)event;
    return DEODR_B200_OK;
}

int64_t deodr_b200_view_generation(const DeodrWorkspace *ws, int view) {
    if (!ws || view < 0 || view >= (int)ws->slots.size() || !ws->slots[view]) return 0;
    return ws->slots[view]->generation;
}

int deodr_b200_check_scene(DeodrWorkspace *ws, const DeodrSceneView *scene, void *stream) {
    if (!ws) return set_error(DEODR_B200_EINVAL, "ws == NULL");
    if (int rc = validate_view(scene, false)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaSetDevice(ws->device));
    SceneView s;
    memcpy(&s, scene, sizeof(s));
    int *flag = ws->scalars.as<int>();
    CUDA_TRY(cudaMemsetAsync(flag, 0, sizeof(int), st));
    if (s.nb_triangles > 0) {
        k_check_scene<<<grid_for(3 * (size_t)s.nb_triangles, 256), 256, 0, st>>>(s, flag);
        ws->launches++;
    }
    CUDA_TRY(cudaMemcpyAsync(ws->host_scratch, flag, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (ws->host_scratch[0] & 1) return set_error(DEODR_B200_EINVAL, "scene.faces value greater than scene.nb_vertices");
    if (ws->host_scratch[0] & 2) return set_error(DEODR_B200_EINVAL, "scene.faces_uv value greater than scene.nb_uv");
    return DEODR_B200_OK;
}

int deodr_b200_render_views(DeodrWorkspace *ws, int n_views, const DeodrSceneView *views, const DeodrViewIO *io,
                            double sigma, int flags, void *stream) {
    return render_views_impl(ws, n_views, views, io, sigma, flags, stream, false);
}

int deodr_b200_render_b_views(DeodrWorkspace *ws, int n_views, const DeodrSceneView *views, const DeodrViewIO *io,
                              const DeodrGrads *grads, double sigma, int flags, void *stream) {
    return render_b_views_impl(ws, n_views, views, io, grads, nullptr, false, sigma, flags, stream);
}

int deodr_b200_render_b_views_depths(DeodrWorkspace *ws, int n_views, const DeodrSceneView *views,
                                     const DeodrViewIO *io, const DeodrGrads *grads, float *const *depths_b,
                                     double sigma, int flags, void *stream) {
    if (n_views > 0 && !depths_b) return set_error(DEODR_B200_EINVAL, "depths_b == NULL (pass an array of NULLs)");
    return render_b_views_impl(ws, n_views, views, io, grads, depths_b, true, sigma, flags, stream);
}

int deodr_b200_render(DeodrWorkspace *ws, const DeodrSceneView *scene, double sigma, float *image, double *z_buffer,
                      int32_t *owner, int32_t *face_id, void *stream) {
    DeodrViewIO io;
    memset(&io, 0, sizeof(io));
    io.image = image;
    io.z_buffer = z_buffer;
    io.owner = owner;
    io.face_id = face_id;
    return render_views_impl(ws, 1, scene, &io, sigma, 0, stream, false);
}

int deodr_b200_render_b(DeodrWorkspace *ws, const DeodrSceneView *scene, double sigma, const double *z_buffer,
                        const int32_t *owner, const float *image_b, const DeodrGrads *grads, void *stream) {
    if (!grads) return set_error(DEODR_B200_EINVAL, "grads == NULL");
    DeodrViewIO io;
    memset(&io, 0, sizeof(io));
    io.z_buffer = const_cast<double *>(z_buffer);
    io.owner = const_cast<int32_t *>(owner);
    io.image_b = image_b;
    return render_b_views_impl(ws, 1, scene, &io, grads, nullptr, false, sigma, 0, stream);
}

}  // extern "C"

int deodr_render_checked(DeodrWorkspace *ws, const DeodrSceneView *scene, const DeodrViewIO *io, double sigma, int flags,
                         void *stream) {
    const bool was = ws->deferred;
    ws->deferred = false;
    const int rc = render_views_impl(ws, 1, scene, io, sigma, flags, stream, true);
    ws->deferred = was;
    return rc;
}
