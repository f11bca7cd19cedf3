// Barrier-separated phases of the binning and tile-raster kernels, written as __host__ __device__ functions of the
// thread index.  kernels.cu strings them together with __syncthreads() in between; the CPU emulation harness under
// tests/emul (test infrastructure) calls the same functions in `for (tid ...)` loops, which is how the kernel logic
// is checked against the oracle in a container without a GPU.
//
// `Env` supplies the few operations that differ between the two worlds (atomics, warp aggregation).
#pragma once

#include "shade.h"

namespace deodr {

constexpr int TS = 16;            // tile side in pixels
constexpr int NT = TS * TS;       // threads per tile CTA, one per pixel
constexpr int PRE_CHUNK = 128;    // pre-masked records per TMA bulk copy (double-buffered landing zone: 2 x 8 KB)
#ifndef DEODR_LARGE_CHUNK
#define DEODR_LARGE_CHUNK 64
#endif
constexpr int LARGE_CHUNK = DEODR_LARGE_CHUNK;  // large triangles staged per pass (stencil records kept in shared memory)
constexpr int PIX_SLOTS = 8;      // candidate small triangles kept per pixel and chunk before the pixel falls back to a scan
constexpr int EDGE_CHUNK = 64;    // edge records staged in shared memory per pass
#ifndef DEODR_EDGE_ROWS
#define DEODR_EDGE_ROWS 16
#endif
// Rows of a tile handled by one CTA of the edge kernels.  16 = whole tile; 4 (16x4 strips, 4 CTAs per tile) was measured
// slower on B200 (edge_fwd 79 vs 56 us, edge_bwd 164 vs 118 us on the 1M-triangle scene: the per-CTA record fetch and span
// set-up are replicated per strip).
constexpr int EDGE_ROWS = DEODR_EDGE_ROWS;
constexpr int EDGE_NT = TS * EDGE_ROWS;

// What the z test needs from a triangle once its coverage masks exist.
struct TriRec {
    double zp[3];  // z (or 1/z) plane
    int32_t id;
    int32_t pad;
};

struct alignas(16) Mask4 {
    uint32_t m[4];
};

// Pre-masked tile record of a SMALL triangle (bounding box that fits a 64-bit mask), written by the fill pass: the exact
// coverage of the 16x16 tile (8 row pairs x 32 bits) + what the z test needs.  64 bytes, so a tile's list is one
// contiguous, 16-byte aligned array that the raster kernel pulls into shared memory with one bulk (TMA) copy.
struct alignas(16) PreRec {
    uint32_t mask[TS / 2];
    double zp[3];
    int32_t id;
    int32_t pad;
};
static_assert(sizeof(PreRec) == 64, "PreRec must be 64 bytes");


// owner codes: triangle index | SMALL_FLAG when the triangle went through the small (pre-masked) path; the adjoint of
// such pixels is taken by the triangle-parallel kernel.  -1 = background, <= -2 = entry of the exact-tie table.
constexpr int SMALL_FLAG = 0x40000000;
constexpr int TRI_INDEX_MASK = 0x3fffffff;

// Shared-memory working set of the tile kernels.  The z pass only uses `tri` and allocates just that part (it is what
// bounds its CTAs per SM, see k_tile_z); the edge kernels only use `edge`.
struct TileShared {
    struct TriPart {
        TriGeom geo[LARGE_CHUNK];  // large triangles: stencils, so that their row spans are computed by 8 threads each
        TriRec rec[LARGE_CHUNK];
        // mask[p][t]: coverage of tile rows 2p (bits 0-15) and 2p+1 (bits 16-31) by triangle t, i.e. one bit per
        // lane of warp p; row-pair-major so that a warp streams its own masks four triangles at a time
        alignas(16) uint32_t mask[TS / 2][LARGE_CHUNK];
        // small triangles: per-pixel candidate lists filled by the record threads (phase_pre_scatter)
        int pix_cnt[NT];
        uint8_t pix_list[PIX_SLOTS][NT];
    };
    struct EdgePart {
        EdgeRec rec[EDGE_CHUNK];
        uint32_t span[EDGE_CHUNK][TS];  // x_begin | x_end << 16 (absolute, int16 each); empty if begin > end
    };
    union {
        TriPart tri;
        EdgePart edge;
    };
};

struct Tile {
    int x0, y0;  // pixel origin
};

// tile_id / tiles_x without the integer division (a runtime divisor costs ~20 instructions per thread and tile: 6 % of
// the z pass): q = (tile_id * mul) >> 40 with mul = ceil(2^40 / tiles_x), exact while tile_id * tiles_x < 2^40
// (tiles_x <= 2048, tile_id < 2^22 for the largest admitted image).
struct TileDiv {
    unsigned long long mul;
    int tiles_x;
};
DEODR_HD TileDiv make_tile_div(int tiles_x) {
    TileDiv d;
    d.tiles_x = tiles_x;
    d.mul = (((unsigned long long)1 << 40) + (unsigned long long)tiles_x - 1) / (unsigned long long)tiles_x;
    return d;
}
DEODR_HD Tile tile_of(int tile_id, TileDiv d) {
    const int row = (int)(((unsigned long long)(unsigned)tile_id * d.mul) >> 40);
    Tile t;
    t.y0 = row * TS;
    t.x0 = (tile_id - row * d.tiles_x) * TS;
    return t;
}

DEODR_HD Tile tile_of(int tile_id, int tiles_x) {
    Tile t;
    t.y0 = (tile_id / tiles_x) * TS;
    t.x0 = (tile_id % tiles_x) * TS;
    return t;
}

// ---------------------------------------------------------------------------------------------------- binning

// Tiles overlapped by the exact bounding box of a drawn triangle (rows/cols the reference can touch).
struct TileBox {
    int tx0, tx1, ty0, ty1;  // inclusive; empty if tx0 > tx1
};

struct TileBox;
DEODR_HD TileBox tri_tile_box(const double V[3][2], bool strict, int width, int height, int *box_w = nullptr,
                              int *box_h = nullptr);

DEODR_HD TileBox tri_tile_box(const double V[3][2], bool strict, int width, int height, int *box_w, int *box_h) {
    TileBox b;
    int x0, x1, y0, y1;
    tri_bounds(V, strict, &x0, &x1, &y0, &y1);
    if (x0 < 0) x0 = 0;
    if (x1 > width - 1) x1 = width - 1;
    if (y0 < 0) y0 = 0;
    if (y1 > height - 1) y1 = height - 1;
    if (box_w) *box_w = x1 - x0 + 1;
    if (box_h) *box_h = y1 - y0 + 1;
    if (y0 > y1 || x0 > x1) { b.tx0 = 1; b.tx1 = 0; b.ty0 = 1; b.ty1 = 0; return b; }
    b.tx0 = x0 / TS; b.tx1 = x1 / TS; b.ty0 = y0 / TS; b.ty1 = y1 / TS;
    return b;
}

DEODR_HD TileBox edge_tile_box(const double V[2][2], double sigma, int width, int height) {
    TileBox b;
    int y_begin, y_end;
    edge_row_range(V, height, sigma, &y_begin, &y_end);
    double lo = fmin(V[0][0], V[1][0]) - sigma, hi = fmax(V[0][0], V[1][0]) + sigma;
    int x0 = (int)floor(fmax(lo, -1.0)) - 1, x1 = (int)ceil(fmin(hi, (double)width)) + 1;
    if (x0 < 0) x0 = 0;
    if (x1 > width - 1) x1 = width - 1;
    if (y_begin > y_end || x0 > x1) { b.tx0 = 1; b.tx1 = 0; b.ty0 = 1; b.ty1 = 0; return b; }
    b.tx0 = x0 / TS; b.tx1 = x1 / TS; b.ty0 = y_begin / TS; b.ty1 = y_end / TS;
    return b;
}

// ---- the plan of a forward pass -----------------------------------------------------------------------------
// Every per-tile list lives in a SEGMENT whose capacity was reserved by the plan (exclusive scan, with slack, of the
// counts of an earlier pass over a scene of the same shape).  The forward pass appends with one atomic per item and
// never waits for the host: an append that does not fit raises a bit of the verdict word instead of writing, every
// later kernel of that forward returns at once when the word is non-zero, and the host - which reads the word from
// pinned memory AFTER it has enqueued the whole pass - re-plans and re-runs (kernels.cu: build_plan / verify).
enum {
    OVF_SMALL = 1,      // pre-masked records of a tile
    OVF_LARGE = 2,      // large-triangle references of a tile
    OVF_EDGES = 4,      // silhouette edges of the view
    OVF_EDGE_REFS = 8,  // edge references of a tile
    OVF_TEXTURE = 16,   // a textured triangle met by kernel instances compiled without the texture paths
    OVF_EDGE_TILES = 32 // more tiles with silhouette edges than the edge kernels were launched for
};

// device scalars of one forward pass (zeroed together with the segment cursors, one memset)
enum {
    SC_OVERFLOW = 0,     // verdict word (OVF_* bits)
    SC_EDGES = 1,        // silhouette edges appended
    SC_SMALL = 2,        // drawn small triangles appended to the compact list
    SC_TIES = 3,         // entries of the exact-tie table
    SC_BAD_INDEX = 4,    // checkSceneValid: 1 = faces, 2 = faces_uv out of range
    SC_TEXTURED = 5,     // the scene holds a textured (and shaded) triangle
    SC_HEAVY_TILES = 6,  // edge tiles with more than one chunk of edges (front of the two-ended list)
    SC_LIGHT_TILES = 7,  // the other edge tiles (back of the list)
    SC_LARGE_TILES = 8,  // tiles that hold large triangles
    SC_TICKET = 9,       // scan kernel: arrival counter of its CTAs
    SC_EDGE_TILES = 13,  // tiles that received at least one silhouette edge (unordered list of k_bin_edges)
    SC_TOTAL_SMALL = 10, // plan building: reserved record / reference totals (with slack)
    SC_TOTAL_LARGE = 11,
    SC_TOTAL_EDGE_REFS = 12,
    SC_PLAN_LARGE_TILES = 14, // plan building: tiles with large triangles / with silhouette edges (launch hints)
    SC_PLAN_EDGE_TILES = 15,
    SC_WORDS = 32
};

struct TileSegments {
    const int *offset;  // [tiles + 1] reserved by the plan
    int *cursor;        // [tiles] items appended (or, in the count-only pass, counted) so far
};

DEODR_HD int segment_size(const TileSegments &seg, int t) {
    const int cap = seg.offset[t + 1] - seg.offset[t], n = seg.cursor[t];
    return n < cap ? n : cap;
}

// position of a new item of tile t, or -1 (verdict bit raised) when the segment is full
template <class Env>
DEODR_HD int segment_reserve(const TileSegments &seg, int t, int *verdict, int bit) {
    const int pos = seg.offset[t] + Env::atomic_add(&seg.cursor[t], 1);
    if (pos < seg.offset[t + 1]) return pos;
    Env::atomic_or(verdict, bit);
    return -1;
}

// Unordered list of the silhouette edges to overdraw (DR.h:2839-2853: sigma > 0, signedArea > 0, flag set), appended
// by the binning pass together with the depth-sum sort key of their triangle.
struct EdgeList {
    int *count;       // number of appended edges (may exceed `capacity`: verdict bit OVF_EDGES)
    int *ids;         // 3 * triangle + n
    uint64_t *keys;   // depth_desc_key(sum of the triangle's vertex depths)
    int capacity;
};

DEODR_HD void gather_edge(const SceneView &s, int edge_id, double V[2][2]) {
    int k = edge_id / 3, n = edge_id - 3 * k;
    for (int i = 0; i < 2; i++) {
        uint32_t v = s.faces[3 * k + edge_vertex(n, i)];
        V[i][0] = s.ij[2 * (size_t)v];
        V[i][1] = s.ij[2 * (size_t)v + 1];
    }
    remove_offset(V, 2, pixel_offset(s));
}

// Per-tile lists of the drawn triangles.  SMALL triangles (bounding box fitting a 64-bit pixel mask: the micro-
// triangle regime) get a pre-masked PreRec per tile they actually cover; LARGE ones are binned by index into every
// tile of their bounding box and their row spans are computed by the tile CTA in parallel.
struct TriBins {
    TileSegments small;
    PreRec *small_recs;
    TileSegments large;
    int *large_refs;
    int *verdict;      // scal + SC_OVERFLOW
    int record_rows;   // height limit of the record path for triangles that are not small (see takes_record_path)
    // May a TEXTURED triangle be "small" (adjoint by the triangle-parallel kernel)?  Its per-pixel adjoint is a chain of
    // dependent texture fetches and twelve texel atomics; one thread walking up to 64 such pixels is only worth it when
    // the scene has enough small triangles to fill the chip with threads (kernels.cu: small_textured_for).  0: textured
    // triangles keep the record path of the forward pass but are owned without SMALL_FLAG (pixel-parallel adjoint).
    int small_textured;
};

// "small" = micro-triangle: at most 2 x 2 tiles and a bounding box that fits a 64-bit mask with a power-of-two row
// stride (pixel <-> bit without a division), so that one thread can afford to walk it (binning pass, adjoint).
DEODR_HD int small_shift(int box_w) {  // log2 of the row stride
    int sh = 0;
    while ((1 << sh) < box_w) sh++;
    return sh;
}
DEODR_HD bool is_small(const TileBox &b, int box_w, int box_h) {
    return b.tx1 - b.tx0 <= 1 && b.ty1 - b.ty0 <= 1 && box_w <= 32 && (box_h << small_shift(box_w)) <= 64;
}
// Triangles that take the RECORD path of the forward pass (exact coverage masks computed once, by the binning thread):
// at most two tile columns and RECORD_ROWS (16) rows.  The small ones (above) are a subset - they also fit the 64-bit
// ownership mask of the triangle-parallel adjoint; the others ("medium": e.g. 12 x 8 pixel triangles, 7 % of the drawn
// triangles of the 1M-triangle scene) are owned without SMALL_FLAG and go through the pixel-parallel adjoint.
// Everything else ("large") is binned by reference and set up inside the tile kernel: one binning thread walking the
// 30+ rows of a 1k-triangle scene's triangles is slower than the tile kernel's parallel set-up (measured: the 640x480
// hand-sized scene 0.154 -> 0.207 ms with a 64-row limit), so the record path stops at one tile height.
#ifndef DEODR_RECORD_ROWS
#define DEODR_RECORD_ROWS 16
#endif
constexpr int RECORD_ROWS = DEODR_RECORD_ROWS;
// `rows` = RECORD_ROWS, or 0 for scenes of a few thousand triangles (TriBins::record_rows): with too few binning threads
// to fill the chip, a thread walking 16 rows is the kernel's critical path and the tile kernel's parallel set-up wins
// (small triangles always take the record path: it is what their adjoint relies on).
DEODR_HD bool takes_record_path(const TileBox &b, int box_w, int box_h, int rows) {
    return is_small(b, box_w, box_h) || (b.tx1 - b.tx0 <= 1 && box_w <= 32 && box_h <= rows);
}

// 16-bit coverage mask of tile row y for one triangle (exact spans of rmath.h, clipped to the tile).
DEODR_HD uint32_t tri_row_mask(const SceneView &s, const TriGeom &g, int y, int tile_x0) {
    int xb, xe;
    tri_row_span(g, y, s.width, s.height, s.strict_edge != 0, &xb, &xe);
    xb -= tile_x0;
    xe -= tile_x0;
    if (xb < 0) xb = 0;
    if (xe > TS - 1) xe = TS - 1;
    return xb <= xe ? (((1u << (xe - xb + 1)) - 1u) << xb) : 0u;
}

// Coverage of row pair p of the tile at (tile_x0, tile_y0): rows 2p (bits 0-15) and 2p+1 (bits 16-31).
DEODR_HD uint32_t tri_pair_mask(const SceneView &s, const TriGeom &g, int y_first, int y_last, int tile_x0, int tile_y0,
                                int p) {
    const int y = tile_y0 + 2 * p;
    uint32_t m = 0;
    if (y + 1 >= y_first && y <= y_last) {
        if (y >= y_first) m = tri_row_mask(s, g, y, tile_x0);
        if (y + 1 <= y_last) m |= tri_row_mask(s, g, y + 1, tile_x0) << 16;
    }
    return m;
}

template <class Env>
DEODR_HD void bin_flush_small(int code, const TriGeom &g, int tiles_x, int tx, int ty, const uint32_t *mask,
                              const TriBins &bins) {
    uint32_t any = 0;
    for (int p = 0; p < TS / 2; p++) any |= mask[p];
    if (!any) return;  // the bounding box touches the tile, the triangle does not
    const int pos = segment_reserve<Env>(bins.small, ty * tiles_x + tx, bins.verdict, OVF_SMALL);
    if (pos < 0) return;
    PreRec rec;
    for (int p = 0; p < TS / 2; p++) rec.mask[p] = mask[p];
    canonical_plane(g.zp, rec.zp);
    rec.id = code;  // triangle index, | SMALL_FLAG when the triangle-parallel adjoint takes it
    rec.pad = 0;
    bins.small_recs[pos] = rec;
}

// Exact coverage masks of every tile a record-path triangle really covers, one pre-masked record per such tile.
// SIMT note: the loop runs over the triangle's ROWS (consecutive for every lane, so the lanes of a warp execute the
// expensive span body together) and scatters each span into the masks of the <= 2 tile columns; a (tile, row-pair)
// loop would make every lane wait for the bodies of all the others.
template <class Env>
DEODR_HD void bin_small(const SceneView &s, int k, const double V[3][2], const double Zv[3], const TileBox &b,
                        int tiles_x, const TriBins &bins) {  // k = owner code of the triangle
    TriGeom g;
    tri_geom(V, Zv, s.strict_edge != 0, s.perspective_correct != 0, &g, nullptr);
    int y_first, y_last;
    tri_row_range(g, s.height, &y_first, &y_last);
    uint32_t mask[2][TS / 2];
    for (int c = 0; c < 2; c++)
        for (int p = 0; p < TS / 2; p++) mask[c][p] = 0u;
    int cur_ty = y_first >> 4;
    for (int y = y_first; y <= y_last; y++) {
        const int ty = y >> 4;
        if (ty != cur_ty) {
            for (int c = 0; c < 2; c++) {
                if (b.tx0 + c <= b.tx1) bin_flush_small<Env>(k, g, tiles_x, b.tx0 + c, cur_ty, mask[c], bins);
                for (int p = 0; p < TS / 2; p++) mask[c][p] = 0u;
            }
            cur_ty = ty;
        }
        int xb, xe;
        tri_row_span(g, y, s.width, s.height, s.strict_edge != 0, &xb, &xe);
        if (xb > xe) continue;
        const int p = (y & (TS - 1)) >> 1, shift = (y & 1) * 16;
        for (int c = 0; c < 2; c++) {
            const int x0 = (b.tx0 + c) * TS;
            int lb = xb - x0, le = xe - x0;
            if (lb < 0) lb = 0;
            if (le > TS - 1) le = TS - 1;
            if (lb <= le) mask[c][p] |= (((1u << (le - lb + 1)) - 1u) << lb) << shift;
        }
    }
    if (y_first <= y_last)
        for (int c = 0; c < 2; c++)
            if (b.tx0 + c <= b.tx1) bin_flush_small<Env>(k, g, tiles_x, b.tx0 + c, cur_ty, mask[c], bins);
}

// The binning pass, one thread per triangle: ONE gather of its vertices serves the classification (DR.h:2751-2779), the
// append of its silhouette edges, and - for a drawn triangle - its pre-masked records (small) or tile references
// (large).  COUNT_ONLY is the plan-building variant: the same decisions, but it only counts the items per tile
// (bounding-box tiles for the small triangles: an upper bound of the records the real pass emits) and the edges per
// tile of their band, so that the plan can reserve the segments.
template <class Env, bool COUNT_ONLY>
DEODR_HD void bin_triangle(const SceneView &s, int k, double sigma, int tiles_x, const TriBins &bins, int *num_small,
                           int *small_ids, const EdgeList &edges, int *edge_tile_count) {
    uint32_t vid[3];
    double V[3][2], Zv[3];
    gather_tri(s, k, vid, V, Zv);
    const TriClass c = classify_tri(s, k, V, Zv);
    if (sigma > 0 && c.area_positive) {
        for (int n = 0; n < 3; n++) {
            if (!s.edgeflags[3 * k + n]) continue;
            const int slot = Env::atomic_add(edges.count, 1);
            if (COUNT_ONLY) {
                double E[2][2];
                for (int i = 0; i < 2; i++) {
                    E[i][0] = V[edge_vertex(n, i)][0];
                    E[i][1] = V[edge_vertex(n, i)][1];
                }
                remove_offset(E, 2, pixel_offset(s));
                const TileBox b = edge_tile_box(E, sigma, s.width, s.height);
                for (int ty = b.ty0; ty <= b.ty1; ty++)
                    for (int tx = b.tx0; tx <= b.tx1; tx++) Env::atomic_add(&edge_tile_count[ty * tiles_x + tx], 1);
            } else if (slot < edges.capacity) {
                edges.ids[slot] = 3 * k + n;
                edges.keys[slot] = depth_desc_key(c.sum_depth);
            } else {
                Env::atomic_or(bins.verdict, OVF_EDGES);
            }
        }
    }
    if (!c.drawn) return;
    remove_offset(V, 3, pixel_offset(s));
    int box_w, box_h;
    const TileBox b = tri_tile_box(V, s.strict_edge != 0, s.width, s.height, &box_w, &box_h);
    if (b.tx0 > b.tx1) return;  // off screen
    const bool records = takes_record_path(b, box_w, box_h, bins.record_rows);
    // small = the triangle-parallel adjoint takes it (textured triangles only when the plan says so)
    const bool small = is_small(b, box_w, box_h) && (bins.small_textured || !(s.textured[k] && s.shaded[k]));
    if (COUNT_ONLY) {
        int *count = records ? bins.small.cursor : bins.large.cursor;
        // a record-path triangle that is not small is owned through the pixel-parallel adjoint: bit 30 of the tile's
        // large counter marks the tile for the plan's launch hint (k_scan_tiles masks it out of the capacity)
        const bool medium = records && !small;
        for (int ty = b.ty0; ty <= b.ty1; ty++)
            for (int tx = b.tx0; tx <= b.tx1; tx++) {
                Env::atomic_add(&count[ty * tiles_x + tx], 1);
                if (medium) Env::atomic_or(&bins.large.cursor[ty * tiles_x + tx], 0x40000000);
            }
        return;
    }
    if (records) {
        // the compact list of the drawn small triangles is what the triangle-parallel adjoint walks (capacity T)
        if (small) small_ids[Env::atomic_add(num_small, 1)] = k;
        bin_small<Env>(s, small ? (k | SMALL_FLAG) : k, V, Zv, b, tiles_x, bins);
    } else {
        for (int ty = b.ty0; ty <= b.ty1; ty++)
            for (int tx = b.tx0; tx <= b.tx1; tx++) {
                const int pos = segment_reserve<Env>(bins.large, ty * tiles_x + tx, bins.verdict, OVF_LARGE);
                if (pos >= 0) bins.large_refs[pos] = k;
            }
    }
}

// Edge pass, one thread per appended silhouette edge (slot = position in the unordered list): the band stencil record
// (DR.h:1366-1460 + z plane + end-point colours) is built ONCE per forward, and the slot goes to every tile of the band.
struct EdgeBins {
    TileSegments seg;
    int *refs;
    int *verdict;
    int *tile_list;    // tiles that hold at least one edge, in arrival order (appended by the first edge of each tile)
    int *tile_count;
    int tile_capacity;
};

// edge `slot` -> list of tile t
template <class Env>
DEODR_HD void bin_edge_tile(int slot, int t, const EdgeBins &bins) {
    const int pos = segment_reserve<Env>(bins.seg, t, bins.verdict, OVF_EDGE_REFS);
    if (pos < 0) return;
    bins.refs[pos] = slot;
    if (pos == bins.seg.offset[t]) {  // first edge of the tile: the tile joins the list the edge kernels walk
        const int at = Env::atomic_add(bins.tile_count, 1);
        if (at < bins.tile_capacity) bins.tile_list[at] = t;
        else Env::atomic_or(bins.verdict, OVF_EDGE_TILES);
    }
}

// (one thread per edge: the CPU emulation's form; the device kernel spreads the tiles of the band over a warp)
template <class Env>
DEODR_HD void bin_edge(const SceneView &s, int slot, double sigma, int tiles_x, const EdgeList &edges,
                       const EdgeBins &bins, EdgeRec *recs) {
    const int id = edges.ids[slot];
    double V[2][2];
    edge_record(s, id, slot, edges.keys[slot], sigma, &recs[slot], V);
    const TileBox b = edge_tile_box(V, sigma, s.width, s.height);
    for (int ty = b.ty0; ty <= b.ty1; ty++)
        for (int tx = b.tx0; tx <= b.tx1; tx++) bin_edge_tile<Env>(slot, ty * tiles_x + tx, bins);
}

// Far-to-near position of item i of a tile's edge list: the reference walks the edges in descending order of their
// triangle's depth sum (DR.h:2656-2662, 2781), ties by ascending (triangle, edge) id.  Only the RELATIVE order of the
// edges that meet in a pixel matters, and those share the tile: no global sort.
DEODR_HD int tile_edge_position(int i, int n, const int *refs, const EdgeRec *recs) {
    const EdgeRec &mine = recs[refs[i]];
    int pos = 0;
    for (int j = 0; j < n; j++) {
        const EdgeRec &o = recs[refs[j]];
        pos += (o.key < mine.key) || (o.key == mine.key && o.id < mine.id);
    }
    return pos;
}

// ------------------------------------------------------------------------------------------- tile kernel phases

template <int MAXC>
struct PixelState {
    double z;        // running z-buffer value of the pixel
    int own;         // forward owner: lowest index among the triangles reaching the minimum z (strict '<', DR.h:961)
    int bown;        // adjoint owner: highest such index (DR.h:1024 walked in reverse index order)
    float col[MAXC];
};

// Phase T1a: two threads per small-triangle record `pre[rec]` walk the set bits of its coverage words (pulled into shared memory by the bulk
// copy) and appends its index to the candidate list of every pixel it covers.  A record covers ~4 pixels, a pixel is
// covered by ~1.3 records: the z test then runs over a pixel's own candidates instead of over every record of the tile.
// pix_cnt[] must be zero on entry (phase_pix_test leaves it so).  One flat loop over the bits (SIMT: lanes with few
// bits idle only for max-over-lanes iterations).
template <class Env>
DEODR_HD void phase_pre_scatter(int tid, int n, const PreRec *pre, TileShared *sh) {
    // two threads per record (rows 0-7 and 8-15 of the tile): all eight warps take part in a 128-record chunk
    static_assert(NT == 2 * PRE_CHUNK, "two threads per record of a chunk");
    const int rec = tid % PRE_CHUNK, half = tid / PRE_CHUNK;
    if (rec >= n) return;
    const PreRec &r = pre[rec];
    uint32_t words = 0u;  // bit p set <=> mask word p (of this thread's half) is not empty
    for (int p = 4 * half; p < 4 * half + 4; p++) words |= (uint32_t)(r.mask[p] != 0u) << p;
    int p = 0;
    uint32_t w = 0u;
    for (;;) {
        if (w == 0u) {
            if (words == 0u) break;
            p = lowest_bit(words);
            words &= words - 1;
            w = r.mask[p];
        }
        const int px = p * 32 + lowest_bit(w);
        w &= w - 1;
        const int slot = Env::shared_inc(&sh->tri.pix_cnt[px]);
        if (slot < PIX_SLOTS) sh->tri.pix_list[slot][px] = (uint8_t)rec;
    }
}

// One candidate against the running state of a pixel, order-independently:
//   own = min index among ties (what a strict '<' walk in ascending index order leaves, DR.h:961),
//   bown = max index among ties (what the '==' walk in descending index order finds first, DR.h:1024).
template <int MAXC>
DEODR_HD void z_candidate(const double *zp, int id, double xd, double yd, int x, int y, bool persp, PixelState<MAXC> *p) {
    double z = plane_z(zp, xd, yd, x, y);
    if (persp) z = DDIV(1.0, z);
    if (z < p->z) { p->z = z; p->own = id; p->bown = id; }
    else if (z == p->z && p->own >= 0) {
        if ((id & TRI_INDEX_MASK) < (p->own & TRI_INDEX_MASK)) p->own = id;
        if ((id & TRI_INDEX_MASK) > (p->bown & TRI_INDEX_MASK)) p->bown = id;
    }
}

// Phase T2a: each pixel z-tests its candidates of this chunk (any order: ties are resolved by index) and clears its
// counter for the next chunk.  A pixel with more than PIX_SLOTS candidates scans the chunk's masks instead.
template <int MAXC>
DEODR_HD void phase_pix_test(const SceneView &s, int tid, int n, Tile tile, const PreRec *pre, TileShared *sh,
                             PixelState<MAXC> *p) {
    const int count = sh->tri.pix_cnt[tid];
    sh->tri.pix_cnt[tid] = 0;
    if (count == 0) return;
    const int x = tile.x0 + tid % TS, y = tile.y0 + tid / TS;
    const double xd = (double)x, yd = (double)y;
    const bool persp = s.perspective_correct != 0;
    if (count <= PIX_SLOTS) {
        for (int i = 0; i < count; i++) {
            const PreRec &r = pre[sh->tri.pix_list[i][tid]];
            z_candidate<MAXC>(r.zp, r.id, xd, yd, x, y, persp, p);
        }
    } else {
        const int lane = tid % 32, pair = tid / 32;
        for (int t = 0; t < n; t++)
            if ((pre[t].mask[pair] >> lane) & 1u) z_candidate<MAXC>(pre[t].zp, pre[t].id, xd, yd, x, y, persp, p);
    }
}

// Phase T1b: thread tid < n sets up the stencil of LARGE triangle list[tid] into shared memory (n <= LARGE_CHUNK).
DEODR_HD void phase_tri_setup(const SceneView &s, int tid, int n, const int *list, TileShared *sh) {
    if (tid >= n) return;
    const int k = list[tid];
    uint32_t vid[3];
    double V[3][2], Zv[3];
    gather_tri(s, k, vid, V, Zv);
    remove_offset(V, 3, pixel_offset(s));
    TriGeom &g = sh->tri.geo[tid];
    tri_geom(V, Zv, s.strict_edge != 0, s.perspective_correct != 0, &g, nullptr);
    TriRec &rec = sh->tri.rec[tid];
    canonical_plane(g.zp, rec.zp);
    rec.id = k;
}

// Phase T1c: (triangle, row pair) items -> coverage masks; 8 threads per large triangle instead of one, which shortens
// the critical path of every tile that holds a large triangle 4x (measured: that barrier was 32 % of k_tile_z's stalls).
// Triangles up to the next multiple of 4 get empty masks (padding).
DEODR_HD void phase_tri_masks(const SceneView &s, int tid, int n, Tile tile, TileShared *sh) {
    const int n4 = (n + 3) & ~3;
    for (int item = tid; item < n4 * (TS / 2); item += NT) {
        const int t = item / (TS / 2), p = item % (TS / 2);
        uint32_t m = 0u;
        if (t < n) {
            const TriGeom &g = sh->tri.geo[t];
            int y_first, y_last;
            tri_row_range(g, s.height, &y_first, &y_last);
            m = tri_pair_mask(s, g, y_first, y_last, tile.x0, tile.y0, p);
        }
        sh->tri.mask[p][t] = m;
    }
}

// Phase T2: each pixel walks the chunk and keeps the minimum z, order-independently:
//   own = min index among ties (what a strict '<' walk in ascending index order leaves, DR.h:961),
//   bown = max index among ties (what the '==' walk in descending index order finds first, DR.h:1024).
// Lane l of warp p owns pixel (col l % 16, row 2p + l / 16) = bit l of mask[p][t].
template <int MAXC>
DEODR_HD void phase_tri_test(const SceneView &s, int tid, int n, Tile tile, const TileShared *sh, PixelState<MAXC> *p) {
    const int lane = tid % 32, pair = tid / 32;
    const int x = tile.x0 + tid % TS, y = tile.y0 + tid / TS;
    const double xd = (double)x, yd = (double)y;
    const bool persp = s.perspective_correct != 0;
    for (int t0 = 0; t0 < n; t0 += 4) {
        const Mask4 m4 = *reinterpret_cast<const Mask4 *>(&sh->tri.mask[pair][t0]);
        if ((m4.m[0] | m4.m[1] | m4.m[2] | m4.m[3]) == 0u) continue;
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int j = 0; j < 4; j++) {
            if (!((m4.m[j] >> lane) & 1u)) continue;
            const TriRec &rec = sh->tri.rec[t0 + j];
            z_candidate<MAXC>(rec.zp, rec.id, xd, yd, x, y, persp, p);
        }
    }
}

// Phase S: background + owner colour.
template <int MAXC>
DEODR_HD void phase_shade(const SceneView &s, int x, int y, PixelState<MAXC> *p, float *w_out = nullptr) {
    const int C = s.nb_colors;
    if (w_out) w_out[0] = w_out[1] = w_out[2] = 0.0f;
    if (p->own < 0) {
        if (s.background_image) {
            const float *bg = s.background_image + ((size_t)y * s.width + x) * C;
            for (int c = 0; c < C; c++) p->col[c] = bg[c];
        } else {
            for (int c = 0; c < C; c++) p->col[c] = s.background_color[c];
        }
        return;
    }
    TriAttr t;
    tri_attr(s, p->own & TRI_INDEX_MASK, &t);
    PixelEval<MAXC> e;
    pixel_colour<MAXC>(s, t, x, y, p->z, &e, p->col);
    if (w_out) { w_out[0] = e.w[0]; w_out[1] = e.w[1]; w_out[2] = e.w[2]; }  // G-buffer: interpolation weights
}

// Phase E1: the CTA fetches the records of the edges list[0..n) of its tile, in far-to-near order (built once per
// forward pass by bin_edge: the stencil's sqrt / divisions are not redone per tile); 8-byte words, all threads.
DEODR_HD void phase_edge_setup(int tid, int nthreads, int n, const int *list, const EdgeRec *edge_recs, TileShared *sh) {
    constexpr int WORDS = (int)(sizeof(EdgeRec) / 8);
    static_assert(sizeof(EdgeRec) % 8 == 0, "EdgeRec is copied as 8-byte words");
    // four words per thread and pass, every load issued before the first store: the compiler cannot hoist a
    // generic-pointer load above a shared-memory store itself, and one word per pass costs a memory round trip each
    constexpr int BATCH = 4;
    const int total = n * WORDS;
    for (int first = tid; first < total; first += BATCH * nthreads) {
        unsigned long long v[BATCH];
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int j = 0; j < BATCH; j++) {
            const int item = first + j * nthreads;
            if (item < total)
                v[j] = reinterpret_cast<const unsigned long long *>(&edge_recs[list[item / WORDS]])[item % WORDS];
        }
#if defined(__CUDA_ARCH__)
#pragma unroll
#endif
        for (int j = 0; j < BATCH; j++) {
            const int item = first + j * nthreads;
            if (item < total) reinterpret_cast<unsigned long long *>(&sh->edge.rec[item / WORDS])[item % WORDS] = v[j];
        }
    }
}

// Phase E2: (edge, row) items of rows [row0, row0 + nrows) of the tile -> x spans.
DEODR_HD void phase_edge_spans(const SceneView &s, int tid, int nthreads, int n, Tile tile, int row0, int nrows,
                               TileShared *sh) {
    for (int item = tid; item < n * nrows; item += nthreads) {
        int e = item / nrows, r = row0 + item % nrows;
        int y = tile.y0 + r;
        uint32_t packed = 1u;  // begin = 1, end = 0: empty
        const EdgeGeom &g = sh->edge.rec[e].g;
        if (y >= g.y_begin && y <= g.y_end) {
            int xb, xe;
            edge_row_span(g, s.width, y, &xb, &xe);
            if (xb <= xe) packed = ((uint32_t)(uint16_t)(int16_t)xb) | (((uint32_t)(uint16_t)(int16_t)xe) << 16);
        }
        sh->edge.span[e][r] = packed;
    }
}

DEODR_HD bool edge_covers(const TileShared *sh, int e, int r, int x) {
    uint32_t packed = sh->edge.span[e][r];
    int xb = (int16_t)(packed & 0xffffu), xe = (int16_t)(packed >> 16);
    return x >= xb && x <= xe;
}

// Bit e set <=> edge e of the chunk (n <= EDGE_CHUNK = 64) has pixel (x, row r) inside its band.  A short uniform loop;
// the per-edge work then runs over the set bits only, so the lanes of a warp step through DIFFERENT edges side by side
// (a warp takes max-over-lanes hits, not the number of distinct edges that touch its 32 pixels).
DEODR_HD unsigned long long edge_hit_mask(const TileShared *sh, int n, int r, int x) {
    static_assert(EDGE_CHUNK <= 64, "one bit per edge of a chunk");
    unsigned long long mask = 0ull;
    for (int e = 0; e < n; e++)
        if (edge_covers(sh, e, r, x)) mask |= 1ull << e;
    return mask;
}

// Phase E3 (forward): overdraw in list order.  image = T*image + (1-T)*A where Z_edge < z_buffer (DR.h:1632-1641).
template <int MAXC>
DEODR_HD void phase_edge_blend(const SceneView &s, int x, int y, int r, int n, const TileShared *sh, PixelState<MAXC> *p) {
    const int C = s.nb_colors;
    for (unsigned long long mask = edge_hit_mask(sh, n, r, x); mask; mask &= mask - 1) {
        const EdgeRec &rec = sh->edge.rec[lowest_bit64(mask)];
        double ze = edge_z(rec, x, y, s.perspective_correct != 0);
        if (!(ze < p->z)) continue;
        EdgeHit<MAXC> h;
        edge_hit<MAXC>(s, rec, x, y, ze, &h);
        float T = (float)h.T, omT = (float)(1.0 - h.T);
        for (int c = 0; c < C; c++) p->col[c] = p->col[c] * T + omT * h.A[c];
    }
}

// ----------------------------------------------------------------------------------------------------- adjoint

// Running state of a pixel during the backward edge sweep.  The colour is tracked in fp64 so that the un-blend
// (DR.h:1738) recovers the colour each edge saw as accurately as the reference does.
template <int MAXC>
struct AdjointState {
    double col[MAXC];   // colour of the pixel after the edges processed so far (forward) / before them (reverse)
    float g[MAXC];      // adjoint of the pixel colour
    bool has_colour;    // col[] initialised (done lazily: only pixels inside an edge band need it)
};

// Forward replay over one chunk (edges in list order) in fp64: col <- T*col + (1-T)*A.
template <int MAXC>
DEODR_HD void phase_edge_replay(const SceneView &s, int x, int y, int r, int n, const TileShared *sh,
                                const PixelState<MAXC> &p, AdjointState<MAXC> *a) {
    const int C = s.nb_colors;
    for (unsigned long long mask = edge_hit_mask(sh, n, r, x); mask; mask &= mask - 1) {
        const EdgeRec &rec = sh->edge.rec[lowest_bit64(mask)];
        double ze = edge_z(rec, x, y, s.perspective_correct != 0);
        if (!(ze < p.z)) continue;
        if (!a->has_colour) {
            PixelState<MAXC> q = p;
            phase_shade<MAXC>(s, x, y, &q);
            for (int c = 0; c < C; c++) a->col[c] = (double)q.col[c];
            a->has_colour = true;
        }
        EdgeHit<MAXC> h;
        edge_hit<MAXC>(s, rec, x, y, ze, &h);
        for (int c = 0; c < C; c++) a->col[c] = a->col[c] * h.T + (1.0 - h.T) * (double)h.A[c];
    }
}

// Reverse sweep over one chunk (edges in reverse list order): un-blend, per-edge plane adjoints, g <- T*g.
// DR.h:1726-1749 (interpolated) / DR.h:2008-2032 (textured), accumulated per edge as moments over (x, y, 1).
template <int MAXC, class Env>
DEODR_HD void phase_edge_adjoint(const SceneView &s, int x, int y, int r, int n, const TileShared *sh,
                                 const PixelState<MAXC> &p, AdjointState<MAXC> *a, double *edge_acc, float *texture_b) {
    const int C = s.nb_colors;
    const int stride = s.perspective_correct ? edge_acc_stride_persp(C) : edge_acc_stride(C);
    for (unsigned long long mask = edge_hit_mask(sh, n, r, x); mask;) {  // near to far: highest bit first
        const int e = highest_bit64(mask);
        mask &= ~(1ull << e);
        const EdgeRec &rec = sh->edge.rec[e];
        double ze = edge_z(rec, x, y, s.perspective_correct != 0);
        if (!(ze < p.z)) continue;
        EdgeHit<MAXC> h;
        edge_hit<MAXC>(s, rec, x, y, ze, &h);
        double *acc = edge_acc + (size_t)rec.slot * stride;
        const double T = h.T, omT = 1.0 - h.T;
        double T_B = 0;
        const double t3[3] = {(double)x, (double)y, 1.0};
        if (s.perspective_correct) {
            // the edge's attribute a = w_0 a_0 + w_1 a_1, w_q = b_q q_q Ze: the same adjoint as pixel_adjoint_persp
            // over the two end points (edge_acc_stride_persp gives the layout)
            const double w[2] = {h.b[0] * rec.inv_z[0] * ze, h.b[1] * rec.inv_z[1] * ze};
            double sd[2] = {0.0, 0.0};
            if (s.texture != nullptr && rec.textured) {
                double L_B = 0;
                float e0_B = 0, e1_B = 0;
                for (int c = 0; c < C; c++) {
                    double gc = (double)a->g[c];
                    double prev = (a->col[c] - omT * (double)h.A[c]) / T;
                    T_B += gc * (prev - (double)h.A[c]);
                    a->col[c] = prev;
                    float A_B = (float)(omT * gc) * h.L;
                    L_B += omT * gc * (double)h.texval[c];
                    texture_fetch_duv(h.tap, s.texture, c, A_B, &e0_B, &e1_B);
                    if (texture_b) {
                        float w00 = (1.0f - h.tap.e0) * (1.0f - h.tap.e1), w10 = h.tap.e0 * (1.0f - h.tap.e1);
                        float w01 = (1.0f - h.tap.e0) * h.tap.e1, w11 = h.tap.e0 * h.tap.e1;
                        Env::atomic_add(texture_b + h.tap.i00 + c, w00 * A_B);
                        Env::atomic_add(texture_b + h.tap.i10 + c, w10 * A_B);
                        Env::atomic_add(texture_b + h.tap.i01 + c, w01 * A_B);
                        Env::atomic_add(texture_b + h.tap.i11 + c, w11 * A_B);
                    }
                    a->g[c] = (float)(gc * T);
                }
                const double U_B = h.tap.out0 ? 0.0 : (double)e0_B, V_B = h.tap.out1 ? 0.0 : (double)e1_B;
                const double L = w[0] * (double)s.shade[rec.vid[0]] + w[1] * (double)s.shade[rec.vid[1]];
                for (int q = 0; q < 2; q++) {
                    const double uq = s.uv[2 * (size_t)rec.uvid[q]], vq = s.uv[2 * (size_t)rec.uvid[q] + 1];
                    sd[q] = U_B * (uq - h.u) + V_B * (vq - h.v) + L_B * ((double)s.shade[rec.vid[q]] - L);
                    Env::atomic_add(acc + 11 + 3 * q, w[q] * U_B);
                    Env::atomic_add(acc + 12 + 3 * q, w[q] * V_B);
                    Env::atomic_add(acc + 13 + 3 * q, w[q] * L_B);
                }
            } else {
                for (int c = 0; c < C; c++) {
                    double gc = (double)a->g[c];
                    double prev = (a->col[c] - omT * (double)h.A[c]) / T;
                    T_B += gc * (prev - (double)h.A[c]);
                    a->col[c] = prev;
                    const double A_B = omT * gc;
                    const double a0 = (double)s.colors[(size_t)rec.vid[0] * C + c],
                                 a1 = (double)s.colors[(size_t)rec.vid[1] * C + c];
                    const double A = w[0] * a0 + w[1] * a1;
                    sd[0] += A_B * (a0 - A);
                    sd[1] += A_B * (a1 - A);
                    Env::atomic_add(acc + 11 + c, w[0] * A_B);
                    Env::atomic_add(acc + 11 + C + c, w[1] * A_B);
                    a->g[c] = (float)(gc * T);
                }
            }
            for (int q = 0; q < 2; q++) {
                const double bq_B = rec.inv_z[q] * ze * sd[q];
                for (int j = 0; j < 3; j++) Env::atomic_add(acc + 3 + 3 * q + j, bq_B * t3[j]);
                Env::atomic_add(acc + 9 + q, -w[q] * sd[q] * rec.inv_z[q]);
            }
        } else if (s.texture != nullptr && rec.textured) {
            double L_B = 0;
            float e0_B = 0, e1_B = 0;
            for (int c = 0; c < C; c++) {
                double gc = (double)a->g[c];
                double prev = (a->col[c] - omT * (double)h.A[c]) / T;  // colour before this edge
                T_B += gc * (prev - (double)h.A[c]);
                a->col[c] = prev;
                float A_B = (float)(omT * gc) * h.L;                    // adjoint of the texture sample
                L_B += omT * gc * (double)h.texval[c];
                texture_fetch_duv(h.tap, s.texture, c, A_B, &e0_B, &e1_B);
                if (texture_b) {
                    float w00 = (1.0f - h.tap.e0) * (1.0f - h.tap.e1), w10 = h.tap.e0 * (1.0f - h.tap.e1);
                    float w01 = (1.0f - h.tap.e0) * h.tap.e1, w11 = h.tap.e0 * h.tap.e1;
                    Env::atomic_add(texture_b + h.tap.i00 + c, w00 * A_B);
                    Env::atomic_add(texture_b + h.tap.i10 + c, w10 * A_B);
                    Env::atomic_add(texture_b + h.tap.i01 + c, w01 * A_B);
                    Env::atomic_add(texture_b + h.tap.i11 + c, w11 * A_B);
                }
                a->g[c] = (float)(gc * T);
            }
            double U_B = h.tap.out0 ? 0.0 : (double)e0_B, V_B = h.tap.out1 ? 0.0 : (double)e1_B;
            for (int j = 0; j < 3; j++) {
                Env::atomic_add(acc + 3 + j, L_B * t3[j]);
                Env::atomic_add(acc + 6 + j, U_B * t3[j]);
                Env::atomic_add(acc + 9 + j, V_B * t3[j]);
            }
        } else {
            for (int c = 0; c < C; c++) {
                double gc = (double)a->g[c];
                double prev = (a->col[c] - omT * (double)h.A[c]) / T;
                T_B += gc * (prev - (double)h.A[c]);
                a->col[c] = prev;
                double A_B = omT * gc;
                for (int j = 0; j < 3; j++) Env::atomic_add(acc + 12 + 3 * c + j, A_B * t3[j]);
                a->g[c] = (float)(gc * T);
            }
        }
        for (int j = 0; j < 3; j++) Env::atomic_add(acc + j, T_B * t3[j]);
    }
}

// ------------------------------------------------------------------------ antialiase_error mode (row f3, DR.h:2066-2618)
//
// The silhouette edges overdraw the squared residual err = sum_c (image_c - obs_c)^2 instead of the colours: the image
// keeps its aliased edges, err <- T * err + (1 - T) * Err_edge with Err_edge = sum_c (A_c - obs_c)^2 where
// Z_edge < z_buffer.  These phases mirror phase_edge_blend / replay / adjoint on that scalar.  They are exercised by the
// CPU emulation against the oracle (tests/test_emul.py); the CUDA entry points still report the mode as unsupported
// until the kernels that call them have been validated on a GPU.

// residual of one pixel before the edges (DR.h:2824-2837)
template <int MAXC>
DEODR_HD double pixel_residual(const SceneView &s, const float *col, const float *obs) {
    double r = 0;
    for (int c = 0; c < s.nb_colors; c++) {
        const double d = (double)col[c] - (double)obs[c];
        r += d * d;
    }
    return r;
}

template <int MAXC>
DEODR_HD double edge_residual(const SceneView &s, const EdgeHit<MAXC> &h, const float *obs) {
    double r = 0;
    for (int c = 0; c < s.nb_colors; c++) {
        const double d = (double)h.A[c] - (double)obs[c];
        r += d * d;
    }
    return r;
}

// forward: overdraw of the residual in list order (DR.h:2186-2187, 2467-2468)
template <int MAXC>
DEODR_HD void phase_edge_blend_error(const SceneView &s, int x, int y, int r, int n, const TileShared *sh, double z,
                                     const float *obs, float *err) {
    for (unsigned long long mask = edge_hit_mask(sh, n, r, x); mask; mask &= mask - 1) {
        const EdgeRec &rec = sh->edge.rec[lowest_bit64(mask)];
        double ze = edge_z(rec, x, y, s.perspective_correct != 0);
        if (!(ze < z)) continue;
        EdgeHit<MAXC> h;
        edge_hit<MAXC>(s, rec, x, y, ze, &h);
        *err = *err * (float)h.T + (float)(1.0 - h.T) * (float)edge_residual<MAXC>(s, h, obs);
    }
}

// Running state of a pixel during the backward edge sweep of the error mode.
template <int MAXC>
struct ErrorAdjointState {
    double err;        // residual after the edges processed so far (forward) / before them (reverse), fp64
    double g;          // adjoint of the residual
    float col[MAXC];   // the pixel's (aliased) colour
    bool has;          // err / col initialised (lazily: only pixels inside an edge band need them)
};

template <int MAXC>
DEODR_HD void phase_edge_replay_error(const SceneView &s, int x, int y, int r, int n, const TileShared *sh,
                                      const PixelState<MAXC> &p, const float *obs, ErrorAdjointState<MAXC> *a) {
    for (unsigned long long mask = edge_hit_mask(sh, n, r, x); mask; mask &= mask - 1) {
        const EdgeRec &rec = sh->edge.rec[lowest_bit64(mask)];
        double ze = edge_z(rec, x, y, false);
        if (!(ze < p.z)) continue;
        if (!a->has) {
            PixelState<MAXC> q = p;
            phase_shade<MAXC>(s, x, y, &q);
            for (int c = 0; c < s.nb_colors; c++) a->col[c] = q.col[c];
            a->err = pixel_residual<MAXC>(s, a->col, obs);
            a->has = true;
        }
        EdgeHit<MAXC> h;
        edge_hit<MAXC>(s, rec, x, y, ze, &h);
        a->err = a->err * h.T + (1.0 - h.T) * edge_residual<MAXC>(s, h, obs);
    }
}

// Reverse sweep (near to far): un-blend the residual, per-edge plane adjoints, g <- T * g.
// DR.h:2296-2336 (textured) / DR.h:2542-2576 (interpolated).  `compat` reproduces the reference's defect #2: for
// interpolated edges only the x moment of the colour-plane adjoint is kept (the per-row A0y_B is never propagated,
// DR.h:2577-2583); with compat = false the mathematically complete adjoint is accumulated.
template <int MAXC, class Env>
DEODR_HD void phase_edge_adjoint_error(const SceneView &s, int x, int y, int r, int n, const TileShared *sh,
                                       const PixelState<MAXC> &p, const float *obs, ErrorAdjointState<MAXC> *a,
                                       double *edge_acc, float *texture_b, bool compat) {
    const int C = s.nb_colors;
    const int stride = edge_acc_stride(C);
    for (unsigned long long mask = edge_hit_mask(sh, n, r, x); mask;) {
        const int e = highest_bit64(mask);
        mask &= ~(1ull << e);
        const EdgeRec &rec = sh->edge.rec[e];
        double ze = edge_z(rec, x, y, false);
        if (!(ze < p.z)) continue;
        EdgeHit<MAXC> h;
        edge_hit<MAXC>(s, rec, x, y, ze, &h);
        double *acc = edge_acc + (size_t)rec.slot * stride;
        const double T = h.T, omT = 1.0 - h.T;
        const double Err = edge_residual<MAXC>(s, h, obs);
        const double prev = (a->err - omT * Err) / T;  // residual before this edge
        const double T_B = a->g * (prev - Err);
        const double Err_B = omT * a->g;
        a->err = prev;
        a->g = a->g * T;
        const double t3[3] = {(double)x, (double)y, 1.0};
        if (s.texture != nullptr && rec.textured) {
            double L_B = 0;
            float e0_B = 0, e1_B = 0;
            for (int c = 0; c < C; c++) {
                const double diff_B = 2.0 * ((double)h.A[c] - (double)obs[c]) * Err_B;  // A_c = texval_c * L
                const float A_B = (float)diff_B * h.L;                                   // adjoint of the texture sample
                L_B += diff_B * (double)h.texval[c];
                texture_fetch_duv(h.tap, s.texture, c, A_B, &e0_B, &e1_B);
                if (texture_b) {
                    float w00 = (1.0f - h.tap.e0) * (1.0f - h.tap.e1), w10 = h.tap.e0 * (1.0f - h.tap.e1);
                    float w01 = (1.0f - h.tap.e0) * h.tap.e1, w11 = h.tap.e0 * h.tap.e1;
                    Env::atomic_add(texture_b + h.tap.i00 + c, w00 * A_B);
                    Env::atomic_add(texture_b + h.tap.i10 + c, w10 * A_B);
                    Env::atomic_add(texture_b + h.tap.i01 + c, w01 * A_B);
                    Env::atomic_add(texture_b + h.tap.i11 + c, w11 * A_B);
                }
            }
            double U_B = h.tap.out0 ? 0.0 : (double)e0_B, V_B = h.tap.out1 ? 0.0 : (double)e1_B;
            for (int j = 0; j < 3; j++) {
                Env::atomic_add(acc + 3 + j, L_B * t3[j]);
                Env::atomic_add(acc + 6 + j, U_B * t3[j]);
                Env::atomic_add(acc + 9 + j, V_B * t3[j]);
            }
        } else {
            for (int c = 0; c < C; c++) {
                const double A_B = 2.0 * ((double)h.A[c] - (double)obs[c]) * Err_B;
                for (int j = 0; j < (compat ? 1 : 3); j++) Env::atomic_add(acc + 12 + 3 * c + j, A_B * t3[j]);
            }
        }
        for (int j = 0; j < 3; j++) Env::atomic_add(acc + j, T_B * t3[j]);
    }
}

// colour adjoint of a pixel from the adjoint of its residual (DR.h:3054-3060)
template <int MAXC>
DEODR_HD void residual_adjoint(const SceneView &s, const float *col, const float *obs, double g, float *image_b) {
    for (int c = 0; c < s.nb_colors; c++) image_b[c] = (float)(-2.0 * ((double)obs[c] - (double)col[c]) * g);
}

// Interior adjoint of one pixel (pixel-parallel kernels): the residual colour adjoint g goes to the vertices of the
// adjoint owner.  `env.emit(ptr, v)` adds v to a vertex-gradient slot; the device version sums over the warp first when
// the whole warp shares the owner triangle.  (The device kernels use interior_adjoint_warp of kernels.cu, which sums
// per owner inside the warp first; this per-pixel form is what the CPU emulation runs.)
template <int MAXC, class Env>
DEODR_HD void phase_interior_adjoint(const SceneView &s, int x, int y, const PixelState<MAXC> &p, const float *g,
                                     float *ij_b, float *colors_b, float *uv_b, float *shade_b, float *texture_b,
                                     const Env &env, float *depths_b = nullptr) {
    TriAttr t;
    tri_attr(s, p.bown & TRI_INDEX_MASK, &t);
    VertexGrads<MAXC> acc;
    zero_vertex_grads<MAXC>(s, &acc);
    float dz[3] = {0.0f, 0.0f, 0.0f};
    pixel_adjoint<MAXC, Env>(s, t, x, y, g, &acc, texture_b, dz);
    flush_vertex_grads<MAXC, Env>(s, t, acc, ij_b, colors_b, uv_b, shade_b, env, dz, depths_b);
}

// Plain atomics for the triangle-parallel adjoint.
template <class Env>
struct AtomicEmit {
    DEODR_HD void emit(float *p, float v) const { Env::atomic_add(p, v); }
};

// Triangle-parallel interior adjoint of one SMALL triangle (micro-triangle regime): the thread walks the triangle's
// bounding box, takes the pixels whose adjoint owner it is (the reference's `Z == z_buffer` walk, DR.h:1024, resolved
// to an owner id by the forward pass), accumulates its vertex gradients in registers and scatters them ONCE: 15
// atomics per triangle instead of 15 per pixel, one barycentric set-up per triangle instead of one per pixel.
// Pixels of tiles that contain silhouette edges are left to k_raster_bwd (their adjoint colour is not image_b).
template <int MAXC, class Env>
DEODR_HD void small_triangle_adjoint(const SceneView &s, int k, int tiles_x, const int *edge_tile_count,
                                     const int *owner, const int *tie_pairs, const float *image_b, float *ij_b,
                                     float *colors_b, float *uv_b, float *shade_b, float *texture_b,
                                     float *depths_b = nullptr) {
    const int C = s.nb_colors;
    double V[3][2];
    for (int i = 0; i < 3; i++) {
        const uint32_t v = s.faces[3 * k + i];
        V[i][0] = s.ij[2 * (size_t)v];
        V[i][1] = s.ij[2 * (size_t)v + 1];
    }
    remove_offset(V, 3, pixel_offset(s));
    int x0, x1, y0, y1;
    tri_bounds(V, s.strict_edge != 0, &x0, &x1, &y0, &y1);
    if (x0 < 0) x0 = 0;
    if (y0 < 0) y0 = 0;
    if (x1 > s.width - 1) x1 = s.width - 1;
    if (y1 > s.height - 1) y1 = s.height - 1;
    const int code = k | SMALL_FLAG;
    // bit index of pixel (x, y) = ((y - y0) << shift) + (x - x0); fits 64 bits by construction of the small list
    const int shift = small_shift(x1 - x0 + 1), stride_mask = (1 << shift) - 1;
    // phase 1 (cheap, uniform): which pixels of the bounding box does this triangle own?  One bit per pixel.
    // Loads of a row are independent: unrolled so that several are in flight.
    unsigned long long mine = 0ull;
    for (int y = y0; y <= y1; y++) {
        const int *row = owner + (size_t)y * s.width;
        const int bit0 = ((y - y0) << shift) - x0;
#if defined(__CUDA_ARCH__)
#pragma unroll 4
#endif
        for (int x = x0; x <= x1; x++) {
            const int c = row[x];
            bool hit = c == code;
            if (c <= -2) hit = tie_pairs[2 * (-2 - c) + 1] == code;
            if (hit) mine |= 1ull << (bit0 + x);
        }
    }
    if (!mine) return;  // hidden triangle
    if (edge_tile_count) {  // pixels of tiles with silhouette edges belong to k_raster_bwd
        for (int ty = y0 / TS; ty <= y1 / TS; ty++)
            for (int tx = x0 / TS; tx <= x1 / TS; tx++) {
                if (edge_tile_count[ty * tiles_x + tx] == 0) continue;
                for (int y = (ty * TS > y0 ? ty * TS : y0); y <= y1 && y < (ty + 1) * TS; y++)
                    for (int x = (tx * TS > x0 ? tx * TS : x0); x <= x1 && x < (tx + 1) * TS; x++)
                        mine &= ~(1ull << (((y - y0) << shift) + (x - x0)));
            }
        if (!mine) return;
    }
    // phase 2: lanes take their i-th owned pixel together; the adjoint colour of the NEXT pixel is loaded while the
    // current one is processed
    TriAttr t;
    tri_attr(s, k, &t);
    float g_next[MAXC];
    int i_next = lowest_bit64(mine);
    mine &= mine - 1;
    {
        const size_t idx = (size_t)(y0 + (i_next >> shift)) * s.width + x0 + (i_next & stride_mask);
        for (int q = 0; q < C; q++) g_next[q] = image_b[idx * C + q];
    }
    // The two kinds of triangle keep different accumulators (vertex colours vs uv + shade): separate loops, so that the
    // common interpolated case holds 15 running sums in registers instead of a 24-float structure in local memory.
    // Perspective-correct triangles take the general loop (pixel_adjoint_persp).
    if (t.textured || s.perspective_correct) {
        VertexGrads<MAXC> acc;
        zero_vertex_grads<MAXC>(s, &acc);
        float dz[3] = {0.0f, 0.0f, 0.0f};
        for (;;) {
            const int i = i_next;
            float g[MAXC];
            for (int q = 0; q < C; q++) g[q] = g_next[q];
            const bool more = mine != 0ull;
            if (more) {
                i_next = lowest_bit64(mine);
                mine &= mine - 1;
                const size_t idx = (size_t)(y0 + (i_next >> shift)) * s.width + x0 + (i_next & stride_mask);
                for (int q = 0; q < C; q++) g_next[q] = image_b[idx * C + q];
            }
            pixel_adjoint<MAXC, Env>(s, t, x0 + (i & stride_mask), y0 + (i >> shift), g, &acc, texture_b, dz);
            if (!more) break;
        }
        flush_vertex_grads<MAXC, AtomicEmit<Env>>(s, t, acc, ij_b, colors_b, uv_b, shade_b, AtomicEmit<Env>(), dz,
                                                  depths_b);
        return;
    }
    // interpolated triangle: per-triangle constants = vertex colours' screen-space gradient
    float dadx[MAXC], dady[MAXC];
    for (int q = 0; q < C; q++) {
        const float a0 = s.colors[(size_t)t.vid[0] * C + q], a1 = s.colors[(size_t)t.vid[1] * C + q],
                    a2 = s.colors[(size_t)t.vid[2] * C + q];
        // (fp64: three terms of size |colour| / area that cancel - a sliver would lose every digit in fp32)
        dadx[q] = (float)(t.gx[0] * (double)a0 + t.gx[1] * (double)a1 + t.gx[2] * (double)a2);
        dady[q] = (float)(t.gy[0] * (double)a0 + t.gy[1] * (double)a1 + t.gy[2] * (double)a2);
    }
    float gij[3][2] = {{0.0f, 0.0f}, {0.0f, 0.0f}, {0.0f, 0.0f}};
    float gcol[3][MAXC];
    for (int q = 0; q < C; q++) gcol[0][q] = gcol[1][q] = gcol[2][q] = 0.0f;
    for (;;) {
        const int i = i_next;
        float g[MAXC];
        for (int q = 0; q < C; q++) g[q] = g_next[q];
        const bool more = mine != 0ull;
        if (more) {
            i_next = lowest_bit64(mine);
            mine &= mine - 1;
            const size_t idx = (size_t)(y0 + (i_next >> shift)) * s.width + x0 + (i_next & stride_mask);
            for (int q = 0; q < C; q++) g_next[q] = image_b[idx * C + q];
        }
        double wd[3];
        tri_weights(s, t, x0 + (i & stride_mask), y0 + (i >> shift), 0.0, wd);
        const float w0 = (float)wd[0], w1 = (float)wd[1], w2 = (float)wd[2];
        float dcdx = 0, dcdy = 0;
        for (int q = 0; q < C; q++) {
            dcdx += g[q] * dadx[q];
            dcdy += g[q] * dady[q];
            gcol[0][q] += g[q] * w0;
            gcol[1][q] += g[q] * w1;
            gcol[2][q] += g[q] * w2;
        }
        gij[0][0] -= w0 * dcdx; gij[0][1] -= w0 * dcdy;
        gij[1][0] -= w1 * dcdx; gij[1][1] -= w1 * dcdy;
        gij[2][0] -= w2 * dcdx; gij[2][1] -= w2 * dcdy;
        if (!more) break;
    }
    for (int i = 0; i < 3; i++) {  // same scatter as flush_vertex_grads, interpolated branch
        Env::atomic_add(ij_b + 2 * (size_t)t.vid[i], gij[i][0]);
        Env::atomic_add(ij_b + 2 * (size_t)t.vid[i] + 1, gij[i][1]);
        for (int q = 0; q < C; q++) Env::atomic_add(colors_b + (size_t)t.vid[i] * C + q, gcol[i][q]);
    }
}

// ---- record-parallel form of the same adjoint -------------------------------------------------------------------
// The forward's pre-masked records already say WHICH pixels of a tile a small triangle covers (3.6 on average on the
// 1M-triangle scene, against the 33 pixels of the bounding box the triangle-parallel form reads to find them).  One
// thread per record of a tile without silhouette edges: the covered pixels are tested for ownership against the tile's
// owner block, the owned ones accumulate into registers, and the record's triangle scatters once (a triangle that
// straddles two tiles scatters twice: 15 % more atomics, none of the bounding-box reads).  `Fetch` hides where the
// tile's owner codes and colour adjoints live: shared memory (staged by TMA tile loads, kernels_bwd.cu) or the global
// arrays (CPU emulation, wide-channel instances).
struct GlobalTileFetch {
    const int *owner_map;
    const float *image_b;
    Tile tile;
    int width, height, C;
    DEODR_HD int owner(int px) const {
        const int x = tile.x0 + (px & (TS - 1)), y = tile.y0 + (px >> 4);
        return x < width && y < height ? owner_map[(size_t)y * width + x] : -1;
    }
    DEODR_HD float g(int px, int q) const {
        const int x = tile.x0 + (px & (TS - 1)), y = tile.y0 + (px >> 4);
        return image_b[((size_t)y * width + x) * C + q];  // (only asked for owned pixels: inside the image)
    }
};

template <int MAXC, class Env, class Fetch>
DEODR_HD void small_record_adjoint(const SceneView &s, const PreRec &r, Tile tile, const Fetch &fetch,
                                   const int *tie_pairs, float *ij_b, float *colors_b, float *uv_b, float *shade_b,
                                   float *texture_b) {
    static_assert(TS == 16, "pixel index of a mask bit: word * 32 + bit = row * 16 + column");
    const int C = s.nb_colors;
    const int code = r.id;
    if (!(code & SMALL_FLAG)) return;  // medium triangle: its pixels belong to the pixel-parallel adjoint
    // phase 1 (cheap): which of the covered pixels does this triangle own?  One flat loop over the set bits.
    uint32_t mine[TS / 2];
    uint32_t words = 0u, own_words = 0u;
    for (int p = 0; p < TS / 2; p++) {
        mine[p] = 0u;
        words |= (uint32_t)(r.mask[p] != 0u) << p;
    }
    {
        int p = 0;
        uint32_t w = 0u;
        for (;;) {
            if (w == 0u) {
                if (words == 0u) break;
                p = lowest_bit(words);
                words &= words - 1;
                w = r.mask[p];
            }
            const int bit = lowest_bit(w);
            w &= w - 1;
            const int c = fetch.owner(p * 32 + bit);
            bool hit = c == code;
            if (c <= -2) hit = tie_pairs[2 * (-2 - c) + 1] == code;
            if (hit) {
                mine[p] |= 1u << bit;
                own_words |= 1u << p;
            }
        }
    }
    if (!own_words) return;  // hidden here
    // phase 2: one set-up per record, then the owned pixels
    const int k = code & TRI_INDEX_MASK;
    TriAttr t;
    tri_attr(s, k, &t);
    int p = 0;
    uint32_t w = 0u;
    if (t.textured) {
        VertexGrads<MAXC> acc;
        zero_vertex_grads<MAXC>(s, &acc);
        for (;;) {
            if (w == 0u) {
                if (own_words == 0u) break;
                p = lowest_bit(own_words);
                own_words &= own_words - 1;
                w = mine[p];
            }
            const int px = p * 32 + lowest_bit(w);
            w &= w - 1;
            float g[MAXC];
            for (int q = 0; q < C; q++) g[q] = fetch.g(px, q);
            pixel_adjoint<MAXC, Env>(s, t, tile.x0 + (px & (TS - 1)), tile.y0 + (px >> 4), g, &acc, texture_b);
        }
        flush_vertex_grads<MAXC, AtomicEmit<Env>>(s, t, acc, ij_b, colors_b, uv_b, shade_b, AtomicEmit<Env>());
        return;
    }
    float dadx[MAXC], dady[MAXC];
    for (int q = 0; q < C; q++) {
        const float a0 = s.colors[(size_t)t.vid[0] * C + q], a1 = s.colors[(size_t)t.vid[1] * C + q],
                    a2 = s.colors[(size_t)t.vid[2] * C + q];
        // (fp64: three terms of size |colour| / area that cancel - a sliver would lose every digit in fp32)
        dadx[q] = (float)(t.gx[0] * (double)a0 + t.gx[1] * (double)a1 + t.gx[2] * (double)a2);
        dady[q] = (float)(t.gy[0] * (double)a0 + t.gy[1] * (double)a1 + t.gy[2] * (double)a2);
    }
    float gij[3][2] = {{0.0f, 0.0f}, {0.0f, 0.0f}, {0.0f, 0.0f}};
    float gcol[3][MAXC];
    for (int q = 0; q < C; q++) gcol[0][q] = gcol[1][q] = gcol[2][q] = 0.0f;
    for (;;) {
        if (w == 0u) {
            if (own_words == 0u) break;
            p = lowest_bit(own_words);
            own_words &= own_words - 1;
            w = mine[p];
        }
        const int px = p * 32 + lowest_bit(w);
        w &= w - 1;
        double wd[3];
        tri_weights(s, t, tile.x0 + (px & (TS - 1)), tile.y0 + (px >> 4), 0.0, wd);
        const float w0 = (float)wd[0], w1 = (float)wd[1], w2 = (float)wd[2];
        float dcdx = 0, dcdy = 0;
        for (int q = 0; q < C; q++) {
            const float g = fetch.g(px, q);
            dcdx += g * dadx[q];
            dcdy += g * dady[q];
            gcol[0][q] += g * w0;
            gcol[1][q] += g * w1;
            gcol[2][q] += g * w2;
        }
        gij[0][0] -= w0 * dcdx; gij[0][1] -= w0 * dcdy;
        gij[1][0] -= w1 * dcdx; gij[1][1] -= w1 * dcdy;
        gij[2][0] -= w2 * dcdx; gij[2][1] -= w2 * dcdy;
    }
    for (int i = 0; i < 3; i++) {  // same scatter as flush_vertex_grads, interpolated branch
        Env::atomic_add(ij_b + 2 * (size_t)t.vid[i], gij[i][0]);
        Env::atomic_add(ij_b + 2 * (size_t)t.vid[i] + 1, gij[i][1]);
        for (int q = 0; q < C; q++) Env::atomic_add(colors_b + (size_t)t.vid[i] * C + q, gcol[i][q]);
    }
}

// One thread per sorted silhouette edge: turn the accumulated plane adjoints into vertex adjoints.
// DR.h:1758-1773 / 2045-2060 followed by get_edge_stencil_equations_B DR.h:1462-1539.
template <class Env>
DEODR_HD void finalize_edge(const SceneView &s, int edge_id, double sigma, const double *acc, float *ij_b,
                            float *colors_b, float *uv_b, float *shade_b, float *depths_b = nullptr) {
    const int C = s.nb_colors;
    int k = edge_id / 3, n = edge_id - 3 * k;
    uint32_t vid[2], uvid[2];
    double V[2][2], Zv[2];
    for (int i = 0; i < 2; i++) {
        int loc = edge_vertex(n, i);
        vid[i] = s.faces[3 * k + loc];
        uvid[i] = s.faces_uv[3 * k + loc];
        V[i][0] = s.ij[2 * (size_t)vid[i]];
        V[i][1] = s.ij[2 * (size_t)vid[i] + 1];
        Zv[i] = s.depths[vid[i]];
    }
    remove_offset(V, 2, pixel_offset(s));
    EdgeGeom g;
    double E[9], Einv[9], nt[3];
    edge_geom(V, Zv, s.height, sigma, s.clockwise != 0, false, &g, E, Einv, nt);
    const bool textured = s.textured[k] && s.shaded[k];
    double Einv_B[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int j = 0; j < 3; j++) Einv_B[6 + j] += acc[j] * (1.0 / sigma);  // T = (row 2 of Einv) / sigma
    if (s.perspective_correct) {  // layout of edge_acc_stride_persp: b_q = (row q of Einv) . (x, y, 1)
        for (int q = 0; q < 2; q++) {
            for (int j = 0; j < 3; j++) Einv_B[3 * q + j] += acc[3 + 3 * q + j];
            if (depths_b) Env::atomic_add(depths_b + vid[q], (float)acc[9 + q]);
            if (textured) {
                Env::atomic_add(uv_b + 2 * (size_t)uvid[q], (float)acc[11 + 3 * q]);
                Env::atomic_add(uv_b + 2 * (size_t)uvid[q] + 1, (float)acc[12 + 3 * q]);
                Env::atomic_add(shade_b + vid[q], (float)acc[13 + 3 * q]);
            } else {
                for (int c = 0; c < C; c++) Env::atomic_add(colors_b + (size_t)vid[q] * C + c, (float)acc[11 + q * C + c]);
            }
        }
    } else if (textured) {
        for (int q = 0; q < 2; q++) {  // edge vertex q
            double sh_b = 0, u_b = 0, v_b = 0;
            double shade_q = (double)s.shade[vid[q]];
            double uq = s.uv[2 * (size_t)uvid[q]], vq = s.uv[2 * (size_t)uvid[q] + 1];
            for (int j = 0; j < 3; j++) {
                sh_b += acc[3 + j] * Einv[3 * q + j];
                u_b += acc[6 + j] * Einv[3 * q + j];
                v_b += acc[9 + j] * Einv[3 * q + j];
                Einv_B[3 * q + j] += acc[3 + j] * shade_q + acc[6 + j] * uq + acc[9 + j] * vq;
            }
            Env::atomic_add(shade_b + vid[q], (float)sh_b);
            Env::atomic_add(uv_b + 2 * (size_t)uvid[q], (float)u_b);
            Env::atomic_add(uv_b + 2 * (size_t)uvid[q] + 1, (float)v_b);
        }
    } else {
        for (int q = 0; q < 2; q++)
            for (int c = 0; c < C; c++) {
                double col_b = 0, a = (double)s.colors[(size_t)vid[q] * C + c];
                for (int j = 0; j < 3; j++) {
                    col_b += acc[12 + 3 * c + j] * Einv[3 * q + j];
                    Einv_B[3 * q + j] += a * acc[12 + 3 * c + j];
                }
                Env::atomic_add(colors_b + (size_t)vid[q] * C + c, (float)col_b);
            }
    }
    double E_B[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    inv3x3_adjoint(Einv, Einv_B, E_B);
    double V_B[2][2] = {{E_B[0], E_B[3]}, {E_B[1], E_B[4]}};
    // normal n = nt * inv_norm, inv_norm = 1/|nt|  (DR.h:1508-1538)
    double n_B[2] = {E_B[2], E_B[5]};
    double inv_norm = nt[2];
    double nt_B[2] = {n_B[0] * inv_norm, n_B[1] * inv_norm};
    double inv_norm_B = n_B[0] * nt[0] + n_B[1] * nt[1];
    double nor_s_B = -inv_norm_B * (inv_norm * inv_norm) * 0.5 * inv_norm;
    nt_B[0] += 2 * nt[0] * nor_s_B;
    nt_B[1] += 2 * nt[1] * nor_s_B;
    if (s.clockwise) { V_B[0][1] += nt_B[0]; V_B[1][1] -= nt_B[0]; V_B[1][0] += nt_B[1]; V_B[0][0] -= nt_B[1]; }
    else             { V_B[0][1] -= nt_B[0]; V_B[1][1] += nt_B[0]; V_B[1][0] -= nt_B[1]; V_B[0][0] += nt_B[1]; }
    for (int i = 0; i < 2; i++) {
        Env::atomic_add(ij_b + 2 * (size_t)vid[i], (float)V_B[i][0]);
        Env::atomic_add(ij_b + 2 * (size_t)vid[i] + 1, (float)V_B[i][1]);
    }
}

}  // namespace deodr
