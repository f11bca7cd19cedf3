// TEST INFRASTRUCTURE ONLY: the CPU emulation of the kernel phases (tests/emul/emul.cpp, included unchanged) with the
// entry point of the perspective-correct adjoint, emul_render_b_depths - the same contract as
// deodr_b200_render_b_views_depths for one view.  Compiled into a library of its own by tests/perspective_support.py.
#include "../emul/emul.cpp"

// The adjoint pass of raster_bwd (colour mode) with the gradient of the vertex depths: the same phase sequence as
// k_raster_bwd + k_interior_bwd + k_small_tri_bwd.  Perspective-correct views always take the triangle-parallel
// small-triangle adjoint (launch_bwd does the same), whatever emul_set_small_records asked for.
template <int MAXC>
static void raster_bwd_depths(const SceneView &s, EmulState &st, const double *z_buffer, const int *owner,
                              const float *image_b, const DeodrGrads &g, double *edge_acc, float *depths_b) {
    std::vector<PixelState<MAXC>> px(NT);
    std::vector<AdjointState<MAXC>> adj(NT);
    TileShared *sh = new TileShared;
    for (int tile_id = 0; tile_id < st.nt; tile_id++) {
        const Tile tile = tile_of(tile_id, st.tiles_x);
        auto inside = [&](int tid) { return tile.x0 + tid % TS < s.width && tile.y0 + tid / TS < s.height; };
        for (int tid = 0; tid < NT; tid++) {
            PixelState<MAXC> &p = px[tid];
            adj[tid].has_colour = false;
            p.z = std::numeric_limits<double>::infinity();
            p.own = p.bown = -1;
            if (!inside(tid)) continue;
            const size_t idx = (size_t)(tile.y0 + tid / TS) * s.width + tile.x0 + tid % TS;
            p.z = z_buffer[idx];
            int code = owner[idx];
            if (code <= -2) { p.own = st.tie_pairs[2 * (-2 - code)]; p.bown = st.tie_pairs[2 * (-2 - code) + 1]; }
            else p.own = p.bown = code;
            for (int k = 0; k < s.nb_colors; k++) adj[tid].g[k] = image_b[idx * s.nb_colors + k];
        }
        const int n_edge = st.E > 0 ? segment_size(st.edge_seg(), tile_id) : 0;
        if (n_edge > 0) {
            const int edge_base = st.edge_offset[tile_id];
            const bool single = n_edge <= EDGE_CHUNK;
            auto stage = [&](int base, int m) {
                for (int tid = 0; tid < NT; tid++)
                    phase_edge_setup(tid, NT, m, st.edge_refs.data() + edge_base + base, st.edge_recs.data(), sh);
                for (int tid = 0; tid < NT; tid++) phase_edge_spans(s, tid, NT, m, tile, 0, TS, sh);
            };
            for (int base = 0; base < n_edge; base += EDGE_CHUNK) {  // forward replay, far to near
                const int m = std::min(EDGE_CHUNK, n_edge - base);
                stage(base, m);
                for (int tid = 0; tid < NT; tid++) {
                    if (!inside(tid)) continue;
                    const int x = tile.x0 + tid % TS, y = tile.y0 + tid / TS;
                    phase_edge_replay<MAXC>(s, x, y, tid / TS, m, sh, px[tid], &adj[tid]);
                    if (single && adj[tid].has_colour)
                        phase_edge_adjoint<MAXC, HostEnv>(s, x, y, tid / TS, m, sh, px[tid], &adj[tid], edge_acc, g.texture_b);
                }
            }
            if (!single) {  // reverse sweep, chunks in reverse order
                const int last = ((n_edge - 1) / EDGE_CHUNK) * EDGE_CHUNK;
                for (int base = last; base >= 0; base -= EDGE_CHUNK) {
                    const int m = std::min(EDGE_CHUNK, n_edge - base);
                    stage(base, m);
                    for (int tid = 0; tid < NT; tid++) {
                        if (!inside(tid) || !adj[tid].has_colour) continue;
                        phase_edge_adjoint<MAXC, HostEnv>(s, tile.x0 + tid % TS, tile.y0 + tid / TS, tid / TS, m, sh,
                                                          px[tid], &adj[tid], edge_acc, g.texture_b);
                    }
                }
            }
        }
        for (int tid = 0; tid < NT; tid++) {  // pixel-parallel interior adjoint
            if (!inside(tid) || px[tid].bown < 0) continue;
            if (n_edge == 0 && (px[tid].bown & SMALL_FLAG)) continue;
            phase_interior_adjoint<MAXC, HostEnv>(s, tile.x0 + tid % TS, tile.y0 + tid / TS, px[tid], adj[tid].g,
                                                  g.ij_b, g.colors_b, g.uv_b, g.shade_b, g.texture_b, HostEnv(),
                                                  depths_b);
        }
    }
    delete sh;
    const int *edge_count = st.E > 0 ? st.edge_cursor.data() : nullptr;
    const bool by_record = g_small_records && !s.perspective_correct;
    if (by_record) {  // k_small_rec_bwd (views without perspective_correct only)
        for (int tile_id = 0; tile_id < st.nt; tile_id++) {
            if (edge_count && edge_count[tile_id] > 0) continue;
            const Tile tile = tile_of(tile_id, st.tiles_x);
            const GlobalTileFetch fetch{owner, image_b, tile, s.width, s.height, s.nb_colors};
            const int n = segment_size(st.small_seg(), tile_id);
            for (int i = 0; i < n; i++)
                small_record_adjoint<MAXC, HostEnv>(s, st.small_recs[st.small_offset[tile_id] + i], tile, fetch,
                                                    st.tie_pairs.data(), g.ij_b, g.colors_b, g.uv_b, g.shade_b, g.texture_b);
        }
        return;
    }
    for (int k : st.small_ids)  // k_small_tri_bwd
        small_triangle_adjoint<MAXC, HostEnv>(s, k, st.tiles_x, edge_count, owner, st.tie_pairs.data(), image_b, g.ij_b,
                                              g.colors_b, g.uv_b, g.shade_b, g.texture_b, depths_b);
}

extern "C" {

// Must follow emul_render on the same scene.  perspective_correct scenes are accepted and the gradient of the vertex
// depths is accumulated into depths_b [V] (left untouched without perspective_correct).
int emul_render_b_depths(const DeodrSceneView *scene, double sigma, const double *z_buffer, const int32_t *owner,
                         const float *image_b, const DeodrGrads *grads, float *depths_b) {
    SceneView s;
    memcpy(&s, scene, sizeof(s));
    EmulState &st = g_state;
    const int C = s.nb_colors;
    const int stride = s.perspective_correct ? edge_acc_stride_persp(C) : edge_acc_stride(C);
    if (!s.perspective_correct) depths_b = nullptr;
    std::vector<double> acc((size_t)std::max(st.E, 1) * stride, 0.0);
    if (C == 1) raster_bwd_depths<1>(s, st, z_buffer, owner, image_b, *grads, acc.data(), depths_b);
    else if (C <= 3) raster_bwd_depths<3>(s, st, z_buffer, owner, image_b, *grads, acc.data(), depths_b);
    else if (C <= 4) raster_bwd_depths<4>(s, st, z_buffer, owner, image_b, *grads, acc.data(), depths_b);
    else raster_bwd_depths<16>(s, st, z_buffer, owner, image_b, *grads, acc.data(), depths_b);
    for (int r = 0; r < st.E; r++)
        finalize_edge<HostEnv>(s, st.edge_ids[r], sigma, acc.data() + (size_t)r * stride, grads->ij_b, grads->colors_b,
                               grads->uv_b, grads->shade_b, depths_b);
    return 0;
}

}  // extern "C"
