/*
 * TEST INFRASTRUCTURE ONLY - the perspective-correct adjoint of the CPU restatement ("port", oracle/deodr_oracle.c).
 *
 * The reference has no such adjoint: its _B rasterisers refuse perspective_correct (DR.h:808-811).  This file adds our
 * own fp64 one, deodr_oracle_render_b_depths, to the port: it includes the port's source unchanged (setup records,
 * row spans, texture taps, depth ordering and the inv3x3 / edge-stencil adjoints are shared) and is compiled into a
 * library of its own by tests/perspective_support.py, with the port's flags (-ffp-contract=off).
 * Nothing in the product (deodr_b200/) links, loads or calls it.
 */
#include "../../oracle/deodr_oracle.c"

/* ------------------------------------------------------------------------------ perspective-correct adjoint */
/*
 * Not in the reference (its _B rasterisers refuse perspective_correct, DR.h:808-811): our own adjoint, the per-pixel
 * formulas of DESIGN.md section 4 written out as plain loops.  For a pixel with plain barycentrics b_i, q_i = 1/z_i,
 * Z = 1 / sum_k b_k q_k (the forward's z) and weights w_i = b_i q_i Z, an attribute a = sum_i w_i a_i with adjoint a_B
 * gives  a_i_B += w_i a_B,  s_i = sum_attr a_B (a_i - a),  b_i_B = q_i Z s_i,  depths_b_i += -w_i s_i q_i.  The
 * barycentric adjoints then go to the vertices through the setup matrices (the same inv3x3 adjoints as above).
 * The z-buffer test only decides ownership and has no adjoint.
 */

/* Attribute adjoint of one pixel: colour adjoint col_B[C] of the attribute interpolated with weights w over nv end
 * points; accumulates the attribute gradients and returns s[nv].  A textured element also feeds texture_b. */
static void persp_attr_adjoint(const Ctx *c, int textured, int nv, const uint32_t *vid, const uint32_t *uvid,
                               const double *w, const double *col_B, double *A, double *A_B, double *s, double *depths_b,
                               const double *q) {
    const OracleScene *sc = c->sc;
    const int C = sc->nb_colors;
    for (int i = 0; i < nv; i++) s[i] = 0;
    if (textured) {
        double UV[2] = {0, 0}, L = 0, L_B = 0, UV_B[2] = {0, 0};
        for (int i = 0; i < nv; i++) {
            UV[0] += w[i] * sc->uv[uvid[i] * 2];
            UV[1] += w[i] * sc->uv[uvid[i] * 2 + 1];
            L += w[i] * sc->shade[vid[i]];
        }
        Tap tap = texture_tap(UV, c->tex_size[0], c->tex_size[1], C);
        texture_fetch(&tap, sc->texture, C, A);
        for (int k = 0; k < C; k++) { A_B[k] = col_B[k] * L; L_B += col_B[k] * A[k]; }
        texture_fetch_adj(&tap, sc->texture, sc->texture_b, C, A_B, UV_B);
        for (int i = 0; i < nv; i++) {
            sc->uv_b[uvid[i] * 2] += w[i] * UV_B[0];
            sc->uv_b[uvid[i] * 2 + 1] += w[i] * UV_B[1];
            sc->shade_b[vid[i]] += w[i] * L_B;
            s[i] = UV_B[0] * (sc->uv[uvid[i] * 2] - UV[0]) + UV_B[1] * (sc->uv[uvid[i] * 2 + 1] - UV[1]) +
                   L_B * (sc->shade[vid[i]] - L);
        }
    } else {
        for (int k = 0; k < C; k++) {
            double a = 0;
            for (int i = 0; i < nv; i++) a += w[i] * sc->colors[(size_t)vid[i] * C + k];
            for (int i = 0; i < nv; i++) {
                sc->colors_b[(size_t)vid[i] * C + k] += w[i] * col_B[k];
                s[i] += col_B[k] * (sc->colors[(size_t)vid[i] * C + k] - a);
            }
        }
    }
    for (int i = 0; i < nv; i++) depths_b[vid[i]] += -w[i] * s[i] * q[i];
}

/* colour of one element at a pixel (forward of persp_attr_adjoint) */
static void persp_colour(const Ctx *c, int textured, int nv, const uint32_t *vid, const uint32_t *uvid,
                         const double *w, double *A, double *col) {
    const OracleScene *sc = c->sc;
    const int C = sc->nb_colors;
    if (textured) {
        double UV[2] = {0, 0}, L = 0;
        for (int i = 0; i < nv; i++) {
            UV[0] += w[i] * sc->uv[uvid[i] * 2];
            UV[1] += w[i] * sc->uv[uvid[i] * 2 + 1];
            L += w[i] * sc->shade[vid[i]];
        }
        Tap tap = texture_tap(UV, c->tex_size[0], c->tex_size[1], C);
        texture_fetch(&tap, sc->texture, C, A);
        for (int k = 0; k < C; k++) col[k] = A[k] * L;
    } else {
        for (int k = 0; k < C; k++) {
            col[k] = 0;
            for (int i = 0; i < nv; i++) col[k] += w[i] * sc->colors[(size_t)vid[i] * C + k];
        }
    }
}

/* silhouette edge: un-blend + adjoint, same walk as edge_adjoint */
static void edge_adjoint_persp(const Ctx *c, double *image_b, int k, int n, double sigma, double off, double *depths_b) {
    const OracleScene *sc = c->sc;
    const int C = sc->nb_colors, W = sc->width;
    double V[2][2], Zv[3], V_B[2][2] = {{0, 0}, {0, 0}};
    uint32_t vid[2], uvid[2];
    EdgeRec r;
    r.planeA = (double *)calloc((size_t)3 * C, sizeof(double));
    double *col = (double *)calloc((size_t)C, sizeof(double)), *col_B = (double *)calloc((size_t)C, sizeof(double));
    double *A = (double *)calloc((size_t)C, sizeof(double)), *A_B = (double *)calloc((size_t)C, sizeof(double));
    edge_gather(sc, k, n, off, V, Zv, vid, uvid);
    const int textured = sc->textured[k] && sc->shaded[k];
    edge_planes(sc, V, Zv, vid, uvid, textured, sigma, &r);
    const double q[2] = {1 / Zv[0], 1 / Zv[1]};
    double bary_B[6] = {0}, transp_B[3] = {0};
    for (short y = (short)r.s.y_begin; y <= r.s.y_end; y++) {
        int xb, xe;
        edge_row_span(r.s.ineq, W, y, &xb, &xe);
        int idx = y * W + xb;
        for (short x = (short)xb; x <= xe; x++, idx++) {
            double Z = row_value(r.planeZ, y) + r.planeZ[0] * x;
            Z = 1 / Z;
            if (!(Z < c->z_buffer[idx])) continue;
            const double t[3] = {(double)x, (double)y, 1};
            double b[2], w[2], s[2];
            for (int i = 0; i < 2; i++) {
                b[i] = r.s.Einv[3 * i] * t[0] + r.s.Einv[3 * i + 1] * t[1] + r.s.Einv[3 * i + 2] * t[2];
                w[i] = b[i] * q[i] * Z;
            }
            double T = row_value(r.s.transp, y) + r.s.transp[0] * x, T_B = 0;
            double *px = c->image + (size_t)C * idx, *px_b = image_b + (size_t)C * idx;
            persp_colour(c, textured, 2, vid, uvid, w, A, col);
            for (int i = 0; i < C; i++) {
                T_B += -px_b[i] * col[i];
                col_B[i] = (1 - T) * px_b[i];
                px[i] = (px[i] - (1 - T) * col[i]) / T;
                T_B += px_b[i] * px[i];
                px_b[i] *= T;
            }
            persp_attr_adjoint(c, textured, 2, vid, uvid, w, col_B, A, A_B, s, depths_b, q);
            for (int i = 0; i < 2; i++)
                for (int j = 0; j < 3; j++) bary_B[3 * i + j] += q[i] * Z * s[i] * t[j];
            for (int j = 0; j < 3; j++) transp_B[j] += T_B * t[j];
        }
    }
    edge_setup_adj(&r.s, V_B, sigma, bary_B, transp_B, sc->clockwise);
    for (int i = 0; i < 2; i++)
        for (int j = 0; j < 2; j++) sc->ij_b[vid[i] * 2 + j] += V_B[i][j];
    free(r.planeA); free(col); free(col_B); free(A); free(A_B);
}

/* triangle: adjoint of the pixels it owns (`Z == z_buffer`, same walk as triangle_adjoint) */
static void triangle_adjoint_persp(const Ctx *c, double *image_b, int k, double off, double *depths_b) {
    const OracleScene *sc = c->sc;
    const int C = sc->nb_colors, W = sc->width, H = sc->height, strict = sc->strict_edge;
    const uint32_t *face = &sc->faces[3 * k], *fuv = &sc->faces_uv[3 * k];
    const int textured = sc->textured[k] && sc->shaded[k];
    if (sc->textured[k] && !textured) return;
    double V[3][2], Zv[3];
    gather_face(sc, k, off, V, Zv);
    TriSetup s;
    tri_setup(V, strict, &s);
    const double q[3] = {1 / Zv[0], 1 / Zv[1], 1 / Zv[2]};
    double planeZ[3], V_B[3][2] = {{0, 0}, {0, 0}, {0, 0}};
    vec_times_rows(3, q, s.Minv, planeZ);
    double *col_B = (double *)calloc((size_t)C, sizeof(double));
    double *A = (double *)calloc((size_t)C, sizeof(double)), *A_B = (double *)calloc((size_t)C, sizeof(double));
    for (int half = 0; half < 2; half++) {
        int y0 = s.y_begin[half], y1 = s.y_end[half];
        if (y0 < 0) y0 = 0;
        if (y1 > H - 1) y1 = H - 1;
        for (short y = (short)y0; y <= y1; y++) {
            short xb, xe;
            tri_row_span(&s, half, y, W, strict, &xb, &xe);
            int idx = y * W + xb;
            for (short x = xb; x <= xe; x++, idx++) {
                double Z = row_value(planeZ, y) + planeZ[0] * x;
                Z = 1 / Z;
                if (Z != c->z_buffer[idx]) continue;
                const double t[3] = {(double)x, (double)y, 1};
                double b[3], w[3], sv[3], gx = 0, gy = 0;
                for (int i = 0; i < 3; i++) {
                    b[i] = s.Minv[3 * i] * t[0] + s.Minv[3 * i + 1] * t[1] + s.Minv[3 * i + 2] * t[2];
                    w[i] = b[i] * q[i] * Z;
                }
                double *px_b = image_b + (size_t)C * idx;
                for (int i = 0; i < C; i++) col_B[i] = px_b[i];
                if (!textured)  /* the interpolated walk consumes the pixel's adjoint (DR.h:1024-1031) */
                    for (int i = 0; i < C; i++) px_b[i] = 0;
                persp_attr_adjoint(c, textured, 3, face, fuv, w, col_B, A, A_B, sv, depths_b, q);
                for (int j = 0; j < 3; j++) {  /* sum_j b_j_B grad b_j */
                    double bj_B = q[j] * Z * sv[j];
                    gx += bj_B * s.Minv[3 * j];
                    gy += bj_B * s.Minv[3 * j + 1];
                }
                for (int v = 0; v < 3; v++) { V_B[v][0] += -b[v] * gx; V_B[v][1] += -b[v] * gy; }
            }
        }
    }
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 2; j++) sc->ij_b[face[i] * 2 + j] += V_B[i][j];
    free(col_B); free(A); free(A_B);
}

/* Adjoint pass that also accepts perspective_correct scenes and accumulates the gradient of the vertex depths into
 * depths_b [V].  Without perspective_correct it is deodr_oracle_render_b (depths_b untouched).  Same walk as
 * deodr_oracle_render_b: edges in reverse depth order with un-blend, then triangles in reverse index order.
 * `image` and `image_b` are MUTATED. */
int deodr_oracle_render_b_depths(const OracleScene *sc, double *image, double *z_buffer, double *image_b, double sigma,
                                 double *depths_b) {
    if (!sc->perspective_correct) return deodr_oracle_render_b(sc, image, z_buffer, image_b, sigma, 0, NULL, NULL, NULL);
    if (check_scene(sc, 1)) return 1;
    if (!depths_b || !image_b) return fail("depths_b and image_b are needed");
    if (!sc->backface_culling) return fail("You have to use backface_culling true if you ant to compute gradients");
    const int T = sc->nb_triangles;
    Ctx c = {sc, image, z_buffer, {sc->texture_width, sc->texture_height}, NULL, NULL, NULL};
    DepthKey *keys = (DepthKey *)malloc(sizeof(DepthKey) * (size_t)(T > 0 ? T : 1));
    double *area = (double *)malloc(sizeof(double) * (size_t)(T > 0 ? T : 1));
    classify(sc, keys, area);
    const float off_f = sc->integer_pixel_centers ? 0 : 0.5;
    const double off = off_f;
    if (sigma > 0)
        for (int it = T - 1; it >= 0; it--) {
            int k = (int)keys[it].index;
            if (area[k] > 0)
                for (int n = 2; n >= 0; n--)
                    if (sc->edgeflags[n + k * 3]) edge_adjoint_persp(&c, image_b, k, n, sigma, off, depths_b);
        }
    for (int k = T - 1; k >= 0; k--)
        if (area[k] > 0) triangle_adjoint_persp(&c, image_b, k, off, depths_b);
    free(keys);
    free(area);
    return 0;
}
