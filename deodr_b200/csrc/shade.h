// Per-pixel attribute math of the raster hot path (colours fp32, geometry / uv fp64): barycentrics of the owner
// triangle, Gouraud / textured-Gouraud colour, bilinear texture tap, silhouette-edge blend, and the per-pixel
// adjoint contributions.  Coverage and z are decided by rmath.h; nothing here changes WHICH pixel is drawn, so this
// file may use FMA freely.  __host__ __device__ for the same reason as rmath.h (tests/emul runs it on the CPU).
//
// Reference semantics restated here: DR.h:779-785 + 960-965 (interpolated), DR.h:1079-1087 + 1243-1251 (textured
// gouraud), DR.h:521-560 / 562-631 (bilinear sample and its adjoint), DR.h:1629-1644 / 1877-1902 (edge blend),
// DR.h:841-858 / 1138-1156 (triangle adjoint), expressed per pixel instead of per scan-line.
#pragma once

#include "rmath.h"

namespace deodr {

struct SceneView {
    const uint32_t *faces;             // [T,3]
    const uint32_t *faces_uv;          // [T,3]
    const double *ij;                  // [V,2]  col 0 = x (column), col 1 = y (row)
    const double *depths;              // [V]
    const double *uv;                  // [Nuv,2] texel coordinates (col 0 = texture column)
    const float *colors;               // [V,C]
    const float *shade;                // [V]
    const uint8_t *edgeflags;          // [T,3]
    const uint8_t *textured;           // [T]
    const uint8_t *shaded;             // [T]
    const float *texture;              // [Ht,Wt,C]
    const float *background_image;     // [H,W,C] or null
    const float *background_color;     // [C] or null
    int nb_triangles, nb_vertices, nb_uv;
    int height, width, nb_colors;
    int texture_height, texture_width;
    int clockwise, backface_culling, strict_edge, perspective_correct, integer_pixel_centers;
};

DEODR_HD double pixel_offset(const SceneView &s) { return s.integer_pixel_centers ? 0.0 : 0.5; }

// Classification of DR.h:2751-2779: depth-sum key, all-vertices-in-front test, signed area on the UN-offset ij.
struct TriClass {
    double sum_depth;
    bool area_positive;  // signedArea > 0 (0 when a vertex is behind the camera)
    bool drawn;          // rasterised by pass 1 (DR.h:2786, 2798, 2813)
    bool textured;       // textured && shaded
};

DEODR_HD void gather_tri(const SceneView &s, int k, uint32_t vid[3], double V[3][2], double Zv[3]) {
    for (int i = 0; i < 3; i++) {
        vid[i] = s.faces[3 * k + i];
        V[i][0] = s.ij[2 * (size_t)vid[i]];
        V[i][1] = s.ij[2 * (size_t)vid[i] + 1];
        Zv[i] = s.depths[vid[i]];
    }
}

DEODR_HD TriClass classify_tri(const SceneView &s, int k, const double V[3][2], const double Zv[3]) {
    TriClass c;
    c.sum_depth = DADD(DADD(DADD(0.0, Zv[0]), Zv[1]), Zv[2]);
    bool in_front = !(Zv[0] < 0) && !(Zv[1] < 0) && !(Zv[2] < 0);
    c.area_positive = in_front && (signed_area(V, s.clockwise != 0) > 0);
    c.textured = s.textured[k] && s.shaded[k];
    c.drawn = (c.area_positive || !s.backface_culling) && (c.textured || !s.textured[k]);
    return c;
}

DEODR_HD void remove_offset(double V[][2], int n, double off) {
    for (int i = 0; i < n; i++) { V[i][0] = DSUB(V[i][0], off); V[i][1] = DSUB(V[i][1], off); }
}

// Vertex pair of silhouette edge n of a face: (1,0), (2,1), (0,2)  (DR.h:2822)
DEODR_HD int edge_vertex(int n, int i) { return i == 0 ? (n + 1) % 3 : n; }

// ------------------------------------------------------------------------------------------------ barycentrics

struct Bary {
    double b[3];        // barycentric coordinates of the pixel centre
    double gx[3], gy[3];  // d b / d x, d b / d y
};

// Barycentrics in the frame of vertex 0 (well conditioned for small triangles far from the origin).
DEODR_HD void tri_bary(const double V[3][2], int x, int y, Bary *o) {
    double e1x = V[1][0] - V[0][0], e1y = V[1][1] - V[0][1];
    double e2x = V[2][0] - V[0][0], e2y = V[2][1] - V[0][1];
    double px = (double)x - V[0][0], py = (double)y - V[0][1];
    double inv = 1.0 / (e1x * e2y - e2x * e1y);
    o->gx[1] = e2y * inv;  o->gy[1] = -e2x * inv;
    o->gx[2] = -e1y * inv; o->gy[2] = e1x * inv;
    o->gx[0] = -(o->gx[1] + o->gx[2]);
    o->gy[0] = -(o->gy[1] + o->gy[2]);
    o->b[1] = px * o->gx[1] + py * o->gy[1];
    o->b[2] = px * o->gx[2] + py * o->gy[2];
    o->b[0] = 1.0 - o->b[1] - o->b[2];
}

// ------------------------------------------------------------------------------------------------------ texture

struct Tap {
    int i00, i10, i01, i11;  // texel offsets, already multiplied by C
    float e0, e1;
    bool out0, out1;
};

// DR.h:527-556: clamp-to-edge bilinear tap at texel coordinate (u = column, v = row)
DEODR_HD Tap texture_tap(double u, double v, int tex_w, int tex_h, int C) {
    Tap t;
    double fu = floor(u), fv = floor(v);
    int f0 = (int)fu, f1 = (int)fv;
    double e0 = u - fu, e1 = v - fv;
    t.out0 = t.out1 = false;
    if (f0 < 0) { t.out0 = true; f0 = 0; e0 = 0; }
    if (f0 > tex_w - 2) { t.out0 = true; f0 = tex_w - 2; e0 = 1; }
    if (f1 < 0) { t.out1 = true; f1 = 0; e1 = 0; }
    if (f1 > tex_h - 2) { t.out1 = true; f1 = tex_h - 2; e1 = 1; }
    t.i00 = C * (f0 + tex_w * f1);
    t.i10 = t.i00 + C;
    t.i01 = C * (f0 + tex_w * (f1 + 1));
    t.i11 = t.i01 + C;
    t.e0 = (float)e0;
    t.e1 = (float)e1;
    return t;
}

DEODR_HD float texture_fetch(const Tap &t, const float *tex, int k) {
    float top = (1.0f - t.e0) * tex[t.i00 + k] + t.e0 * tex[t.i10 + k];
    float bot = (1.0f - t.e0) * tex[t.i01 + k] + t.e0 * tex[t.i11 + k];
    return top * (1.0f - t.e1) + bot * t.e1;
}

// adjoint of texture_fetch w.r.t. (u, v): accumulates into e_B (DR.h:609-619); the caller applies the clamp masks
DEODR_HD void texture_fetch_duv(const Tap &t, const float *tex, int k, float a_B, float *e0_B, float *e1_B) {
    float top = (1.0f - t.e0) * tex[t.i00 + k] + t.e0 * tex[t.i10 + k];
    float bot = (1.0f - t.e0) * tex[t.i01 + k] + t.e0 * tex[t.i11 + k];
    *e1_B += a_B * (bot - top);
    *e0_B += a_B * (1.0f - t.e1) * (tex[t.i10 + k] - tex[t.i00 + k]) + a_B * t.e1 * (tex[t.i11 + k] - tex[t.i01 + k]);
}

// -------------------------------------------------------------------------------------------- owner-triangle data

// Per-triangle constants of the attribute interpolation: gathered once per triangle (once per pixel in the
// pixel-parallel kernels, once per triangle in the triangle-parallel adjoint).
struct TriAttr {
    uint32_t vid[3], uvid[3];
    double x0, y0;        // vertex 0, pixel-centre offset removed: barycentrics are evaluated in its frame
    double gx[3], gy[3];  // d b_i / dx, d b_i / dy
    double inv_z[3];      // 1 / depth of the vertices (perspective_correct only)
    bool textured;
};

// 1/d for the barycentric set-up (colour path only: nothing exact depends on it).  An fp64 division costs ~40 issue
// slots; fp32 reciprocal + two Newton steps gives ~1e-15 relative error in 8.
DEODR_HD double attr_recip(double d) {
#if defined(__CUDA_ARCH__)
    double r = (double)__frcp_rn((float)d);
    r = r * (2.0 - d * r);
    r = r * (2.0 - d * r);
    return r;
#else
    return 1.0 / d;
#endif
}

DEODR_HD void tri_attr(const SceneView &s, int k, TriAttr *t) {
    double V[3][2];
    for (int i = 0; i < 3; i++) {
        t->vid[i] = s.faces[3 * k + i];
        V[i][0] = s.ij[2 * (size_t)t->vid[i]];
        V[i][1] = s.ij[2 * (size_t)t->vid[i] + 1];
    }
    remove_offset(V, 3, pixel_offset(s));
    const double e1x = V[1][0] - V[0][0], e1y = V[1][1] - V[0][1];
    const double e2x = V[2][0] - V[0][0], e2y = V[2][1] - V[0][1];
    const double inv = attr_recip(e1x * e2y - e2x * e1y);
    t->x0 = V[0][0];
    t->y0 = V[0][1];
    t->gx[1] = e2y * inv;  t->gy[1] = -e2x * inv;
    t->gx[2] = -e1y * inv; t->gy[2] = e1x * inv;
    t->gx[0] = -(t->gx[1] + t->gx[2]);
    t->gy[0] = -(t->gy[1] + t->gy[2]);
    // (`s.texture != nullptr` is how a kernel instance compiled for scenes WITHOUT textured triangles folds every
    // texture branch away: it nulls its copy of the pointer, see fix_scene_flags in kernels.cu)
    t->textured = s.texture != nullptr && s.textured[k] && s.shaded[k];
    if (t->textured)
        for (int i = 0; i < 3; i++) t->uvid[i] = s.faces_uv[3 * k + i];
    if (s.perspective_correct)
        for (int i = 0; i < 3; i++) t->inv_z[i] = 1.0 / s.depths[t->vid[i]];
}

// Interpolation weights of pixel (x, y): barycentrics in the frame of vertex 0 (well conditioned for small triangles
// far from the origin); times (1/z_i) * Z with perspective_correct (DR.h:943-955), Z = the pixel's z-buffer value.
DEODR_HD void tri_weights(const SceneView &s, const TriAttr &t, int x, int y, double Z, double w[3]) {
    const double px = (double)x - t.x0, py = (double)y - t.y0;
    w[1] = px * t.gx[1] + py * t.gy[1];
    w[2] = px * t.gx[2] + py * t.gy[2];
    w[0] = 1.0 - w[1] - w[2];
    if (s.perspective_correct)
        for (int i = 0; i < 3; i++) w[i] = w[i] * t.inv_z[i] * Z;
}

// What the adjoint needs from the evaluation of one pixel.
template <int MAXC>
struct PixelEval {
    float w[3];
    // textured path
    float L;
    Tap tap;
    float texval[MAXC];
};

// Colour of pixel (x, y) inside triangle `t` (DR.h:960-965 interpolated, DR.h:1243-1251 textured gouraud).
template <int MAXC>
DEODR_HD void pixel_colour(const SceneView &s, const TriAttr &t, int x, int y, double Z, PixelEval<MAXC> *e,
                           float *colour) {
    const int C = s.nb_colors;
    double wd[3];
    tri_weights(s, t, x, y, Z, wd);
    for (int i = 0; i < 3; i++) e->w[i] = (float)wd[i];
    if (t.textured) {
        double u = 0, v = 0;
        e->L = 0;
        for (int i = 0; i < 3; i++) {
            u += wd[i] * s.uv[2 * (size_t)t.uvid[i]];
            v += wd[i] * s.uv[2 * (size_t)t.uvid[i] + 1];
            e->L += e->w[i] * s.shade[t.vid[i]];
        }
        e->tap = texture_tap(u, v, s.texture_width, s.texture_height, C);
        for (int c = 0; c < C; c++) {
            e->texval[c] = texture_fetch(e->tap, s.texture, c);
            colour[c] = e->texval[c] * e->L;
        }
    } else {
        const float *a0 = s.colors + (size_t)t.vid[0] * C, *a1 = s.colors + (size_t)t.vid[1] * C,
                    *a2 = s.colors + (size_t)t.vid[2] * C;
        for (int c = 0; c < C; c++) colour[c] = e->w[0] * a0[c] + e->w[1] * a1[c] + e->w[2] * a2[c];
    }
}

// Gradients of one triangle's vertices, accumulated over its pixels before they are scattered.
template <int MAXC>
struct VertexGrads {
    float ij[3][2];
    float attr[3][MAXC];  // colours (interpolated triangles)
    float uv[3][2];       // textured triangles
    float shade[3];
};

template <int MAXC>
DEODR_HD void zero_vertex_grads(const SceneView &s, VertexGrads<MAXC> *a) {
    for (int i = 0; i < 3; i++) {
        a->ij[i][0] = a->ij[i][1] = 0.0f;
        a->uv[i][0] = a->uv[i][1] = 0.0f;
        a->shade[i] = 0.0f;
        for (int c = 0; c < s.nb_colors; c++) a->attr[i][c] = 0.0f;
    }
}

// Adjoint of pixel_colour for one pixel with colour adjoint g (closed form of DR.h:841-858 / 1138-1156):
//   attr_b[v]  += (d colour / d attr) g * b_v          ij_b[v][d] -= b_v * sum_c g_c * d colour_c / d x_d
// accumulated into `acc`; texel adjoints go straight to texture_b (summed, see INTEGRATION.md).
template <int MAXC, class Env>
DEODR_HD void pixel_adjoint_persp(const SceneView &s, const TriAttr &t, int x, int y, const float *g,
                                  VertexGrads<MAXC> *acc, float *depth_acc, float *texture_b);

// (depth_acc: [3] running depths_b of the vertices, perspective_correct only; kept out of VertexGrads so that the
// instances without perspective carry nothing more)
template <int MAXC, class Env>
DEODR_HD void pixel_adjoint(const SceneView &s, const TriAttr &t, int x, int y, const float *g, VertexGrads<MAXC> *acc,
                            float *texture_b, float *depth_acc = nullptr) {
    if (s.perspective_correct) {
        pixel_adjoint_persp<MAXC, Env>(s, t, x, y, g, acc, depth_acc, texture_b);
        return;
    }
    const int C = s.nb_colors;
    PixelEval<MAXC> e;
    float colour[MAXC];
    pixel_colour<MAXC>(s, t, x, y, 0.0, &e, colour);
    float dcdx = 0, dcdy = 0;  // sum_c g_c * d colour_c / dx, dy
    if (t.textured) {
        float L_B = 0, e0_B = 0, e1_B = 0;
        for (int c = 0; c < C; c++) {
            float A_B = g[c] * e.L;
            L_B += g[c] * e.texval[c];
            texture_fetch_duv(e.tap, s.texture, c, A_B, &e0_B, &e1_B);
            if (texture_b) {
                float w00 = (1.0f - e.tap.e0) * (1.0f - e.tap.e1), w10 = e.tap.e0 * (1.0f - e.tap.e1);
                float w01 = (1.0f - e.tap.e0) * e.tap.e1, w11 = e.tap.e0 * e.tap.e1;
                Env::atomic_add(texture_b + e.tap.i00 + c, w00 * A_B);
                Env::atomic_add(texture_b + e.tap.i10 + c, w10 * A_B);
                Env::atomic_add(texture_b + e.tap.i01 + c, w01 * A_B);
                Env::atomic_add(texture_b + e.tap.i11 + c, w11 * A_B);
            }
        }
        float U_B = e.tap.out0 ? 0.0f : e0_B, V_B = e.tap.out1 ? 0.0f : e1_B;
        // screen-space gradients of u, v, L: sums of three terms of size |attribute| / area that cancel - in fp64, or a
        // sliver triangle (area 1e-3 px^2) loses every digit of them
        double dudx = 0, dudy = 0, dvdx = 0, dvdy = 0, dLdx = 0, dLdy = 0;
        for (int i = 0; i < 3; i++) {
            const double gx = t.gx[i], gy = t.gy[i];
            const double ui = s.uv[2 * (size_t)t.uvid[i]], vi = s.uv[2 * (size_t)t.uvid[i] + 1];
            const double li = (double)s.shade[t.vid[i]];
            dudx += gx * ui; dudy += gy * ui; dvdx += gx * vi; dvdy += gy * vi; dLdx += gx * li; dLdy += gy * li;
            acc->uv[i][0] += U_B * e.w[i];
            acc->uv[i][1] += V_B * e.w[i];
            acc->shade[i] += L_B * e.w[i];
        }
        dcdx = (float)((double)U_B * dudx + (double)V_B * dvdx + (double)L_B * dLdx);
        dcdy = (float)((double)U_B * dudy + (double)V_B * dvdy + (double)L_B * dLdy);
    } else {
        const float *a0 = s.colors + (size_t)t.vid[0] * C, *a1 = s.colors + (size_t)t.vid[1] * C,
                    *a2 = s.colors + (size_t)t.vid[2] * C;
        double sx = 0, sy = 0;  // (fp64: the three terms cancel, see above)
        for (int c = 0; c < C; c++) {
            const double c0 = (double)a0[c], c1 = (double)a1[c], c2 = (double)a2[c];
            sx += (double)g[c] * (t.gx[0] * c0 + t.gx[1] * c1 + t.gx[2] * c2);
            sy += (double)g[c] * (t.gy[0] * c0 + t.gy[1] * c1 + t.gy[2] * c2);
            for (int i = 0; i < 3; i++) acc->attr[i][c] += g[c] * e.w[i];
        }
        dcdx = (float)sx;
        dcdy = (float)sy;
    }
    for (int i = 0; i < 3; i++) {
        acc->ij[i][0] -= e.w[i] * dcdx;
        acc->ij[i][1] -= e.w[i] * dcdy;
    }
}

// Perspective-correct form of pixel_adjoint (DESIGN.md section 4).  With the plain barycentrics b_i, q_i = 1/z_i,
// Z = 1 / sum_k b_k q_k and the weights w_i = b_i q_i Z, every attribute is a = sum_i w_i a_i, and for its adjoint a_B:
//   a_i_B += w_i a_B      s_i = sum_attributes a_B (a_i - a)      b_i_B = q_i Z s_i      depths_b_i += -w_i s_i / z_i
//   ij_b[v] -= b_v sum_j b_j_B grad b_j          (d b_j / d V_v = -b_v grad b_j: the PLAIN b_v, not w_v)
// Z is recomputed from b and q (one fp64 reciprocal) rather than read from the z-buffer: every adjoint kernel can do
// that, only the edge-tile kernel has the z-buffer at hand.  s_i and the screen-space sums are formed in fp64 (the
// cancellation of pixel_adjoint).
template <int MAXC, class Env>
DEODR_HD void pixel_adjoint_persp(const SceneView &s, const TriAttr &t, int x, int y, const float *g,
                                  VertexGrads<MAXC> *acc, float *depth_acc, float *texture_b) {
    const int C = s.nb_colors;
    const double px = (double)x - t.x0, py = (double)y - t.y0;
    double b[3], w[3], sd[3] = {0.0, 0.0, 0.0};
    b[1] = px * t.gx[1] + py * t.gy[1];
    b[2] = px * t.gx[2] + py * t.gy[2];
    b[0] = 1.0 - b[1] - b[2];
    const double Z = 1.0 / (b[0] * t.inv_z[0] + b[1] * t.inv_z[1] + b[2] * t.inv_z[2]);
    for (int i = 0; i < 3; i++) w[i] = b[i] * t.inv_z[i] * Z;
    if (t.textured) {
        double u = 0, v = 0, L = 0, ui[3], vi[3], li[3];
        for (int i = 0; i < 3; i++) {
            ui[i] = s.uv[2 * (size_t)t.uvid[i]];
            vi[i] = s.uv[2 * (size_t)t.uvid[i] + 1];
            li[i] = (double)s.shade[t.vid[i]];
            u += w[i] * ui[i];
            v += w[i] * vi[i];
            L += w[i] * li[i];
        }
        const Tap tap = texture_tap(u, v, s.texture_width, s.texture_height, C);
        float L_B = 0, e0_B = 0, e1_B = 0;
        for (int c = 0; c < C; c++) {
            const float A_B = g[c] * (float)L;
            L_B += g[c] * texture_fetch(tap, s.texture, c);
            texture_fetch_duv(tap, s.texture, c, A_B, &e0_B, &e1_B);
            if (texture_b) {
                float w00 = (1.0f - tap.e0) * (1.0f - tap.e1), w10 = tap.e0 * (1.0f - tap.e1);
                float w01 = (1.0f - tap.e0) * tap.e1, w11 = tap.e0 * tap.e1;
                Env::atomic_add(texture_b + tap.i00 + c, w00 * A_B);
                Env::atomic_add(texture_b + tap.i10 + c, w10 * A_B);
                Env::atomic_add(texture_b + tap.i01 + c, w01 * A_B);
                Env::atomic_add(texture_b + tap.i11 + c, w11 * A_B);
            }
        }
        const double U_B = tap.out0 ? 0.0 : (double)e0_B, V_B = tap.out1 ? 0.0 : (double)e1_B;
        for (int i = 0; i < 3; i++) {
            sd[i] = U_B * (ui[i] - u) + V_B * (vi[i] - v) + (double)L_B * (li[i] - L);
            acc->uv[i][0] += (float)(U_B * w[i]);
            acc->uv[i][1] += (float)(V_B * w[i]);
            acc->shade[i] += (float)((double)L_B * w[i]);
        }
    } else {
        for (int c = 0; c < C; c++) {
            const double a0 = (double)s.colors[(size_t)t.vid[0] * C + c], a1 = (double)s.colors[(size_t)t.vid[1] * C + c],
                         a2 = (double)s.colors[(size_t)t.vid[2] * C + c];
            const double a = w[0] * a0 + w[1] * a1 + w[2] * a2, gc = (double)g[c];
            sd[0] += gc * (a0 - a);
            sd[1] += gc * (a1 - a);
            sd[2] += gc * (a2 - a);
            for (int i = 0; i < 3; i++) acc->attr[i][c] += (float)(gc * w[i]);
        }
    }
    double dx = 0, dy = 0;  // sum_j b_j_B grad b_j
    for (int j = 0; j < 3; j++) {
        const double bj_B = t.inv_z[j] * Z * sd[j];
        dx += bj_B * t.gx[j];
        dy += bj_B * t.gy[j];
        depth_acc[j] -= (float)(w[j] * sd[j] * t.inv_z[j]);
    }
    for (int i = 0; i < 3; i++) {
        acc->ij[i][0] -= (float)(b[i] * dx);
        acc->ij[i][1] -= (float)(b[i] * dy);
    }
}

// Scatter of one triangle's accumulated vertex gradients; `emit.emit(ptr, value)` adds value to *ptr.  depths_b is only
// written by the perspective-correct instances.
template <int MAXC, class Emit>
DEODR_HD void flush_vertex_grads(const SceneView &s, const TriAttr &t, const VertexGrads<MAXC> &acc, float *ij_b,
                                 float *colors_b, float *uv_b, float *shade_b, const Emit &emit,
                                 const float *depth_acc = nullptr, float *depths_b = nullptr) {
    const int C = s.nb_colors;
    for (int i = 0; i < 3; i++) {
        emit.emit(ij_b + 2 * (size_t)t.vid[i], acc.ij[i][0]);
        emit.emit(ij_b + 2 * (size_t)t.vid[i] + 1, acc.ij[i][1]);
        if (s.perspective_correct && depths_b) emit.emit(depths_b + t.vid[i], depth_acc[i]);
        if (t.textured) {
            emit.emit(uv_b + 2 * (size_t)t.uvid[i], acc.uv[i][0]);
            emit.emit(uv_b + 2 * (size_t)t.uvid[i] + 1, acc.uv[i][1]);
            emit.emit(shade_b + t.vid[i], acc.shade[i]);
        } else {
            for (int c = 0; c < C; c++) emit.emit(colors_b + (size_t)t.vid[i] * C + c, acc.attr[i][c]);
        }
    }
}

// ------------------------------------------------------------------------------------------------ edge records

// Record of one silhouette edge: built once per forward pass (bin_edge), staged in shared memory by the tile kernels.
struct EdgeRec {
    EdgeGeom g;
    uint64_t key;     // depth_desc_key of the edge's triangle: ascending key = far to near (DR.h:2781)
    uint32_t vid[2], uvid[2];
    int32_t id;       // 3 * triangle + n: breaks the ties of the key
    int32_t slot;     // position in the view's unordered edge list (index of the record and of its accumulators)
    uint8_t textured;
    uint8_t has_col;  // col[][] holds the end-point colours (C <= 4): no gathers in the blend loop
    uint8_t pad[6];
    double inv_z[2];  // 1/z of the end points (perspective_correct only)
    float col[2][4];
};
static_assert(sizeof(EdgeRec) % 8 == 0, "EdgeRec is copied as 8-byte words");

// V receives the two end points with the pixel-centre offset removed (what the band's tile box is computed from).
DEODR_HD void edge_record(const SceneView &s, int edge_id, int slot, uint64_t key, double sigma, EdgeRec *r,
                          double V[2][2]) {
    int k = edge_id / 3, n = edge_id - 3 * k;
    double Zv[2];
    for (int i = 0; i < 2; i++) {
        int loc = edge_vertex(n, i);
        r->vid[i] = s.faces[3 * k + loc];
        r->uvid[i] = s.faces_uv[3 * k + loc];
        V[i][0] = s.ij[2 * (size_t)r->vid[i]];
        V[i][1] = s.ij[2 * (size_t)r->vid[i] + 1];
        Zv[i] = s.depths[r->vid[i]];
        r->inv_z[i] = 1.0 / Zv[i];
    }
    remove_offset(V, 2, pixel_offset(s));
    edge_geom(V, Zv, s.height, sigma, s.clockwise != 0, s.perspective_correct != 0, &r->g, nullptr, nullptr, nullptr);
    r->key = key;
    r->id = edge_id;
    r->slot = slot;
    r->textured = (uint8_t)(s.textured[k] && s.shaded[k]);
    r->has_col = (uint8_t)(s.nb_colors <= 4);
    for (int i = 0; i < 6; i++) r->pad[i] = 0;
    for (int i = 0; i < 2; i++)
        for (int c = 0; c < 4; c++) r->col[i][c] = c < s.nb_colors ? s.colors[(size_t)r->vid[i] * s.nb_colors + c] : 0.0f;
}

// What one edge contributes at one pixel of its band.
template <int MAXC>
struct EdgeHit {
    double T;        // transparency of the overdraw: image = T*image + (1-T)*A   (DR.h:1634-1641)
    double b[2];     // edge barycentrics of the pixel
    float w[2];      // attribute weights (b, or b/z*Z when perspective_correct)
    float A[MAXC];   // edge colour at the pixel
    // textured
    double u, v;
    float L;
    Tap tap;
    float texval[MAXC];
};

// Z of the edge at the pixel (DR.h:1631 / 1611-1612) - the exact quantity compared with the z-buffer.
DEODR_HD double edge_z(const EdgeRec &r, int x, int y, bool persp) {
    double z = plane_at(r.g.zp, plane_row(r.g.zp, y), x);
    return persp ? DDIV(1.0, z) : z;
}

template <int MAXC>
DEODR_HD void edge_hit(const SceneView &s, const EdgeRec &r, int x, int y, double Ze, EdgeHit<MAXC> *h) {
    const int C = s.nb_colors;
    const double *q = r.g.ineq;
    h->b[0] = q[0] * x + q[1] * y + q[2];
    h->b[1] = q[3] * x + q[4] * y + q[5];
    h->T = plane_at(q + 6, plane_row(q + 6, y), x);
    double wd[2] = {h->b[0], h->b[1]};
    if (s.perspective_correct) { wd[0] = wd[0] * r.inv_z[0] * Ze; wd[1] = wd[1] * r.inv_z[1] * Ze; }
    h->w[0] = (float)wd[0];
    h->w[1] = (float)wd[1];
    if (s.texture != nullptr && r.textured) {
        h->u = wd[0] * s.uv[2 * (size_t)r.uvid[0]] + wd[1] * s.uv[2 * (size_t)r.uvid[1]];
        h->v = wd[0] * s.uv[2 * (size_t)r.uvid[0] + 1] + wd[1] * s.uv[2 * (size_t)r.uvid[1] + 1];
        h->L = h->w[0] * s.shade[r.vid[0]] + h->w[1] * s.shade[r.vid[1]];
        h->tap = texture_tap(h->u, h->v, s.texture_width, s.texture_height, C);
        for (int c = 0; c < C; c++) {
            h->texval[c] = texture_fetch(h->tap, s.texture, c);
            h->A[c] = h->texval[c] * h->L;
        }
    } else {
        const float *a0 = r.has_col ? r.col[0] : s.colors + (size_t)r.vid[0] * C;
        const float *a1 = r.has_col ? r.col[1] : s.colors + (size_t)r.vid[1] * C;
        for (int c = 0; c < C; c++) h->A[c] = h->w[0] * a0[c] + h->w[1] * a1[c];
    }
}

// ------------------------------------------------------------------------------------ per-edge adjoint finalisation

// Layout of the per-edge fp64 accumulators filled by the backward tile kernel (one row per sorted edge):
//   [0..2]   transp_B : sum T_B * (x, y, 1)
//   [3..5]   L_B      : sum L_B * (x, y, 1)                 (textured)
//   [6..11]  UV_B     : sum UV_B[q] * (x, y, 1), q = 0, 1   (textured)
//   [12..]   A_B      : sum A_B[c] * (x, y, 1), c < C       (interpolated)
DEODR_HD int edge_acc_stride(int C) { return 12 + 3 * C; }

// Layout of the same accumulators in the perspective-correct instances: the attribute weights w_i = b_i q_i Ze are not
// planes over (x, y, 1) any more, so the rows hold the adjoints of the two barycentric planes and per-end-point sums.
//   [0..2]   transp_B : sum T_B * (x, y, 1)
//   [3..8]   b_B      : sum b_q_B * (x, y, 1), q = 0, 1
//   [9..10]  depths_b : sum -w_q s_q / z_q, q = 0, 1
//   [11..]   a_B      : sum w_q a_B: colours [q * C + c] (interpolated) or (u, v, L) [3 q + 0..2] (textured)
DEODR_HD int edge_acc_stride_persp(int C) { return 11 + (2 * C > 6 ? 2 * C : 6); }

// Adjoint of inv3x3 (DR.h:124-232): S_B += d(inv)/dS^T T_B, with Tinv = inv(S):  S_B = -Tinv^T T_B Tinv^T.
DEODR_HD void inv3x3_adjoint(const double *Tinv, const double *T_B, double *S_B) {
    double tmp[9];
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
            double a = 0;
            for (int k = 0; k < 3; k++) a += Tinv[3 * k + i] * T_B[3 * k + j];
            tmp[3 * i + j] = a;
        }
    for (int i = 0; i < 3; i++)
        for (int j = 0; j < 3; j++) {
            double a = 0;
            for (int k = 0; k < 3; k++) a += tmp[3 * i + k] * Tinv[3 * j + k];
            S_B[3 * i + j] -= a;
        }
}

}  // namespace deodr
