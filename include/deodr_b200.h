/*
 * deodr_b200 - C-ABI of the B200 (sm_100a) differentiable rasteriser.
 *
 * This is the drop-in boundary for the reference's only native entry points,
 *     void renderScene  (Scene, double* image, double* z_buffer, double sigma, bool antialiaseError,
 *                        double* obs, double* err_buffer)                C++/DifferentiableRenderer.h:2717
 *     void renderScene_B(Scene, double* image, double* z_buffer, double* image_b, double sigma, bool,
 *                        double* obs, double* err_buffer, double* err_buffer_b)   C++/DifferentiableRenderer.h:2903
 * which the reference reaches through its Cython shim (deodr/differentiable_renderer_cython.pyx:50 renderSceneCpp,
 * :206 renderSceneBCpp; extern block :11-45).  Plain pointers and sizes only; no torch / numpy types.
 *
 * Two levels:
 *   - deodr_b200_render_host / deodr_b200_render_b_host take the reference's own `struct Scene`
 *     (DifferentiableRenderer.h:56-90: HOST pointers, fp64) and have the reference semantics (image / z_buffer
 *     fully overwritten; gradients ACCUMULATED into scene.*_b; image_b scaled in place is NOT reproduced - it is
 *     left untouched).  Host<->device copies happen inside the call.
 *   - deodr_b200_render / deodr_b200_render_b work on DEVICE-resident buffers in the canonical layout
 *     (fp64 ij / depths / uv / z_buffer, fp32 colours / shade / texture / image / gradients, int32 face ids) on a
 *     caller-supplied CUDA stream; this is what the PyTorch surface uses.
 *
 * All functions return 0 on success or a DEODR_B200_E* code; deodr_b200_last_error() gives the message of the last
 * failure on the calling thread (the reference throws `const char*` instead: DifferentiableRenderer.h:2664-2715,
 * 810, 2924).
 */
#ifndef DEODR_B200_H
#define DEODR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
    DEODR_B200_OK = 0,
    DEODR_B200_EINVAL = 1,      /* null pointer / bad size / index out of range (checkSceneValid, DR.h:2664) */
    DEODR_B200_EUNSUPPORTED = 2,/* backward without backface_culling (DR.h:2924); backward with perspective_correct
                                   through any adjoint entry point but deodr_b200_render_b_views_depths (DR.h:810),
                                   and there together with antialiase_error */
    DEODR_B200_ECUDA = 3,       /* CUDA runtime failure */
    DEODR_B200_ENOMEM = 4,
    DEODR_B200_EREPLAN = 5      /* deferred mode only: a forward overflowed the lists its plan had reserved; the
                                   results of that pass are void, the plan has been rebuilt: run the pass again */
};

/* flags of the *_views entry points */
enum {
    DEODR_B200_ANTIALIASE_ERROR = 1, /* renderScene(..., antialiaseError = true): the silhouette edges overdraw the
                                        squared residual err_buffer instead of the image (DR.h:2066-2618, 2824-2837) */
    DEODR_B200_ERROR_ADJOINT_COMPLETE = 2, /* adjoint of the mode above WITHOUT the reference's dropped row term
                                        (DR.h:2577-2583 never propagates A0y_B): the mathematically complete gradient.
                                        Default (flag clear) = bug-compatible with the reference. */
    /* A forward pass in two calls (deodr_b200_render_views only), for callers that overlap a collective with it:
     * GEOMETRY enqueues the head of the pass - list reset, index check, binning (with DEODR_B200_GEOMETRY_Z=1 in the
     * environment also the z pass, unfused): kernels that read only faces, ij, depths and the flags - and returns;
     * RESUME, with the same arguments, enqueues the rest (edge records, z pass + shading, edge overdraw: the readers of
     * colours / uv / shade / texture).  Between the two the caller makes `stream`
     * wait for whatever produces the colours (cudaStreamWaitEvent on its communication stream's event): unlike the
     * colours-ready event below, that wait is an ordinary stream dependency, so both halves can be captured in CUDA
     * graphs of their own and replayed with the wait in between.  The verdict of the pass belongs to the RESUME call. */
    DEODR_B200_FORWARD_GEOMETRY = 4,
    DEODR_B200_FORWARD_RESUME = 8
};

/* Device-resident scene ("SceneView"): the fields of struct Scene (DR.h:56-90) in the canonical device layout. */
typedef struct DeodrSceneView {
    const uint32_t *faces;            /* [T,3] */
    const uint32_t *faces_uv;         /* [T,3] */
    const double *ij;                 /* [V,2] col 0 = x (image column), col 1 = y (image row) */
    const double *depths;             /* [V] */
    const double *uv;                 /* [Nuv,2] texel coordinates, col 0 = texture column */
    const float *colors;              /* [V,C] */
    const float *shade;               /* [V] */
    const uint8_t *edgeflags;         /* [T,3] */
    const uint8_t *textured;          /* [T] */
    const uint8_t *shaded;            /* [T] */
    const float *texture;             /* [Ht,Wt,C] */
    const float *background_image;    /* [H,W,C] or NULL */
    const float *background_color;    /* [C] (device) or NULL; exactly one of the two backgrounds is set */
    int32_t nb_triangles, nb_vertices, nb_uv;
    int32_t height, width, nb_colors;
    int32_t texture_height, texture_width;
    int32_t clockwise, backface_culling, strict_edge, perspective_correct, integer_pixel_centers;
} DeodrSceneView;

/* Device-resident gradient slots (scene.*_b of DR.h:82-86), fp32, ACCUMULATED into.  Any pointer may be NULL. */
typedef struct DeodrGrads {
    float *ij_b;       /* [V,2] */
    float *colors_b;   /* [V,C] */
    float *uv_b;       /* [Nuv,2] */
    float *shade_b;    /* [V] */
    float *texture_b;  /* [Ht,Wt,C]  (summed: the reference's `=` defect DR.h:621-624 is not reproduced) */
} DeodrGrads;

/* The fields of the reference's scene struct (DR.h:56-90) in the SAME ORDER, with HOST pointers.  NOT layout-compatible
 * with `struct Scene`: the reference's five `bool` members are int32_t here (a C ABI has no C++ bool), so offsets and
 * size differ - a caller fills the fields one by one (as the pyx does, pyx:117-171), it cannot pass its Scene through. */
typedef struct DeodrHostScene {
    const uint32_t *faces;
    const uint32_t *faces_uv;
    const double *depths;
    const double *uv;
    const double *ij;
    const double *shade;
    const double *colors;
    const uint8_t *edgeflags;
    const uint8_t *textured;
    const uint8_t *shaded;
    int32_t nb_triangles;
    int32_t nb_vertices;
    int32_t clockwise;
    int32_t backface_culling;
    int32_t nb_uv;
    int32_t height;
    int32_t width;
    int32_t nb_colors;
    const double *texture;
    int32_t texture_height;
    int32_t texture_width;
    const double *background_image;
    const double *background_color;
    double *uv_b;
    double *ij_b;
    double *shade_b;
    double *colors_b;
    double *texture_b;
    int32_t strict_edge;
    int32_t perspective_correct;
    int32_t integer_pixel_centers;
} DeodrHostScene;

/* Opaque per-device workspace.  It holds VIEW SLOTS: the forward pass of view i leaves in slot i the state its adjoint
 * pass replays (tile edge lists, row-span cache, exact-tie table, compact triangle lists) together with the PLAN of the
 * pass - the capacities reserved for every per-tile list, learnt from an earlier pass over a scene of the same shape.
 * deodr_b200_render / _render_b use slot 0; the *_views entry points use slots 0 .. n_views-1.
 * Not thread-safe: one workspace per host thread (the Python layer serialises its calls with a lock). */
typedef struct DeodrWorkspace DeodrWorkspace;

int deodr_b200_workspace_create(DeodrWorkspace **ws, int device);
void deodr_b200_workspace_destroy(DeodrWorkspace *ws);
/* bytes of device memory currently held by the workspace */
int64_t deodr_b200_workspace_bytes(const DeodrWorkspace *ws);
/* number of kernels launched by the library on behalf of this workspace since creation */
int64_t deodr_b200_workspace_launches(const DeodrWorkspace *ws);

/* Forward pass on device buffers (replaces renderScene, DR.h:2717, antialiaseError = false).
 *   image   [H,W,C] fp32, fully overwritten
 *   z_buffer[H,W]   fp64, fully overwritten (bit-identical to the reference; +inf = background)
 *   owner   [H,W]   int32, adjoint-owner triangle per pixel (-1 = background); state consumed by the backward pass
 *   face_id [H,W]   int32 or NULL: forward owner (lowest index at the minimum z), i.e. rint() of the reference's
 *                   render_deferred face-id channel
 * `stream` is a cudaStream_t.  The pass is enqueued without waiting for the device; before returning the call reads
 * the verdict word the binning kernels publish in pinned memory (they are the first kernels of the pass, the rest of
 * it is already queued behind them) and, if a list outgrew its plan, re-plans and runs the pass again - the caller
 * always gets a valid result.  The first pass over a new shape builds the plan (one count pass + one read-back). */
int deodr_b200_render(DeodrWorkspace *ws, const DeodrSceneView *scene, double sigma, float *image, double *z_buffer,
                      int32_t *owner, int32_t *face_id, void *stream);

/* Adjoint pass on device buffers (replaces renderScene_B, DR.h:2903, antialiaseError = false).
 * Must follow deodr_b200_render on the same workspace, scene and sigma, with the z_buffer / owner arrays that pass
 * wrote (checked: DEODR_B200_EINVAL otherwise).  image_b [H,W,C] fp32 is read-only.  Gradients are accumulated (+=)
 * into `grads`.  No host synchronisation. */
int deodr_b200_render_b(DeodrWorkspace *ws, const DeodrSceneView *scene, double sigma, const double *z_buffer,
                        const int32_t *owner, const float *image_b, const DeodrGrads *grads, void *stream);

/* ---- batch of views (SURVEY 8b/8e; the frames loop of deodr/mesh_fitter.py:511-549) ---------------------------
 * Per-view device framebuffers.  Forward outputs: image, z_buffer, owner (required), face_id, barycentric (optional);
 * antialiase_error mode: obs [H,W,C] in, err_buffer [H,W] out.  Adjoint inputs: image_b [H,W,C] (normal mode) or
 * err_buffer_b [H,W] + obs + the forward's image (antialiase_error mode). */
typedef struct DeodrViewIO {
    float *image;              /* [H,W,C] */
    double *z_buffer;          /* [H,W] */
    int32_t *owner;            /* [H,W] */
    int32_t *face_id;          /* [H,W] or NULL */
    float *barycentric;        /* [H,W,3] or NULL: interpolation weights of the forward owner's three vertices (0 on the
                                  background): with face_id, the G-buffer of Scene3D.render_deferred
                                  (deodr/differentiable_renderer.py:1053-1174) without its C = 14 interpolated channels */
    const float *obs;          /* [H,W,C] or NULL */
    float *err_buffer;         /* [H,W] or NULL */
    const float *image_b;      /* [H,W,C] or NULL */
    const float *err_buffer_b; /* [H,W] or NULL */
} DeodrViewIO;

/* Forward passes of n_views views (views[i] -> slot i), interleaved on a few internal streams forked from / joined
 * to `stream`.  Same verdict handling as deodr_b200_render, after ALL the views have been enqueued. */
int deodr_b200_render_views(DeodrWorkspace *ws, int n_views, const DeodrSceneView *views, const DeodrViewIO *io,
                            double sigma, int flags, void *stream);

/* Adjoint passes of the same views.  grads[i] may alias each other: gradients of the parameters the views share
 * (colors_b, uv_b, shade_b, texture_b) accumulate in place - the `+=` of deodr/mesh_fitter.py:518-527 - while each view
 * gets its own ij_b. */
int deodr_b200_render_b_views(DeodrWorkspace *ws, int n_views, const DeodrSceneView *views, const DeodrViewIO *io,
                              const DeodrGrads *grads, double sigma, int flags, void *stream);

/* Adjoint passes of the views, as deodr_b200_render_b_views, that also accept perspective_correct scenes and return
 * the gradient of the vertex depths: depths_b[i] is a device pointer to [V] fp32 of view i (or NULL), accumulated
 * into.  For views without perspective_correct the depths do not reach the image and depths_b[i] is left untouched.
 * With perspective_correct the interpolation weights depend on the depths; the z-buffer test only decides which
 * triangle or edge owns a pixel and has no adjoint.  DEODR_B200_ANTIALIASE_ERROR together with a perspective_correct
 * view is refused (DEODR_B200_EUNSUPPORTED). */
int deodr_b200_render_b_views_depths(DeodrWorkspace *ws, int n_views, const DeodrSceneView *views,
                                     const DeodrViewIO *io, const DeodrGrads *grads, float *const *depths_b,
                                     double sigma, int flags, void *stream);

/* Deferred mode (on = 1): the entry points never read the verdict themselves - nothing in them touches the host side
 * of the device, so a forward + adjoint sequence can be captured in a CUDA graph (they also behave this way whenever
 * `stream` is being captured).  The caller then asks deodr_b200_workspace_status() after synchronising: OK, or
 * DEODR_B200_EREPLAN when a pass overflowed its plan (its outputs are void - gradients were not accumulated -, the plan
 * has been rebuilt; re-capture and run again). */
int deodr_b200_workspace_set_deferred(DeodrWorkspace *ws, int on);
int deodr_b200_workspace_status(DeodrWorkspace *ws);

/* "Colours ready" event (a cudaEvent_t, or NULL): the NEXT forward call makes only the kernels that read the vertex
 * colours (k_shade, the silhouette-edge records) wait for it; the geometry half of the pass - binning and the z pass,
 * more than half of its duration - starts at once.  This is how the all-reduce of the shared colour gradient and the
 * optimiser update that follows it (on the caller's communication stream, which records the event) overlap the next
 * step instead of sitting between two steps (DESIGN.md section 8).  One-shot: consumed by that call. */
int deodr_b200_workspace_set_colors_ready(DeodrWorkspace *ws, void *event);

/* Stamp of the last forward pass that ran in slot `view` (0 = none yet): lets a caller that keeps several forward
 * results alive (autograd) detect that the slot has been reused before it runs the adjoint. */
int64_t deodr_b200_view_generation(const DeodrWorkspace *ws, int view);

/* Reference-shaped host entry points (fp64 host buffers in, fp64 host buffers out). */
int deodr_b200_render_host(DeodrWorkspace *ws, const DeodrHostScene *scene, double *image, double *z_buffer,
                           double sigma, int antialiase_error, const double *obs, double *err_buffer);
int deodr_b200_render_b_host(DeodrWorkspace *ws, const DeodrHostScene *scene, double *image, double *z_buffer,
                             double *image_b, double sigma, int antialiase_error, const double *obs,
                             double *err_buffer, double *err_buffer_b);

/* Zero-fills `n` host buffers (ptrs[i], bytes[i]) with the host path's copy threads: what Scene2D.clear_gradients
 * (deodr/differentiable_renderer.py:599-610, five numpy `fill(0)` calls = 30+ MB on a 1M-triangle scene) does before
 * every adjoint call, at memory speed instead of one core's. */
int deodr_b200_host_zero(DeodrWorkspace *ws, void *const *ptrs, const int64_t *bytes, int n);

/* Index-range validation of a device scene (checkSceneValid, DR.h:2703-2714); synchronises the stream. */
int deodr_b200_check_scene(DeodrWorkspace *ws, const DeodrSceneView *scene, void *stream);

/* ---- the steps either side of the raster (SURVEY 8f1 / 8f2), on device buffers ------------------------------- */

/* Pinhole camera with the reference's OpenCV-style distortion (deodr/differentiable_renderer.py:341-438):
 * extrinsic [3,4] row-major, intrinsic [3,3] row-major, distortion k1 k2 p1 p2 k3 (has_distortion = 0: ignored). */
typedef struct DeodrCamera {
    double extrinsic[12];
    double intrinsic[9];
    double distortion[5];
    int32_t has_distortion;
    int32_t pad;
} DeodrCamera;

/* Camera.project_points (differentiable_renderer.py:391-418): points [N,3] fp64 -> ij [N,2] (col 0 = x), depths [N]. */
int deodr_b200_project_points(const double *points, int n, const DeodrCamera *camera, double *ij, double *depths,
                              void *stream);
/* Camera.project_points_backward (:420-438): points_b [N,3] fp64 += J^T (ij_b, depths_b); ij_b fp32 [N,2] is the
 * rasteriser's gradient, depths_b fp64 [N] or NULL.  reference_transpose = 1 reproduces the reference's last line
 * `p_camera_b.dot(extrinsic[:3,:3].T)` (:438), which is the adjoint of world_to_camera only for a symmetric rotation
 * (INTEGRATION.md, defect #3); 0 multiplies by the rotation itself (matches finite differences). */
int deodr_b200_project_points_b(const double *points, int n, const DeodrCamera *camera, const float *ij_b,
                                const double *depths_b, double *points_b, int reference_transpose, void *stream);

/* Gouraud luminosity of Scene3D.compute_vertices_luminosity + _compute_vertices_colors_with_illumination (:814-833):
 *   luminosity[v] = max(0, -dot(normals[v], light_directional)) + ambient;  colors[v,c] = vertex_colors[v,c] * luminosity[v]
 * normals [V,3] fp64, vertex_colors [V,C] fp64 or NULL (then only the luminosity is written); outputs fp32 (the
 * rasteriser's attribute type), either may be NULL.  light_directional: three doubles in HOST memory, NULL = no
 * directional light. */
int deodr_b200_vertex_luminosity(const double *normals, const double *vertex_colors, int n_vertices, int nb_colors,
                                 const double *light_directional, double ambient, float *luminosity, float *colors,
                                 void *stream);
/* adjoint (:835-850) from colors_b [V,C] fp32 (and / or luminosity_b [V] fp32, added to it):
 * vertex_colors_b [V,C] = colors_b * luminosity (overwritten, as the reference assigns it), normals_b [V,3] overwritten,
 * light_b[4] (device, fp64) += (light_directional_b[3], light_ambient_b).  Any output may be NULL. */
int deodr_b200_vertex_luminosity_b(const double *normals, const double *vertex_colors, int n_vertices, int nb_colors,
                                   const double *light_directional, double ambient, const float *colors_b,
                                   const float *luminosity_b, double *normals_b, double *vertex_colors_b,
                                   double *light_b, void *stream);

/* Static adjacency of a triangulated mesh (device pointers; built once per mesh on the host, e.g. by
 * deodr_b200.mesh_ops.MeshTopology from the same arrays as TriMeshAdjacencies, deodr/triangulated_mesh.py:21-98). */
typedef struct DeodrMeshTopology {
    const uint32_t *faces;            /* [T,3] */
    const int32_t *faces_edges;       /* [T,3] unique-edge id of the face's edges (v0,v1), (v1,v2), (v2,v0) */
    const int32_t *edge_face_offset;  /* [E+1] CSR: faces incident to every unique edge ... */
    const int32_t *edge_face_index;   /* ... (length 3T) */
    const int32_t *vertex_face_offset;/* [V+1] CSR: faces incident to every vertex (ascending), with multiplicity ... */
    const int32_t *vertex_face_index; /* ... (length 3T) */
    int32_t nb_faces, nb_edges, nb_vertices, clockwise;
} DeodrMeshTopology;

/* TriMeshAdjacencies.edge_on_silhouette (triangulated_mesh.py:153-166): edgeflags[T,3] = "exactly one of the faces
 * that share the edge is visible", visibility from the 2D winding of ij [V,2] (exact: same products and difference as
 * np.cross).  face_visible [T] u8 is scratch / by-product. */
int deodr_b200_edge_on_silhouette(const DeodrMeshTopology *mesh, const double *ij, uint8_t *face_visible,
                                  uint8_t *edgeflags, void *stream);

/* compute_face_normals + compute_vertex_normals (triangulated_mesh.py:113-143): unit face normals [T,3] (sign by
 * `clockwise`), summed over the faces incident to each vertex and normalised -> vertex_normals [V,3]. */
int deodr_b200_vertex_normals(const DeodrMeshTopology *mesh, const double *vertices, double *face_normals,
                              double *vertex_normals, void *stream);
/* compute_vertex_normals_backward + compute_face_normals_backward (:145-151, :125-135): vertex_normals_b [V,3] ->
 * vertices_b [V,3] (accumulated, fp64 atomics).  vertex_scratch [V,3] fp64 is scratch. */
int deodr_b200_vertex_normals_b(const DeodrMeshTopology *mesh, const double *vertices, const double *vertex_normals_b,
                                double *vertex_scratch, double *vertices_b, void *stream);

/* Per-kernel device timing with CUDA events recorded on the launching stream (for bench.py's roofline).
 * enable: pre-creates `max_records` event pairs (0 disables and frees them).  Every instrumented launch group of the
 * following render / render_b calls then records one (phase, start, stop) triple until the pool is exhausted.
 * collect: synchronises the recorded events, writes up to `capacity` (phase, milliseconds) pairs in launch order,
 * resets the pool and returns the number of records written (negative on error). */
enum {
    DEODR_B200_PH_PLAN = 0,         /* plan building only: count-only binning pass + k_scan_tiles + read-back */
    DEODR_B200_PH_EDGE_BIN = 1,     /* k_bin_edges: stencil records of the silhouette edges + their tile lists */
    DEODR_B200_PH_BIN = 2,          /* memset + (index check) + k_bin: the single binning pass over the triangles */
    DEODR_B200_PH_EDGE_TILE_SORT = 3,/* k_sort_tile_edges: far-to-near order inside every tile */
    DEODR_B200_PH_TILE_Z = 4,       /* k_tile_z: z-buffer + owner ids */
    DEODR_B200_PH_SHADE = 5,        /* k_shade: colour of every pixel */
    DEODR_B200_PH_EDGE_FWD = 6,     /* k_edge_fwd: ordered silhouette-edge overdraw */
    DEODR_B200_PH_SMALL_BWD = 7,    /* k_small_tri_bwd: triangle-parallel interior adjoint */
    DEODR_B200_PH_INTERIOR_BWD = 8, /* k_interior_bwd: pixel-parallel interior adjoint (large triangles) */
    DEODR_B200_PH_EDGE_BWD = 9,     /* accumulator memset + k_raster_bwd: tiles with silhouette edges */
    DEODR_B200_PH_EDGE_FINALIZE = 10,/* k_finalize_edges */
    DEODR_B200_PH_COUNT = 11
};
int deodr_b200_timing_enable(DeodrWorkspace *ws, int max_records);
int deodr_b200_timing_collect(DeodrWorkspace *ws, int32_t *phase, float *ms, int capacity);
const char *deodr_b200_phase_name(int phase);

const char *deodr_b200_last_error(void);
const char *deodr_b200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* DEODR_B200_H */
