/*
 * bihrt.h -- C ABI of libbihrt.so: B200-native (sm_100a) BIH build + ray traversal + ray/triangle
 * intersection, a drop-in for the hot path of rehakvoj1/BIH-GPU-Raytracer.
 *
 * The reference has no FFI/plugin interface: the path sits behind three C++ classes with
 * thrust-typed members (App, Renderer, GPUArrayManager).  The boundary kept here is the set of
 * entry points and their data contracts (SURVEY.md 8(b)); each export cites what it replaces.
 * R/ = BIH_Raytracer/BIH_Raytracer/ of the reference tree.
 *
 * Conventions
 *   - plain pointers and sizes only; every function returns BIHRT_OK (0) or a negative code and
 *     never exits the process (the reference prints and calls exit(99), R/src/Renderer.cpp:63-73);
 *     bihrt_last_error() gives the message of the last failure on that context.
 *   - pointer arguments marked "host or device" are classified with cudaPointerGetAttributes.
 *   - one context = one GPU, one stream; calls are asynchronous on that stream unless they return
 *     data to host memory.  One context per host thread.
 *   - there is NO CPU fallback: every compute entry point fails if no sm_100-class GPU is present.
 */
#ifndef BIHRT_H
#define BIHRT_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define BIHRT_API __attribute__((visibility("default")))
#else
#define BIHRT_API
#endif

#define BIHRT_VERSION 100

#define BIHRT_OK             0
#define BIHRT_ERR_INVALID   -1   /* bad argument */
#define BIHRT_ERR_CUDA      -2   /* CUDA runtime error (message has the CUDA string) */
#define BIHRT_ERR_NOMEM     -3   /* device or host allocation failed (reference: Allocate* -> false) */
#define BIHRT_ERR_STATE     -4   /* call order: no scene loaded / BIH not built */
#define BIHRT_ERR_IO        -5   /* OBJ file unreadable or malformed */
#define BIHRT_ERR_INTERNAL  -6   /* device-side watchdog tripped (never expected) */

typedef struct bihrt_ctx bihrt_ctx;

/* Run-time replacement of the compile-time macros in R/src/Constants.h:4-8. */
typedef struct bihrt_config {
    int32_t  device;        /* CUDA device ordinal */
    uint32_t flags;         /* reserved, 0 */
    int32_t  reserved[6];
} bihrt_config;

/* Camera, same four vectors as R/src/Camera.h:14-17; ray(u,v) = (origin,
 * lower_left + u*horizontal + v*vertical - origin), NOT normalised (R/src/Camera.cu:18-20). */
typedef struct bihrt_camera {
    float origin[3];
    float lower_left[3];
    float horizontal[3];
    float vertical[3];
} bihrt_camera;

/* Ray = origin + direction (R/src/Ray.h:19-20); invDir/sign are derived inside (R/src/Ray.cu:3-10). */
typedef struct bihrt_ray {
    float o[3];
    float d[3];
} bihrt_ray;

/* bihrt_render flags */
#define BIHRT_RENDER_JITTER   1u   /* jittered samples (reference behaviour); otherwise pixel centres */
#define BIHRT_RENDER_COUNTS   2u   /* framebuffer receives per-pixel hit counts instead of packed colours */

/* Reference view of a built BIH: arrays with the exact field meaning of the reference's device
 * arrays (SURVEY.md 2.3).  Caller allocates; any pointer may be NULL to skip that array.
 * Capacities: [n] for the per-triangle arrays, [nu] / [nu-1] for the per-cell / per-node ones
 * (allocating n entries for each is always enough). */
typedef struct bihrt_refview {
    int64_t   n;                    /* out: triangles */
    int64_t   nu;                   /* out: unique Morton cells = leaves (GetUniqueMCSize) */
    float     scene_lo[3];          /* out: AABBs::sceneBBoxLo, R/src/AABB.h:15 */
    float     scene_hi[3];          /* out: AABBs::sceneBBoxHi */
    uint32_t* morton_codes;         /* [n]    m_mortonCodes after the sort */
    uint32_t* tris_indexes;         /* [n]    m_trisIndexes: sorted slot -> input triangle */
    uint32_t* unique_morton_codes;  /* [nu]   m_uniqueMortonCodes */
    uint32_t* duplicates_cnts;      /* [nu]   m_duplicatesCnts */
    int32_t*  first_idxs;           /* [nu]   m_firstIdxs */
    float*    clip_planes;          /* [2*(nu-1)] TreeInternalNode::t_clipPlanes, R/src/Tree.cuh:17 */
    int32_t*  axis;                 /* [nu-1] t_axis */
    uint8_t*  is_leaf;              /* [2*(nu-1)] isLeaf */
    int32_t*  children;             /* [2*(nu-1)] children */
    int32_t*  parent;               /* [nu-1] parent (root: -1) */
    int32_t*  leaf_parents;         /* [nu]   m_leafParents */
} bihrt_refview;

typedef struct bihrt_build_info {
    int64_t n;                /* triangles */
    int64_t nu;               /* leaves */
    int64_t node_bytes;       /* compact nodes, 16 B each */
    int64_t tri_bytes;        /* leaf-ordered triangles, 48 B each */
    float   last_build_ms;    /* device time of the last bihrt_build (CUDA events) */
    int32_t sort_passes;
    int32_t reserved[6];
} bihrt_build_info;

/* ---- lifetime ------------------------------------------------------------------------------ */
BIHRT_API int         bihrt_version(void);
BIHRT_API int         bihrt_create(bihrt_ctx** out, const bihrt_config* cfg);   /* replaces Renderer::Init + GPUArrayManager ctor, R/src/Renderer.cpp:87-105 */
BIHRT_API void        bihrt_destroy(bihrt_ctx* ctx);
BIHRT_API const char* bihrt_last_error(const bihrt_ctx* ctx);                   /* replaces checkCudaErrors' stderr print */
/* Stream of the context.  A new context runs on its OWN private non-blocking stream.  bihrt_set_stream takes a
 * cudaStream_t with CUDA's own meaning -- NULL (0) is the legacy default stream, exactly what
 * torch.cuda.current_stream().cuda_stream is while torch runs on its default stream -- or BIHRT_STREAM_OWN to go back
 * to the private stream.  Work of a caller that runs on ANOTHER stream is not ordered with the library's: either hand
 * that stream to bihrt_set_stream, or order the two with events on the handle bihrt_get_stream returns (the Python
 * mirror does this for torch tensors). */
#define BIHRT_STREAM_OWN ((void*)(intptr_t)-1)
BIHRT_API int         bihrt_set_stream(bihrt_ctx* ctx, void* cuda_stream);
BIHRT_API int         bihrt_get_stream(bihrt_ctx* ctx, void** cuda_stream);     /* the cudaStream_t the context launches on */
BIHRT_API int         bihrt_sync(bihrt_ctx* ctx);                               /* replaces the cudaDeviceSynchronize after each step, R/src/Renderer.cpp:428-503 */
/* Options (INTEGRATION.md, "Options", lists them all; an unknown name is BIHRT_ERR_INVALID).  The two that change WHAT is built:
 *   "morton_bits" 30 (default): the reference's 10-bit grid per axis, R/src/Renderer.cpp:116-136 -- the parity path, bit-exact tree.
 *                 63: QUALITY MODE, not a parity path (SURVEY.md 8(f) f4): 21 bits per axis, ties broken by sorted position,
 *                 every subtree of at most "leaf_cap" (default 4, 1..64) triangles collapsed into one leaf.  Hits equal brute force
 *                 (including on axis-aligned geometry where the reference's strict comparisons lose hits); bihrt_refit and
 *                 bihrt_export_reference_view are not available.  A context that adopts a replicated BIH (bihrt_bih_adopt) must
 *                 have the builder's value; bihrt_bih_copy and bihrt_bih_import carry it over themselves. */
BIHRT_API int         bihrt_set_option(bihrt_ctx* ctx, const char* name, int64_t value);
BIHRT_API int         bihrt_get_stat(bihrt_ctx* ctx, const char* name, int64_t* value);   /* "kernel_launches": kernels of this library launched so far */

/* ---- scene load: App::LoadModels + GPUArrayManager::Allocate*, R/src/App.cpp:65-167,
 *      R/src/GPUArrayManager.cpp:7-91.  xyz9 = n x (v0,v1,v2) floats in model->mesh->face order,
 *      host or device; the library copies. ------------------------------------------------------ */
BIHRT_API int bihrt_scene_load_triangles(bihrt_ctx* ctx, const float* xyz9, int64_t n);
BIHRT_API int bihrt_scene_update_vertices(bihrt_ctx* ctx, const float* xyz9, int64_t n);  /* animation: same n, BIH becomes stale */
BIHRT_API int bihrt_scene_load_obj(bihrt_ctx* ctx, const char* path);          /* minimal Wavefront reader replacing Model(path), R/src/Model.cpp:10-29 */

/* ---- build: first half of Renderer::Render (Morton transform, sort, RLE, Launch_BuildTree,
 *      Launch_FindClipPlanes), R/src/Renderer.cpp:422-503.  No host sync inside. ------------------ */
BIHRT_API int bihrt_build(bihrt_ctx* ctx);
/* NOT a parity path (SURVEY.md 8(f) f3): after bihrt_scene_update_vertices keep the order, leaves and topology of the
 * last full build and recompute scene box, triangle records, children boxes and clip planes only (about half the time of
 * a build).  Every plane and box bounds its subtree of the moved vertices, but the tree is not the one the reference would
 * build for them.  What the queries give on it:
 *   - bihrt_closest_point and bihrt_winding_number prune with the children boxes: they equal brute force over the moved
 *     triangles on every refit tree (winding: the exact sum at beta = inf, the far-field walk otherwise).
 *   - Ray queries (trace, trace_any, intersect, the renders) walk with the parity tree's strict plane test.  They equal
 *     brute force unless the motion flattens geometry onto an axis-aligned plane that the old topology splits across: a
 *     node whose two sides now meet in that plane gets clip0 == clip1, the far side's ray interval is a single point, and
 *     the strict test drops it.  There the parity walk's flat-geometry misses become frequent, and a ray that loses its
 *     nearest triangle may report a farther one.  Measured on a displaced sphere of 18 432 triangles, 20 000 random rays
 *     (hits of brute force -> of the refit tree): y clamped to a floor at 0, 12 589 -> 10 267, 51 of them farther than the
 *     nearest; at y = 0.5, 11 099 -> 8 305 (276 farther); the whole mesh flattened onto x = 0.25, 12 076 -> 324.
 *     A full bihrt_build of the moved vertices finds every hit again: use it after such motions. */
BIHRT_API int bihrt_refit(bihrt_ctx* ctx);
BIHRT_API int bihrt_get_build_info(bihrt_ctx* ctx, bihrt_build_info* out);     /* synchronises */
BIHRT_API int bihrt_export_reference_view(bihrt_ctx* ctx, bihrt_refview* view); /* synchronises; see bihrt_refview */

/* ---- trace: Launch_cudaRender -> cudaRender -> TraverseTree, R/src/CUDAKernels.cu:227-447.
 *      Per ray: t in units of |d| (FLT_MAX on miss), slot = index into the Morton-sorted triangle
 *      order (the reference's HitRecord::triangleIdx, R/src/CUDAKernels.cu:215-221; -1 on miss),
 *      prim = input triangle index = tris_indexes[slot].  rays / outputs: host or device; any
 *      output may be NULL. ---------------------------------------------------------------------- */
BIHRT_API int bihrt_trace(bihrt_ctx* ctx, const bihrt_ray* rays, int64_t n, float* t, int32_t* slot, int32_t* prim);
/* Occlusion query (shadow rays): blocker[i] = slot of SOME triangle ray i hits with 0 < t < tmax, or -1 (host or
 * device).  The traversal is cut at tmax and ends at the first such hit, so blocker[i] >= 0 exactly when the closest
 * hit bihrt_trace reports has t < tmax; which blocker is found is unspecified.  With the shadow rays of
 * bihrt_secondary_rays (direction = light - origin) tmax = 1 asks "is the light hidden". */
BIHRT_API int bihrt_trace_any(bihrt_ctx* ctx, const bihrt_ray* rays, int64_t n, float tmax, int32_t* blocker);
/* ---- ray queries: rays with their own parametric interval, full hit records.
 *      A triangle is ACCEPTED when max(tmin, 0) < t < min(tmax, FLT_MAX), both comparisons strict (like bihrt_trace's
 *      0 < t < best): a negative tmin acts as 0, a tmax of FLT_MAX or more (+inf included) as FLT_MAX.  A ray with
 *      !(max(tmin, 0) < tmax) -- a NaN in either bound included -- misses without being traced.
 *      flags 0 (closest hit): the accepted triangle with the smallest t that bihrt_trace's walk reaches.  The walk is
 *        bihrt_trace's (the reference's strict plane test with the scene-box entry, far-leaf-first order, and its misses on
 *        axis-aligned flat geometry); the interval only narrows it.  So with tmin = 0 and tmax >= FLT_MAX, t / slot / prim
 *        are bihrt_trace's bit for bit, and with tmin = 0 a ray hits exactly when bihrt_trace's t < tmax, with the same
 *        triangle.  Peeling (next query with tmin = the last t) visits a ray's distinct hit distances front to back.
 *      BIHRT_INTERSECT_ANY (occlusion): the walk ends with the leaf in which a triangle is first accepted.  A ray hits exactly when the
 *        closest-hit query with the same interval hits; the record describes the triangle found (which one: unspecified).
 *      Record per ray (every output pointer of bihrt_hits may be NULL; each one host or device):
 *        t     Moller-Trumbore t, bit-identical to what bihrt_trace reports for that triangle;
 *        u, v  the reference's Moller-Trumbore u, v (R/src/CUDAKernels.cu:35,42, same IEEE binary32 operations): the hit
 *              point is ~ (1-u-v) v0 + u v1 + v v2 in the triangle's input vertex order;
 *        slot, prim  as bihrt_trace;
 *        ng    geometric normal e1 x e2, e1 = v1 - v0, e2 = v2 - v0, NOT normalised, binary32 with every product rounded and
 *              no FMA: (e1y*e2z - e1z*e2y, e1z*e2x - e1x*e2z, e1x*e2y - e1y*e2x), 3 floats per ray.  ng keeps the input
 *              winding, so it tells the side that was hit: dot(d, ng) < 0 on a front face, > 0 on a back face (the
 *              convention Embree uses).  Without BIHRT_INTERSECT_TWO_SIDED hits are front faces only (det >= 1e-6, as in
 *              the reference), so dot(d, ng) < 0.
 *        miss: t = FLT_MAX, slot = prim = -1, u = v = 0, ng = (0, 0, 0).
 *      BIHRT_INTERSECT_TWO_SIDED (combines with BIHRT_INTERSECT_ANY): back faces count too.  A triangle is a candidate when
 *        !(|det| < 1e-6) instead of !(det < 1e-6) -- Moller-Trumbore's non-culling branch -- and everything after that test is
 *        the same arithmetic (1 / det rounds symmetrically), so u, v, t of a front face are computed bit for bit as without the
 *        flag.  The walk is unchanged (strict plane test, far-leaf-first order, the flat-geometry misses of the parity tree,
 *        the quality tree's rules); only more triangles are accepted.  Hence:
 *          - every ray the one-sided query hits, the two-sided query hits, with t <= the one-sided t;
 *          - where the two-sided record's triangle is front-facing, the record equals the one-sided one (slot and prim
 *            may differ only between triangles at exactly the same t);
 *          - on quality-mode trees, hits equal two-sided brute force over the interval, except where triangles of
 *            different leaves lie in one plane (coincident surfaces, such as the bottom face of a box resting on a floor,
 *            which only a two-sided query can hit from above): their t differ only by rounding, and the walk may report
 *            the one whose t is an ulp larger.
 *        A ray from inside a closed mesh sees its inner (back) faces; peeling visits entry and exit hits in order.
 *      Quality-mode trees (morton_bits 63): same contract without the reference's quirks; hits equal brute force over the
 *      interval.  The option trace_sort_rays does not apply (rays are traced in list order).  rays: host or device; device
 *      rays must be 16-byte aligned (a ray is read as two 128-bit loads).  Host outputs: the call synchronises and leaves them
 *      untouched if the build's watchdog tripped; device outputs are written asynchronously on the context's stream.
 *      Errors: BIHRT_ERR_INVALID for unknown flag bits, rays == NULL with n > 0, out == NULL, n < 0, n >= 2^32 - 2^24 or
 *      misaligned device rays; BIHRT_ERR_STATE without a built BIH. ------------------------------------------------------ */
/* ray with its own parametric interval: 32 B, two 128-bit loads */
typedef struct bihrt_ray_interval { float o[3]; float tmin; float d[3]; float tmax; } bihrt_ray_interval;
/* outputs of bihrt_intersect: any pointer may be NULL; each one host or device */
typedef struct bihrt_hits {
    float*   t;     /* [n] */
    float*   u;     /* [n] barycentric weight of v1 */
    float*   v;     /* [n] barycentric weight of v2 */
    int32_t* slot;  /* [n] */
    int32_t* prim;  /* [n] */
    float*   ng;    /* [3n] geometric normal, xyz per ray */
} bihrt_hits;
#define BIHRT_INTERSECT_ANY 1u   /* occlusion: end at the first accepted triangle of the interval */
#define BIHRT_INTERSECT_TWO_SIDED 4u   /* back faces count too (|det| >= 1e-6); flag values 0, 1, 4 and 5 are valid */
BIHRT_API int bihrt_intersect(bihrt_ctx* ctx, const bihrt_ray_interval* rays, int64_t n, uint32_t flags, const bihrt_hits* out);
/* ---- multi-hit ray queries: the k nearest accepted triangles of each ray's interval, front to back, and the number of all
 *      of them (the ray's crossing count).
 *      Acceptance is bihrt_intersect's: max(tmin, 0) < t < min(tmax, FLT_MAX), both strict, and the det test of the flags;
 *      a ray with !(max(tmin, 0) < tmax), NaN bounds included, has no candidates and is not walked.
 *      flags 0: one-sided; BIHRT_INTERSECT_TWO_SIDED: back faces count too.  BIHRT_INTERSECT_ANY and every other bit:
 *        BIHRT_ERR_INVALID.
 *      The walk is bihrt_intersect's (scene-box entry; on parity trees the strict plane test, the children boxes with their
 *      margin and the far-leaf-first order, hence the same misses on axis-aligned flat geometry; on quality trees the closed
 *      tests).  Only the cut differs: once k triangles are held it is the t of the k-th of them, before that -- and always when
 *      total is asked for -- the interval's upper end.  The cut is CLOSED for ties: a node whose interval starts exactly at the
 *      k-th t is still visited, and a triangle at exactly that t with a smaller slot still enters.
 *      Result for ray i: the accepted triangles the walk reaches, ordered by (t, slot) ascending, ties to the smaller slot (the
 *      key t_bits << 32 | slot orders them exactly: every accepted t is > 0).  The first min(k, that many) go to rows i*k + 0,
 *      1, ... of the arrays of rec, each row a full bihrt_hits record (t, u, v, slot, prim, ng) computed after the walk from
 *      its slot with the walk's own arithmetic, so t, u, v are bit for bit what bihrt_intersect reports for that triangle.
 *      The rows after them hold the miss record (t = FLT_MAX, slot = prim = -1, u = v = 0, ng = 0).  count[i] is the number of
 *      rows written; total[i] the number of ALL accepted triangles the walk reaches over the whole interval (with
 *      BIHRT_INTERSECT_TWO_SIDED on a closed mesh its parity is an inside test).  Consequences:
 *        - k == 1: t, u, v and ng of the row are bihrt_intersect's record; slot and prim may differ only between triangles
 *          at exactly the same t, where this call takes the smaller slot;
 *        - quality-mode trees: the rows equal brute force over the interval, except the classes bihrt_intersect documents
 *          (DESIGN.md section 2, and the two-sided coplanar-leaves note above);
 *        - the rows at k are the first k rows at any larger k;
 *        - where total <= k, the distinct t of the rows are exactly the sequence the peeling loop (bihrt_intersect again with
 *          tmin = the last t) visits -- and unlike peeling the rows keep triangles that share a t.  With
 *          BIHRT_INTERSECT_TWO_SIDED this holds up to the coplanar-leaves class above, on both tree kinds: where coincident
 *          faces of different leaves are hit at t an ulp apart, a peeling step (a closest-hit walk from a raised tmin) may
 *          skip one of them that the rows hold (DESIGN.md section 11);
 *        - refit trees: as the other ray queries, see bihrt_refit.
 *      Cost: without total the walk prunes at the k-th t, like bihrt_intersect at k = 1.  With total it visits every leaf the
 *      interval crosses, so the cost grows with the ray's depth complexity.
 *      k: 0 .. BIHRT_INTERSECT_K_MAX.  k == 0 writes no rows: with total the call is a pure crossing count, without it the call
 *      only fills count with 0.
 *      rec: arrays of n*k entries (ng: 3*n*k floats), any of them NULL; count, total: n entries, either NULL.  Each one host or
 *      device.  rays, staging, synchronisation, watchdog and replica behaviour as bihrt_intersect.
 *      Errors: those of bihrt_intersect, and BIHRT_ERR_INVALID for k < 0, k > BIHRT_INTERSECT_K_MAX, rec == NULL or
 *      BIHRT_INTERSECT_ANY; BIHRT_ERR_NOMEM when the staging buffer of host outputs cannot be allocated. ------------------ */
#define BIHRT_INTERSECT_K_MAX 64
BIHRT_API int bihrt_intersect_k(bihrt_ctx* ctx, const bihrt_ray_interval* rays, int64_t n, int32_t k, uint32_t flags,
                                const bihrt_hits* rec, int32_t* count, int32_t* total);
/* ---- closest-point queries: the triangle nearest to a point within the point's own search radius, full records.
 *      Distance of point p to a triangle: one IEEE binary32 function, every product, sum and quotient rounded, no FMA,
 *      computed from the triangle record's v0, e1 = v1 - v0, e2 = v2 - v0 (fl(v1 - v0), fl(v2 - v0), as bihrt_intersect
 *      uses them).  It is Ericson's ClosestPtPointTriangle (Real-Time Collision Detection, 5.1.5) with a = v0, b = v1, c = v2:
 *        ap = p - v0;  d1 = e1.ap, d2 = e2.ap                   (a.b = (ax*bx + ay*by) + az*bz throughout)
 *        d1 <= 0 && d2 <= 0                          -> (u, v) = (0, 0)
 *        bp = ap - e1; d3 = e1.bp, d4 = e2.bp
 *        d3 >= 0 && d4 <= d3                          -> (1, 0)
 *        vc = d1*d4 - d3*d2;  vc <= 0 && d1 >= 0 && d3 <= 0  -> (d1 / (d1 - d3), 0)                  [if d1 - d3 > 0]
 *        cp = ap - e2; d5 = e1.cp, d6 = e2.cp
 *        d6 >= 0 && d5 <= d6                          -> (0, 1)
 *        vb = d5*d2 - d1*d6;  vb <= 0 && d2 >= 0 && d6 <= 0  -> (0, d2 / (d2 - d6))                  [if d2 - d6 > 0]
 *        va = d3*d6 - d5*d4;  va <= 0 && d4 - d3 >= 0 && d5 - d6 >= 0
 *                                                     -> w = (d4 - d3) / ((d4 - d3) + (d5 - d6)), (1 - w, w)
 *                                                                                       [if (d4 - d3) + (d5 - d6) > 0]
 *        s = (va + vb) + vc;  s > 0                   -> (vb / s, vc / s)   (quotients, not products with 1 / s: a zero
 *                                                        weight stays 0 when 1 / s would overflow)
 *        otherwise, and when an edge branch's bracketed condition fails (an edge of zero length, e.g. a repeated vertex):
 *        zero or near-zero area, the nearest of the three edge segments, ties to AB, then AC, then BC.  Segment
 *        from a with direction e (AB: ap, e1; AC: ap, e2; BC: bp, e2 - e1): t = (ap.e) / (e.e), t = 0 unless t > 0 (so also
 *        for 0 / 0), t = 1 if t > 1; (u, v) = (t, 0), (0, t), (1 - t, t); each one's d2 as below.
 *      then q = (v0 + u*e1) + v*e2 and d2 = ((p-q).x^2 + (p-q).y^2) + (p-q).z^2.  u, v are the barycentric weights of v1, v2.
 *      For finite vertices and points whose differences and squares stay finite the result is never NaN.
 *      A triangle is a CANDIDATE when d2 <= min(fl(rmax*rmax), FLT_MAX): rmax = +inf, or any rmax whose square overflows, is
 *      unbounded; a triangle whose d2 overflows to +inf is never a candidate.  A query with a NaN or negative rmax, or a NaN or
 *      infinite coordinate of p, misses without being walked.
 *      Result: the candidate with the smallest (d2, slot), compared lexicographically -- ties go to the smaller slot -- so the
 *      result does not depend on the walk's order and EQUALS BRUTE FORCE OVER ALL SLOTS BIT FOR BIT, in every output, on parity
 *      and quality-mode trees alike.  The walk prunes with the children's exact boxes widened by a margin that covers the
 *      rounding of the distance function (DESIGN.md section 8), so no candidate is ever pruned.
 *      Record per query (every output pointer of bihrt_closest may be NULL; each one host or device):
 *        d2, u, v   as above; slot, prim as bihrt_trace; q = (v0 + u*e1) + v*e2, 3 floats; ng = e1 x e2, as bihrt_hits.ng.
 *        miss: d2 = FLT_MAX, slot = prim = -1, u = v = 0, q = ng = (0, 0, 0).
 *      The trace options (trace_tile_order, trace_sm_queues, trace_sort_rays, trace_lane_groups, ...) do not apply: points are
 *      taken in list order.  pts: host or device; device points must be 16-byte aligned (one 128-bit load per point).  Host
 *      outputs: the call synchronises and leaves them untouched if the build's watchdog tripped; device outputs are written
 *      asynchronously on the context's stream.
 *      Errors: BIHRT_ERR_INVALID for out == NULL, n < 0, pts == NULL with n > 0, n >= 2^32 - 2^24 or misaligned device points;
 *      BIHRT_ERR_STATE without a built BIH or for a replica of the other tree kind; BIHRT_ERR_INTERNAL after a tripped build
 *      watchdog. ---------------------------------------------------------------------------------------------------------- */
/* point with its own search radius: 16 B, one 128-bit load */
typedef struct bihrt_point_query { float p[3]; float rmax; } bihrt_point_query;
/* outputs of bihrt_closest_point: any pointer may be NULL; each one host or device */
typedef struct bihrt_closest {
    float*   d2;    /* [n]  squared distance to the closest point */
    float*   u;     /* [n]  barycentric weight of v1 */
    float*   v;     /* [n]  barycentric weight of v2 */
    int32_t* slot;  /* [n]  as bihrt_trace */
    int32_t* prim;  /* [n]  input triangle */
    float*   q;     /* [3n] the closest point, xyz */
    float*   ng;    /* [3n] geometric normal e1 x e2 of that triangle, as bihrt_hits.ng */
} bihrt_closest;
BIHRT_API int bihrt_closest_point(bihrt_ctx* ctx, const bihrt_point_query* pts, int64_t n, const bihrt_closest* out);
/* ---- k-nearest-triangle queries: the k triangles nearest to a point within the point's own search radius, nearest first, and
 *      the number of all triangles within that radius.
 *      Points, the distance function and the candidates are those of bihrt_closest_point: a triangle is a candidate when its
 *      d2 <= min(fl(rmax*rmax), FLT_MAX); a query with a NaN or negative rmax, or a NaN or infinite coordinate, has none and is
 *      not walked.
 *      Result for point i: its candidates ordered by (d2, slot) ascending, ties to the smaller slot; the first min(k, candidates)
 *      of them go to rows i*k + 0, 1, ... of the arrays of rec (each row as bihrt_closest_point's record: d2, u, v, slot, prim,
 *      q, ng).  The rows after them hold the miss record (d2 = FLT_MAX, slot = prim = -1, u = v = q = ng = 0).  count[i] is
 *      the number of rows written; total[i] the number of ALL candidates of point i, also where that is more than k (a radius
 *      query whose total[i] > k overflowed: ask again with a larger k).  Every output EQUALS BRUTE FORCE OVER ALL SLOTS BIT FOR
 *      BIT, on parity, quality-mode and refit trees alike; with k == 1 every row is bihrt_closest_point's record.
 *      Cost: without total the walk prunes at the current k-th best (d2, slot), like bihrt_closest_point at k = 1.  With total
 *      it prunes at the radius only, so it visits every leaf that holds a triangle in range: the records are the same, but the
 *      cost grows with the number of triangles within the radius (rmax = +inf visits every leaf).
 *      k == 0 writes no rows: with total it counts the triangles within the radius, without it the call only fills count with 0.
 *      rec: arrays of n*k entries (q and ng: 3*n*k floats), any of them NULL; count, total: n entries, either NULL.  Each one
 *      host or device.  pts, staging, synchronisation, watchdog and replica behaviour as bihrt_closest_point.
 *      Errors: those of bihrt_closest_point, and BIHRT_ERR_INVALID for k < 0, k > BIHRT_CLOSEST_K_MAX or rec == NULL;
 *      BIHRT_ERR_NOMEM when the staging buffer of host outputs cannot be allocated. ------------------------------------------- */
#define BIHRT_CLOSEST_K_MAX 64
BIHRT_API int bihrt_closest_k(bihrt_ctx* ctx, const bihrt_point_query* pts, int64_t n, int32_t k, const bihrt_closest* rec,
                              int32_t* count, int32_t* total);
/* ---- winding-number queries: inside / outside of closed meshes, and with bihrt_closest_point a signed distance.
 *      w(p) = (1/4pi) x the sum over all triangles of the signed solid angle the triangle subtends at p (the generalized winding
 *      number, Jacobson et al. 2013): 1 inside and 0 outside a closed mesh wound counter-clockwise seen from outside (the
 *      orientation ng = e1 x e2 points away from the inside), -1 inside an inward-wound one, k where k closed meshes overlap,
 *      and a smooth value in between for open meshes and soups.  Points are bihrt_point_query; rmax is not read, so one buffer
 *      serves bihrt_closest_point and bihrt_winding_number.
 *      Solid angle of a triangle (Van Oosterom & Strackee), binary32, every operation rounded, no FMA, from the record:
 *        a = v0 - p, b = a + e1, c = a + e2                     (x.y = (x0*y0 + x1*y1) + x2*y2; |x| = sqrt(x.x))
 *        det = a.(b x c), b x c = (by*cz - bz*cy, bz*cx - bx*cz, bx*cy - by*cx)
 *        den = (((|a|*|b|)*|c| + (a.b)*|c|) + (a.c)*|b|) + (b.c)*|a|
 *        Omega/2 = atan2f_bihrt(det, den); a triangle with det == 0 (p in its plane, or no area) contributes 0.
 *      atan2f_bihrt(y, x): mx = max(|x|, |y|), mn = min(|x|, |y|), t = mn / mx; if t > 0.41421356f: t = (t - 1) / (t + 1),
 *        off = 0.78539819f (pi/4 in binary32), else off = 0; z = t*t;
 *        r = (((((0.0805374449538f*z - 0.138776856032f)*z + 0.199777106478f)*z - 0.333329491539f)*z)*t + t) + off;
 *        if |y| > |x|: r = 1.57079637f - r; if x < 0: r = 3.14159274f - r; if y < 0: r = -r.
 *        Its largest error against binary64 atan2 is 2.7e-7 rad (DESIGN.md section 9: measured on 2^22 arguments).
 *      Far field (Barill et al. 2018): the walk treats a child (leaf or subtree) whose box has centre c = (lo + hi) * 0.5 and
 *      half-diagonal r as one cluster when |p - c|^2 > beta^2 r^2, computed as dot(c - p, c - p) > fl(beta*beta) *
 *      (dot(hi - lo, hi - lo) * 0.25); its term is the order-2 Taylor expansion of its triangles' solid angles about c
 *      (area vector N, first moments M, second moments Q: DESIGN.md section 9, which states its operation order).  A child that
 *      is not far is descended, a leaf's triangles are summed exactly.  The walk is depth first, the left child before the
 *      right, and terms are accumulated in binary64 in that order (an exact term adds 2 x Omega/2, a far term its Omega);
 *      w = (float)(sum x (1 / (4 pi) in binary64)).  beta = +INFINITY visits every leaf in slot order: the exact sum, bit for
 *      bit the brute force over slots 0 .. n-1, at O(n) work per point (a reference mode).  beta = 2 is the recommended value:
 *      its error against the exact sum is stated in DESIGN.md section 9.
 *      A point with a NaN or infinite coordinate is not walked and gets w = 0; so does every point of an empty scene.  A tree of
 *      one leaf is summed exactly.  For finite vertices and points whose differences and squares stay finite, w is never NaN.
 *      The far-field table (256 bytes per node slot) is built on the device by the first call with n > 0 after the BIH changed
 *      (build, refit, import, adopt, copy, broadcast), and freed with the context.
 *      pts: host or device, device points 16-byte aligned; w: host or device; staging, synchronisation and watchdog behaviour as
 *      bihrt_closest_point.
 *      Errors: BIHRT_ERR_INVALID for w == NULL, n < 0, pts == NULL with n > 0, n >= 2^32 - 2^24, misaligned device points, or
 *      beta NaN or <= 1; BIHRT_ERR_STATE without a built BIH or for a replica of the other tree kind; BIHRT_ERR_INTERNAL after a
 *      tripped build watchdog; BIHRT_ERR_NOMEM when the table cannot be allocated. ---------------------------------------- */
BIHRT_API int bihrt_winding_number(bihrt_ctx* ctx, const bihrt_point_query* pts, int64_t n, float beta, float* w);
/* instrumented trace: counters[0]=internal nodes visited, [1]=triangle tests, [2]=max stack depth,
 * [3]=rays; same results as bihrt_trace (outputs may be NULL). */
BIHRT_API int bihrt_trace_counted(bihrt_ctx* ctx, const bihrt_ray* rays, int64_t n, float* t, int32_t* slot,
                        int32_t* prim, uint64_t counters[4]);

/* Render w x h pixels, spp samples each, into the context's framebuffer with the reference's
 * colouring: hit (255,255,0), miss (20,20,40), mean over samples, packed r | g<<8 | b<<16, row 0 =
 * bottom (R/src/CUDAKernels.cu:82-88,385-387,391-423).  Jitter comes from a counter-based hash of
 * (seed, pixel, sample) instead of per-pixel XORWOW state (documented difference). */
BIHRT_API int bihrt_render(bihrt_ctx* ctx, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp,
                 uint64_t seed, uint32_t flags);
/* Same as bihrt_render through the instrumented kernel: counters as in bihrt_trace_counted. */
BIHRT_API int bihrt_render_counted(bihrt_ctx* ctx, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp,
                         uint64_t seed, uint32_t flags, uint64_t counters[4]);
/* Multi-GPU: render only the 32x32-pixel tiles with tile_id % shard_count == shard_index; every
 * other pixel of the framebuffer is set to 0, so a sum (or bitwise OR) of the shards' framebuffers
 * is the full image. */
BIHRT_API int bihrt_render_shard(bihrt_ctx* ctx, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp,
                       uint64_t seed, uint32_t flags, int32_t shard_index, int32_t shard_count);
/* Multi-GPU, sample sharding: trace only samples [sample_begin, sample_end) of every pixel of a
 * spp-sample frame and store per-pixel HIT COUNTS in the framebuffer.  Summing the counts of all ranks
 * and calling bihrt_framebuffer_resolve(spp) gives exactly the image bihrt_render(spp) produces; every
 * rank walks the whole image, so warp coherence is that of the single-GPU render. */
BIHRT_API int bihrt_render_samples(bihrt_ctx* ctx, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp,
                         uint64_t seed, uint32_t flags, int32_t sample_begin, int32_t sample_end);
BIHRT_API int bihrt_framebuffer_resolve(bihrt_ctx* ctx, int32_t spp);   /* counts -> packed colours, in place */
/* Multi-GPU, unit interleave (preferred): every rank walks every 32x32 tile but traces only every count-th
 * 32-ray unit of it (unit = a few neighbouring pixels with ALL their samples), writing per-pixel hit counts and 0
 * for the pixels it does not own.  Balanced by construction, same tile locality as the single-GPU render, and a
 * pixel's samples stay together in consecutive lanes.  count must divide 32 << k, k = log2 of the lane groups. */
BIHRT_API int bihrt_render_interleaved(bihrt_ctx* ctx, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp,
                             uint64_t seed, uint32_t flags, int32_t index, int32_t count);
/* Multi-GPU, unit interleave fused with the framebuffer gather: same partition as bihrt_render_interleaved, but the
 * final packed colour of every pixel this rank owns is stored by the trace kernel itself straight into `target_fb`
 * (w*h uint32; NULL = this context's own framebuffer) and no other pixel is touched.  With target_fb = the
 * framebuffer of the gathering GPU (a device pointer of another context of this process, or one opened with
 * bihrt_framebuffer_ipc_open in a one-process-per-GPU job) the stores travel over NVLink while the kernel runs:
 * no per-rank framebuffer clear, no hit-count reduce, no resolve pass.  The frame is complete once every rank's
 * launch has finished (a barrier, not a data collective).  Requires the lane-group layout every rank uses for
 * the same spp, so a pixel's samples never leave one rank. */
BIHRT_API int bihrt_render_interleaved_to(bihrt_ctx* ctx, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp,
                                uint64_t seed, uint32_t flags, int32_t index, int32_t count, uint32_t* target_fb);
/* Sharing the gathering GPU's framebuffer with the other processes of the job (CUDA IPC): export allocates the
 * context's w x h framebuffer and writes a 64-byte handle; open maps it in another process (peer access over
 * NVLink) and returns the pointer to pass as target_fb; close unmaps it. */
BIHRT_API int bihrt_framebuffer_ipc_export(bihrt_ctx* ctx, int32_t w, int32_t h, void* handle64);
BIHRT_API int bihrt_framebuffer_ipc_open(bihrt_ctx* ctx, const void* handle64, uint32_t** peer_fb);
BIHRT_API int bihrt_framebuffer_ipc_close(bihrt_ctx* ctx, uint32_t* peer_fb);
/* While a handle is out the exporting context refuses (BIHRT_ERR_STATE) to reallocate its framebuffer for a larger
 * frame -- the peers would keep storing into freed memory.  Call this once every peer has closed its mapping.  (The
 * same care is the caller's for a raw bihrt_framebuffer() pointer handed to another context as target_fb.) */
BIHRT_API int bihrt_framebuffer_ipc_unexport(bihrt_ctx* ctx);
/* Per-sample hit buffers of the same rays bihrt_render traces (index = (j*w+i)*spp + s); device or
 * host outputs, any may be NULL.  Used by the parity tests. */
BIHRT_API int bihrt_render_hits(bihrt_ctx* ctx, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp,
                      uint64_t seed, uint32_t flags, float* t, int32_t* slot, int32_t* prim);

/* ---- secondary rays (the stage after the path; the reference's Color() is a stub, R/src/CUDAKernels.cu:370-389).
 *      From the primary hits of a camera frame (the w*h*spp samples bihrt_render traces) build the next ray
 *      batch ON THE DEVICE: every sample that hits emits one ray from the hit point (moved 1e-3 along the
 *      geometric normal) to `light` (SHADOW; direction = light - origin, so t = 1 at the light) or in a
 *      cosine-weighted direction about the normal (DIFFUSE; counter-based hash of seed, pixel, sample).  Rays
 *      are written compacted and in sample order to out_rays (DEVICE, capacity w*h*spp); out_sample[i] (device,
 *      may be NULL) = source sample.  *count (host) receives the number of rays.  Synchronises. */
#define BIHRT_SECONDARY_SHADOW  0
#define BIHRT_SECONDARY_DIFFUSE 1
BIHRT_API int bihrt_secondary_rays(bihrt_ctx* ctx, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp, uint64_t seed,
                         uint32_t flags, int32_t kind, const float light[3], bihrt_ray* out_rays, int32_t* out_sample,
                         int64_t* count);

/* ---- framebuffer: Renderer::m_cudaDestResource, R/src/Renderer.h:46, R/src/Renderer.cpp:762-768 */
BIHRT_API int bihrt_framebuffer(bihrt_ctx* ctx, uint32_t** dev_ptr, int32_t* w, int32_t* h);  /* device pointer, owned by ctx */
BIHRT_API int bihrt_framebuffer_read(bihrt_ctx* ctx, uint32_t* host_dst);                      /* synchronises */

/* ---- BIH replication across GPUs (one broadcast of this blob per build, SURVEY.md 8(e)) ------- */
BIHRT_API int bihrt_bih_blob_bytes(bihrt_ctx* ctx, uint64_t* bytes);                     /* synchronises (needs Nu) */
BIHRT_API int bihrt_bih_export(bihrt_ctx* ctx, void* dev_dst, uint64_t bytes);           /* device buffer, D2D on the ctx stream */
BIHRT_API int bihrt_bih_import(bihrt_ctx* ctx, const void* dev_src, uint64_t bytes);     /* adopt a blob built on another GPU */

/* In place: the blob of an n-triangle scene is one contiguous device region whose size follows from n alone, so it can be
 * the buffer of the broadcast on every rank (no export / import copies, no host read of Nu).  bihrt_bih_region lays the
 * context's blob out for n triangles and returns the region (a no-op on the rank that built an n-triangle scene);
 * receivers call bihrt_bih_adopt(n) once the broadcast has been enqueued on the context's stream. */
BIHRT_API int bihrt_bih_region(bihrt_ctx* ctx, int64_t n, void** dev_ptr, uint64_t* bytes);
BIHRT_API int bihrt_bih_adopt(bihrt_ctx* ctx, int64_t n);
/* The same inside ONE process (a C host driving several GPUs, no NCCL): peer copy of src's BIH into dst over NVLink,
 * ordered after the work enqueued on src's stream and before dst's next call. */
BIHRT_API int bihrt_bih_copy(bihrt_ctx* dst, bihrt_ctx* src);

/* ---- several GPUs in ONE process (SURVEY.md 8(b): "Multi-GPU adds bihrt_create_multi(ctx**, int ngpu) which internally holds
 *      one NCCL communicator").  The reference is single-GPU; rays are independent given a replicated tree (8(e)).
 *      bihrt_create_multi fills ctxs[0..ngpu) with one context per device 0..ngpu-1 that share an NCCL communicator set
 *      (ncclCommInitAll; NCCL is bound at run time from libnccl.so.2).  Context 0 is the builder and the gatherer: load the
 *      scene and bihrt_build on it as usual, then per frame
 *          bihrt_multi_broadcast(ctxs[0]);                    one ncclBroadcast of the BIH blob, in place, no host copy
 *          bihrt_multi_render(ctxs[0], cam, w, h, spp, ...);   unit interleave; every device's trace kernel stores its finished
 *                                                             pixels straight into context 0's framebuffer over NVLink
 *          bihrt_framebuffer_read(ctxs[0], host);             ordered after every device's launch (events), same image as
 *                                                             bihrt_render on one GPU, bit for bit
 *      Everything is asynchronous on the contexts' streams; bihrt_multi_sync waits for all of them.  Contexts of a group are
 *      released together with bihrt_destroy_multi (not bihrt_destroy). ----------------------------------------------------- */
BIHRT_API int  bihrt_create_multi(bihrt_ctx** ctxs, int32_t ngpu);
BIHRT_API void bihrt_destroy_multi(bihrt_ctx** ctxs, int32_t ngpu);
BIHRT_API int  bihrt_multi_size(const bihrt_ctx* ctx);                       /* contexts in ctx's group (1 for a plain context) */
BIHRT_API int  bihrt_multi_nccl_version(void);                               /* e.g. 22809; 0 if libnccl.so.2 cannot be bound */
BIHRT_API int  bihrt_multi_broadcast(bihrt_ctx* ctx0);
BIHRT_API int  bihrt_multi_render(bihrt_ctx* ctx0, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp,
                                  uint64_t seed, uint32_t flags);
BIHRT_API int  bihrt_multi_sync(bihrt_ctx* ctx0);

#ifdef __cplusplus
}
#endif
#endif /* BIHRT_H */
