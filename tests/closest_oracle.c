/*
 * closest_oracle.c -- CPU restatement of bihrt_closest_point (csrc/closest.cu, k_closest) on the blob bihrt_bih_export writes,
 * for both tree kinds.  TEST INFRASTRUCTURE ONLY, built by tests/closest_oracle.py into a temporary directory, with
 * -ffp-contract=off so that every product and sum is rounded on its own, as the kernel's explicit __f*_rn are.
 *
 * The distance function is written from its statement in include/bihrt.h, not from the kernel's source: Ericson's
 * ClosestPtPointTriangle on the triangle record's v0, e1, e2, with the zero-length-edge and zero-area cases going to the nearest
 * of the three edge segments.  The walk is the kernel's best-first descent over the children's boxes widened by the query's
 * margin (DESIGN.md section 8); brute force tests every slot in slot order.
 *
 * The blob: header (16 words: n, nu, scene lo.xyz, hi.xyz, status, root_axis, quality, 5 spare), node slots (16 words:
 * clip0, clip1, the two child references, the left and the right child's box lo.xyz hi.xyz), n triangle records (12 words:
 * v0, e1, e2, prim, last, slot).  A child reference is REF_LEAF | its first slot << 2 for a leaf and its node index << 2 | its
 * split axis for a node; node 0 is the root (its reference is header word 9: node 0 with its axis).
 */
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define ORC_API __attribute__((visibility("default")))
#define C_STACK 128
#define C_REF_LEAF 0x80000000u

typedef struct { uint64_t nodes, tris; int max_stack; } c_counters;

/* CUDA's fminf / fmaxf: a NaN operand loses, -0 < +0 */
static inline float c_fminf(float a, float b) {
    if (a != a) return b;
    if (b != b) return a;
    if (a == 0.0f && b == 0.0f) return signbit(a) ? a : b;
    return a < b ? a : b;
}
static inline float c_fmaxf(float a, float b) {
    if (a != a) return b;
    if (b != b) return a;
    if (a == 0.0f && b == 0.0f) return signbit(a) ? b : a;
    return a > b ? a : b;
}

static inline float c_dot(const float a[3], const float b[3]) { return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]; }

/* q = (v0 + u*e1) + v*e2; returns |p - q|^2 */
static float c_q(const float* p, const float* r, float u, float v, float q[3]) {
    float d[3];
    for (int k = 0; k < 3; k++) { q[k] = (r[k] + u * r[3 + k]) + v * r[6 + k]; d[k] = p[k] - q[k]; }
    return c_dot(d, d);
}

static float c_seg(const float rel[3], const float e[3]) {
    float t = c_dot(rel, e) / c_dot(e, e);
    return t > 0.0f ? fminf(t, 1.0f) : 0.0f;
}

/* r: the record's first 9 words (v0, e1, e2); returns d2, sets u, v */
static float c_pt_tri(const float* p, const float* r, float* u, float* v) {
    const float *e1 = r + 3, *e2 = r + 6;
    float ap[3], bp[3], cp[3], q[3];
    for (int k = 0; k < 3; k++) { ap[k] = p[k] - r[k]; bp[k] = ap[k] - e1[k]; cp[k] = ap[k] - e2[k]; }
    float d1 = c_dot(e1, ap), d2 = c_dot(e2, ap);
    float d3 = c_dot(e1, bp), d4 = c_dot(e2, bp);
    float d5 = c_dot(e1, cp), d6 = c_dot(e2, cp);
    float vc = d1 * d4 - d3 * d2, vb = d5 * d2 - d1 * d6, va = d3 * d6 - d5 * d4;
    float s = (va + vb) + vc;
    int degen = 0;              /* an edge branch with a zero-length edge, or the interior branch without area */
    *u = 0.0f; *v = 0.0f;
    if (d1 <= 0.0f && d2 <= 0.0f) { }
    else if (d3 >= 0.0f && d4 <= d3) *u = 1.0f;
    else if (vc <= 0.0f && d1 >= 0.0f && d3 <= 0.0f) { if (d1 - d3 > 0.0f) *u = d1 / (d1 - d3); else degen = 1; }
    else if (d6 >= 0.0f && d5 <= d6) *v = 1.0f;
    else if (vb <= 0.0f && d2 >= 0.0f && d6 <= 0.0f) { if (d2 - d6 > 0.0f) *v = d2 / (d2 - d6); else degen = 1; }
    else if (va <= 0.0f && d4 - d3 >= 0.0f && d5 - d6 >= 0.0f) {
        if ((d4 - d3) + (d5 - d6) > 0.0f) { float w = (d4 - d3) / ((d4 - d3) + (d5 - d6)); *u = 1.0f - w; *v = w; } else degen = 1;
    }
    else if (s > 0.0f) { *u = vb / s; *v = vc / s; }
    else degen = 1;
    if (degen) {
        float bc[3] = { e2[0] - e1[0], e2[1] - e1[1], e2[2] - e1[2] };
        float cand[3][2] = { { c_seg(ap, e1), 0.0f }, { 0.0f, c_seg(ap, e2) }, { 0.0f, c_seg(bp, bc) } };
        cand[2][0] = 1.0f - cand[2][1];
        int pick = 0;
        float best = c_q(p, r, cand[0][0], cand[0][1], q);
        for (int j = 1; j < 3; j++) {
            float dj = c_q(p, r, cand[j][0], cand[j][1], q);
            if (dj < best) { best = dj; pick = j; }
        }
        *u = cand[pick][0]; *v = cand[pick][1];
    }
    return c_q(p, r, *u, *v, q);
}

/* squared distance from p to the box (lo.xyz, hi.xyz) widened by m on every side */
static float c_box(const float* b, const float* p, float m) {
    float g[3];
    for (int k = 0; k < 3; k++) g[k] = c_fmaxf(c_fmaxf(b[k] - p[k], p[k] - b[3 + k]) - m, 0.0f);
    return c_dot(g, g);
}

/* slot i against the best so far: smallest (d2, slot) with d2 <= cut */
static inline void c_test(const uint32_t* tris, const float* p, uint32_t i, float* cut, uint32_t* best, c_counters* c) {
    float u, v;
    c->tris++;
    float d2 = c_pt_tri(p, (const float*)(tris + 12 * (int64_t)i), &u, &v);
    if (d2 < *cut || (d2 == *cut && i < *best)) { *cut = d2; *best = i; }
}

/* pts4: p.xyz rmax per query.  brute_force 0: the kernel's walk (margin = margin_scale x the largest magnitude among the
 * point's and the scene box's coordinates; the kernel's is 2^-16); 1: every slot in slot order.  Outputs (each may be NULL):
 * d2, u, v, slot, prim, q (3), ng (3); a miss is (FLT_MAX, 0, 0, -1, -1, 0 0 0, 0 0 0).  counters3: node fetches, distance
 * evaluations, deepest stack. */
ORC_API void orc_closest(const uint32_t* hdr, const uint32_t* nodes, const uint32_t* tris, int brute_force, float margin_scale,
                         const float* pts4, int64_t npts, float* out_d2, float* out_u, float* out_v, int32_t* out_slot,
                         int32_t* out_prim, float* out_q, float* out_ng, uint64_t* counters3, int nthreads) {
    const float* sb = (const float*)(hdr + 2);        /* scene lo.xyz hi.xyz */
    float smag = 0.0f;
    for (int k = 0; k < 6; k++) smag = c_fmaxf(smag, fabsf(sb[k]));
    const uint32_t n = hdr[0], nu = hdr[1];
    uint64_t tot_nodes = 0, tot_tris = 0; int max_stack = 0;
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 256) num_threads(nthreads) reduction(+:tot_nodes, tot_tris) reduction(max:max_stack)
#else
    (void)nthreads;
#endif
    for (int64_t i = 0; i < npts; i++) {
        const float* p = pts4 + 4 * i;
        const float rmax = p[3];
        float cut = c_fminf(rmax * rmax, FLT_MAX);
        uint32_t best = 0xFFFFFFFFu;
        c_counters c = { 0, 0, 0 };
        int live = rmax >= 0.0f && fabsf(p[0]) <= FLT_MAX && fabsf(p[1]) <= FLT_MAX && fabsf(p[2]) <= FLT_MAX;
        if (live && brute_force) {
            for (uint32_t s = 0; s < n; s++) c_test(tris, p, s, &cut, &best, &c);
        } else if (live && nu > 0) {
            const float m = margin_scale * c_fmaxf(smag, c_fmaxf(c_fmaxf(fabsf(p[0]), fabsf(p[1])), fabsf(p[2])));
            struct { uint32_t ref; float bound; } stack[C_STACK];
            int sp = 0;
            uint32_t cur = 0xFFFFFFFFu;
            if (!(c_box(sb, p, m) > cut)) cur = nu == 1 ? C_REF_LEAF : hdr[9];
            while (cur != 0xFFFFFFFFu) {
                if (cur & C_REF_LEAF) {
                    for (uint32_t s = (cur & 0x7FFFFFFFu) >> 2;; s++) {
                        c_test(tris, p, s, &cut, &best, &c);
                        if (tris[12 * (int64_t)s + 10] & 1u) break;
                    }
                    cur = 0xFFFFFFFFu;
                } else {
                    c.nodes++;
                    const uint32_t* nw = nodes + 16 * (int64_t)(cur >> 2);
                    const float* nd = (const float*)nw;
                    float b[2] = { c_box(nd + 4, p, m), c_box(nd + 10, p, m) };
                    int near = b[1] < b[0], far = 1 - near;
                    if (b[near] > cut) cur = 0xFFFFFFFFu;
                    else {
                        if (!(b[far] > cut)) {
                            if (sp == C_STACK) { c.max_stack = INT32_MAX; break; }
                            stack[sp].ref = nw[2 + far]; stack[sp].bound = b[far]; sp++;
                            if (sp > c.max_stack) c.max_stack = sp;
                        }
                        cur = nw[2 + near];
                    }
                }
                while (cur == 0xFFFFFFFFu && sp > 0) {
                    sp--;
                    if (!(stack[sp].bound > cut)) cur = stack[sp].ref;
                }
            }
        }
        float u = 0.0f, v = 0.0f, q[3] = { 0.0f, 0.0f, 0.0f }, g[3] = { 0.0f, 0.0f, 0.0f };
        int32_t prim = -1;
        if (best != 0xFFFFFFFFu) {
            const float* r = (const float*)(tris + 12 * (int64_t)best);
            const float *e1 = r + 3, *e2 = r + 6;
            c_pt_tri(p, r, &u, &v);
            c_q(p, r, u, v, q);
            g[0] = e1[1] * e2[2] - e1[2] * e2[1];
            g[1] = e1[2] * e2[0] - e1[0] * e2[2];
            g[2] = e1[0] * e2[1] - e1[1] * e2[0];
            prim = (int32_t)tris[12 * (int64_t)best + 9];
        }
        if (out_d2) out_d2[i] = best != 0xFFFFFFFFu ? cut : FLT_MAX;
        if (out_u) out_u[i] = u;
        if (out_v) out_v[i] = v;
        if (out_slot) out_slot[i] = (int32_t)best;
        if (out_prim) out_prim[i] = prim;
        if (out_q) { out_q[3 * i] = q[0]; out_q[3 * i + 1] = q[1]; out_q[3 * i + 2] = q[2]; }
        if (out_ng) { out_ng[3 * i] = g[0]; out_ng[3 * i + 1] = g[1]; out_ng[3 * i + 2] = g[2]; }
        tot_nodes += c.nodes; tot_tris += c.tris;
        if (c.max_stack > max_stack) max_stack = c.max_stack;
    }
    if (counters3) { counters3[0] = tot_nodes; counters3[1] = tot_tris; counters3[2] = (uint64_t)max_stack; }
}
