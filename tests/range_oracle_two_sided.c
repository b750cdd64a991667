/*
 * range_oracle_two_sided.c -- CPU restatement of bihrt_intersect with BIHRT_INTERSECT_TWO_SIDED (csrc/trace.cu MODE 4).
 * TEST INFRASTRUCTURE ONLY, built by tests/test_gpu_intersect_two_sided.py into a temporary directory.
 *
 * It includes tests/range_oracle.c unchanged (the one-sided restatement, orc_trace_range, which the tests use for the
 * one-sided query) and adds orc_trace_range_two_sided: the same box walk, brute force and record computation, with one
 * change -- ray_triangle_uvt2 takes back faces too, fabs((double)det) < 0.000001 instead of (double)det < 0.000001.  The
 * walk, the interval, the ANY exit and the record are range_oracle.c's, line for line.
 */
#include "range_oracle.c"

static inline int ray_triangle_uvt2(const float* tri, const orc_ray* r, float* out_t, float* out_u, float* out_v) {
    float e1[3], e2[3], pvec[3], tvec[3], qvec[3];
    for (int k = 0; k < 3; k++) { e1[k] = tri[3 + k] - tri[k]; e2[k] = tri[6 + k] - tri[k]; }
    cross3(r->d, e2, pvec);
    float det = dot3(e1, pvec);
    if (fabs((double)det) < 0.000001) return 0;                 /* the only difference from ray_triangle_uvt */
    float inv_det = (float)(1.0 / (double)det);
    for (int k = 0; k < 3; k++) tvec[k] = r->o[k] - tri[k];
    float u = dot3(tvec, pvec) * inv_det;
    if (u < 0 || u > 1) return 0;
    cross3(tvec, e1, qvec);
    float v = dot3(r->d, qvec) * inv_det;
    if (v < 0 || u + v > 1) return 0;
    *out_t = dot3(e2, qvec) * inv_det;
    *out_u = u; *out_v = v;
    return 1;
}

static inline void find_range2(const orc_scene* s, const orc_ray* r, float tlo, int leaf, orc_hit* rec, orc_counters* c) {
    float t = FLT_MAX, u, v;
    for (int64_t i = s->first[leaf]; i < (int64_t)s->first[leaf] + s->cnt[leaf]; i++) {
        c->tris++;
        if (ray_triangle_uvt2(s->tri9 + 9 * (int64_t)s->tris_idx[i], r, &t, &u, &v))
            if (t > tlo && t < rec->t) { rec->t = t; rec->slot = (int)i; }
    }
}

static void traverse_range2(const orc_scene* s, const float* cbox, const orc_ray* r, float tlo, int any, orc_hit* rec, orc_counters* c) {
    float rMin, sMax;
    if (s->nu <= 0) return;
    if (!scene_slab(s, r, &rMin, &sMax)) return;
    if (s->nu == 1) { find_range2(s, r, tlo, 0, rec, c); return; }
    float pMin = dev_fmaxf(rMin, tlo), pMax = sMax;
    struct { int ref; float rMin, pMin, pMax; } stack[64];
    int sp = 0;
    int cur = 0;
    orc_boxray q;
    make_boxray(&q, r, rMin, sMax);
    for (;;) {
        int next = 0;
        if (pMin <= dev_fminf(pMax, (float)rec->t)) {
            pMax = dev_fminf(pMax, (float)rec->t);
            if (cur < 0) {
                find_range2(s, r, tlo, ~cur, rec, c);
                if (any && rec->slot >= 0) break;                   /* occlusion: nothing else to learn */
            } else {
                c->nodes++;
                int ax = s->axis[cur];
                float org = r->o[ax], inv = r->inv[ax];
                int near = r->sign[ax], far = 1 - near;
                float t0 = (s->clip[2 * cur] - org) * inv;
                float t1 = (s->clip[2 * cur + 1] - org) * inv;
                float tn = near ? t1 : t0, tf = near ? t0 : t1;
                const uint8_t* lf = s->is_leaf + 2 * cur;
                const int32_t* ch = s->children + 2 * cur;
                int refn = lf[near] ? ~ch[near] : ch[near], reff = lf[far] ? ~ch[far] : ch[far];
                float nMax = dev_fminf(pMax, tn);
                float fMin = dev_fmaxf(pMin, tf);
                float bn[2], bf[2];
                box_slab(cbox + 12 * (int64_t)cur, r, &q, &bn[0], &bf[0]);
                box_slab(cbox + 12 * (int64_t)cur + 6, r, &q, &bn[1], &bf[1]);
                float nLo = dev_fmaxf(pMin, bn[near]), nHi = dev_fminf(nMax, bf[near]);
                float fLo = dev_fmaxf(fMin, bn[far]), fHi = dev_fminf(pMax, bf[far]);
                int go_near = (rMin < tn) && (nLo <= nHi);
                int go_far = (fLo <= fHi);
                if (go_near && go_far) {
                    if (refn >= 0 && reff < 0) {
                        stack[sp].ref = refn; stack[sp].rMin = rMin; stack[sp].pMin = nLo; stack[sp].pMax = nHi;
                        cur = reff; rMin = tf; pMin = fLo; pMax = fHi;
                    } else {
                        stack[sp].ref = reff; stack[sp].rMin = tf; stack[sp].pMin = fLo; stack[sp].pMax = fHi;
                        cur = refn; pMin = nLo; pMax = nHi;
                    }
                    sp++;
                    if (sp > c->max_stack) c->max_stack = sp;
                    next = 1;
                } else if (go_near) { cur = refn; pMin = nLo; pMax = nHi; next = 1; }
                else if (go_far) { cur = reff; rMin = tf; pMin = fLo; pMax = fHi; next = 1; }
            }
        }
        if (next) continue;
        if (sp == 0) break;
        sp--;
        cur = stack[sp].ref; rMin = stack[sp].rMin; pMin = stack[sp].pMin; pMax = stack[sp].pMax;
    }
}

static void brute_range2(const orc_scene* s, const orc_ray* r, float tlo, orc_hit* rec, orc_counters* c) {
    float t = FLT_MAX, u, v;
    for (int64_t i = 0; i < s->n; i++) {
        c->tris++;
        if (ray_triangle_uvt2(s->tri9 + 9 * (int64_t)s->tris_idx[i], r, &t, &u, &v))
            if (t > tlo && t < rec->t) { rec->t = t; rec->slot = (int)i; }
    }
}

/* orc_trace_range with two-sided triangles: same arguments, mode 0 = traverse_range2 (the kernel), 1 = brute_range2;
 * flags 1 = ANY (traverse_range2 only). */
ORC_API void orc_trace_range_two_sided(int mode, uint32_t flags, const float* tri9, int64_t n, int64_t nu,
                                       const uint32_t* tris_idx, const uint32_t* cnt, const int32_t* first,
                                       const float* clip, const int32_t* axis, const uint8_t* is_leaf,
                                       const int32_t* children, const float* scene_lo, const float* scene_hi,
                                       const float* rays8, int64_t nrays, float* out_t, float* out_u, float* out_v,
                                       int32_t* out_slot, int32_t* out_prim, float* out_ng, uint64_t* counters3, int nthreads) {
    orc_scene s = { tri9, n, nu, tris_idx, cnt, first, clip, axis, is_leaf, children, {0, 0, 0}, {0, 0, 0} };
    for (int k = 0; k < 3; k++) { s.scene_lo[k] = scene_lo[k]; s.scene_hi[k] = scene_hi[k]; }
    uint64_t tot_nodes = 0, tot_tris = 0; int max_stack = 0;
    float* cbox = NULL;
    if (mode == 0) { cbox = (float*)malloc(sizeof(float) * 12 * (size_t)(nu > 1 ? nu - 1 : 1)); children_boxes(&s, cbox); }
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 256) num_threads(nthreads) reduction(+:tot_nodes, tot_tris) reduction(max:max_stack)
#else
    (void)nthreads;
#endif
    for (int64_t i = 0; i < nrays; i++) {
        const float* r8 = rays8 + 8 * i;
        orc_ray r;
        make_ray(&r, r8, r8 + 4);
        const float tmin = r8[3], tmax = r8[7];
        const float tlo = dev_fmaxf(tmin, 0.0f);
        orc_hit rec = { dev_fminf(tmax, FLT_MAX), -1 };
        orc_counters c = { 0, 0, 0 };
        if (tmin == tmin && tlo < tmax) {
            if (mode == 0) traverse_range2(&s, cbox, &r, tlo, (int)(flags & 1u), &rec, &c);
            else brute_range2(&s, &r, tlo, &rec, &c);
        }
        float t = FLT_MAX, u = 0.0f, v = 0.0f, g[3] = { 0.0f, 0.0f, 0.0f };
        if (rec.slot >= 0) {
            const float* tri = tri9 + 9 * (int64_t)tris_idx[rec.slot];
            float tt;
            ray_triangle_uvt2(tri, &r, &tt, &u, &v);
            t = (float)rec.t;
            float e1[3], e2[3];
            for (int k = 0; k < 3; k++) { e1[k] = tri[3 + k] - tri[k]; e2[k] = tri[6 + k] - tri[k]; }
            g[0] = e1[1] * e2[2] - e1[2] * e2[1];
            g[1] = e1[2] * e2[0] - e1[0] * e2[2];
            g[2] = e1[0] * e2[1] - e1[1] * e2[0];
        }
        if (out_t) out_t[i] = t;
        if (out_u) out_u[i] = u;
        if (out_v) out_v[i] = v;
        if (out_slot) out_slot[i] = rec.slot;
        if (out_prim) out_prim[i] = rec.slot >= 0 ? (int32_t)tris_idx[rec.slot] : -1;
        if (out_ng) { out_ng[3 * i] = g[0]; out_ng[3 * i + 1] = g[1]; out_ng[3 * i + 2] = g[2]; }
        tot_nodes += c.nodes; tot_tris += c.tris;
        if (c.max_stack > max_stack) max_stack = c.max_stack;
    }
    free(cbox);
    if (counters3) { counters3[0] = tot_nodes; counters3[1] = tot_tris; counters3[2] = (uint64_t)max_stack; }
}
