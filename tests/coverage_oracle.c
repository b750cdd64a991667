/*
 * coverage_oracle.c -- CPU restatement of the framebuffer renders of csrc/trace.cu (MODE 1: bihrt_render and its
 * shard / sample / interleave variants, bihrt_render_counted), which are coverage queries: a sample ends at the first
 * triangle it accepts.  TEST INFRASTRUCTURE ONLY, built by tests/test_gpu_coverage.py into a temporary directory.
 *
 * It includes the oracle's source unchanged (oracle/bih_oracle.c, whose outputs tests/golden/golden_scenes.json
 * freezes) and adds one traversal next to its modes:
 *
 * mode "first" -- traverse_box that stops at the first accepted triangle.  find_first returns at the first triangle of a
 * leaf with 0 < t < best (best is still FLT_MAX: nothing has been accepted yet), and the walk ends after the leaf that
 * found it.  Up to that leaf the walk is traverse_box's step for step, because traverse_box too has rec->t == FLT_MAX
 * until its first accepted triangle: same entry checks, same strict test (rMin < t[near]), same far-leaf-first order,
 * same misses on axis-aligned flat geometry.  So a ray hits in "first" exactly when it hits in "box" -- and hence in
 * "ref", which box equals -- while its node and triangle counters can only be smaller.  The slot and t it returns are
 * those of the FIRST accepted triangle, not the closest one; only hit / miss is meaningful.
 */
#include "bih_oracle.c"

static inline void find_first(const orc_scene* s, const orc_ray* r, int leaf, orc_hit* rec, orc_counters* c) {
    float t = FLT_MAX;
    for (int64_t i = s->first[leaf]; i < (int64_t)s->first[leaf] + s->cnt[leaf]; i++) {
        uint32_t tri = s->tris_idx[i];
        c->tris++;
        if (ray_triangle(s->tri9 + 9 * (int64_t)tri, r, &t)) {
            if (t > 0 && t < rec->t) { rec->t = t; rec->slot = (int)i; return; }
        }
    }
}

static void traverse_first(const orc_scene* s, const float* cbox, const orc_ray* r, orc_hit* rec, orc_counters* c) {
    float rMin, sMax;
    if (s->nu <= 0) return;
    if (!scene_slab(s, r, &rMin, &sMax)) return;
    if (s->nu == 1) { find_first(s, r, 0, rec, c); return; }
    float pMin = dev_fmaxf(rMin, 0.0f), pMax = sMax;
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
                find_first(s, r, ~cur, rec, c);
                if (rec->slot >= 0) break;                          /* covered: the only difference to traverse_box */
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

/* orc_trace's arguments without the mode: the "first" traversal over every ray */
ORC_API void orc_trace_first(const float* tri9, int64_t n, int64_t nu,
                             const uint32_t* tris_idx, const uint32_t* cnt, const int32_t* first,
                             const float* clip, const int32_t* axis, const uint8_t* is_leaf,
                             const int32_t* children, const float* scene_lo, const float* scene_hi,
                             const float* rays6, int64_t nrays, float* out_t, int32_t* out_slot,
                             int32_t* out_prim, uint64_t* counters3, int nthreads) {
    orc_scene s = { tri9, n, nu, tris_idx, cnt, first, clip, axis, is_leaf, children, {0, 0, 0}, {0, 0, 0} };
    for (int k = 0; k < 3; k++) { s.scene_lo[k] = scene_lo[k]; s.scene_hi[k] = scene_hi[k]; }
    uint64_t tot_nodes = 0, tot_tris = 0; int max_stack = 0;
    float* cbox = (float*)malloc(sizeof(float) * 12 * (size_t)(nu > 1 ? nu - 1 : 1));
    children_boxes(&s, cbox);
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 256) num_threads(nthreads) reduction(+:tot_nodes, tot_tris) reduction(max:max_stack)
#else
    (void)nthreads;
#endif
    for (int64_t i = 0; i < nrays; i++) {
        orc_ray r;
        make_ray(&r, rays6 + 6 * i, rays6 + 6 * i + 3);
        orc_hit rec = { FLT_MAX, -1 };
        orc_counters c = { 0, 0, 0 };
        traverse_first(&s, cbox, &r, &rec, &c);
        out_t[i] = (float)rec.t;
        out_slot[i] = rec.slot;
        if (out_prim) out_prim[i] = rec.slot >= 0 ? (int32_t)tris_idx[rec.slot] : -1;
        tot_nodes += c.nodes; tot_tris += c.tris;
        if (c.max_stack > max_stack) max_stack = c.max_stack;
    }
    free(cbox);
    if (counters3) { counters3[0] = tot_nodes; counters3[1] = tot_tris; counters3[2] = (uint64_t)max_stack; }
}
