/*
 * intersect_k_oracle.c -- CPU restatement of the multi-hit ray query (bihrt_intersect_k, csrc/trace.cu k_trace MODE 5 and 6)
 * on the blob bihrt_bih_export writes.  TEST INFRASTRUCTURE ONLY, built by tests/intersect_k_oracle.py into a temporary
 * directory.
 *
 * It includes walk_oracle.c unchanged, so the triangle test (ray_tri), the blob builders, the scene slab and the children-box
 * slab are stated once.  It adds:
 *
 * walk_k   walk_oracle.c's walk (the same entry, node step, strict test on parity trees, far-leaf-first order and stack),
 *          with a list of up to k keys t_bits << 32 | slot in place of the closest hit.  A triangle is accepted for
 *          tlo < t < thi (tlo = max(tmin, 0), thi = min(tmax, FLT_MAX)); it enters the list while the list is short or when
 *          its key is below the k-th one.  The cut the node test reads (pMin <= min(pMax, cut), closed) is thi, or the k-th
 *          key's t once k keys are held and the total is not asked for.  tests/test_intersect_k_oracle.py ties it to walk's
 *          t and slot at k = 1.
 * brute_k  every slot, the accepted triangles sorted by key (qsort), the first k of them.
 *
 * Both count every accepted triangle they meet (the total: over the whole interval when the total is asked for).
 */
#include "walk_oracle.c"

#define K_MAX 64

typedef struct {
    uint64_t keys[K_MAX];
    int k, cnt, prune;            /* prune: the cut follows the k-th key (no total asked for) */
    uint32_t tot;
    float thi;
} klist;

static inline uint64_t tkey(float t, uint32_t slot) {
    uint32_t b;
    memcpy(&b, &t, 4);
    return (uint64_t)b << 32 | slot;
}

/* the cut the node test and the leaves read: thi, or the k-th key's t once the list is full and prunes */
static inline float klist_cut(const klist* L) {
    if (!(L->prune && L->k > 0 && L->cnt == L->k)) return L->thi;
    uint32_t b = (uint32_t)(L->keys[L->k - 1] >> 32);
    float t;
    memcpy(&t, &b, 4);
    return t;
}

/* an accepted triangle: counted, and kept when the list is short or its key is below the k-th one */
static void klist_add(klist* L, uint64_t key) {
    L->tot++;
    if (L->k == 0 || (L->cnt == L->k && key >= L->keys[L->k - 1])) return;
    int j = L->cnt < L->k ? L->cnt++ : L->k - 1;
    for (; j > 0 && L->keys[j - 1] > key; j--) L->keys[j] = L->keys[j - 1];
    L->keys[j] = key;
}

static void leaf_k(const blob* T, const orc_ray* r, uint32_t slot, int two_sided, float tlo, klist* L, orc_counters* c) {
    for (uint32_t i = slot;; i++) {
        float t, u, v;
        c->tris++;
        if (ray_tri(T->tri9 + 9 * (int64_t)T->tris[12 * (int64_t)i + 9], r, two_sided, &t, &u, &v) && t > tlo && t < L->thi)
            klist_add(L, tkey(t, i));
        if (T->tris[12 * (int64_t)i + 10] & 1u) break;
    }
}

/* walk_oracle.c's walk, step for step, with leaf_k and the list's cut in place of leaf and h.t */
static void walk_k(const blob* T, const orc_ray* r, int two_sided, float tlo, klist* L, orc_counters* c) {
    float rMin, sMax;
    const uint32_t nu = T->hdr[1];
    const int strict = T->hdr[10] == 0;
    if (nu == 0) return;
    if (!scene_slab(&T->s, r, &rMin, &sMax)) return;
    if (nu == 1) { leaf_k(T, r, 0, two_sided, tlo, L, c); return; }
    float pMin = dev_fmaxf(rMin, tlo), pMax = sMax;
    struct { uint32_t ref; float rMin, pMin, pMax; } stack[W_STACK];
    int sp = 0;
    uint32_t cur = T->hdr[9];
    orc_boxray q;
    make_boxray(&q, r, rMin, sMax);
    for (;;) {
        int next = 0;
        const float cut = klist_cut(L);
        if (pMin <= dev_fminf(pMax, cut)) {
            pMax = dev_fminf(pMax, cut);
            if (cur & REF_LEAF) {
                leaf_k(T, r, (cur & 0x7FFFFFFFu) >> 2, two_sided, tlo, L, c);
            } else {
                c->nodes++;
                const uint32_t* nw = T->nodes + 16 * (int64_t)(cur >> 2);
                const float* nd = (const float*)nw;
                int ax = (int)(cur & 3u);
                float org = r->o[ax], inv = r->inv[ax];
                int near = r->sign[ax], far = 1 - near;
                float t0 = (nd[0] - org) * inv;
                float t1 = (nd[1] - org) * inv;
                float tn = near ? t1 : t0, tf = near ? t0 : t1;
                uint32_t refn = nw[2 + near], reff = nw[2 + far];
                float nMax = dev_fminf(pMax, tn);
                float fMin = dev_fmaxf(pMin, tf);
                float bn[2], bf[2];
                box_slab(nd + 4, r, &q, &bn[0], &bf[0]);
                box_slab(nd + 10, r, &q, &bn[1], &bf[1]);
                float nLo = dev_fmaxf(pMin, bn[near]), nHi = dev_fminf(nMax, bf[near]);
                float fLo = dev_fmaxf(fMin, bn[far]), fHi = dev_fminf(pMax, bf[far]);
                int go_near = (!strict || rMin < tn) && (nLo <= nHi);
                int go_far = (fLo <= fHi);
                if (go_near && go_far) {
                    if (sp == W_STACK) { c->max_stack = INT32_MAX; break; }
                    if (!(refn & REF_LEAF) && (reff & REF_LEAF)) {
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

static int key_cmp(const void* x, const void* y) {
    uint64_t a = *(const uint64_t*)x, b = *(const uint64_t*)y;
    return a < b ? -1 : (a > b);
}

static void brute_k(const blob* T, const orc_ray* r, int two_sided, float tlo, klist* L, orc_counters* c) {
    const uint32_t n = T->hdr[0];
    uint64_t* all = (uint64_t*)malloc(8 * (size_t)(n ? n : 1));
    uint32_t m = 0;
    for (uint32_t i = 0; i < n; i++) {
        float t, u, v;
        c->tris++;
        if (ray_tri(T->tri9 + 9 * (int64_t)T->tris[12 * (int64_t)i + 9], r, two_sided, &t, &u, &v) && t > tlo && t < L->thi)
            all[m++] = tkey(t, i);
    }
    qsort(all, m, 8, key_cmp);
    L->tot = m;
    L->cnt = (int)(m < (uint32_t)L->k ? m : (uint32_t)L->k);
    memcpy(L->keys, all, 8 * (size_t)L->cnt);
    free(all);
}

/* brute_force 0: walk_k, 1: brute_k.  rays8: o.xyz tmin d.xyz tmax per ray.  want_total: the total is asked for (the walk
 * cuts at thi only).  A ray with !(max(tmin, 0) < tmax), NaN bounds included, or with k == 0 and no total, is not walked.
 * Rows i*k + j (each may be NULL): t, u, v, slot, prim, ng (3 per row); the record of a kept slot is computed after the walk
 * as walk_oracle.c's orc_walk computes it; a miss row is (FLT_MAX, 0, 0, -1, -1, 0 0 0).  count, total: per ray.
 * counters3: total nodes, total triangle tests, deepest stack. */
ORC_API void orc_walk_k(const float* tri9, const uint32_t* hdr, const uint32_t* nodes, const uint32_t* tris, int brute_force,
                        int two_sided, int k, int want_total, const float* rays8, int64_t nrays, float* out_t, float* out_u,
                        float* out_v, int32_t* out_slot, int32_t* out_prim, float* out_ng, int32_t* out_count,
                        int32_t* out_total, uint64_t* counters3, int nthreads) {
    blob T;
    memset(&T, 0, sizeof T);
    T.tri9 = tri9; T.hdr = hdr; T.nodes = nodes; T.tris = tris;
    memcpy(T.s.scene_lo, hdr + 2, 12); memcpy(T.s.scene_hi, hdr + 5, 12);
    uint64_t tot_nodes = 0, tot_tris = 0; int max_stack = 0;
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 64) num_threads(nthreads) reduction(+:tot_nodes, tot_tris) reduction(max:max_stack)
#else
    (void)nthreads;
#endif
    for (int64_t i = 0; i < nrays; i++) {
        const float* r8 = rays8 + 8 * i;
        orc_ray r;
        make_ray(&r, r8, r8 + 4);
        const float tmin = r8[3], tmax = r8[7], tlo = dev_fmaxf(tmin, 0.0f);
        klist L;
        L.k = k; L.cnt = 0; L.prune = !want_total; L.tot = 0; L.thi = dev_fminf(tmax, FLT_MAX);
        orc_counters c = { 0, 0, 0 };
        if (tmin == tmin && tlo < tmax && (k > 0 || want_total)) {
            if (brute_force) brute_k(&T, &r, two_sided, tlo, &L, &c);
            else walk_k(&T, &r, two_sided, tlo, &L, &c);
        }
        for (int j = 0; j < k; j++) {
            const int64_t row = i * k + j;
            float t = FLT_MAX, u = 0.0f, v = 0.0f, g[3] = { 0.0f, 0.0f, 0.0f };
            int32_t slot = -1, prim = -1;
            if (j < L.cnt) {
                const uint32_t tb = (uint32_t)(L.keys[j] >> 32);
                memcpy(&t, &tb, 4);
                slot = (int32_t)(uint32_t)L.keys[j];
                prim = (int32_t)tris[12 * (int64_t)slot + 9];
                const float* tri = tri9 + 9 * (int64_t)prim;
                float tt;
                ray_tri(tri, &r, two_sided, &tt, &u, &v);
                float e1[3], e2[3];
                for (int m = 0; m < 3; m++) { e1[m] = tri[3 + m] - tri[m]; e2[m] = tri[6 + m] - tri[m]; }
                g[0] = e1[1] * e2[2] - e1[2] * e2[1];
                g[1] = e1[2] * e2[0] - e1[0] * e2[2];
                g[2] = e1[0] * e2[1] - e1[1] * e2[0];
            }
            if (out_t) out_t[row] = t;
            if (out_u) out_u[row] = u;
            if (out_v) out_v[row] = v;
            if (out_slot) out_slot[row] = slot;
            if (out_prim) out_prim[row] = prim;
            if (out_ng) { out_ng[3 * row] = g[0]; out_ng[3 * row + 1] = g[1]; out_ng[3 * row + 2] = g[2]; }
        }
        if (out_count) out_count[i] = L.cnt;
        if (out_total) out_total[i] = (int32_t)L.tot;
        tot_nodes += c.nodes; tot_tris += c.tris;
        if (c.max_stack > max_stack) max_stack = c.max_stack;
    }
    if (counters3) { counters3[0] = tot_nodes; counters3[1] = tot_tris; counters3[2] = (uint64_t)max_stack; }
}
