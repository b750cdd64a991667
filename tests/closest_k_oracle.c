/*
 * closest_k_oracle.c -- CPU restatement of bihrt_closest_k (csrc/closest.cu, k_closest_k) on the blob bihrt_bih_export writes,
 * for both tree kinds.  TEST INFRASTRUCTURE ONLY, built by tests/closest_k_oracle.py into a temporary directory, with
 * -ffp-contract=off.  The distance function, the box bound and the blob layout are those of closest_oracle.c, included here
 * so that they are stated once (its orc_closest is exported from the same library).
 *
 * A candidate is a triangle with d2 <= min(fl(rmax^2), FLT_MAX); its key is (d2 bits << 32) | slot, which orders as (d2, slot)
 * because d2 is never negative or NaN.  The walk keeps the kernel's sorted list of up to k keys and prunes at min(radius cut,
 * k-th d2) once the list is full (at the radius cut alone when the total is wanted).  Brute force tests every slot, keeps the k
 * smallest keys in an unsorted pool and sorts them at the end: the same result by other means.
 */
#include <stdlib.h>

#include "closest_oracle.c"

#define CK_MAX 64

typedef unsigned long long ck_key;

static int ck_cmp(const void* a, const void* b) {
    const ck_key x = *(const ck_key*)a, y = *(const ck_key*)b;
    return x < y ? -1 : x > y;
}

/* the walk's list: insert key into the ascending list of *cnt keys (capacity k), dropping the k-th when full */
static void ck_insert(ck_key* list, int* cnt, int k, ck_key key) {
    int j = *cnt < k ? (*cnt)++ : k - 1;
    for (; j > 0 && list[j - 1] > key; j--) list[j] = list[j - 1];
    list[j] = key;
}

/* one point by the kernel's walk: fills list / cnt, returns the number of candidates met */
static uint32_t ck_walk(const uint32_t* hdr, const uint32_t* nodes, const uint32_t* tris, float margin_scale, float smag, int k,
                        int want_total, const float* p, ck_key* list, int* cnt, c_counters* c) {
    const float* sb = (const float*)(hdr + 2);
    const uint32_t nu = hdr[1];
    const float rcut = c_fminf(p[3] * p[3], FLT_MAX);
    float cut = rcut;
    ck_key kkey = k > 0 ? ~0ull : 0ull;
    uint32_t tot = 0;
    if (nu == 0 || (k == 0 && !want_total)) return 0;
    const float m = margin_scale * c_fmaxf(smag, c_fmaxf(c_fmaxf(fabsf(p[0]), fabsf(p[1])), fabsf(p[2])));
    struct { uint32_t ref; float bound; } stack[C_STACK];
    int sp = 0;
    uint32_t cur = 0xFFFFFFFFu;
    if (!(c_box(sb, p, m) > cut)) cur = nu == 1 ? C_REF_LEAF : hdr[9];
    while (cur != 0xFFFFFFFFu) {
        if (cur & C_REF_LEAF) {
            for (uint32_t s = (cur & 0x7FFFFFFFu) >> 2;; s++) {
                float u, v;
                c->tris++;
                const float d2 = c_pt_tri(p, (const float*)(tris + 12 * (int64_t)s), &u, &v);
                if (d2 <= rcut) {
                    tot++;
                    uint32_t bits;
                    memcpy(&bits, &d2, 4);
                    const ck_key key = (ck_key)bits << 32 | s;
                    if (key < kkey) {
                        ck_insert(list, cnt, k, key);
                        if (*cnt == k) {
                            kkey = list[k - 1];
                            if (!want_total) { bits = (uint32_t)(kkey >> 32); memcpy(&cut, &bits, 4); }
                        }
                    }
                }
                if (tris[12 * (int64_t)s + 10] & 1u) break;
            }
            cur = 0xFFFFFFFFu;
        } else {
            c->nodes++;
            const uint32_t* nw = nodes + 16 * (int64_t)(cur >> 2);
            const float* nd = (const float*)nw;
            float b[2] = { c_box(nd + 4, p, m), c_box(nd + 10, p, m) };
            int near = b[1] < b[0], far = 1 - near;
            if (b[near] > cut) cur = 0xFFFFFFFFu;
            else {
                if (!(b[far] > cut)) {
                    if (sp == C_STACK) { c->max_stack = INT32_MAX; break; }
                    stack[sp].ref = nw[2 + far]; stack[sp].bound = b[far]; sp++;
                    if (sp > c->max_stack) c->max_stack = sp;
                }
                cur = nw[2 + near];
            }
        }
        while (cur == 0xFFFFFFFFu && sp > 0) {
            sp--;
            if (!(stack[sp].bound > cut)) cur = stack[sp].ref;
        }
    }
    return tot;
}

/* one point by brute force: every slot; the k smallest keys in an unsorted pool (the largest replaced), sorted at the end */
static uint32_t ck_brute(const uint32_t* tris, uint32_t n, int k, const float* p, ck_key* list, int* cnt, c_counters* c) {
    const float rcut = c_fminf(p[3] * p[3], FLT_MAX);
    uint32_t tot = 0;
    int top = 0;                                   /* index of the largest key in a full pool */
    for (uint32_t s = 0; s < n; s++) {
        float u, v;
        c->tris++;
        const float d2 = c_pt_tri(p, (const float*)(tris + 12 * (int64_t)s), &u, &v);
        if (!(d2 <= rcut)) continue;
        tot++;
        uint32_t bits;
        memcpy(&bits, &d2, 4);
        const ck_key key = (ck_key)bits << 32 | s;
        if (*cnt < k) list[(*cnt)++] = key;
        else if (k > 0 && key < list[top]) list[top] = key;
        else continue;
        if (*cnt == k)
            for (int j = 0; j < k; j++) if (list[j] > list[top]) top = j;
    }
    qsort(list, (size_t)*cnt, sizeof(ck_key), ck_cmp);
    return tot;
}

/* pts4: p.xyz rmax per query.  brute_force 0: the kernel's walk (margin = margin_scale x the largest magnitude among the
 * point's and the scene box's coordinates; the kernel's is 2^-16), pruning at the k-th best unless total is wanted (out_total
 * not NULL), as the kernel does; 1: every slot.
 * Outputs (each may be NULL): rows i*k + j of d2, u, v, slot, prim, q (3), ng (3), a miss after the count[i] kept ones;
 * count[i]; total[i], the number of candidates.  counters3: node fetches,
 * distance evaluations, deepest stack. */
ORC_API void orc_closest_k(const uint32_t* hdr, const uint32_t* nodes, const uint32_t* tris, int brute_force, float margin_scale,
                           int k, const float* pts4, int64_t npts, float* out_d2, float* out_u, float* out_v,
                           int32_t* out_slot, int32_t* out_prim, float* out_q, float* out_ng, int32_t* out_count, int32_t* out_total,
                           uint64_t* counters3, int nthreads) {
    const float* sb = (const float*)(hdr + 2);
    float smag = 0.0f;
    for (int j = 0; j < 6; j++) smag = c_fmaxf(smag, fabsf(sb[j]));
    const uint32_t n = hdr[0];
    if (k < 0) k = 0;
    if (k > CK_MAX) k = CK_MAX;
    uint64_t tot_nodes = 0, tot_tris = 0; int max_stack = 0;
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 256) num_threads(nthreads) reduction(+:tot_nodes, tot_tris) reduction(max:max_stack)
#else
    (void)nthreads;
#endif
    for (int64_t i = 0; i < npts; i++) {
        const float* p = pts4 + 4 * i;
        c_counters c = { 0, 0, 0 };
        ck_key list[CK_MAX];
        int cnt = 0;
        uint32_t tot = 0;
        const int live = p[3] >= 0.0f && fabsf(p[0]) <= FLT_MAX && fabsf(p[1]) <= FLT_MAX && fabsf(p[2]) <= FLT_MAX;
        if (live && brute_force) tot = ck_brute(tris, n, k, p, list, &cnt, &c);
        else if (live) tot = ck_walk(hdr, nodes, tris, margin_scale, smag, k, out_total != NULL, p, list, &cnt, &c);
        for (int j = 0; j < k; j++) {
            const int64_t row = i * (int64_t)k + j;
            float d2 = FLT_MAX, u = 0.0f, v = 0.0f, q[3] = { 0.0f, 0.0f, 0.0f }, g[3] = { 0.0f, 0.0f, 0.0f };
            int32_t slot = -1, prim = -1;
            if (j < cnt) {
                const uint32_t s = (uint32_t)list[j], bits = (uint32_t)(list[j] >> 32);
                const float* r = (const float*)(tris + 12 * (int64_t)s);
                const float *e1 = r + 3, *e2 = r + 6;
                memcpy(&d2, &bits, 4);
                c_pt_tri(p, r, &u, &v);
                c_q(p, r, u, v, q);
                g[0] = e1[1] * e2[2] - e1[2] * e2[1];
                g[1] = e1[2] * e2[0] - e1[0] * e2[2];
                g[2] = e1[0] * e2[1] - e1[1] * e2[0];
                slot = (int32_t)s;
                prim = (int32_t)tris[12 * (int64_t)s + 9];
            }
            if (out_d2) out_d2[row] = d2;
            if (out_u) out_u[row] = u;
            if (out_v) out_v[row] = v;
            if (out_slot) out_slot[row] = slot;
            if (out_prim) out_prim[row] = prim;
            if (out_q) { out_q[3 * row] = q[0]; out_q[3 * row + 1] = q[1]; out_q[3 * row + 2] = q[2]; }
            if (out_ng) { out_ng[3 * row] = g[0]; out_ng[3 * row + 1] = g[1]; out_ng[3 * row + 2] = g[2]; }
        }
        if (out_count) out_count[i] = cnt;
        if (out_total) out_total[i] = (int32_t)tot;
        tot_nodes += c.nodes; tot_tris += c.tris;
        if (c.max_stack > max_stack) max_stack = c.max_stack;
    }
    if (counters3) { counters3[0] = tot_nodes; counters3[1] = tot_tris; counters3[2] = (uint64_t)max_stack; }
}
