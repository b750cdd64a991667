/*
 * walk_oracle.c -- CPU restatement of the walk every trace entry point takes (csrc/trace.cu, k_trace), on the blob
 * bihrt_bih_export writes, for both tree kinds.  TEST INFRASTRUCTURE ONLY, built by tests/walk_oracle.py into a temporary
 * directory.
 *
 * It includes the oracle's source unchanged (oracle/bih_oracle.c, whose outputs tests/golden/golden_scenes.json freezes)
 * and reuses its ray setup, scene slab, children-box slab and children boxes.  Its traverse_box stays the reference the walk
 * here is tied to (tests/test_gpu_intersect.py: over (0, inf) the parity walk IS traverse_box, counters included).
 *
 * The blob: header (16 words: n, nu, scene lo.xyz, hi.xyz, status, root_axis, quality, 5 spare), node slots (16 words:
 * clip0, clip1, the two child references, the left and the right child's box lo.xyz hi.xyz), n triangle records (12 words:
 * v0, e1, e2, prim, last, slot).  A child reference is REF_LEAF | its first slot << 2 for a leaf, whose last slot is flagged,
 * and its node index << 2 | its own split axis for a node.  Two builders write it:
 *
 * orc_parity_blob  the oracle's parity tree (the arrays oracle.Bih holds): quality = 0, root_axis = axis[0], nu - 1 node
 *                  slots; node i is the oracle's node i with its clip planes and children_boxes' two boxes.
 * orc_q_build      the quality-mode tree (morton_bits 63 and leaf_cap, csrc/build.cu), written from the definition of the
 *                  tree, not from k_nodes_q:
 *   scene box    exact min / max of all vertex coordinates (-0 < +0);
 *   keys         per axis centre = (min + max) * 0.5, nrm = (centre - lo) / (hi - lo), q = min(max(nrm * 2^21, 0), 2^21 - 1) with
 *                NaN-dropping min / max (a flat axis gives 0), truncated; key = x << 2 | y << 1 | z of the bit-interleaved axes;
 *   order        stable by key: slot order is (key, input index);
 *   tree         the binary radix tree over the distinct strings (64 key bits, then 32 bits of the slot position).  Range
 *                [a, b] splits after the last slot whose string agrees with slot a's beyond the common prefix p of a and b; the
 *                left child [a, s] is node s, the right child [s + 1, b] is node s + 1, the root [0, n - 1] is node 0; the node
 *                splits on axis (p + 2) % 3.  A child of at most `cap` slots is a leaf.  n <= cap: one leaf, no node;
 *   node record  clip0 = max hi[axis] of the left child's vertices, clip1 = min lo[axis] of the right child's, the two refs,
 *                and the exact boxes of both children.  n - 1 node slots; only reachable ones are written.
 *
 * walk   traverse_box on a blob, with the ray's interval and a long stack.  A triangle is accepted for tlo < t < h.t, where
 *        tlo = max(tmin, 0) and h.t starts where the caller says; the root's tight interval starts at max(rMin, tlo).  The
 *        closed tight interval decides the near child, and on parity trees (hdr[10] == 0) so does the reference's strict test
 *        rMin < t[near] (rMin: the scene-box entry, overwritten on far descents); quality trees drop the strict test.  Exits:
 *          W_CLOSEST  the closest hit (bihrt_trace, bihrt_render_hits, bihrt_intersect);
 *          W_FIRST    the first accepted triangle (the framebuffer renders, which are coverage queries);
 *          W_ANY      the first leaf that accepts a triangle, keeping that leaf's closest (bihrt_trace_any, bihrt_intersect ANY).
 *        Until a triangle is accepted nothing but the narrower interval separates the parity walk from traverse_box, so over
 *        (0, >= FLT_MAX) with h.t = FLT_MAX it IS traverse_box, counters included.  W_FIRST takes traverse_box's decisions up
 *        to its first hit (same entry checks, strict test, far-leaf-first order and misses on axis-aligned flat geometry), so
 *        it hits exactly where traverse_box -- and hence traverse_ref -- hits, with no more work; its t and slot are those of
 *        the FIRST accepted triangle.  A walk that would stack more than W_STACK items ends and reports max_stack INT32_MAX.
 * brute  every slot in slot order, the closest accepted triangle.
 */
#include "bih_oracle.c"

#define W_CLOSEST 0
#define W_FIRST 1
#define W_ANY 2
#define W_STACK 128
#define REF_LEAF 0x80000000u

/* ray_triangle (bih_oracle.c) operation for operation, also returning u and v; two_sided takes back faces too:
 * fabs((double)det) < 0.000001 instead of (double)det < 0.000001 (csrc/trace.cu MODE 4) */
static inline int ray_tri(const float* tri, const orc_ray* r, int two_sided, float* out_t, float* out_u, float* out_v) {
    float e1[3], e2[3], pvec[3], tvec[3], qvec[3];
    for (int k = 0; k < 3; k++) { e1[k] = tri[3 + k] - tri[k]; e2[k] = tri[6 + k] - tri[k]; }
    cross3(r->d, e2, pvec);
    float det = dot3(e1, pvec);
    if ((two_sided ? fabs((double)det) : (double)det) < 0.000001) return 0;
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

/* triangle records in slot order (prim: slot -> input triangle), no leaf flagged yet */
static void tri_records(const float* tri9, int64_t n, const uint32_t* prim, uint32_t* tris) {
    for (int64_t i = 0; i < n; i++) {
        const float* t = tri9 + 9 * (int64_t)prim[i];
        float* r = (float*)(tris + 12 * i);
        for (int k = 0; k < 3; k++) { r[k] = t[k]; r[3 + k] = t[3 + k] - t[k]; r[6 + k] = t[6 + k] - t[k]; }
        tris[12 * i + 9] = prim[i]; tris[12 * i + 10] = 0; tris[12 * i + 11] = (uint32_t)i;
    }
}

/* ------------------------------------------------------------------------------------------------------ parity blob */
/* hdr: 16 words; nodes: 16 x max(nu - 1, 0) words; tris: 12 x n words */
ORC_API void orc_parity_blob(const float* tri9, int64_t n, int64_t nu, const uint32_t* tris_idx, const uint32_t* cnt,
                             const int32_t* first, const float* clip, const int32_t* axis, const uint8_t* is_leaf,
                             const int32_t* children, const float* scene_lo, const float* scene_hi, uint32_t* hdr,
                             uint32_t* nodes, uint32_t* tris) {
    orc_scene s = { tri9, n, nu, tris_idx, cnt, first, clip, axis, is_leaf, children, {0, 0, 0}, {0, 0, 0} };
    memset(hdr, 0, 64);
    hdr[0] = (uint32_t)n; hdr[1] = (uint32_t)nu;
    memcpy(hdr + 2, scene_lo, 12); memcpy(hdr + 5, scene_hi, 12);
    hdr[9] = nu > 1 ? (uint32_t)axis[0] : 0u;
    tri_records(tri9, n, tris_idx, tris);
    for (int64_t l = 0; l < nu; l++) tris[12 * ((int64_t)first[l] + cnt[l] - 1) + 10] = 1u;
    if (nu < 2) return;
    float* cbox = (float*)malloc(sizeof(float) * 12 * (size_t)(nu - 1));
    children_boxes(&s, cbox);
    for (int64_t i = 0; i < nu - 1; i++) {
        float* nd = (float*)(nodes + 16 * i);
        nd[0] = clip[2 * i]; nd[1] = clip[2 * i + 1];
        for (int c = 0; c < 2; c++) {
            int32_t ch = children[2 * i + c];
            nodes[16 * i + 2 + c] = is_leaf[2 * i + c] ? REF_LEAF | (uint32_t)first[ch] << 2 : (uint32_t)ch << 2 | (uint32_t)axis[ch];
        }
        memcpy(nd + 4, cbox + 12 * i, 48);
    }
    free(cbox);
}

/* ------------------------------------------------------------------------------------------------------- quality build */
typedef struct {
    const float* tri9; int64_t n; int cap;
    const uint64_t* key;      /* by slot */
    const uint32_t* prim;     /* slot -> input triangle */
    uint32_t* nodes;          /* 16 words per node slot */
    uint32_t* tris;           /* 12 words per slot */
    uint8_t* reach;           /* node slot written */
    int64_t nu; int depth;
} q_build;

static inline uint64_t spread21(uint32_t q) {
    uint64_t x = 0;
    for (int b = 0; b < 21; b++) x |= (uint64_t)((q >> b) & 1u) << (3 * b);
    return x;
}

/* length of the common prefix of the strings of slots i and j: 64 key bits, then 32 bits of the slot position */
static inline int q_delta(const q_build* B, int64_t i, int64_t j) {
    uint64_t x = B->key[i] ^ B->key[j];
    if (x) return __builtin_clzll(x);
    uint32_t y = (uint32_t)i ^ (uint32_t)j;
    return 64 + (y ? __builtin_clz(y) : 32);
}

static void q_range_box(const q_build* B, int64_t a, int64_t b, float box[6]) {
    for (int k = 0; k < 3; k++) { box[k] = INFINITY; box[3 + k] = -INFINITY; }
    for (int64_t i = a; i <= b; i++) {
        const float* t = B->tri9 + 9 * (int64_t)B->prim[i];
        for (int v = 0; v < 3; v++) for (int k = 0; k < 3; k++) {
            box[k] = dev_fminf(box[k], t[3 * v + k]); box[3 + k] = dev_fmaxf(box[3 + k], t[3 * v + k]);
        }
    }
}

static inline uint32_t q_axis(const q_build* B, int64_t a, int64_t b) { return (uint32_t)((q_delta(B, a, b) + 2) % 3); }

/* node `idx` over slots [a, b] (more than cap of them) at depth `depth` (root = 1); writes its subtree, returns its box */
static void q_node(q_build* B, int64_t a, int64_t b, int64_t idx, int depth, float box[6]) {
    if (depth > B->depth) B->depth = depth;
    const int p = q_delta(B, a, b);
    int64_t lo = a, hi = b - 1;                       /* largest s in [a, b) with delta(a, s) > p: delta(a, .) is non-increasing */
    while (lo < hi) {
        int64_t mid = lo + (hi - lo + 1) / 2;
        if (q_delta(B, a, mid) > p) lo = mid; else hi = mid - 1;
    }
    const int64_t s = lo;
    const int64_t ca[2] = { a, s + 1 }, cb[2] = { s, b }, cn[2] = { s, s + 1 };
    float cbox[2][6];
    uint32_t ref[2];
    for (int c = 0; c < 2; c++) {
        if (cb[c] - ca[c] + 1 <= B->cap) {
            ref[c] = REF_LEAF | (uint32_t)ca[c] << 2;
            B->tris[12 * cb[c] + 10] = 1u;
            B->nu++;
            q_range_box(B, ca[c], cb[c], cbox[c]);
        } else {
            ref[c] = (uint32_t)cn[c] << 2 | q_axis(B, ca[c], cb[c]);
            q_node(B, ca[c], cb[c], cn[c], depth + 1, cbox[c]);
        }
    }
    const int ax = (p + 2) % 3;
    float* nd = (float*)(B->nodes + 16 * idx);
    nd[0] = cbox[0][3 + ax];
    nd[1] = cbox[1][ax];
    B->nodes[16 * idx + 2] = ref[0];
    B->nodes[16 * idx + 3] = ref[1];
    memcpy(nd + 4, cbox[0], 24);
    memcpy(nd + 10, cbox[1], 24);
    B->reach[idx] = 1;
    for (int k = 0; k < 3; k++) { box[k] = dev_fminf(cbox[0][k], cbox[1][k]); box[3 + k] = dev_fmaxf(cbox[0][3 + k], cbox[1][3 + k]); }
}

static const uint64_t* g_sort_key;
static int q_cmp(const void* x, const void* y) {
    uint32_t i = *(const uint32_t*)x, j = *(const uint32_t*)y;
    uint64_t a = g_sort_key[i], b = g_sort_key[j];
    if (a != b) return a < b ? -1 : 1;
    return i < j ? -1 : (i > j);
}

/* hdr: 16 words; nodes: 16 x max(n - 1, 0) words (zeroed here, reach[i] = 1 where written); tris: 12 x n words;
 * keys: n sorted keys (may be NULL).  Returns the depth in nodes of the deepest leaf (0: no node). */
ORC_API int orc_q_build(const float* tri9, int64_t n, int cap, uint32_t* hdr, uint32_t* nodes, uint8_t* reach, uint32_t* tris,
                        uint64_t* keys_out) {
    memset(hdr, 0, 64);
    if (n <= 0) return 0;
    float lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
    for (int64_t i = 0; i < 9 * n; i++) { lo[i % 3] = dev_fminf(lo[i % 3], tri9[i]); hi[i % 3] = dev_fmaxf(hi[i % 3], tri9[i]); }
    uint64_t* key = (uint64_t*)malloc(8 * (size_t)n);
    uint64_t* skey = (uint64_t*)malloc(8 * (size_t)n);
    uint32_t* prim = (uint32_t*)malloc(4 * (size_t)n);
    for (int64_t i = 0; i < n; i++) {
        const float* t = tri9 + 9 * i;
        uint64_t q3[3];
        for (int k = 0; k < 3; k++) {
            float mn = dev_fminf(dev_fminf(t[k], t[3 + k]), t[6 + k]), mx = dev_fmaxf(dev_fmaxf(t[k], t[3 + k]), t[6 + k]);
            float centre = (mn + mx) * 0.5f;
            float nrm = (centre - lo[k]) / (hi[k] - lo[k]);
            float q = dev_fminf(dev_fmaxf(nrm * 2097152.0f, 0.0f), 2097151.0f);
            q3[k] = spread21((uint32_t)q);
        }
        key[i] = q3[0] << 2 | q3[1] << 1 | q3[2];
        prim[i] = (uint32_t)i;
    }
    g_sort_key = key;
    qsort(prim, (size_t)n, 4, q_cmp);
    for (int64_t i = 0; i < n; i++) skey[i] = key[prim[i]];
    if (keys_out) memcpy(keys_out, skey, 8 * (size_t)n);
    tri_records(tri9, n, prim, tris);
    if (n > 1) { memset(nodes, 0, 64 * (size_t)(n - 1)); memset(reach, 0, (size_t)(n - 1)); }
    q_build B = { tri9, n, cap, skey, prim, nodes, tris, reach, 0, 0 };
    uint32_t root_axis = 0;
    if (n <= cap) { B.nu = 1; tris[12 * (n - 1) + 10] = 1u; }
    else { float box[6]; root_axis = q_axis(&B, 0, n - 1); q_node(&B, 0, n - 1, 0, 1, box); }
    hdr[0] = (uint32_t)n; hdr[1] = (uint32_t)B.nu;
    memcpy(hdr + 2, lo, 12); memcpy(hdr + 5, hi, 12);
    hdr[8] = 0; hdr[9] = root_axis; hdr[10] = 1;
    free(key); free(skey); free(prim);
    return B.depth;
}

/* -------------------------------------------------------------------------------------------------------------- walk */
typedef struct {
    const float* tri9; const uint32_t* hdr; const uint32_t* nodes; const uint32_t* tris;
    orc_scene s;              /* the scene box, for scene_slab */
} blob;

/* tests slot i: an accepted triangle becomes the hit; returns 1 when it was accepted */
static inline int test_slot(const blob* T, const orc_ray* r, uint32_t i, int two_sided, float tlo, float* ht, int* hs,
                            orc_counters* c) {
    float t, u, v;
    c->tris++;
    if (ray_tri(T->tri9 + 9 * (int64_t)T->tris[12 * (int64_t)i + 9], r, two_sided, &t, &u, &v) && t > tlo && t < *ht) {
        *ht = t; *hs = (int)i;
        return 1;
    }
    return 0;
}

/* the leaf starting at `slot`, up to its last-flagged triangle; returns 1 when the walk ends here */
static int leaf(const blob* T, const orc_ray* r, uint32_t slot, int exit_mode, int two_sided, float tlo, float* ht, int* hs,
                orc_counters* c) {
    for (uint32_t i = slot;; i++) {
        if (test_slot(T, r, i, two_sided, tlo, ht, hs, c) && exit_mode == W_FIRST) return 1;
        if (T->tris[12 * (int64_t)i + 10] & 1u) break;
    }
    return exit_mode != W_CLOSEST && *hs >= 0;
}

static void walk(const blob* T, const orc_ray* r, int exit_mode, int two_sided, float tlo, float* ht, int* hs, orc_counters* c) {
    float rMin, sMax;
    const uint32_t nu = T->hdr[1];
    const int strict = T->hdr[10] == 0;
    if (nu == 0) return;
    if (!scene_slab(&T->s, r, &rMin, &sMax)) return;
    if (nu == 1) { leaf(T, r, 0, exit_mode, two_sided, tlo, ht, hs, c); return; }
    float pMin = dev_fmaxf(rMin, tlo), pMax = sMax;
    struct { uint32_t ref; float rMin, pMin, pMax; } stack[W_STACK];
    int sp = 0;
    uint32_t cur = T->hdr[9];                         /* root: node 0 with its axis */
    orc_boxray q;
    make_boxray(&q, r, rMin, sMax);
    for (;;) {
        int next = 0;
        if (pMin <= dev_fminf(pMax, *ht)) {
            pMax = dev_fminf(pMax, *ht);
            if (cur & REF_LEAF) {
                if (leaf(T, r, (cur & 0x7FFFFFFFu) >> 2, exit_mode, two_sided, tlo, ht, hs, c)) break;
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
                    if (!(refn & REF_LEAF) && (reff & REF_LEAF)) {    /* a far LEAF next to a near NODE is tested first */
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

static void brute(const blob* T, const orc_ray* r, int two_sided, float tlo, float* ht, int* hs, orc_counters* c) {
    for (uint32_t i = 0; i < T->hdr[0]; i++) test_slot(T, r, i, two_sided, tlo, ht, hs, c);
}

/* brute_force 0: the walk with exit_mode (W_*), 1: brute force.  rays8: o.xyz tmin d.xyz tmax per ray; h.t starts at
 * min(tmax, ht_max): bihrt_intersect passes FLT_MAX, bihrt_trace_any tmax as given (ht_max = inf).  A ray with
 * !(max(tmin, 0) < tmax), NaN bounds included, misses without a walk.  The record of a hit is computed after the walk from
 * its slot, as the kernel's epilogue does: u, v by ray_tri, ng = e1 x e2 with rounded products.  Outputs (each may be
 * NULL): t, u, v, slot, prim, ng (3 per ray), a miss is (FLT_MAX, 0, 0, -1, -1, 0 0 0); stack: the deepest stack of each ray;
 * counters3: total nodes, total triangle tests, deepest stack. */
ORC_API void orc_walk(const float* tri9, const uint32_t* hdr, const uint32_t* nodes, const uint32_t* tris, int brute_force,
                      int exit_mode, int two_sided, float ht_max, const float* rays8, int64_t nrays, float* out_t,
                      float* out_u, float* out_v, int32_t* out_slot, int32_t* out_prim, float* out_ng, int32_t* out_stack,
                      uint64_t* counters3, int nthreads) {
    blob T;
    memset(&T, 0, sizeof T);
    T.tri9 = tri9; T.hdr = hdr; T.nodes = nodes; T.tris = tris;
    memcpy(T.s.scene_lo, hdr + 2, 12); memcpy(T.s.scene_hi, hdr + 5, 12);
    uint64_t tot_nodes = 0, tot_tris = 0; int max_stack = 0;
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
        const float tmin = r8[3], tmax = r8[7], tlo = dev_fmaxf(tmin, 0.0f);
        float ht = dev_fminf(tmax, ht_max); int hs = -1;
        orc_counters c = { 0, 0, 0 };
        if (tmin == tmin && tlo < tmax) {
            if (brute_force) brute(&T, &r, two_sided, tlo, &ht, &hs, &c);
            else walk(&T, &r, exit_mode, two_sided, tlo, &ht, &hs, &c);
        }
        float t = FLT_MAX, u = 0.0f, v = 0.0f, g[3] = { 0.0f, 0.0f, 0.0f };
        if (hs >= 0) {
            const float* tri = tri9 + 9 * (int64_t)tris[12 * (int64_t)hs + 9];
            float tt;
            ray_tri(tri, &r, two_sided, &tt, &u, &v);
            t = ht;
            float e1[3], e2[3];
            for (int k = 0; k < 3; k++) { e1[k] = tri[3 + k] - tri[k]; e2[k] = tri[6 + k] - tri[k]; }
            g[0] = e1[1] * e2[2] - e1[2] * e2[1];
            g[1] = e1[2] * e2[0] - e1[0] * e2[2];
            g[2] = e1[0] * e2[1] - e1[1] * e2[0];
        }
        if (out_t) out_t[i] = t;
        if (out_u) out_u[i] = u;
        if (out_v) out_v[i] = v;
        if (out_slot) out_slot[i] = hs;
        if (out_prim) out_prim[i] = hs >= 0 ? (int32_t)tris[12 * (int64_t)hs + 9] : -1;
        if (out_ng) { out_ng[3 * i] = g[0]; out_ng[3 * i + 1] = g[1]; out_ng[3 * i + 2] = g[2]; }
        if (out_stack) out_stack[i] = c.max_stack;
        tot_nodes += c.nodes; tot_tris += c.tris;
        if (c.max_stack > max_stack) max_stack = c.max_stack;
    }
    if (counters3) { counters3[0] = tot_nodes; counters3[1] = tot_tris; counters3[2] = (uint64_t)max_stack; }
}
