/*
 * winding_oracle.c -- CPU restatement of bihrt_winding_number (csrc/winding.cu: the far-field table and k_winding) on the blob
 * bihrt_bih_export writes, for both tree kinds.  TEST INFRASTRUCTURE ONLY, built by tests/winding_oracle.py into a temporary
 * directory, with -ffp-contract=off so that every product and sum is rounded on its own, as the kernel's explicit __f*_rn are.
 *
 * Written from the statement in include/bihrt.h (solid angle, atan2, far test, walk order, accumulation) and DESIGN.md section 9
 * (the table's content and construction order, the far-field term's operation order), not from the kernel's source.  The table
 * is built here by a recursion from the root (the kernel: a top-down queue pass and a bottom-up pass with arrival counters);
 * both give every record by the same fixed-order arithmetic.
 *
 * Blob words as in closest_oracle.c: header (16 words: n, nu, scene box, status, root_axis, quality, ...), node slots (16
 * words: clip0, clip1, left and right child references, the left and right child's box lo.xyz hi.xyz), triangle records (12
 * words: v0, e1, e2, prim, last, slot).
 */
#include <math.h>
#include <stdint.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

#define ORC_API __attribute__((visibility("default")))
#define W_STACK 128
#define W_REF_LEAF 0x80000000u
#define W_REC 32                       /* floats per child record: N[3], M[9] row-major, Q[i][00 01 02 11 12 22], 2 unused */

static const int JJ[6] = { 0, 0, 0, 1, 1, 2 }, KK[6] = { 0, 1, 2, 1, 2, 2 };

static inline float w_dot(const float a[3], const float b[3]) { return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]; }

/* the header's atan2f_bihrt */
ORC_API float orc_atan2(float y, float x) {
    float ax = fabsf(x), ay = fabsf(y);
    float mx = ax > ay ? ax : ay, mn = ax > ay ? ay : ax;
    float t = mn / mx, off = 0.0f;
    if (t > 0.41421356f) { t = (t - 1.0f) / (t + 1.0f); off = 0.78539819f; }
    float z = t * t;
    float r = (((((0.0805374449538f * z - 0.138776856032f) * z + 0.199777106478f) * z - 0.333329491539f) * z) * t + t) + off;
    if (ay > ax) r = 1.57079637f - r;
    if (x < 0.0f) r = 3.14159274f - r;
    return y < 0.0f ? -r : r;
}

ORC_API void orc_atan2_many(const float* y, const float* x, float* out, int64_t n) {
    for (int64_t i = 0; i < n; i++) out[i] = orc_atan2(y[i], x[i]);
}

/* Omega / 2 of triangle record r (v0, e1, e2) at p */
static float w_half_angle(const float* p, const float* r) {
    float a[3], b[3], c[3], bc[3];
    for (int k = 0; k < 3; k++) { a[k] = r[k] - p[k]; b[k] = a[k] + r[3 + k]; c[k] = a[k] + r[6 + k]; }
    bc[0] = b[1] * c[2] - b[2] * c[1];
    bc[1] = b[2] * c[0] - b[0] * c[2];
    bc[2] = b[0] * c[1] - b[1] * c[0];
    float det = w_dot(a, bc);
    if (det == 0.0f) return 0.0f;
    float la = sqrtf(w_dot(a, a)), lb = sqrtf(w_dot(b, b)), lc = sqrtf(w_dot(c, c));
    float den = (((la * lb) * lc + w_dot(a, b) * lc) + w_dot(a, c) * lb) + w_dot(b, c) * la;
    return orc_atan2(det, den);
}

static void w_centre(const float* box, float c[3]) {
    for (int k = 0; k < 3; k++) c[k] = (box[k] + box[3 + k]) * 0.5f;
}

/* record of a leaf: its triangles from slot s to the `last` flag, in slot order, about centre c */
static void w_leaf_rec(const uint32_t* tris, uint32_t s, const float c[3], float* e) {
    memset(e, 0, W_REC * sizeof(float));
    for (;; s++) {
        const float* r = (const float*)(tris + 12 * (int64_t)s);
        const float *e1 = r + 3, *e2 = r + 6;
        float h[3] = { (e1[1] * e2[2] - e1[2] * e2[1]) * 0.5f, (e1[2] * e2[0] - e1[0] * e2[2]) * 0.5f,
                       (e1[0] * e2[1] - e1[1] * e2[0]) * 0.5f };
        float v[3][3], S[3], m[3], E[6];
        for (int k = 0; k < 3; k++) {
            v[0][k] = r[k] - c[k];
            v[1][k] = v[0][k] + e1[k];
            v[2][k] = v[0][k] + e2[k];
            S[k] = (v[0][k] + v[1][k]) + v[2][k];
            m[k] = S[k] / 3.0f;
        }
        for (int t = 0; t < 6; t++) {
            int j = JJ[t], k = KK[t];
            E[t] = (((v[0][j] * v[0][k] + v[1][j] * v[1][k]) + v[2][j] * v[2][k]) + S[j] * S[k]) / 12.0f;
        }
        for (int i = 0; i < 3; i++) {
            e[i] += h[i];
            for (int k = 0; k < 3; k++) e[3 + 3 * i + k] += h[i] * m[k];
            for (int t = 0; t < 6; t++) e[12 + 6 * i + t] += h[i] * E[t];
        }
        if (tris[12 * (int64_t)s + 10] & 1u) break;
    }
}

/* record of an internal child X about centre cx: X's two records (left, then right) shifted by d = their centre - cx */
static void w_combine(const float* recs, const float* xnode, const float cx[3], float* e) {
    memset(e, 0, W_REC * sizeof(float));
    for (int side = 0; side < 2; side++) {
        const float* r = recs + W_REC * side;
        float cc[3], d[3];
        w_centre(xnode + 4 + 6 * side, cc);
        for (int k = 0; k < 3; k++) d[k] = cc[k] - cx[k];
        for (int i = 0; i < 3; i++) {
            e[i] += r[i];
            for (int k = 0; k < 3; k++) e[3 + 3 * i + k] += r[3 + 3 * i + k] + r[i] * d[k];
            for (int t = 0; t < 6; t++) {
                int j = JJ[t], k = KK[t];
                e[12 + 6 * i + t] += ((r[12 + 6 * i + t] + r[3 + 3 * i + j] * d[k]) + r[3 + 3 * i + k] * d[j]) + r[i] * (d[j] * d[k]);
            }
        }
    }
}

/* the records of both children of node x (recursively below it) */
static void w_table_node(const uint32_t* nodes, const uint32_t* tris, uint32_t x, float* tab) {
    const uint32_t* nw = nodes + 16 * (int64_t)x;
    for (int side = 0; side < 2; side++) {
        uint32_t ref = nw[2 + side];
        float c[3];
        w_centre((const float*)nw + 4 + 6 * side, c);
        float* dst = tab + (2 * (int64_t)x + side) * W_REC;
        if (ref & W_REF_LEAF) w_leaf_rec(tris, (ref & 0x7FFFFFFFu) >> 2, c, dst);
        else {
            uint32_t y = (ref & 0x7FFFFFFFu) >> 2;
            w_table_node(nodes, tris, y, tab);
            w_combine(tab + 2 * (int64_t)y * W_REC, (const float*)(nodes + 16 * (int64_t)y), c, dst);
        }
    }
}

/* tab: (number of node slots) x 2 x W_REC floats; slots the tree does not reach are left as they are */
ORC_API void orc_wtab(const uint32_t* hdr, const uint32_t* nodes, const uint32_t* tris, float* tab) {
    if (hdr[1] >= 2) w_table_node(nodes, tris, 0, tab);
}

/* the far-field term of record e at p, with R = c - p, d2 = R.R (DESIGN.md section 9) */
static float w_far(const float* e, const float R[3], float d2) {
    float ir = 1.0f / sqrtf(d2);
    float u[3] = { R[0] * ir, R[1] * ir, R[2] * ir };
    float t0 = (w_dot(u, e) * ir) * ir;
    float mu[3] = { w_dot(e + 3, u), w_dot(e + 6, u), w_dot(e + 9, u) };
    float trm = (e[3] + e[7]) + e[11];
    float t1 = (((trm - 3.0f * w_dot(u, mu)) * ir) * ir) * ir;
    float qu[3][3], trq[3], uqu[3];
    for (int i = 0; i < 3; i++) {
        const float* q = e + 12 + 6 * i;
        float row0[3] = { q[0], q[1], q[2] }, row1[3] = { q[1], q[3], q[4] }, row2[3] = { q[2], q[4], q[5] };
        qu[i][0] = w_dot(row0, u); qu[i][1] = w_dot(row1, u); qu[i][2] = w_dot(row2, u);
        trq[i] = (q[0] + q[3]) + q[5];
        uqu[i] = w_dot(u, qu[i]);
    }
    float A = (qu[0][0] + qu[1][1]) + qu[2][2];
    float B = w_dot(u, trq), Cc = w_dot(u, uqu);
    float g = 15.0f * Cc - 3.0f * (2.0f * A + B);
    float t2 = ((((g * 0.5f) * ir) * ir) * ir) * ir;
    return (t0 + t1) + t2;
}

/* far test of a child box: sets R = c - p and d2 */
static int w_is_far(const float* box, const float* p, float b2, float R[3], float* d2) {
    float c[3], ext[3];
    w_centre(box, c);
    for (int k = 0; k < 3; k++) { R[k] = c[k] - p[k]; ext[k] = box[3 + k] - box[k]; }
    *d2 = w_dot(R, R);
    return *d2 > b2 * (w_dot(ext, ext) * 0.25f);
}

/* pts4: p.xyz (rmax ignored).  brute 1: every slot in slot order, exactly.  b2 = fl(beta * beta).  counters3: internal nodes
 * stepped, far-field terms, exact triangle terms. */
ORC_API void orc_winding(const uint32_t* hdr, const uint32_t* nodes, const uint32_t* tris, const float* tab, int brute, float b2,
                         const float* pts4, int64_t npts, float* out_w, uint64_t* counters3, int nthreads) {
    const uint32_t n = hdr[0], nu = hdr[1];
    uint64_t tot_nodes = 0, tot_far = 0, tot_exact = 0;
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 64) num_threads(nthreads) reduction(+:tot_nodes, tot_far, tot_exact)
#else
    (void)nthreads;
#endif
    for (int64_t i = 0; i < npts; i++) {
        const float* p = pts4 + 4 * i;
        double acc = 0.0;
        if (fabsf(p[0]) <= 3.402823466e38f && fabsf(p[1]) <= 3.402823466e38f && fabsf(p[2]) <= 3.402823466e38f) {
            if (brute) {
                for (uint32_t s = 0; s < n; s++) acc += 2.0 * (double)w_half_angle(p, (const float*)(tris + 12 * (int64_t)s));
                tot_exact += n;
            } else if (nu == 1) {
                for (uint32_t s = 0;; s++) {
                    acc += 2.0 * (double)w_half_angle(p, (const float*)(tris + 12 * (int64_t)s));
                    tot_exact++;
                    if (tris[12 * (int64_t)s + 10] & 1u) break;
                }
            } else if (nu > 1) {
                /* stack items: a child reference to walk, or (kind 1) a far child (node, side) whose term is still due */
                struct { int kind; uint32_t ref, node, side; } st[W_STACK];
                int sp = 0;
                st[sp].kind = 0; st[sp].ref = 0; sp++;               /* the root: node 0 */
                while (sp > 0) {
                    sp--;
                    if (st[sp].kind == 1) {
                        const float* box = (const float*)(nodes + 16 * (int64_t)st[sp].node) + 4 + 6 * st[sp].side;
                        float R[3], d2;
                        w_is_far(box, p, b2, R, &d2);
                        acc += (double)w_far(tab + (2 * (int64_t)st[sp].node + st[sp].side) * W_REC, R, d2);
                        tot_far++;
                        continue;
                    }
                    uint32_t ref = st[sp].ref;
                    if (ref & W_REF_LEAF) {
                        for (uint32_t s = (ref & 0x7FFFFFFFu) >> 2;; s++) {
                            acc += 2.0 * (double)w_half_angle(p, (const float*)(tris + 12 * (int64_t)s));
                            tot_exact++;
                            if (tris[12 * (int64_t)s + 10] & 1u) break;
                        }
                        continue;
                    }
                    uint32_t x = ref >> 2;
                    const uint32_t* nw = nodes + 16 * (int64_t)x;
                    tot_nodes++;
                    /* depth first, left before right: push right, then left; a far child is pushed as its term */
                    for (int side = 1; side >= 0; side--) {
                        float R[3], d2;
                        if (sp == W_STACK) { sp = 0; acc = NAN; break; }
                        if (w_is_far((const float*)nw + 4 + 6 * side, p, b2, R, &d2)) {
                            st[sp].kind = 1; st[sp].node = x; st[sp].side = (uint32_t)side;
                        } else {
                            st[sp].kind = 0; st[sp].ref = nw[2 + side];
                        }
                        sp++;
                    }
                }
            }
        }
        out_w[i] = (float)(acc * 0.079577471545947673);
    }
    if (counters3) { counters3[0] = tot_nodes; counters3[1] = tot_far; counters3[2] = tot_exact; }
}

/* float64 reference: the exact solid-angle sum over the input triangles (n x 9 floats, v0 v1 v2), binary64 and libm atan2 */
ORC_API void orc_winding64(const float* tri9, int64_t n, const float* pts3, int64_t npts, double* out_w, int nthreads) {
#ifdef _OPENMP
    if (nthreads <= 0) nthreads = omp_get_max_threads();
#pragma omp parallel for schedule(dynamic, 16) num_threads(nthreads)
#else
    (void)nthreads;
#endif
    for (int64_t i = 0; i < npts; i++) {
        const double px = pts3[3 * i], py = pts3[3 * i + 1], pz = pts3[3 * i + 2];
        double acc = 0.0;
        for (int64_t t = 0; t < n; t++) {
            const float* v = tri9 + 9 * t;
            double a[3] = { v[0] - px, v[1] - py, v[2] - pz }, b[3] = { v[3] - px, v[4] - py, v[5] - pz },
                   c[3] = { v[6] - px, v[7] - py, v[8] - pz };
            double det = a[0] * (b[1] * c[2] - b[2] * c[1]) + a[1] * (b[2] * c[0] - b[0] * c[2]) + a[2] * (b[0] * c[1] - b[1] * c[0]);
            double la = sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]), lb = sqrt(b[0] * b[0] + b[1] * b[1] + b[2] * b[2]),
                   lc = sqrt(c[0] * c[0] + c[1] * c[1] + c[2] * c[2]);
            double den = la * lb * lc + (a[0] * b[0] + a[1] * b[1] + a[2] * b[2]) * lc + (a[0] * c[0] + a[1] * c[1] + a[2] * c[2]) * lb +
                         (b[0] * c[0] + b[1] * c[1] + b[2] * c[2]) * la;
            if (det != 0.0) acc += 2.0 * atan2(det, den);
        }
        out_w[i] = acc / (4.0 * 3.14159265358979323846);
    }
}
