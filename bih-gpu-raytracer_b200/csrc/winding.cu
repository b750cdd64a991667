// Winding-number queries on sm_100a (bihrt_winding_number, include/bihrt.h): for every point, (1/4pi) x the sum of the signed
// solid angles of all triangles, with far clusters replaced by an order-2 Taylor expansion (Barill et al. 2018).
//
// Far-field table (built lazily, DESIGN.md section 9)
//   * per node slot, one 128-byte record per child: the child's area vector N, first moments M and second moments Q about the
//     centre of the child's box in the parent's BihNode (WTAB_FLOATS floats, bihrt_internal.cuh);
//   * k_wtab_down: persistent warps (one active lane each) take the reachable nodes from a device queue in discovery order,
//     starting at the root, and record each internal child's parent and each leaf child's (parent, side).  A quality tree's
//     stale node slots are never queued;
//   * k_wtab_up: one thread per leaf child sums its triangles in slot order into the record, then climbs: the second of the two
//     children of a node to arrive (per-node counter, fences around it) combines them, left then right, shifted to the node's
//     own centre, into the node's record in its parent.  Every combination has a fixed operation order, so the table does not
//     depend on which thread arrives last.
// Query
//   * k_winding<Q>: persistent warps, units of 32 points, one lane per point (the shape of k_closest).  Depth first, left child
//     before right.  At a node, both children's far tests use the boxes of the loaded 64-byte record; a far child's 128-byte
//     table record is fetched only then.  A far right child whose left sibling is descended is pushed as a marker (a leaf
//     reference with a nonzero axis field, which real leaf references never have) so that its term is added after the left
//     subtree's: terms are accumulated in binary64 in walk order.
// Everything that decides a result is IEEE binary32 with explicit __f*_rn (no contraction), restated on the CPU by
// tests/winding_oracle.c.
#include "bihrt_internal.cuh"
#include <float.h>

#define FULL 0xffffffffu
#define NONE 0xFFFFFFFFu
#define WINDING_THREADS 128
#define WINDING_MIN_BLOCKS 8
#define WQ_EMPTY 0xFFFFFFFFu
#define WQ_SPIN_LIMIT (1u << 24)        // polls of an empty queue cell before the table build gives up (a corrupt blob)
#define INV_4PI 0.079577471545947673    // 1 / (4 pi), binary64

__device__ __forceinline__ float wdot(float ax, float ay, float az, float bx, float by, float bz) {
    return __fadd_rn(__fadd_rn(__fmul_rn(ax, bx), __fmul_rn(ay, by)), __fmul_rn(az, bz));
}

// atan2 with a fixed operation order (include/bihrt.h): range reduction to [0, 1], then to [-0.1716, 0.4142], Cephes' atanf
// polynomial
__device__ __forceinline__ float atan2_bihrt(float y, float x) {
    const float ax = fabsf(x), ay = fabsf(y);
    const float mx = fmaxf(ax, ay), mn = fminf(ax, ay);
    float t = __fdiv_rn(mn, mx), off = 0.f;
    if (t > 0.41421356f) { t = __fdiv_rn(__fsub_rn(t, 1.f), __fadd_rn(t, 1.f)); off = 0.78539819f; }
    const float z = __fmul_rn(t, t);
    float p = __fsub_rn(__fmul_rn(0.0805374449538f, z), 0.138776856032f);
    p = __fadd_rn(__fmul_rn(p, z), 0.199777106478f);
    p = __fsub_rn(__fmul_rn(p, z), 0.333329491539f);
    float r = __fadd_rn(__fadd_rn(__fmul_rn(__fmul_rn(p, z), t), t), off);
    if (ay > ax) r = __fsub_rn(1.57079637f, r);
    if (x < 0.f) r = __fsub_rn(3.14159274f, r);
    return y < 0.f ? -r : r;
}

// Omega / 2 of the triangle record (v0, e1, e2) seen from p (Van Oosterom & Strackee); 0 when det == 0
__device__ __forceinline__ float tri_half_angle(float px, float py, float pz, float4 q0, float4 q1, float4 q2) {
    const float ax = __fsub_rn(q0.x, px), ay = __fsub_rn(q0.y, py), az = __fsub_rn(q0.z, pz);
    const float bx = __fadd_rn(ax, q0.w), by = __fadd_rn(ay, q1.x), bz = __fadd_rn(az, q1.y);
    const float cx = __fadd_rn(ax, q1.z), cy = __fadd_rn(ay, q1.w), cz = __fadd_rn(az, q2.x);
    const float X = __fsub_rn(__fmul_rn(by, cz), __fmul_rn(bz, cy));
    const float Y = __fsub_rn(__fmul_rn(bz, cx), __fmul_rn(bx, cz));
    const float Z = __fsub_rn(__fmul_rn(bx, cy), __fmul_rn(by, cx));
    const float det = wdot(ax, ay, az, X, Y, Z);
    if (det == 0.f) return 0.f;
    const float la = __fsqrt_rn(wdot(ax, ay, az, ax, ay, az));
    const float lb = __fsqrt_rn(wdot(bx, by, bz, bx, by, bz));
    const float lc = __fsqrt_rn(wdot(cx, cy, cz, cx, cy, cz));
    float den = __fadd_rn(__fmul_rn(__fmul_rn(la, lb), lc), __fmul_rn(wdot(ax, ay, az, bx, by, bz), lc));
    den = __fadd_rn(den, __fmul_rn(wdot(ax, ay, az, cx, cy, cz), lb));
    den = __fadd_rn(den, __fmul_rn(wdot(bx, by, bz, cx, cy, cz), la));
    return atan2_bihrt(det, den);
}

// the order-2 far-field term of the table record e (about centre c) at p, with R = c - p and d2 = R.R > 0
__device__ __forceinline__ float far_term(const float* e, float Rx, float Ry, float Rz, float d2) {
    const float ir = __fdiv_rn(1.f, __fsqrt_rn(d2));
    const float ux = __fmul_rn(Rx, ir), uy = __fmul_rn(Ry, ir), uz = __fmul_rn(Rz, ir);
    const float t0 = __fmul_rn(__fmul_rn(wdot(ux, uy, uz, e[0], e[1], e[2]), ir), ir);
    const float mu0 = wdot(e[3], e[4], e[5], ux, uy, uz), mu1 = wdot(e[6], e[7], e[8], ux, uy, uz), mu2 = wdot(e[9], e[10], e[11], ux, uy, uz);
    const float umu = wdot(ux, uy, uz, mu0, mu1, mu2);
    const float trm = __fadd_rn(__fadd_rn(e[3], e[7]), e[11]);
    const float t1 = __fmul_rn(__fmul_rn(__fmul_rn(__fsub_rn(trm, __fmul_rn(3.f, umu)), ir), ir), ir);
    float qu[3][3], trq[3];
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const float* q = e + 12 + 6 * i;            // Q_i00 Q_i01 Q_i02 Q_i11 Q_i12 Q_i22
        qu[i][0] = wdot(q[0], q[1], q[2], ux, uy, uz);
        qu[i][1] = wdot(q[1], q[3], q[4], ux, uy, uz);
        qu[i][2] = wdot(q[2], q[4], q[5], ux, uy, uz);
        trq[i] = __fadd_rn(__fadd_rn(q[0], q[3]), q[5]);
    }
    const float A = __fadd_rn(__fadd_rn(qu[0][0], qu[1][1]), qu[2][2]);
    const float B = wdot(ux, uy, uz, trq[0], trq[1], trq[2]);
    const float C = wdot(ux, uy, uz, wdot(ux, uy, uz, qu[0][0], qu[0][1], qu[0][2]), wdot(ux, uy, uz, qu[1][0], qu[1][1], qu[1][2]),
                         wdot(ux, uy, uz, qu[2][0], qu[2][1], qu[2][2]));
    const float g = __fsub_rn(__fmul_rn(15.f, C), __fmul_rn(3.f, __fadd_rn(__fmul_rn(2.f, A), B)));
    const float t2 = __fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(__fmul_rn(g, 0.5f), ir), ir), ir), ir);
    return __fadd_rn(__fadd_rn(t0, t1), t2);
}

// ---------------------------------------------------------------------------------------------- table build

__device__ __forceinline__ void box_centre(const float* b, float& cx, float& cy, float& cz) {
    cx = __fmul_rn(__fadd_rn(b[0], b[3]), 0.5f);
    cy = __fmul_rn(__fadd_rn(b[1], b[4]), 0.5f);
    cz = __fmul_rn(__fadd_rn(b[2], b[5]), 0.5f);
}

__device__ __forceinline__ void store_rec(float* dst, const float* e) {
    float4* d = reinterpret_cast<float4*>(dst);
#pragma unroll
    for (int k = 0; k < WTAB_FLOATS / 4; k++) __stcg(d + k, make_float4(e[4 * k], e[4 * k + 1], e[4 * k + 2], e[4 * k + 3]));
}

__device__ __forceinline__ void load_rec_cg(const float* src, float* e) {
    const float4* s = reinterpret_cast<const float4*>(src);
#pragma unroll
    for (int k = 0; k < WTAB_FLOATS / 4; k++) { const float4 v = __ldcg(s + k); e[4 * k] = v.x; e[4 * k + 1] = v.y; e[4 * k + 2] = v.z; e[4 * k + 3] = v.w; }
}

// scratch words: queue [ns] | parent [ns] | leaf list [ns] | arrivals [ns] | counters (grab, queue tail, leaf tail)
__global__ void __launch_bounds__(WINDING_THREADS) k_wtab_down(const BihHeader* hdr, const BihNode* nodes, uint32_t* scr, uint32_t ns,
                                                               uint32_t* status_map) {
    if (hdr->status != 0 || (threadIdx.x & 31) != 0) return;
    const uint32_t nu = hdr->nu;
    if (nu < 2) return;
    uint32_t* queue = scr; uint32_t* parent = scr + ns; uint32_t* leaves = scr + 2 * (size_t)ns; uint32_t* cnt = scr + 4 * (size_t)ns;
    for (;;) {
        const uint32_t k = atomicAdd(&cnt[0], 1u);
        if (k >= nu - 1) break;                  // a tree of nu leaves has nu - 1 internal nodes, all reachable
        uint32_t node = 0;
        if (k > 0) {
            uint32_t spins = 0;
            while ((node = ld_relaxed(queue + k)) == WQ_EMPTY) {
                if (++spins == WQ_SPIN_LIMIT) { if (status_map) *status_map = 0x200u; return; }
                __nanosleep(64);
            }
        }
        const uint4 nd = __ldg(reinterpret_cast<const uint4*>(nodes + node));
        const uint32_t refs[2] = { nd.z, nd.w };
#pragma unroll
        for (int side = 0; side < 2; side++) {
            const uint32_t ref = refs[side];
            if (ref & BIH_REF_LEAF) leaves[atomicAdd(&cnt[2], 1u)] = node * 2u + side;
            else {
                const uint32_t ch = BIH_REF_INDEX(ref);
                parent[ch] = node * 2u + side;
                st_relaxed(queue + 1 + atomicAdd(&cnt[1], 1u), ch);
            }
        }
    }
}

__global__ void __launch_bounds__(WINDING_THREADS) k_wtab_up(const BihHeader* hdr, const BihNode* nodes, const BihTri* tris, float* wtab,
                                                             uint32_t* scr, uint32_t ns) {
    if (hdr->status != 0) return;
    const uint32_t* parent = scr + ns; const uint32_t* leaves = scr + 2 * (size_t)ns; uint32_t* arrive = scr + 3 * (size_t)ns;
    const uint32_t* cnt = scr + 4 * (size_t)ns;
    const uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    if (hdr->nu < 2 || j >= cnt[2]) return;
    const uint32_t le = leaves[j];
    uint32_t P = le >> 1, side = le & 1u;
    float e[WTAB_FLOATS];
#pragma unroll
    for (int k = 0; k < WTAB_FLOATS; k++) e[k] = 0.f;
    {
        const BihNode* nd = nodes + P;
        float cx, cy, cz;
        box_centre(side ? nd->rbox : nd->lbox, cx, cy, cz);
        const float4* tp = reinterpret_cast<const float4*>(tris) + 3 * (size_t)BIH_REF_INDEX(side ? nd->ref_r : nd->ref_l);
        for (;;) {
            const float4 q0 = __ldg(tp), q1 = __ldg(tp + 1), q2 = __ldg(tp + 2);
            const float e1[3] = { q0.w, q1.x, q1.y }, e2[3] = { q1.z, q1.w, q2.x };
            const float h[3] = { __fmul_rn(__fsub_rn(__fmul_rn(e1[1], e2[2]), __fmul_rn(e1[2], e2[1])), 0.5f),
                                 __fmul_rn(__fsub_rn(__fmul_rn(e1[2], e2[0]), __fmul_rn(e1[0], e2[2])), 0.5f),
                                 __fmul_rn(__fsub_rn(__fmul_rn(e1[0], e2[1]), __fmul_rn(e1[1], e2[0])), 0.5f) };
            const float s0[3] = { __fsub_rn(q0.x, cx), __fsub_rn(q0.y, cy), __fsub_rn(q0.z, cz) };
            float s1[3], s2[3], S[3], m[3];
#pragma unroll
            for (int k = 0; k < 3; k++) {
                s1[k] = __fadd_rn(s0[k], e1[k]); s2[k] = __fadd_rn(s0[k], e2[k]);
                S[k] = __fadd_rn(__fadd_rn(s0[k], s1[k]), s2[k]);
                m[k] = __fdiv_rn(S[k], 3.f);
            }
            float E[6];
            {
                const int jj[6] = { 0, 0, 0, 1, 1, 2 }, kk[6] = { 0, 1, 2, 1, 2, 2 };
#pragma unroll
                for (int t = 0; t < 6; t++) {
                    const int a = jj[t], b = kk[t];
                    const float acc = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(s0[a], s0[b]), __fmul_rn(s1[a], s1[b])), __fmul_rn(s2[a], s2[b])),
                                                __fmul_rn(S[a], S[b]));
                    E[t] = __fdiv_rn(acc, 12.f);
                }
            }
#pragma unroll
            for (int i = 0; i < 3; i++) {
                e[i] = __fadd_rn(e[i], h[i]);
#pragma unroll
                for (int k = 0; k < 3; k++) e[3 + 3 * i + k] = __fadd_rn(e[3 + 3 * i + k], __fmul_rn(h[i], m[k]));
#pragma unroll
                for (int t = 0; t < 6; t++) e[12 + 6 * i + t] = __fadd_rn(e[12 + 6 * i + t], __fmul_rn(h[i], E[t]));
            }
            if (__float_as_uint(q2.z) & 1u) break;
            tp += 3;
        }
    }
    store_rec(wtab + (2 * (size_t)P + side) * WTAB_FLOATS, e);
    // climb: the second child of a node to arrive combines both into the node's record in its parent
    for (uint32_t X = P; X != 0;) {
        __threadfence();
        if (atomicAdd(&arrive[X], 1u) == 0) return;
        __threadfence();
        const BihNode* nx = nodes + X;
        const uint32_t pe = __ldcg(parent + X);
        const uint32_t PP = pe >> 1, ps = pe & 1u;
        const BihNode* np = nodes + PP;
        float xc[3];
        box_centre(ps ? np->rbox : np->lbox, xc[0], xc[1], xc[2]);
#pragma unroll
        for (int k = 0; k < WTAB_FLOATS; k++) e[k] = 0.f;
#pragma unroll
        for (int c = 0; c < 2; c++) {
            float r[WTAB_FLOATS], cc[3], d[3];
            load_rec_cg(wtab + (2 * (size_t)X + c) * WTAB_FLOATS, r);
            box_centre(c ? nx->rbox : nx->lbox, cc[0], cc[1], cc[2]);
#pragma unroll
            for (int k = 0; k < 3; k++) d[k] = __fsub_rn(cc[k], xc[k]);
            const int jj[6] = { 0, 0, 0, 1, 1, 2 }, kk[6] = { 0, 1, 2, 1, 2, 2 };
#pragma unroll
            for (int i = 0; i < 3; i++) {
                e[i] = __fadd_rn(e[i], r[i]);
#pragma unroll
                for (int k = 0; k < 3; k++)
                    e[3 + 3 * i + k] = __fadd_rn(e[3 + 3 * i + k], __fadd_rn(r[3 + 3 * i + k], __fmul_rn(r[i], d[k])));
#pragma unroll
                for (int t = 0; t < 6; t++) {
                    const int a = jj[t], b = kk[t];
                    float q = __fadd_rn(r[12 + 6 * i + t], __fmul_rn(r[3 + 3 * i + a], d[b]));
                    q = __fadd_rn(q, __fmul_rn(r[3 + 3 * i + b], d[a]));
                    q = __fadd_rn(q, __fmul_rn(r[i], __fmul_rn(d[a], d[b])));
                    e[12 + 6 * i + t] = __fadd_rn(e[12 + 6 * i + t], q);
                }
            }
        }
        store_rec(wtab + (2 * (size_t)PP + ps) * WTAB_FLOATS, e);
        X = PP;
    }
}

int bihrt_winding_table_launch(bihrt_ctx* c) {
    const uint32_t ns = (uint32_t)c->wtab_slots;
    uint32_t* scr = c->d_wscratch;
    BIHRT_CUDA(c, cudaMemsetAsync(scr, 0xFF, (size_t)ns * 4, c->stream));                              // empty queue cells
    BIHRT_CUDA(c, cudaMemsetAsync(scr + 3 * (size_t)ns, 0, ((size_t)ns + 16) * 4, c->stream));         // arrivals, counters
    int per_sm = 0;
    BIHRT_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_wtab_down, WINDING_THREADS, 0));
    if (per_sm < 1) per_sm = 1;
    k_wtab_down<<<c->sm_count * per_sm, WINDING_THREADS, 0, c->stream>>>(c->d_hdr, c->d_nodes, scr, ns, c->d_status_map);
    BIHRT_CUDA(c, cudaGetLastError());
    k_wtab_up<<<(ns + WINDING_THREADS - 1) / WINDING_THREADS, WINDING_THREADS, 0, c->stream>>>(c->d_hdr, c->d_nodes, c->d_tris, c->d_wtab, scr, ns);
    BIHRT_CUDA(c, cudaGetLastError());
    c->kernel_launches += 2;
    return BIHRT_OK;
}

// ---------------------------------------------------------------------------------------------- query

// the far test of one child box (lo.xyz hi.xyz): R = c - p, d2 = R.R; far when d2 > b2 * r^2
__device__ __forceinline__ bool far_child(float b0, float b1, float b2_, float b3, float b4, float b5, float px, float py, float pz,
                                          float b2, float& Rx, float& Ry, float& Rz, float& d2) {
    Rx = __fsub_rn(__fmul_rn(__fadd_rn(b0, b3), 0.5f), px);
    Ry = __fsub_rn(__fmul_rn(__fadd_rn(b1, b4), 0.5f), py);
    Rz = __fsub_rn(__fmul_rn(__fadd_rn(b2_, b5), 0.5f), pz);
    d2 = wdot(Rx, Ry, Rz, Rx, Ry, Rz);
    const float ex = __fsub_rn(b3, b0), ey = __fsub_rn(b4, b1), ez = __fsub_rn(b5, b2_);
    const float rr = __fmul_rn(wdot(ex, ey, ez, ex, ey, ez), 0.25f);
    return d2 > __fmul_rn(b2, rr);
}

__device__ __forceinline__ double far_rec(const float* wtab, uint32_t node, uint32_t side, float Rx, float Ry, float Rz, float d2) {
    const float4* s = reinterpret_cast<const float4*>(wtab + (2 * (size_t)node + side) * WTAB_FLOATS);
    float e[WTAB_FLOATS];
#pragma unroll
    for (int k = 0; k < 8; k++) { const float4 v = __ldg(s + k); e[4 * k] = v.x; e[4 * k + 1] = v.y; e[4 * k + 2] = v.z; e[4 * k + 3] = v.w; }
    return (double)far_term(e, Rx, Ry, Rz, d2);
}

// Q: the BIH is a quality-mode tree; it sets only the stack depth
template <bool Q>
__global__ void __launch_bounds__(WINDING_THREADS, WINDING_MIN_BLOCKS) k_winding(WindingArgs a) {
    constexpr int STACK_DEPTH = Q ? STACK_DEPTH_QUALITY : STACK_DEPTH_PARITY;
    if (a.hdr->status != 0) return;             // the build's device watchdog tripped: answer nothing (the host reports it)
    if ((a.hdr->quality != 0) != Q) {           // a tree of the other kind
        if (blockIdx.x == 0 && threadIdx.x == 0 && a.status_map) *a.status_map = 0x100u;
        return;
    }
    const uint32_t nu = a.hdr->nu;
    const uint32_t root_ref = BIH_REF_NODE(0, a.hdr->root_axis);
    const float4* __restrict__ nodes = reinterpret_cast<const float4*>(a.nodes);
    const float4* __restrict__ tris = reinterpret_cast<const float4*>(a.tris);
    const float b2 = a.b2;
    const int lane = threadIdx.x & 31;
    uint32_t stack[STACK_DEPTH];

    for (;;) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(a.work, 32u);
        base = __shfl_sync(FULL, base, 0);
        if ((uint64_t)base >= (uint64_t)a.n) break;
        const uint64_t i = (uint64_t)base + (uint32_t)lane;
        if (i < (uint64_t)a.n) {
            const float4 P = __ldg(reinterpret_cast<const float4*>(a.pts) + i);
            const float px = P.x, py = P.y, pz = P.z;
            const bool live = fabsf(px) <= FLT_MAX && fabsf(py) <= FLT_MAX && fabsf(pz) <= FLT_MAX;
            double acc = 0.0;
            uint32_t cur = (live && nu > 0) ? (nu == 1 ? BIH_REF_LEAFREF(0) : root_ref) : NONE;
            int sp = 0;
            while (cur != NONE) {
                if (cur & BIH_REF_LEAF) {
                    if (cur & 3u) {                          // a far right child whose left sibling was descended
                        const uint32_t node = BIH_REF_INDEX(cur);
                        const float4* np = nodes + 4 * (size_t)node;
                        const float4 b1 = __ldg(np + 2), b2v = __ldg(np + 3);
                        float Rx, Ry, Rz, d2;
                        far_child(b1.z, b1.w, b2v.x, b2v.y, b2v.z, b2v.w, px, py, pz, b2, Rx, Ry, Rz, d2);
                        acc = __dadd_rn(acc, far_rec(a.wtab, node, 1, Rx, Ry, Rz, d2));
                    } else {
                        const float4* tp = tris + 3 * (size_t)BIH_REF_INDEX(cur);
                        for (;;) {
                            const float4 q0 = __ldg(tp), q1 = __ldg(tp + 1), q2 = __ldg(tp + 2);
                            acc = __dadd_rn(acc, __dmul_rn(2.0, (double)tri_half_angle(px, py, pz, q0, q1, q2)));
                            if (__float_as_uint(q2.z) & 1u) break;
                            tp += 3;
                        }
                    }
                    cur = NONE;
                } else {
                    const uint32_t node = BIH_REF_INDEX(cur);
                    const float4* np = nodes + 4 * (size_t)node;
                    const float4 nd = __ldg(np), b0 = __ldg(np + 1), b1 = __ldg(np + 2), b2v = __ldg(np + 3);
                    float lRx, lRy, lRz, ld2, rRx, rRy, rRz, rd2;
                    const bool fl = far_child(b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, px, py, pz, b2, lRx, lRy, lRz, ld2);
                    const bool fr = far_child(b1.z, b1.w, b2v.x, b2v.y, b2v.z, b2v.w, px, py, pz, b2, rRx, rRy, rRz, rd2);
                    const uint32_t rl = __float_as_uint(nd.z), rr = __float_as_uint(nd.w);
                    if (fl) {
                        acc = __dadd_rn(acc, far_rec(a.wtab, node, 0, lRx, lRy, lRz, ld2));
                        if (fr) { acc = __dadd_rn(acc, far_rec(a.wtab, node, 1, rRx, rRy, rRz, rd2)); cur = NONE; }
                        else cur = rr;
                    } else {
                        stack[sp++] = fr ? (BIH_REF_LEAF | (node << 2) | 2u) : rr;     // one push per step, as in k_trace
                        cur = rl;
                    }
                }
                if (cur == NONE && sp > 0) cur = stack[--sp];
            }
            a.out_w[i] = __double2float_rn(__dmul_rn(acc, INV_4PI));
        }
    }
}

template <bool Q>
static int launch(bihrt_ctx* c, const WindingArgs& a) {
    int per_sm = 0;
    BIHRT_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_winding<Q>, WINDING_THREADS, 0));
    if (per_sm < 1) per_sm = 1;
    BIHRT_CUDA(c, cudaMemsetAsync(a.work, 0, 4, c->stream));
    k_winding<Q><<<c->sm_count * per_sm, WINDING_THREADS, 0, c->stream>>>(a);
    c->kernel_launches += 1;
    BIHRT_CUDA(c, cudaGetLastError());
    return BIHRT_OK;
}

int bihrt_winding_launch(bihrt_ctx* c, const WindingArgs& a) {
    return c->built_quality ? launch<true>(c, a) : launch<false>(c, a);
}
