// Closest-point queries on sm_100a (bihrt_closest_point, include/bihrt.h): for every point, the triangle nearest to it within
// the point's own search radius, and where on it.
//
// Kernel shape
//   * persistent warps (grid = SMs x the resident blocks of 4 warps); a warp takes units of 32 points from one global atomic
//     counter and every lane walks its own point to the end before the warp takes the next unit.  The cost of a point varies
//     by orders of magnitude (a point on the surface visits a handful of nodes, a point far away with an unbounded radius
//     descends to the nearest leaves of a whole side of the mesh), so units are small and handed out on demand;
//   * the walk is a best-first descent with a stack of (child reference, lower bound) items in local memory: a node is ONE
//     64-byte record (4 x LDG.128), of which only the two children's exact boxes are used -- the clip planes and the
//     reference's plane logic play no part, so the walk is the same on parity and quality-mode trees.  The lower bound of a
//     child is the squared distance from the point to its box widened by the query's margin; the nearer child is entered
//     (the left one on equal bounds), the other one is pushed unless it is beyond the cut, and items popped from the stack
//     are dropped when the cut has since moved below their bound;
//   * the cut is min(best d2, fl(rmax^2)), one squared value, updated whenever a leaf improves the best;
//   * a leaf is a run of triangle records up to the `last` flag, each one tested with the distance function of the header;
//   * u, v, q and ng are not carried through the walk: when a point ends with a hit its triangle is fetched again and the
//     record recomputed by the same function, bit for bit the walk's values.
// Everything that decides a result is IEEE binary32 with explicit __f*_rn (no contraction), restated on the CPU by
// tests/closest_oracle.c.
//
// The margin (DESIGN.md section 8): a triangle that lies inside a box can have a computed d2 a few ulps BELOW the computed
// distance of its box (the records hold fl(v1 - v0), q is rounded, the box bound is rounded).  Every box is therefore widened
// by m = 2^-16 x M on each side, M = the largest magnitude among the point's coordinates and the scene box's, which bounds
// those errors with a factor of four to spare; with it no candidate is ever pruned and the result equals brute force.
#include "bihrt_internal.cuh"
#include <float.h>

#define FULL 0xffffffffu
#define NONE 0xFFFFFFFFu              // "no item": leaf bit set, never a valid slot
#define CLOSEST_THREADS 128
#define CLOSEST_MIN_BLOCKS 8          // <= 64 registers per thread
#define CLOSEST_EPS 1.52587890625e-05f   /* 2^-16: the boxes' margin is this times the query's largest coordinate magnitude */

__device__ __forceinline__ float dot3(float ax, float ay, float az, float bx, float by, float bz) {
    return __fadd_rn(__fadd_rn(__fmul_rn(ax, bx), __fmul_rn(ay, by)), __fmul_rn(az, bz));
}

// q = (v0 + u*e1) + v*e2 and d2 = |p - q|^2
__device__ __forceinline__ float pt_q(float px, float py, float pz, float v0x, float v0y, float v0z, float e1x, float e1y,
                                      float e1z, float e2x, float e2y, float e2z, float u, float v, float& qx, float& qy, float& qz) {
    qx = __fadd_rn(__fadd_rn(v0x, __fmul_rn(u, e1x)), __fmul_rn(v, e2x));
    qy = __fadd_rn(__fadd_rn(v0y, __fmul_rn(u, e1y)), __fmul_rn(v, e2y));
    qz = __fadd_rn(__fadd_rn(v0z, __fmul_rn(u, e1z)), __fmul_rn(v, e2z));
    const float dx = __fsub_rn(px, qx), dy = __fsub_rn(py, qy), dz = __fsub_rn(pz, qz);
    return dot3(dx, dy, dz, dx, dy, dz);
}

// parameter of the point of segment (start, start + e) nearest to the point at r = p - start: 0 unless > 0 (0 / 0 included), <= 1
__device__ __forceinline__ float seg_t(float rx, float ry, float rz, float ex, float ey, float ez) {
    const float t = __fdiv_rn(dot3(rx, ry, rz, ex, ey, ez), dot3(ex, ey, ez, ex, ey, ez));
    return t > 0.f ? fminf(t, 1.f) : 0.f;
}

// Ericson's ClosestPtPointTriangle on the record (v0, e1, e2), the operation order include/bihrt.h states: (u, v) of the
// closest point, returns its d2
__device__ __forceinline__ float pt_tri(float px, float py, float pz, float v0x, float v0y, float v0z, float e1x, float e1y,
                                        float e1z, float e2x, float e2y, float e2z, float& u, float& v) {
    const float apx = __fsub_rn(px, v0x), apy = __fsub_rn(py, v0y), apz = __fsub_rn(pz, v0z);
    const float d1 = dot3(e1x, e1y, e1z, apx, apy, apz), d2 = dot3(e2x, e2y, e2z, apx, apy, apz);
    const float bpx = __fsub_rn(apx, e1x), bpy = __fsub_rn(apy, e1y), bpz = __fsub_rn(apz, e1z);
    const float d3 = dot3(e1x, e1y, e1z, bpx, bpy, bpz), d4 = dot3(e2x, e2y, e2z, bpx, bpy, bpz);
    const float cpx = __fsub_rn(apx, e2x), cpy = __fsub_rn(apy, e2y), cpz = __fsub_rn(apz, e2z);
    const float d5 = dot3(e1x, e1y, e1z, cpx, cpy, cpz), d6 = dot3(e2x, e2y, e2z, cpx, cpy, cpz);
    const float vc = __fsub_rn(__fmul_rn(d1, d4), __fmul_rn(d3, d2));
    const float vb = __fsub_rn(__fmul_rn(d5, d2), __fmul_rn(d1, d6));
    const float va = __fsub_rn(__fmul_rn(d3, d6), __fmul_rn(d5, d4));
    const float s = __fadd_rn(__fadd_rn(va, vb), vc);
    float qx, qy, qz;
    bool degen = false;         // an edge of zero length (its branch would divide 0 by 0) or no area: the edges decide
    u = 0.f; v = 0.f;
    if (d1 <= 0.f && d2 <= 0.f) { }                                                           // vertex v0
    else if (d3 >= 0.f && d4 <= d3) u = 1.f;                                                  // vertex v1
    else if (vc <= 0.f && d1 >= 0.f && d3 <= 0.f) {                                           // edge v0 v1
        const float den = __fsub_rn(d1, d3);
        if (den > 0.f) u = __fdiv_rn(d1, den); else degen = true;
    }
    else if (d6 >= 0.f && d5 <= d6) v = 1.f;                                                  // vertex v2
    else if (vb <= 0.f && d2 >= 0.f && d6 <= 0.f) {                                           // edge v0 v2
        const float den = __fsub_rn(d2, d6);
        if (den > 0.f) v = __fdiv_rn(d2, den); else degen = true;
    }
    else if (va <= 0.f && __fsub_rn(d4, d3) >= 0.f && __fsub_rn(d5, d6) >= 0.f) {            // edge v1 v2
        const float den = __fadd_rn(__fsub_rn(d4, d3), __fsub_rn(d5, d6));
        if (den > 0.f) { const float w = __fdiv_rn(__fsub_rn(d4, d3), den); u = __fsub_rn(1.f, w); v = w; } else degen = true;
    }
    else if (s > 0.f) { u = __fdiv_rn(vb, s); v = __fdiv_rn(vc, s); }                        // interior
    else degen = true;
    if (degen) {
        // zero or near-zero area: the nearest of the three edge segments, ties to AB, then AC, then BC
        const float tab = seg_t(apx, apy, apz, e1x, e1y, e1z);
        const float tac = seg_t(apx, apy, apz, e2x, e2y, e2z);
        const float tbc = seg_t(bpx, bpy, bpz, __fsub_rn(e2x, e1x), __fsub_rn(e2y, e1y), __fsub_rn(e2z, e1z));
        const float dab = pt_q(px, py, pz, v0x, v0y, v0z, e1x, e1y, e1z, e2x, e2y, e2z, tab, 0.f, qx, qy, qz);
        const float dac = pt_q(px, py, pz, v0x, v0y, v0z, e1x, e1y, e1z, e2x, e2y, e2z, 0.f, tac, qx, qy, qz);
        const float dbc = pt_q(px, py, pz, v0x, v0y, v0z, e1x, e1y, e1z, e2x, e2y, e2z, __fsub_rn(1.f, tbc), tbc, qx, qy, qz);
        u = tab; v = 0.f;
        float best = dab;
        if (dac < best) { u = 0.f; v = tac; best = dac; }
        if (dbc < best) { u = __fsub_rn(1.f, tbc); v = tbc; }
    }
    return pt_q(px, py, pz, v0x, v0y, v0z, e1x, e1y, e1z, e2x, e2y, e2z, u, v, qx, qy, qz);
}

// lower bound on the squared distance from p to the box widened by m on every side
__device__ __forceinline__ float box_d2(float lx, float ly, float lz, float hx, float hy, float hz, float px, float py, float pz, float m) {
    const float gx = fmaxf(__fsub_rn(fmaxf(__fsub_rn(lx, px), __fsub_rn(px, hx)), m), 0.f);
    const float gy = fmaxf(__fsub_rn(fmaxf(__fsub_rn(ly, py), __fsub_rn(py, hy)), m), 0.f);
    const float gz = fmaxf(__fsub_rn(fmaxf(__fsub_rn(lz, pz), __fsub_rn(pz, hz)), m), 0.f);
    return dot3(gx, gy, gz, gx, gy, gz);
}

// Q: the BIH is a quality-mode tree; it sets only the stack depth (the walk reads nothing but the children's boxes)
template <bool Q>
__global__ void __launch_bounds__(CLOSEST_THREADS, CLOSEST_MIN_BLOCKS) k_closest(ClosestArgs a) {
    constexpr int STACK_DEPTH = Q ? STACK_DEPTH_QUALITY : STACK_DEPTH_PARITY;
    if (a.hdr->status != 0) return;             // the build's device watchdog tripped: answer nothing rather than garbage (the host reports it)
    if ((a.hdr->quality != 0) != Q) {           // a tree of the other kind (a replica adopted without the matching morton_bits option)
        if (blockIdx.x == 0 && threadIdx.x == 0 && a.status_map) *a.status_map = 0x100u;
        return;
    }
    const uint32_t nu = a.hdr->nu;
    const float lx = a.hdr->lo[0], ly = a.hdr->lo[1], lz = a.hdr->lo[2], hx = a.hdr->hi[0], hy = a.hdr->hi[1], hz = a.hdr->hi[2];
    const float smag = fmaxf(fmaxf(fmaxf(fabsf(lx), fabsf(ly)), fmaxf(fabsf(lz), fabsf(hx))), fmaxf(fabsf(hy), fabsf(hz)));
    const uint32_t root_ref = BIH_REF_NODE(0, a.hdr->root_axis);
    const float4* __restrict__ nodes = reinterpret_cast<const float4*>(a.nodes);
    const float4* __restrict__ tris = reinterpret_cast<const float4*>(a.tris);
    const int lane = threadIdx.x & 31;
    uint2 stack[STACK_DEPTH];                   // (child reference, its lower bound)

    for (;;) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(a.work, 32u);
        base = __shfl_sync(FULL, base, 0);
        if ((uint64_t)base >= (uint64_t)a.n) break;
        const uint64_t i = (uint64_t)base + (uint32_t)lane;
        if (i < (uint64_t)a.n) {
            const float4 P = __ldg(reinterpret_cast<const float4*>(a.pts) + i);
            const float px = P.x, py = P.y, pz = P.z;
            const bool live = P.w >= 0.f && fabsf(px) <= FLT_MAX && fabsf(py) <= FLT_MAX && fabsf(pz) <= FLT_MAX;
            float cut = fminf(__fmul_rn(P.w, P.w), FLT_MAX);      // min(best d2, fl(rmax^2), FLT_MAX)
            uint32_t best = NONE;                                 // slot of the best candidate so far
            const float m = __fmul_rn(CLOSEST_EPS, fmaxf(smag, fmaxf(fmaxf(fabsf(px), fabsf(py)), fabsf(pz))));
            uint32_t cur = NONE;
            if (live && nu > 0 && !(box_d2(lx, ly, lz, hx, hy, hz, px, py, pz, m) > cut)) cur = nu == 1 ? BIH_REF_LEAFREF(0) : root_ref;
            int sp = 0;
            while (cur != NONE) {
                if (cur & BIH_REF_LEAF) {
                    const float4* tp = tris + 3 * (size_t)BIH_REF_INDEX(cur);
                    for (;;) {
                        const float4 q0 = __ldg(tp), q1 = __ldg(tp + 1), q2 = __ldg(tp + 2);
                        float u, v;
                        const float d2 = pt_tri(px, py, pz, q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, u, v);
                        const uint32_t s = __float_as_uint(q2.w);
                        if (d2 < cut || (d2 == cut && s < best)) { cut = d2; best = s; }
                        if (__float_as_uint(q2.z) & 1u) break;     // last triangle of the leaf
                        tp += 3;
                    }
                    cur = NONE;
                } else {
                    const float4* np = nodes + 4 * (size_t)BIH_REF_INDEX(cur);
                    const float4 nd = __ldg(np), b0 = __ldg(np + 1), b1 = __ldg(np + 2), b2 = __ldg(np + 3);
                    const float bl = box_d2(b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, px, py, pz, m);
                    const float br = box_d2(b1.z, b1.w, b2.x, b2.y, b2.z, b2.w, px, py, pz, m);
                    const bool rfirst = br < bl;                   // the nearer child first; the left one on equal bounds
                    const float bn = rfirst ? br : bl, bf = rfirst ? bl : br;
                    const uint32_t rn = __float_as_uint(rfirst ? nd.w : nd.z), rf = __float_as_uint(rfirst ? nd.z : nd.w);
                    if (bn > cut) cur = NONE;
                    else {
                        // one push per step: the depth is bounded by the tree's, as in k_trace
                        if (!(bf > cut)) { stack[sp] = make_uint2(rf, __float_as_uint(bf)); sp++; }
                        cur = rn;
                    }
                }
                if (cur == NONE) {
                    while (sp > 0) {
                        sp--;
                        const uint2 e = stack[sp];
                        if (!(__uint_as_float(e.y) > cut)) { cur = e.x; break; }
                    }
                }
            }
            // the record: the best triangle again, by the walk's own function
            float u = 0.f, v = 0.f, qx = 0.f, qy = 0.f, qz = 0.f, gx = 0.f, gy = 0.f, gz = 0.f;
            int32_t prim = -1;
            if (best != NONE) {
                const float4* tp = tris + 3 * (size_t)best;
                const float4 q0 = __ldg(tp), q1 = __ldg(tp + 1), q2 = __ldg(tp + 2);
                const float e1x = q0.w, e1y = q1.x, e1z = q1.y, e2x = q1.z, e2y = q1.w, e2z = q2.x;
                pt_tri(px, py, pz, q0.x, q0.y, q0.z, e1x, e1y, e1z, e2x, e2y, e2z, u, v);
                pt_q(px, py, pz, q0.x, q0.y, q0.z, e1x, e1y, e1z, e2x, e2y, e2z, u, v, qx, qy, qz);
                gx = __fsub_rn(__fmul_rn(e1y, e2z), __fmul_rn(e1z, e2y));
                gy = __fsub_rn(__fmul_rn(e1z, e2x), __fmul_rn(e1x, e2z));
                gz = __fsub_rn(__fmul_rn(e1x, e2y), __fmul_rn(e1y, e2x));
                prim = (int32_t)__float_as_uint(q2.y);
            }
            if (a.out_d2) a.out_d2[i] = best != NONE ? cut : FLT_MAX;
            if (a.out_u) a.out_u[i] = u;
            if (a.out_v) a.out_v[i] = v;
            if (a.out_slot) a.out_slot[i] = (int32_t)best;
            if (a.out_prim) a.out_prim[i] = prim;
            if (a.out_q) { float* g = a.out_q + 3 * i; g[0] = qx; g[1] = qy; g[2] = qz; }
            if (a.out_ng) { float* g = a.out_ng + 3 * i; g[0] = gx; g[1] = gy; g[2] = gz; }
        }
    }
}

template <bool Q>
static int launch(bihrt_ctx* c, const ClosestArgs& a) {
    int per_sm = 0;
    BIHRT_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_closest<Q>, CLOSEST_THREADS, 0));
    if (per_sm < 1) per_sm = 1;
    BIHRT_CUDA(c, cudaMemsetAsync(a.work, 0, 4, c->stream));
    k_closest<Q><<<c->sm_count * per_sm, CLOSEST_THREADS, 0, c->stream>>>(a);
    c->kernel_launches += 1;
    BIHRT_CUDA(c, cudaGetLastError());
    return BIHRT_OK;
}

int bihrt_closest_launch(bihrt_ctx* c, const ClosestArgs& a) {
    return c->built_quality ? launch<true>(c, a) : launch<false>(c, a);
}
