// Ray traversal + ray/triangle intersection on sm_100a.  Replaces cudaRender / Color / TraverseTree /
// FindNearestTriangle / RayTriangleIntersection (R/src/CUDAKernels.cu:17-50,206-423) and
// Camera::GetRay / Ray::Ray (R/src/Camera.cu:18-20, R/src/Ray.cu:3-10).
//
// Kernel shape
//   * persistent warps (grid = SMs x 8 resident blocks of 4 warps); a warp takes units of 32 work items from one
//     global atomic counter (or from per-SM queues, 1 spp launches of >= 16 M rays).  Camera modes: an item is a
//     pixel's sample group -- the samples of a pixel sit in CONSECUTIVE LANES, the warp moves from sample to sample
//     in lock step and a pixel is written once, as its final colour, by the lane that completes it (possibly into
//     another GPU's framebuffer: bihrt_render_interleaved_to).  A warp is refilled once every lane's ray has ended: each
//     lane starts its item's next sample or takes a new item.  An option traces a ray list through a sort permutation
//     (csrc/raysort.cu);
//   * the tiles of a camera frame are traced in the order k_tile_order derived from the PREVIOUS launch of the same
//     frame geometry (longest unit per tile, expensive tiles first): the launch is as long as its longest unit;
//   * every lane walks its own ray with a short stack of 16-byte items (child reference + the three
//     interval bounds) in local memory; a leaf is an item like a node, so the hot loop has one shape.  An item in
//     hand is valid by construction; only items popped from the stack are re-checked against the closest hit;
//   * a node is ONE 64-byte record fetched with four 128-bit read-only loads: the reference's two clip planes and
//     child references (the BIH proper) and the bounding boxes of the two children.  The plane logic decides what the
//     reference's decides (strict and closed comparisons included); the boxes only remove visits -- a child whose box the
//     ray misses inside the child's interval is never fetched (39 -> 14 nodes and 13 -> 1.1 triangle tests per primary ray
//     on the 1 M-triangle scene, identical hits).  The per-axis ray constants (origin, 1/dir) of the node's axis come from
//     shared memory by one 64-bit LDS selected with the axis bits the parent's reference carried; 1/dir and -origin/dir of
//     all three axes sit in registers for the boxes (plane distance = one FMA); origin and direction themselves are only
//     read by the triangle test, from shared memory;
//   * leaf-ordered triangles (3 x 16 B) are fetched with 128-bit read-only loads;
//   * two-phase ("while-while") loop: lanes take 4 node steps (unrolled), the warp votes, leaves are tested,
//     repeat; the vote ends the node phase as soon as the lanes waiting with a leaf outnumber the walking ones.
//
// Logical per-ray algorithm = oracle/bih_oracle.c:traverse_box (pruned traversal + children boxes that returns what
// the reference's TraverseTree returns, including on axis-aligned flat geometry where the reference's
// strict comparisons decide); framebuffer renders (MODE 1) end a sample at its first accepted triangle, which
// tests/walk_oracle.c restates as exit "first" (COVER below).  Everything that decides a hit is IEEE binary32 without FMA contraction (explicit __f*_rn)
// so t is bit-identical to the oracle's; the box distances are explicit FMAs, mirrored with fmaf in the oracle.
#include "bihrt_internal.cuh"
#include <float.h>
#include <type_traits>

#define FULL 0xffffffffu
#define NONE 0xFFFFFFFFu        // "no item": leaf bit set, never a valid slot
#define TRACE_THREADS 128
#define TRACE_MIN_BLOCKS 8        // <= 64 registers per thread
// node steps a lane takes between two votes of the node phase (DESIGN §4: 2 / 3 / 6 steps measured -2 / -2 / 0 %)
constexpr int NODE_STEPS = 4;

// Framebuffer renders (MODE 1) as coverage queries: a pixel's colour depends only on WHETHER each sample hits, so a sample
// ends at the first triangle it accepts -- inside the leaf and for the whole walk -- instead of searching on for the
// closest one.  Until that first hit the walk is the closest-hit walk step for step (h.t is FLT_MAX in both: same strict
// test, same far-leaf-first order, same flat-geometry misses), so a sample hits exactly when the closest-hit search hits and
// the image is the same bit for bit.  While a sample is alive every stacked item is still valid (pMin <= pMax <= FLT_MAX
// held when it was pushed), so the pop needs no compare-and-drop loop.  MODE 0 and 2 keep the closest hit.
// Framebuffer renders (MODE 1) with lane groups (spp > 1) walk in one of nine copies of the node phase, chosen per warp after
// every refill: one per ray octant, where every live lane's 1/d has the same sign on each axis, and the generic copy for a warp that mixes signs.  In
// an octant copy a box's near and far distances are taken by compile-time sign, one FMNMX3 each, instead of the per-axis
// min / max of the plane pair.  Exact: with lo <= hi (every child box) and a finite nonzero 1/d, round-to-nearest FMA is
// monotone in the plane, so the sign selects the very distance min / max returns; a NaN 1/d (zero direction component)
// gives two NaN distances, which the three-input min / max drop as the nested calls do, and 1/d == 0 gives two equal
// ones.  Same intervals, same visits, same counters, same pixels.
#define OCT_MIXED 8                         // the generic copy: lanes disagree on the sign of some axis
#define BOX_EPS 2.384185791015625e-07f      /* 2^-22: the box tests' margin is this times (largest finite |o/d| + larger end of the ray's scene interval), one constant per ray */

// (double)det < 0.000001 (R/src/CUDAKernels.cu:28)  <=>  det < 0x358637be as binary32; two-sided ray queries (MODE 4) test
// fabs((double)det) < 0.000001  <=>  fabsf(det) < 0x358637be (the binary32 threshold is symmetric)
#define DET_EPS __uint_as_float(0x358637beu)

struct Hit { float t; int slot; };

__device__ __forceinline__ float fmin3(float a, float b, float c) { float r; asm("min.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c)); return r; }
__device__ __forceinline__ float fmax3(float a, float b, float c) { float r; asm("max.f32 %0, %1, %2, %3;" : "=f"(r) : "f"(a), "f"(b), "f"(c)); return r; }

// Color + rgbToInt, R/src/CUDAKernels.cu:82-88,385-387,420-422: mean over the samples of hit (255,255,0) /
// miss (20,20,40), packed r | g<<8 | b<<16 (sums of 255/20/40 are exact in binary32)
__device__ __forceinline__ uint32_t pack_colour(uint32_t hits, int samples) {
    const float fh = (float)hits, fm = (float)(samples - (int)hits), fs = (float)samples;
    float cr = __fdiv_rn(__fadd_rn(__fmul_rn(fh, 255.f), __fmul_rn(fm, 20.f)), fs);
    float cb = __fdiv_rn(__fmul_rn(fm, 40.f), fs);
    cr = fmaxf(0.f, fminf(255.f, cr));
    cb = fmaxf(0.f, fminf(255.f, cb));
    return ((uint32_t)(int)cb << 16) | ((uint32_t)(int)cr << 8) | (uint32_t)(int)cr;
}

// Moller-Trumbore in three steps (R/src/CUDAKernels.cu:24-42).  The triangle test of the walk and the hit-record epilogue
// of MODE 3 both call these, so the u, v a ray query reports are the ones its walk computed, bit for bit.
// pvec = cross(dir, e2); returns det = dot(e1, pvec)                                           R/src/CUDAKernels.cu:24-26
__device__ __forceinline__ float mt_det(float dx, float dy, float dz, float e1x, float e1y, float e1z, float e2x, float e2y, float e2z,
                                        float& px, float& py, float& pz) {
    px = __fsub_rn(__fmul_rn(dy, e2z), __fmul_rn(e2y, dz));
    py = __fsub_rn(__fmul_rn(dz, e2x), __fmul_rn(e2z, dx));
    pz = __fsub_rn(__fmul_rn(dx, e2y), __fmul_rn(e2x, dy));
    return __fadd_rn(__fadd_rn(__fmul_rn(e1x, px), __fmul_rn(e1y, py)), __fmul_rn(e1z, pz));
}
// tvec = origin - v0; returns u = dot(tvec, pvec) * inv                                        :33-35
__device__ __forceinline__ float mt_u(float ox, float oy, float oz, const float4& q0, float px, float py, float pz, float inv,
                                      float& tx, float& ty, float& tz) {
    tx = __fsub_rn(ox, q0.x); ty = __fsub_rn(oy, q0.y); tz = __fsub_rn(oz, q0.z);
    return __fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(tx, px), __fmul_rn(ty, py)), __fmul_rn(tz, pz)), inv);
}
// qvec = cross(tvec, e1); returns v = dot(dir, qvec) * inv                                     :40-42
__device__ __forceinline__ float mt_v(float dx, float dy, float dz, float e1x, float e1y, float e1z, float tx, float ty, float tz, float inv,
                                      float& qx, float& qy, float& qz) {
    qx = __fsub_rn(__fmul_rn(ty, e1z), __fmul_rn(e1y, tz));
    qy = __fsub_rn(__fmul_rn(tz, e1x), __fmul_rn(e1z, tx));
    qz = __fsub_rn(__fmul_rn(tx, e1y), __fmul_rn(e1x, ty));
    return __fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(dx, qx), __fmul_rn(dy, qy)), __fmul_rn(dz, qz)), inv);
}

// FIRST: stop at the first accepted triangle (coverage queries)
// RANGE: ray queries with an interval (MODE 3): a triangle is accepted for tlo < t < h.t, with tlo = max(tmin, 0) read from
// word 9 of the lane's shared-memory ray record (only when a candidate is found: no register is held through the leaf)
// TWO_SIDED: back faces too (MODE 4): Moller-Trumbore's non-culling branch, |det| >= 1e-6.  Everything after the det test is
// the same arithmetic (1/det rounds symmetrically), so a front-face candidate is computed bit for bit as without it; a NaN
// det still passes here and is rejected by the t compare.
template <bool COUNTED, bool FIRST, bool RANGE = false, bool TWO_SIDED = false>
__device__ __forceinline__ void test_leaf(const char* __restrict__ first_tri, float ox, float oy, float oz,
                                          float dx, float dy, float dz, Hit& h, uint32_t& ntris, uint32_t& wleaf,
                                          const float* tlo_p = nullptr) {
    const float4* p = reinterpret_cast<const float4*>(first_tri);
    for (;;) {
        const float4 q0 = __ldg(p), q1 = __ldg(p + 1), q2 = __ldg(p + 2);
        if (COUNTED) { ntris++; const uint32_t am = __activemask(); wleaf += ((threadIdx.x & 31) == __ffs(am) - 1); }
        const float e1x = q0.w, e1y = q1.x, e1z = q1.y, e2x = q1.z, e2y = q1.w, e2z = q2.x;
        float px, py, pz;
        const float det = mt_det(dx, dy, dz, e1x, e1y, e1z, e2x, e2y, e2z, px, py, pz);
        if (!((TWO_SIDED ? fabsf(det) : det) < DET_EPS)) {
            const float inv = __frcp_rn(det);        // == (float)(1.0 / (double)det), :31 (53 >= 2*24+2 bits)
            float tx, ty, tz;
            const float u = mt_u(ox, oy, oz, q0, px, py, pz, inv, tx, ty, tz);
            if (!(u < 0.f || u > 1.f)) {
                float qx, qy, qz;
                const float v = mt_v(dx, dy, dz, e1x, e1y, e1z, tx, ty, tz, inv, qx, qy, qz);
                if (!(v < 0.f || __fadd_rn(u, v) > 1.f)) {
                    const float t = __fmul_rn(__fadd_rn(__fadd_rn(__fmul_rn(e2x, qx), __fmul_rn(e2y, qy)), __fmul_rn(e2z, qz)), inv);
                    if (t > (RANGE ? *tlo_p : 0.f) && t < h.t) {                              // :218-221, slot = sorted index
                        h.t = t; h.slot = (int)__float_as_uint(q2.w);
                        if (FIRST) break;
                    }
                }
            }
        }
        if (__float_as_uint(q2.z) & 1u) break;      // last triangle of the leaf
        p += 3;
    }
}

// ------------------------------------------------------------------------------------------
// MODE 0: ray list -> (t, slot, prim);  1: camera -> packed framebuffer;  2: camera -> per-sample hits;
// 3: ray list with per-ray intervals [tmin, tmax] -> hit records (t, u, v, slot, prim, ng): bihrt_intersect;
// 4: MODE 3 with two-sided triangles (BIHRT_INTERSECT_TWO_SIDED): only the leaf's det test differs.
// Work item = one ray (MODE 0/3/4) or one pixel with its spp samples (MODE 1/2).
// MODE 3 walks exactly like MODE 0 with a narrower root interval: pMin = max(rMin, tlo) and pMax = min(sMax, h.t), where
// h.t starts at min(tmax, FLT_MAX) (so the item in hand is valid, as for the occlusion query) and tlo = max(tmin, 0) sits in
// word 9 of the ray record, where the triangle test reads it.  u, v and ng are not carried through the walk (the kernel is
// at its register cap): when a hitting ray ends, its triangle is fetched again and u, v recomputed with the walk's own
// arithmetic (mt_det / mt_u / mt_v).
// ------------------------------------------------------------------------------------------
// Q: the BIH is a quality-mode tree (63-bit keys, capped leaves; csrc/build.cu): long stack, and the closed tight-interval
// tests alone decide -- the reference's extra strict test (rMin < t[near], :292), which the parity path reproduces together
// with the hits it loses on axis-aligned geometry, is dropped.
template <int MODE, bool COUNTED, bool Q>
__global__ void __launch_bounds__(TRACE_THREADS, TRACE_MIN_BLOCKS) k_trace(TraceArgs a) {
    constexpr int STACK_DEPTH = Q ? STACK_DEPTH_QUALITY : STACK_DEPTH_PARITY;
    constexpr bool COVER = MODE == 1;                                  // a sample ends at its first hit
    constexpr bool OCTS = MODE == 1;                                   // node phase specialised on the warp's ray octant
    constexpr bool LIST = MODE == 0 || MODE == 3 || MODE == 4;         // work items are rays of a list
    constexpr bool RANGE = MODE == 3 || MODE == 4;                     // rays carry [tmin, tmax]; hit records out
    constexpr bool TWO_SIDED = MODE == 4;                              // back faces accepted too
    // per-axis ray constants (origin, 1/dir), one row of 3 float2 per thread: 24-byte stride keeps a
    // half-warp's 64-bit accesses on distinct banks when the lanes agree on the axis
    // per-thread ray record in shared memory, 10 words: (ox, 1/dx) (oy, 1/dy) (oz, 1/dz) dx dy dz, and word 9: tlo (MODE 3 and 4) or
    // the warp's ray octant (MODE 1: read once per node phase, so no register holds it through the walk).  The node step picks
    // (origin, 1/dir) of the node's axis with one 64-bit LDS (40-byte stride: a half-warp's accesses fall on distinct banks
    // when the lanes agree on the axis); the direction is only needed by the triangle test, so it lives here, not in registers.
    __shared__ __align__(16) float s_ray[TRACE_THREADS * 10];
    const int lane = threadIdx.x & 31;
    const uint32_t lt = (1u << lane) - 1u;
    float* my_ray = s_ray + threadIdx.x * 10;
    const char* __restrict__ nodes_b = reinterpret_cast<const char*>(a.nodes);
    const char* __restrict__ tris_b = reinterpret_cast<const char*>(a.tris);
    const BihTri* __restrict__ tris = a.tris;
    const uint32_t nu = a.hdr->nu;
    if (a.hdr->status != 0) return;             // the build's device watchdog tripped: trace nothing rather than garbage (the host reports it)
    if ((a.hdr->quality != 0) != Q) {           // a tree of the other kind (a replica adopted without the matching morton_bits option)
        if (blockIdx.x == 0 && threadIdx.x == 0 && a.status_map) *a.status_map = 0x100u;
        return;
    }
    const float blo[3] = { a.hdr->lo[0], a.hdr->lo[1], a.hdr->lo[2] }, bhi[3] = { a.hdr->hi[0], a.hdr->hi[1], a.hdr->hi[2] };
    uint32_t nnodes = 0, ntris = 0, maxsp = 0;
    uint32_t wnode = 0, wleaf = 0;              // COUNTED: warp-level executions of the node step / the triangle test (SIMD efficiency = lane steps / 32 / these)

    // work items: 32-bit in the camera modes, whose launches bihrt_trace_launch refuses from 2^32 - 2^24 padded items on
    // (the margin covers every warp's last fetch past the end)
    using item_t = std::conditional_t<LIST, uint64_t, uint32_t>;
    constexpr item_t NO_ITEM = ~item_t(0);
    item_t total;
    // ray lists with cost-ordered chunks: the list is dealt in chunks of 1024 rays (the last one padded)
    if (LIST) total = a.tile_cost ? (((uint64_t)a.nrays + 1023u) >> 10) << 10 : (uint64_t)a.nrays;
    else {
        const int tx = (a.w + 31) / 32;
        const int ty = (a.h + 31) / 32, T = tx * ty;
        const int my_tiles = T > a.shard_index ? (T - a.shard_index + a.shard_count - 1) / a.shard_count : 0;
        total = ((item_t)my_tiles * 1024u) << a.gshift;
    }
    // Camera modes: the samples [s_begin, s_end) of a pixel are split into 2^gshift groups that sit in
    // CONSECUTIVE LANES (item = pixel * groups + group); a lane traces its group's samples one after the
    // other.  More groups = a warp covers fewer pixels = its 32 rays are closer together.
    const int gshift = LIST ? 0 : a.gshift;
    const int nsamp = LIST ? 1 : ((a.s_end - a.s_begin) >> gshift);    // samples per item
    uint32_t my_queue = 0;
    if (a.queues > 1) { asm("mov.u32 %0, %%smid;" : "=r"(my_queue)); my_queue %= (uint32_t)a.queues; }
    item_t pool_next = 0, pool_end = 0;        // warp-uniform
    uint32_t pool_xy = 0;                      // warp-uniform, camera modes: first pixel of the pool's tile, x | y << 16
    long long unit_t0 = 0; uint32_t unit_tile = 0xFFFFFFFFu;   // warp-uniform: start time / tile of the packet being traced
    bool exhausted = false;                    // warp-uniform: the global counter ran past `total`

    // lane state
    item_t item = NO_ITEM;                     // current work item
    int s = 0, s0 = 0;                         // sample of the item being traced, first sample of the item
    uint32_t hits = 0, pixel = 0, pxy = 0;
    // the box tests need all three axes: 1/direction, -origin/direction (plane distance = one FMA) and the absolute rounding
    // margin that goes with it; origin and direction themselves are only needed per axis (plane test) and by the triangle
    // test, and live in shared memory
    float ix = 1.f, iy = 1.f, iz = 1.f, nx = 0.f, ny = 0.f, nz = 0.f, bpad = 0.f;
    uint32_t cur = NONE;                       // item being walked: node index, leaf|slot, or NONE
    float rMin = 0.f, pMin = 0.f, pMax = 0.f;
    Hit h; h.t = FLT_MAX; h.slot = -1;
    bool tracing = false;                      // a ray is in flight (its result has not been recorded)
    uint4 stack[STACK_DEPTH];
    int sp = 0;
#define STACK_RESET() do { sp = 0; } while (0)
#define STACK_PUSH(item) do { stack[sp] = (item); sp++; } while (0)
#define STACK_POP(e) do { sp--; (e) = stack[sp]; } while (0)
    const uint32_t root_ref = BIH_REF_NODE(0, a.hdr->root_axis);
    // colours with a pixel's samples in several lanes: the warp moves from sample to sample in lock step, so the lanes
    // of a pixel hold its complete hit count when they finish and the pixel is written once, without atomics
    const bool direct = MODE == 1 && gshift > 0 && !(a.flags & BIHRT_RENDER_COUNTS);
    const uint32_t ray_smem = (uint32_t)__cvta_generic_to_shared(my_ray);

    for (;;) {
        // ================= refill: once the whole warp has drained, every lane records its ray and gets the next one ========
        // A lane moves on to the next SAMPLE of its own item, or takes a new ITEM when its item is done, so the warp starts
        // each packet together.  (Refilling the idle lanes of a warp that is still walking was measured as a loss with the
        // children boxes: DESIGN §4.)  Lanes that have nothing left park until the launch ends.
        const uint32_t busy = ~__ballot_sync(FULL, cur == NONE);
        if (busy == 0) {
            bool want_item = false, finishing = false;
            if (cur == NONE) {
                if (tracing) {                                   // record the ray that just ended
                    tracing = false;
                    if (MODE == 1) hits += (h.slot >= 0);
                    else if (RANGE) {
                        // hit record epilogue: the hit triangle again (48 bytes just read by the walk, likely in L1), u and v
                        // by the walk's arithmetic on the ray still in shared memory, ng = e1 x e2 (products rounded, no FMA)
                        const bool hit = h.slot >= 0;
                        const bool rec = a.out_u || a.out_v || a.out_ng;
                        float u = 0.f, v = 0.f, gx = 0.f, gy = 0.f, gz = 0.f;
                        int32_t prim = -1;
                        if (hit && (rec || a.out_prim)) {
                            const float4* tq = reinterpret_cast<const float4*>(tris + h.slot);
                            const float4 q0 = __ldg(tq), q1 = __ldg(tq + 1), q2 = __ldg(tq + 2);
                            prim = (int32_t)__float_as_uint(q2.y);
                            if (rec) {
                                const float e1x = q0.w, e1y = q1.x, e1z = q1.y, e2x = q1.z, e2y = q1.w, e2z = q2.x;
                                const float2 dxy = *reinterpret_cast<const float2*>(my_ray + 6);
                                const float dx = dxy.x, dy = dxy.y, dz = my_ray[8];
                                float px, py, pz, tx, ty, tz, qx, qy, qz;
                                const float inv = __frcp_rn(mt_det(dx, dy, dz, e1x, e1y, e1z, e2x, e2y, e2z, px, py, pz));
                                u = mt_u(my_ray[0], my_ray[2], my_ray[4], q0, px, py, pz, inv, tx, ty, tz);
                                v = mt_v(dx, dy, dz, e1x, e1y, e1z, tx, ty, tz, inv, qx, qy, qz);
                                gx = __fsub_rn(__fmul_rn(e1y, e2z), __fmul_rn(e1z, e2y));
                                gy = __fsub_rn(__fmul_rn(e1z, e2x), __fmul_rn(e1x, e2z));
                                gz = __fsub_rn(__fmul_rn(e1x, e2y), __fmul_rn(e1y, e2x));
                            }
                        }
                        // (h.t of a miss may be the cut tmax: the record says FLT_MAX)
                        if (a.out_t) a.out_t[item] = hit ? h.t : FLT_MAX;
                        if (a.out_slot) a.out_slot[item] = h.slot;
                        if (a.out_prim) a.out_prim[item] = prim;
                        if (a.out_u) a.out_u[item] = u;
                        if (a.out_v) a.out_v[item] = v;
                        if (a.out_ng) { float* g = a.out_ng + 3 * item; g[0] = gx; g[1] = gy; g[2] = gz; }
                    } else {
                        const uint64_t o = MODE == 0 ? item : (uint64_t)pixel * (uint32_t)a.spp + (uint32_t)(s0 + s);
                        if (a.out_t) a.out_t[o] = h.t;
                        if (a.out_slot) a.out_slot[o] = h.slot;
                        if (a.out_prim) a.out_prim[o] = h.slot >= 0 ? (int32_t)tris[h.slot].prim : -1;
                    }
                    s++;
                    if (s == nsamp) {
                        if (MODE == 1 && gshift > 0) finishing = true;      // written below, by the pixel's lanes together
                        else if (MODE == 1 && (a.flags & BIHRT_RENDER_COUNTS)) a.fb[pixel] = hits;     // resolved after the reduce
                        else if (MODE == 1) a.fb[pixel] = pack_colour(hits, nsamp);
                        item = NO_ITEM;
                    }
                }
                want_item = (item == NO_ITEM);
            }
            if (MODE == 1 && gshift > 0) {
                // the lanes of one pixel finish together (always, when the warp moves in lock step).  The participants are
                // named by a ballot taken where the whole warp is converged (the refill block is entered warp-uniformly),
                // not by __activemask() inside the divergent branch, which promises nothing about convergence.
                const uint32_t fin = __ballot_sync(FULL, finishing);
                if (finishing) {
                    const uint32_t same = __match_any_sync(fin, pixel);
                    const uint32_t sum = __reduce_add_sync(same, hits);
                    if (lane == __ffs(same) - 1) {
                        // colours: the pixel's lanes hold all its samples -> one plain store of the final value
                        // (a.fb may be another GPU's framebuffer: the store then travels over NVLink);
                        // counts (a pixel's samples are spread over ranks): one atomic per pixel and warp
                        if (direct) a.fb[pixel] = pack_colour(sum, nsamp << gshift);
                        else if (sum) atomicAdd(&a.fb[pixel], sum);
                    }
                }
            }
            // the packet that just drained: its duration is the cost of its tile for the next frame's order
            if (!LIST && a.tile_cost && unit_tile != 0xFFFFFFFFu) {
                if (lane == 0) atomicMax(a.tile_cost + unit_tile, (uint32_t)min((unsigned long long)(clock64() - unit_t0) >> 8, 0xFFFFFFFFull));
                unit_tile = 0xFFFFFFFFu;
            }
            // hand out new items (warp-uniform control flow)
            uint32_t want = __ballot_sync(FULL, want_item);
            while (want && !exhausted) {
                if (pool_next >= pool_end) {
                    // Work comes in units of 32 items, grouped in tiles of 32 units (a 32x32-pixel tile / 1024
                    // rays).  With per-SM queues (a.queues > 1) tile t belongs to queue t % queues and every
                    // warp of an SM drains its own SM's queue first, so the warps resident on one SM walk the
                    // same one or two tiles and share nodes and triangles in L1; an SM that runs dry steals
                    // from the others.  a.queues == 1 is one global counter (one unit per fetch).
                    item_t base = NO_ITEM;
                    uint32_t got = 0, unit_m = 0, unit_xy = 0;
                    if (lane == 0) {
                        // unit interleave across GPUs (il_count ranks): this rank owns every il_count-th 32-item unit
                        // of every tile, so all ranks walk all tiles (same locality, perfect balance) and every
                        // pixel keeps all its samples -- and their lane grouping -- on one GPU
                        const uint32_t ilc = (uint32_t)a.il_count, ili = (uint32_t)a.il_index, ics = (uint32_t)a.il_cshift;
                        if (a.queues <= 1) {
                            const item_t fetched = atomicAdd(a.work, 32u); got = 32;
                            const item_t lu = fetched >> 5;            // this rank's unit -> the frame's unit (runs of 2^il_cshift units)
                            if constexpr (LIST) {
                                base = ilc > 1 ? ((((lu >> ics) * ilc + ili) << ics) | (lu & ((1u << ics) - 1u))) << 5 : fetched;
                                if (base >= total) base = NO_ITEM;
                            } else {
                                // compared as units: past the end of an interleaved launch the frame's unit may reach 2^27,
                                // where its first item would wrap
                                const uint32_t fu = ilc > 1 ? (((lu >> ics) * ilc + ili) << ics) | (lu & ((1u << ics) - 1u)) : lu;
                                if (fu < (total >> 5)) base = fu << 5;
                            }
                        } else {
                            const uint32_t tshift = 10 + gshift, ushift = 5 + gshift;       // items / units per tile
                            const item_t ntile = (total + ((item_t(1) << tshift) - 1)) >> tshift;
                            for (uint32_t k = 0; k < (uint32_t)a.queues; k++) {
                                uint32_t q = my_queue + k; if (q >= (uint32_t)a.queues) q -= (uint32_t)a.queues;
                                if (q >= ntile) continue;
                                const uint32_t upt = (1u << ushift) / ilc;                                  // this rank's units per tile
                                const item_t units = ((ntile - q + a.queues - 1) / a.queues) * upt;         // of queue q
                                if (ld_relaxed(a.work + q) >= units) continue;
                                const uint32_t u = atomicAdd(a.work + q, 1u);
                                if (u >= units) continue;
                                const uint32_t lu = u % upt;
                                const item_t b = (((item_t)(u / upt) * a.queues + q) << tshift) + ((item_t)((((lu >> ics) * ilc + ili) << ics) | (lu & ((1u << ics) - 1u))) << 5);
                                if (b < total) { base = b; got = 32; break; }
                            }
                        }
                        if (!LIST && base != NO_ITEM) {
                            // the unit's tile, once for its 32 items: m-th in cost order, its row and column (tile < 2^22: the
                            // multiply-high is the row or one below it), its first pixel packed as x | y << 16 (w, h <= 65535)
                            const uint32_t mi = (uint32_t)base >> (10 + gshift);
                            unit_m = a.tile_order ? __ldg(a.tile_order + mi) : mi;
                            const uint32_t tile = (uint32_t)a.shard_index + unit_m * (uint32_t)a.shard_count;
                            uint32_t row = __umulhi(tile, a.tile_cols_rcp), col = tile - row * a.tile_cols;
                            if (col >= a.tile_cols) { row++; col -= a.tile_cols; }
                            unit_xy = (col << 5) | (row << 21);
                        }
                    }
                    base = __shfl_sync(FULL, base, 0);
                    if (LIST) got = __shfl_sync(FULL, got, 0);
                    if (LIST && a.tile_cost && unit_tile != 0xFFFFFFFFu) {
                        // ray lists: the time between two fetches of the warp is charged to the chunk of the earlier one
                        if (lane == 0) atomicMax(a.tile_cost + unit_tile, (uint32_t)min((unsigned long long)(clock64() - unit_t0) >> 8, 0xFFFFFFFFull));
                        unit_tile = 0xFFFFFFFFu;
                    }
                    if (base == NO_ITEM) { exhausted = true; break; }
                    pool_next = base;
                    pool_end = LIST ? min(base + got, total) : base + 32u;     // (camera units never straddle the end: whole tiles)
                    if (!LIST) pool_xy = __shfl_sync(FULL, unit_xy, 0);
                    if (a.tile_cost && unit_tile == 0xFFFFFFFFu) {
                        if (LIST) {
                            const uint32_t m = (uint32_t)(base >> (10 + gshift));
                            unit_tile = a.tile_order ? __ldg(a.tile_order + m) : m;
                        } else unit_tile = __shfl_sync(FULL, unit_m, 0);
                        unit_t0 = clock64();
                    }
                }
                const item_t avail = pool_end - pool_next;
                const uint32_t rank = __popc(want & lt);
                const bool served = want_item && (item_t)rank < avail;
                if (served) {
                    item = pool_next + rank; s = 0; hits = 0; want_item = false;
                    if (LIST && a.tile_cost) {
                        // logical item -> ray: chunk (item >> 10) is the chunk traced m-th in cost order
                        const uint32_t mi = (uint32_t)(item >> 10);
                        const uint64_t ray = ((uint64_t)(a.tile_order ? __ldg(a.tile_order + mi) : mi) << 10) | (item & 1023u);
                        item = ray < (uint64_t)a.nrays ? ray : NO_ITEM;      // padding of the last chunk
                        if (item == NO_ITEM) want_item = true;
                    }
                    // sorted ray lists: the i-th item is ray perm[i]; from here on `item` is the ray's own index (load and store)
                    if (MODE == 0 && a.perm && item != NO_ITEM) item = __ldg(a.perm + item);
                    if (!LIST) {
                        // the item's pixel: the unit's first pixel plus the pixel's place in the tile (8x4 blocks of 8x4 pixels)
                        const uint32_t q = (uint32_t)(item >> gshift) & 1023u;
                        s0 = a.s_begin + (int)((uint32_t)item & ((1u << gshift) - 1u)) * nsamp;
                        const uint32_t xy = pool_xy + (((q >> 2) & 0x18u) | (q & 7u)) + ((((q >> 5) & 0x1cu) | ((q >> 3) & 3u)) << 16);
                        const uint32_t px = xy & 0xFFFFu, py = xy >> 16;
                        if (px < (uint32_t)a.w && py < (uint32_t)a.h) { pixel = py * (uint32_t)a.w + px; pxy = xy; }
                        else item = NO_ITEM;                                 // padding pixel of an edge tile
                        if (item == NO_ITEM) want_item = true;
                    }
                }
                pool_next += min((item_t)__popc(want), avail);
                // lanes that drew a padding pixel, or were not served, ask again
                want = __ballot_sync(FULL, want_item);
            }
            // start the next ray of every idle lane that owns an item
            if (cur == NONE && item != NO_ITEM) {
                float ox, oy, oz, dx, dy, dz;
                float tlo = 0.f, thi = FLT_MAX;           // MODE 3: max(tmin, 0), min(tmax, FLT_MAX)
                bool live = true;                         // MODE 3: max(tmin, 0) < tmax (false for a NaN bound): else a miss, not traced
                if (RANGE) {
                    // bihrt_ray_interval, 32 bytes: (o, tmin) (d, tmax) as two 128-bit loads
                    const float4* p = reinterpret_cast<const float4*>(a.rays_iv + item);
                    const float4 r0 = __ldg(p), r1 = __ldg(p + 1);
                    ox = r0.x; oy = r0.y; oz = r0.z; dx = r1.x; dy = r1.y; dz = r1.z;
                    tlo = fmaxf(r0.w, 0.f);
                    live = r0.w == r0.w && tlo < r1.w;
                    thi = fminf(r1.w, FLT_MAX);
                } else if (MODE == 0) {
                    const float* p = reinterpret_cast<const float*>(a.rays + item);
                    ox = __ldg(p); oy = __ldg(p + 1); oz = __ldg(p + 2); dx = __ldg(p + 3); dy = __ldg(p + 4); dz = __ldg(p + 5);
                } else {
                    // u,v per R/src/CUDAKernels.cu:414-415; GetRay per R/src/Camera.cu:18-20
                    const int px = (int)(pxy & 0xFFFFu), py = (int)(pxy >> 16);
                    const float ru = (a.flags & BIHRT_RENDER_JITTER) ? bihrt_jitter(a.seed, pixel, (uint32_t)(s0 + s), 0) : 0.5f;
                    const float rv = (a.flags & BIHRT_RENDER_JITTER) ? bihrt_jitter(a.seed, pixel, (uint32_t)(s0 + s), 1) : 0.5f;
                    const float uu = __fdiv_rn(__fadd_rn((float)px, ru), (float)a.w);
                    const float vv = __fdiv_rn(__fadd_rn((float)py, rv), (float)a.h);
                    ox = a.cam.origin[0]; oy = a.cam.origin[1]; oz = a.cam.origin[2];
                    dx = __fsub_rn(__fadd_rn(__fadd_rn(a.cam.lower_left[0], __fmul_rn(uu, a.cam.horizontal[0])), __fmul_rn(vv, a.cam.vertical[0])), ox);
                    dy = __fsub_rn(__fadd_rn(__fadd_rn(a.cam.lower_left[1], __fmul_rn(uu, a.cam.horizontal[1])), __fmul_rn(vv, a.cam.vertical[1])), oy);
                    dz = __fsub_rn(__fadd_rn(__fadd_rn(a.cam.lower_left[2], __fmul_rn(uu, a.cam.horizontal[2])), __fmul_rn(vv, a.cam.vertical[2])), oz);
                }
                // Ray::Ray, R/src/Ray.cu:3-10
                ix = __frcp_rn(dx); iy = __frcp_rn(dy); iz = __frcp_rn(dz);
                // box planes: t = fma(plane, 1/d, -(o/d)).  The rounding of o/d is an ABSOLUTE error of 2^-24 |o/d| in t (it does not
                // shrink with t): bpad = 2^-22 x the largest finite |o/d| widens every box interval by four times that bound.
                nx = -__fmul_rn(ox, ix); ny = -__fmul_rn(oy, iy); nz = -__fmul_rn(oz, iz);
                bpad = __fmul_rn(BOX_EPS, fmaxf(fmaxf(fabsf(nx) <= FLT_MAX ? fabsf(nx) : 0.f, fabsf(ny) <= FLT_MAX ? fabsf(ny) : 0.f),
                                                fabsf(nz) <= FLT_MAX ? fabsf(nz) : 0.f));
                *reinterpret_cast<float2*>(my_ray) = make_float2(ox, ix); *reinterpret_cast<float2*>(my_ray + 2) = make_float2(oy, iy);
                *reinterpret_cast<float2*>(my_ray + 4) = make_float2(oz, iz); *reinterpret_cast<float2*>(my_ray + 6) = make_float2(dx, dy);
                my_ray[8] = dz;
                if (RANGE) my_ray[9] = tlo;             // the triangle test's lower bound
                // occlusion queries (MODE 0, any_hit): only hits before tmax count, and the first one found ends the ray;
                // ray queries (MODE 3): only hits inside the ray's own interval count
                h.t = RANGE ? thi : (MODE == 0 && a.any_hit) ? a.tmax : FLT_MAX; h.slot = -1; STACK_RESET(); tracing = true;
                // slab test against the scene box, R/src/CUDAKernels.cu:237-262 (same operation order)
                bool in = nu > 0 && live;
                float tMin = __fmul_rn(__fsub_rn(ix < 0.f ? bhi[0] : blo[0], ox), ix);
                float tMax = __fmul_rn(__fsub_rn(ix < 0.f ? blo[0] : bhi[0], ox), ix);
                const float tymin = __fmul_rn(__fsub_rn(iy < 0.f ? bhi[1] : blo[1], oy), iy);
                const float tymax = __fmul_rn(__fsub_rn(iy < 0.f ? blo[1] : bhi[1], oy), iy);
                if ((tMin > tymax) || (tymin > tMax)) in = false;
                if (tymin > tMin) tMin = tymin;
                if (tymax < tMax) tMax = tymax;
                const float tzmin = __fmul_rn(__fsub_rn(iz < 0.f ? bhi[2] : blo[2], oz), iz);
                const float tzmax = __fmul_rn(__fsub_rn(iz < 0.f ? blo[2] : bhi[2], oz), iz);
                if ((tMin > tzmax) || (tzmin > tMax)) in = false;
                if (tzmin > tMin) tMin = tzmin;
                if (tzmax < tMax) tMax = tzmax;
                if (in) {
                    // ... and the rounding of the FMA itself is a RELATIVE error of 2^-24 in t.  A box test can only change its
                    // outcome when the distance in question lies at an end of the ray's interval, i.e. inside the scene box:
                    // 2^-22 x the larger end of the scene interval bounds four times that error for every distance that
                    // matters, and makes the margin ONE constant per ray (one add per bound instead of an add and an FMA)
                    const float tabs = fmaxf(fabsf(tMin), fabsf(tMax));
                    bpad = __fmaf_rn(BOX_EPS, tabs <= FLT_MAX ? tabs : FLT_MAX, bpad);
                    // a zero direction component: fma(plane, inf, -(o * inf)) is inf - inf = NaN or a signed infinity depending on
                    // the signs of plane and origin, never a distance.  The box tests take NaN as 1 / d for that axis, so both its
                    // plane distances are NaN and the NaN-dropping min / max leave the axis out (no constraint: conservative).  The
                    // plane logic of the BIH proper keeps the reference's infinity (it reads 1 / d from shared memory).
                    const float qnan = __uint_as_float(0x7fc00000u);
                    ix = fabsf(ix) <= FLT_MAX ? ix : qnan; iy = fabsf(iy) <= FLT_MAX ? iy : qnan; iz = fabsf(iz) <= FLT_MAX ? iz : qnan;
                    // (coverage: cut at h.t = FLT_MAX too, so that every item's pMax is finite and never needs the pop's check;
                    // ray queries: the interval only narrows the tight interval, rMin -- the reference's strict test -- stays the
                    // scene-box entry)
                    rMin = tMin; pMin = fmaxf(tMin, tlo); pMax = ((MODE == 0 && a.any_hit) || COVER || RANGE) ? fminf(tMax, h.t) : tMax;
                    // Nu == 1: no internal node; the single leaf starts at slot 0 (and must not be
                    // interval-pruned: the reference tests it unconditionally once the box is hit)
                    if (nu == 1) { cur = BIH_REF_LEAFREF(0); pMin = -FLT_MAX; pMax = FLT_MAX; }
                    else if (pMin <= pMax) cur = root_ref;          // box behind the origin: nothing to walk
                }
            }
            if (OCTS) {
                // the octant of the lanes with an item to walk, after every refill; a NaN or zero 1/d fits either sign.  Only
                // warps of pixel sample groups (gshift > 0: at 16 spp a warp holds 2 pixels) take the octant copies: a 1 spp
                // warp spans 8x4 pixels and is refilled lane by lane, and with the copies 1080p x 1 spp lost 11 % (1 M
                // triangles) and 21 % (atrium) against the generic walk alone
                int oct = OCT_MIXED;
                if (gshift > 0) {
                    const bool w = cur != NONE;
                    const uint32_t xn = __ballot_sync(FULL, w && ix < 0.f), xp = __ballot_sync(FULL, w && ix > 0.f);
                    const uint32_t yn = __ballot_sync(FULL, w && iy < 0.f), yp = __ballot_sync(FULL, w && iy > 0.f);
                    const uint32_t zn = __ballot_sync(FULL, w && iz < 0.f), zp = __ballot_sync(FULL, w && iz > 0.f);
                    if (!((xn && xp) || (yn && yp) || (zn && zp))) oct = (xn != 0) | (yn != 0) << 1 | (zn != 0) << 2;
                }
                my_ray[9] = __int_as_float(oct);
            }
            if (__ballot_sync(FULL, cur != NONE || tracing) == 0 && exhausted &&
                __ballot_sync(FULL, item != NO_ITEM) == 0) break;
        }

        // ================= phase 1: internal nodes =====================================================
        // A lane steps through nodes until it holds a leaf, then waits.  The warp leaves the phase when
        // nobody has a node left, or as soon as the waiting lanes outnumber the walking ones: finishing
        // the node phase for a few stragglers with most lanes idle costs more than testing the held
        // leaves first.
        // Invariant: an item held in `cur` has a non-empty tight interval that ends at or before the closest hit
        // (pMin <= pMax <= h.t).  Children inherit it from the tests that select them, so only items that
        // come off the stack -- h.t may have shrunk since they were pushed -- are checked (POP_VALID); an
        // item that fails is dropped without a node fetch.  Same visits, same order, same counters as the
        // entry check of oracle/bih_oracle.c:traverse_proper.
#define BOX_SLAB(lx, ly, lz, hx, hy, hz, bn, bf)                                                            \
        do {                                                                                                \
            const float ax0 = __fmaf_rn((lx), ix, nx), ax1 = __fmaf_rn((hx), ix, nx);                       \
            const float ay0 = __fmaf_rn((ly), iy, ny), ay1 = __fmaf_rn((hy), iy, ny);                       \
            const float az0 = __fmaf_rn((lz), iz, nz), az1 = __fmaf_rn((hz), iz, nz);                       \
            float n_, f_;                                                                                   \
            if (OCT == OCT_MIXED) {                                                                         \
                n_ = fmaxf(fmaxf(fminf(ax0, ax1), fminf(ay0, ay1)), fminf(az0, az1));                       \
                f_ = fminf(fminf(fmaxf(ax0, ax1), fmaxf(ay0, ay1)), fmaxf(az0, az1));                       \
            } else {                           /* 1/d < 0: the hi plane is the near one */                  \
                n_ = fmax3((OCT & 1) ? ax1 : ax0, (OCT & 2) ? ay1 : ay0, (OCT & 4) ? az1 : az0);            \
                f_ = fmin3((OCT & 1) ? ax0 : ax1, (OCT & 2) ? ay0 : ay1, (OCT & 4) ? az0 : az1);            \
            }                                                                                               \
            (bn) = __fsub_rn(n_, bpad);                                                                     \
            (bf) = __fadd_rn(f_, bpad);                                                                     \
        } while (0)
#define POP_VALID()                                                                                         \
        do {                                                                                                \
            cur = NONE;                                                                                     \
            if (COVER) {                       /* h.t is still FLT_MAX: the top item is valid */            \
                if (sp > 0) {                                                                               \
                    uint4 e;                                                                                \
                    STACK_POP(e);                                                                           \
                    cur = e.x; rMin = __uint_as_float(e.y); pMin = __uint_as_float(e.z); pMax = __uint_as_float(e.w); \
                }                                                                                           \
            } else while (sp > 0) {                                                                         \
                uint4 e;                                                                                    \
                STACK_POP(e);                                                                               \
                const float m = fminf(__uint_as_float(e.w), h.t);                                           \
                if (__uint_as_float(e.z) <= m) { cur = e.x; rMin = __uint_as_float(e.y); pMin = __uint_as_float(e.z); pMax = m; break; } \
            }                                                                                               \
        } while (0)
#ifdef BIHRT_DEBUG_STACK
#define DEBUG_STACK_TRAP() do { if (sp >= STACK_DEPTH) __trap(); } while (0)
#else
#define DEBUG_STACK_TRAP() do { } while (0)
#endif
        // The node phase, expanded once per ray octant (OCT = its sign bits) and once generic (OCT_MIXED), see the
        // octant copies at the head of this file.  A macro rather than a function or lambda: the other modes then compile to the code they had.
#define NODE_PHASE(OCT_)                                                                                           \
        do {                                                                                                        \
            constexpr int OCT = (OCT_);                                                                             \
            for (;;) {                                                                                              \
                _Pragma("unroll (NODE_STEPS)")                                                                      \
                for (int rep = 0; rep < NODE_STEPS && (int)cur >= 0; rep++) {                                       \
                    /* (origin, 1/dir) on this node's axis: one 64-bit LDS at ray_smem + axis * 8 */                \
                    float2 oi;                                                                                      \
                    uint32_t ra;                                                                                    \
                    asm("mad.lo.u32 %0, %1, 8, %2;" : "=r"(ra) : "r"(cur & 3u), "r"(ray_smem));                     \
                    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(oi.x), "=f"(oi.y) : "r"(ra));            \
                    /* node address = base + index * 64, as one 32x32->64 multiply-add on the base pointer */       \
                    const float4* np;                                                                               \
                    asm("mad.wide.u32 %0, %1, 64, %2;" : "=l"(np) : "r"(cur >> 2), "l"(nodes_b));                   \
                    /* Ray lists (MODE 0 and 3) fetch the 64-byte node as TWO 256-bit read-only loads (LDG.E.256, new on sm_100) instead of */ \
                    /* four 128-bit ones.  Measured (B200, Mrays/s, 128-bit -> 256-bit): diffuse bounce list on the atrium 2157 -> 2304 */ \
                    /* (there every lane fetches its own node and the L1 tag stage is the busiest unit, 88 %), 1 M triangles 1080p x 1 */ \
                    /* spp 6045 -> 6230, 10 M 3282 -> 3403; but coherent packets lose -- 4K x 16 spp 12014 -> 11833, atrium x 4 spp */ \
                    /* 6613 -> 6475 (the 8-register alignment of the destination costs two spills in a 64-register kernel).  So the */ \
                    /* camera modes keep the 128-bit loads. */                                                      \
                    float4 nd, b0, b1, b2;                                                                          \
                    if (LIST) {                                                                                     \
                        asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"                                  \
                            : "=f"(nd.x), "=f"(nd.y), "=f"(nd.z), "=f"(nd.w), "=f"(b0.x), "=f"(b0.y), "=f"(b0.z), "=f"(b0.w) : "l"(np)); \
                        asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"                                  \
                            : "=f"(b1.x), "=f"(b1.y), "=f"(b1.z), "=f"(b1.w), "=f"(b2.x), "=f"(b2.y), "=f"(b2.z), "=f"(b2.w) : "l"(np + 2)); \
                    } else { nd = __ldg(np); b0 = __ldg(np + 1); b1 = __ldg(np + 2); b2 = __ldg(np + 3); }          \
                    if (COUNTED) { nnodes++; const uint32_t am = __activemask(); wnode += (lane == __ffs(am) - 1); } \
                    const uint32_t rl = __float_as_uint(nd.z), rr = __float_as_uint(nd.w);                          \
                    const bool neg = oi.y < 0.f;                           /* near = sign[axis], :286 */            \
                    const float t0 = __fmul_rn(__fsub_rn(nd.x, oi.x), oi.y);   /* :288-289 */                       \
                    const float t1 = __fmul_rn(__fsub_rn(nd.y, oi.x), oi.y);                                        \
                    const float tn = neg ? t1 : t0, tf = neg ? t0 : t1;                                             \
                    const uint32_t refn = neg ? rr : rl, reff = neg ? rl : rr;                                      \
                    /* the children's boxes: parametric interval of the ray inside each (slab test on all three axes; min / max of */ \
                    /* the two plane distances per axis orders them whatever the sign of the direction -- an octant copy orders */ \
                    /* them by the sign it knows -- and drops the NaN of a zero direction component), widened by the ray's margin */ \
                    /* (bpad) so that rounding never culls a box the exact ray touches.  A child the ray misses is never fetched; a */ \
                    /* child that is entered gets the tighter interval. */                                          \
                    float bnL, bfL, bnR, bfR;                                                                       \
                    BOX_SLAB(b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, bnL, bfL);                                         \
                    BOX_SLAB(b1.z, b1.w, b2.x, b2.y, b2.z, b2.w, bnR, bfR);                                         \
                    /* (three-input min / max, FMNMX3: same NaN and signed-zero behaviour as the nested two-input calls they replace) */ \
                    const float nLo = fmaxf(pMin, neg ? bnR : bnL), nHi = fmin3(pMax, tn, neg ? bfR : bfL);         \
                    const float fLo = fmax3(pMin, tf, neg ? bnL : bnR), fHi = fminf(pMax, neg ? bfL : bfR);         \
                    const bool go_near = (Q || rMin < tn) && (nLo <= nHi);   /* reference's strict test (:292) + closed tight interval */ \
                    const bool go_far = (fLo <= fHi);                                                               \
                    /* (the four cases as SELECTS instead of branch targets were measured: 4K x 16 spp 11997 -> 11259 Mrays/s, atrium -9 %: */ \
                    /* coherent lanes mostly agree on the case, and the selects cost every lane every time) */      \
                    if (go_near && go_far) {                                                                        \
                        /* near before far, except a far LEAF next to a near NODE is tested first (:344-349) */     \
                        if ((int)refn >= 0 && (int)reff < 0) {                                                      \
                            STACK_PUSH(make_uint4(refn, __float_as_uint(rMin), __float_as_uint(nLo), __float_as_uint(nHi))); \
                            cur = reff; rMin = tf; pMin = fLo; pMax = fHi;                                          \
                        } else {                                                                                    \
                            STACK_PUSH(make_uint4(reff, __float_as_uint(tf), __float_as_uint(fLo), __float_as_uint(fHi))); \
                            cur = refn; pMin = nLo; pMax = nHi;                                                     \
                        }                                                                                           \
                        /* depth: a root-to-leaf path pushes at most one item per Morton bit, so sp <= 30 < STACK_DEPTH by */ \
                        /* construction; the instrumented build reports the deepest stack (counters[2]) and refuses to run past */ \
                        /* the array, -DBIHRT_DEBUG_STACK traps in every build */                                   \
                        if (COUNTED) { maxsp = max(maxsp, (uint32_t)sp); if (sp >= STACK_DEPTH) { maxsp = 0x7fffffffu; sp = STACK_DEPTH - 1; } } \
                        DEBUG_STACK_TRAP();                                                                         \
                    } else if (go_near) { cur = refn; pMin = nLo; pMax = nHi; }                                     \
                    else if (go_far) { cur = reff; rMin = tf; pMin = fLo; pMax = fHi; }                             \
                    else POP_VALID();                                                                               \
                }                                                                                                   \
                const uint32_t m_walk = __ballot_sync(FULL, (int)cur >= 0);                                         \
                if (m_walk == 0) break;                                                                             \
                const uint32_t m_wait = __ballot_sync(FULL, cur + 1u > 0x80000000u);  /* a leaf (negative, not NONE) */ \
                if (__popc(m_wait) > __popc(m_walk)) break;                                                         \
            }                                                                                                       \
        } while (0)
        if constexpr (!OCTS) NODE_PHASE(OCT_MIXED);       // (not instantiated in the other modes: their code stays as it was)
        else switch (__float_as_int(my_ray[9])) {        // warp-uniform
            case 0: NODE_PHASE(0); break;
            case 1: NODE_PHASE(1); break;
            case 2: NODE_PHASE(2); break;
            case 3: NODE_PHASE(3); break;
            case 4: NODE_PHASE(4); break;
            case 5: NODE_PHASE(5); break;
            case 6: NODE_PHASE(6); break;
            case 7: NODE_PHASE(7); break;
            default: NODE_PHASE(OCT_MIXED); break;
        }
        // ================= phase 2: the leaf this lane holds ===========================================
        if (cur + 1u > 0x80000000u) {
            const char* tp;
            asm("mad.wide.u32 %0, %1, 12, %2;" : "=l"(tp) : "r"(cur & 0x7FFFFFFCu), "l"(tris_b));
            const float2 dxy = *reinterpret_cast<const float2*>(my_ray + 6);
            test_leaf<COUNTED, COVER, RANGE, TWO_SIDED>(tp, my_ray[0], my_ray[2], my_ray[4], dxy.x, dxy.y, my_ray[8], h, ntris, wleaf, my_ray + 9);
            // occluded / covered: nothing else to learn
            if (((LIST && a.any_hit) || COVER) && h.slot >= 0) { STACK_RESET(); cur = NONE; }
            else POP_VALID();
        }
#undef NODE_PHASE
#undef DEBUG_STACK_TRAP
#undef POP_VALID
#undef BOX_SLAB
#undef STACK_RESET
#undef STACK_PUSH
#undef STACK_POP
        __syncwarp();
    }

    if (COUNTED) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            nnodes += __shfl_xor_sync(FULL, nnodes, o);
            ntris += __shfl_xor_sync(FULL, ntris, o);
            maxsp = max(maxsp, __shfl_xor_sync(FULL, maxsp, o));
        }
        if (lane == 0) {
            atomicAdd(&a.counters[0], (unsigned long long)nnodes);
            atomicAdd(&a.counters[1], (unsigned long long)ntris);
            atomicMax(&a.counters[2], (unsigned long long)maxsp);
        }
        wnode = __reduce_add_sync(FULL, wnode); wleaf = __reduce_add_sync(FULL, wleaf);
        if (lane == 0) { atomicAdd(&a.counters[4], (unsigned long long)wnode); atomicAdd(&a.counters[5], (unsigned long long)wleaf); }
    }
}

// hit counts -> packed colour (Color + rgbToInt, R/src/CUDAKernels.cu:82-88,385-387,420-422), in place
__global__ void k_resolve(uint32_t* fb, int npix, int spp) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npix) return;
    fb[i] = pack_colour(fb[i], spp);
}

// Tile order for the next launch of the same frame geometry, from the costs the launch that just ended measured
// (longest 32-ray unit of each tile).  Tiles are put in TILE_CLASSES classes by cost relative to the frame's longest
// unit (>= 1/2, >= 1/4, >= 1/8, >= 1/16, the rest), most expensive class first, scan order kept inside a class (a
// stable partition: the bulk of the frame is still traced in scan order and neighbouring tiles share L1 / L2).
// A unit on the silhouette of the 1 M-triangle sphere is ~0.4 ms of dependent fetches; started last it is the tail
// of the launch, started first it overlaps everything else.
#define TILE_CLASSES 5
__device__ __forceinline__ int tile_class(uint32_t c, uint32_t mx) {
    int k = 0;
#pragma unroll
    for (int j = 1; j < TILE_CLASSES; j++) k += c < max(1u, mx >> j);
    return k;
}
__global__ void __launch_bounds__(1024) k_tile_order(uint32_t* __restrict__ cost, uint32_t* __restrict__ order, uint32_t ntiles) {
    __shared__ uint32_t s_w[TILE_CLASSES][32];
    __shared__ uint32_t s_max, s_base[TILE_CLASSES];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const uint32_t per = (ntiles + 1023u) / 1024u, i0 = min(ntiles, threadIdx.x * per), i1 = min(ntiles, i0 + per);
    uint32_t mx = 0;
    for (uint32_t i = i0; i < i1; i++) mx = max(mx, cost[i]);
    mx = __reduce_max_sync(0xffffffffu, mx);
    if (lane == 0) s_w[0][w] = mx;
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t m = 0; for (int k = 0; k < 32; k++) m = max(m, s_w[0][k]); s_max = m; }
    __syncthreads();
    mx = s_max;
    uint32_t cnt[TILE_CLASSES], inc[TILE_CLASSES];
#pragma unroll
    for (int k = 0; k < TILE_CLASSES; k++) cnt[k] = 0;
    for (uint32_t i = i0; i < i1; i++) {
        const int cl = tile_class(cost[i], mx);
#pragma unroll
        for (int k = 0; k < TILE_CLASSES; k++) cnt[k] += (cl == k);
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TILE_CLASSES; k++) {                      // block-wide exclusive scan of every class count
        inc[k] = cnt[k];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, inc[k], o); if (lane >= o) inc[k] += t; }
        if (lane == 31) s_w[k][w] = inc[k];
    }
    __syncthreads();
    if (threadIdx.x < TILE_CLASSES) {
        uint32_t run = 0;
        for (int j = 0; j < 32; j++) { const uint32_t x = s_w[threadIdx.x][j]; s_w[threadIdx.x][j] = run; run += x; }
        s_base[threadIdx.x] = run;                                // class total
    }
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t run = 0; for (int k = 0; k < TILE_CLASSES; k++) { const uint32_t x = s_base[k]; s_base[k] = run; run += x; } }
    __syncthreads();
    uint32_t pos[TILE_CLASSES];
#pragma unroll
    for (int k = 0; k < TILE_CLASSES; k++) pos[k] = s_base[k] + s_w[k][w] + inc[k] - cnt[k];
    for (uint32_t i = i0; i < i1; i++) {
        const int cl = tile_class(cost[i], mx);
#pragma unroll
        for (int k = 0; k < TILE_CLASSES; k++) if (cl == k) order[pos[k]++] = i;
    }
    __syncthreads();
    for (uint32_t i = i0; i < i1; i++) cost[i] = 0;
}

// Small launches (a few million rays: every tile holds only a handful of units per warp, and the tail is a large part of
// the launch) get a full descending sort by cost instead: counting sort over 256 buckets of ~2 us, order inside a bucket
// arbitrary.  480x270 x 16 spp: 2630 -> 3000 Mrays/s; at 33 M rays the same sort loses 3 % to the scattered tiles.
__global__ void __launch_bounds__(1024) k_tile_sort(uint32_t* __restrict__ cost, uint32_t* __restrict__ order, uint32_t ntiles) {
    __shared__ uint32_t s_cnt[256], s_off[256];
    if (threadIdx.x < 256) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < ntiles; i += 1024) atomicAdd(&s_cnt[min(255u, cost[i] >> 4)], 1u);
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t run = 0; for (int b = 255; b >= 0; b--) { s_off[b] = run; run += s_cnt[b]; } }
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < ntiles; i += 1024) order[atomicAdd(&s_off[min(255u, cost[i] >> 4)], 1u)] = i;
    __syncthreads();
    for (uint32_t i = threadIdx.x; i < ntiles; i += 1024) cost[i] = 0;
}

int bihrt_tile_order_launch(bihrt_ctx* c, uint32_t* cost, uint32_t* order, uint32_t ntiles, bool full_sort) {
    if (full_sort) k_tile_sort<<<1, 1024, 0, c->stream>>>(cost, order, ntiles);
    else k_tile_order<<<1, 1024, 0, c->stream>>>(cost, order, ntiles);
    c->kernel_launches += 1;
    BIHRT_CUDA(c, cudaGetLastError());
    return BIHRT_OK;
}

int bihrt_resolve_launch(bihrt_ctx* c, uint32_t* fb, int npix, int spp) {
    k_resolve<<<(npix + 255) / 256, 256, 0, c->stream>>>(fb, npix, spp);
    c->kernel_launches += 1;
    BIHRT_CUDA(c, cudaGetLastError());
    return BIHRT_OK;
}

template <int MODE, bool COUNTED, bool Q>
static int launch(bihrt_ctx* c, const TraceArgs& a) {
    int per_sm = c->opt_trace_blocks_per_sm;
    if (per_sm <= 0) {
        BIHRT_CUDA(c, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_trace<MODE, COUNTED, Q>, TRACE_THREADS, 0));
        if (per_sm < 1) per_sm = 1;
    }
    BIHRT_CUDA(c, cudaMemsetAsync(a.work, 0, 4 * 1024, c->stream));
    k_trace<MODE, COUNTED, Q><<<c->sm_count * per_sm, TRACE_THREADS, 0, c->stream>>>(a);
    c->kernel_launches += 1;
    BIHRT_CUDA(c, cudaGetLastError());
    return BIHRT_OK;
}

template <bool Q>
static int launch_mode(bihrt_ctx* c, const TraceArgs& a, int mode, bool counted) {
    switch (mode * 2 + (counted ? 1 : 0)) {
        case 0: return launch<0, false, Q>(c, a);
        case 1: return launch<0, true, Q>(c, a);
        case 2: return launch<1, false, Q>(c, a);
        case 3: return launch<1, true, Q>(c, a);
        case 4: return launch<2, false, Q>(c, a);
        case 5: return launch<2, true, Q>(c, a);
        case 6: return launch<3, false, Q>(c, a);
        case 8: return launch<4, false, Q>(c, a);
        default: return bihrt_fail(c, BIHRT_ERR_INVALID, "bad trace mode %d", mode);
    }
}

int bihrt_trace_launch(bihrt_ctx* c, const TraceArgs& a_in, int mode, bool counted) {
    TraceArgs a = a_in;
    // per-SM queues pay off once a launch is long enough to amortise the end-of-kernel stealing
    // (measured: +7 % at 133 M rays, -9 % at 2 M rays on the 1 M-triangle scene)
    const bool list = mode == 0 || mode == 3 || mode == 4;     // ray lists (3, 4: with intervals and hit records)
    const int64_t rays = list ? a.nrays : (int64_t)a.w * a.h * (a.s_end - a.s_begin) / (a.shard_count > 0 ? a.shard_count : 1) / (a.il_count > 0 ? a.il_count : 1);
    // ... and only when a warp spans many pixels: with a pixel's samples in consecutive lanes a warp is coherent on
    // its own and the queues only add stealing overhead (-5 % at 4K x 16 spp)
    const bool on = a.queues < 0 ? (rays >= (16ll << 20) && (list || a.gshift == 0)) : a.queues != 0;
    a.queues = on ? (c->sm_count < 1024 ? c->sm_count : 1024) : 1;
    // cost-ordered tiles (camera modes, one global counter): reuse the order measured by the previous launch of the same
    // frame geometry; always record the costs of this one
    uint32_t ntiles = 0;
    bihrt_ctx::TileKey key;
    // the 32-bit work counters (global and per-SM) must not wrap: padded items of this launch
    if (!list) {
        const int tx = (a.w + 31) / 32, ty = (a.h + 31) / 32, T = tx * ty;
        const int mine = T > a.shard_index ? (T - a.shard_index + a.shard_count - 1) / a.shard_count : 0;
        if ((((uint64_t)mine * 1024u) << a.gshift) >= (1ull << 32) - (1ull << 24))
            return bihrt_fail(c, BIHRT_ERR_INVALID, "launch of %d tiles x 1024 pixels x %d lane groups exceeds the 32-bit work counter", mine, 1 << a.gshift);
        a.tile_cols = (uint32_t)tx; a.tile_cols_rcp = 0xFFFFFFFFu / (uint32_t)tx;
    }
    // (launches of tens of milliseconds have no tail to speak of and lose ~0.5 % to the changed tile neighbourhood; tiny
    // scenes have no long units -- the Cornell box frame is 25 us -- and only pay for the extra k_tile_order launch)
    const bool order_on = a.queues == 1 && (c->opt_tile_order > 1 || (c->opt_tile_order == 1 && rays >= (64ll << 10) && rays < (48ll << 20) && c->n >= 10000));
    if (order_on) {
        if (list) {
            // ray lists: chunks of 1024 rays play the role of tiles; the order is reused for lists of the same length (the
            // next frame's shadow / bounce batch), stale costs only change the schedule, never a result
            if (a.nrays > 1024 && a.nrays <= (65536ll << 10)) { ntiles = (uint32_t)((a.nrays + 1023) >> 10); key.nrays = a.nrays; }
        } else {
            const int tx = (a.w + 31) / 32, ty = (a.h + 31) / 32, T = tx * ty;
            const int mine = T > a.shard_index ? (T - a.shard_index + a.shard_count - 1) / a.shard_count : 0;
            if (mine > 1 && mine <= 65536) ntiles = (uint32_t)mine;
            key.w = a.w; key.h = a.h; key.gshift = a.gshift; key.nsamp = a.s_end - a.s_begin; key.shard_index = a.shard_index;
            key.shard_count = a.shard_count; key.il_index = a.il_index; key.il_count = a.il_count; key.il_cshift = a.il_cshift;
        }
        key.mode = list ? mode : 1; key.ntiles = ntiles;     // (interval lists, one- and two-sided, keep their own slots)
    }
    bihrt_ctx::TileSlot* slot = nullptr;
    if (ntiles) {
        for (auto& ts : c->tile_slots) if (ts.cap && ts.key == key) slot = &ts;
        if (!slot) {                                  // take the next slot round-robin
            slot = &c->tile_slots[c->tile_next];
            c->tile_next = (c->tile_next + 1) % 4;
            slot->key = key; slot->valid = false;
        }
        if ((size_t)ntiles > slot->cap) {
            if (slot->cost) cudaFree(slot->cost);
            if (slot->order) cudaFree(slot->order);
            slot->cost = slot->order = nullptr; slot->cap = 0; slot->valid = false;
            if (cudaMalloc(&slot->cost, (size_t)ntiles * 4) != cudaSuccess || cudaMalloc(&slot->order, (size_t)ntiles * 4) != cudaSuccess) {
                cudaGetLastError();
                if (slot->cost) { cudaFree(slot->cost); slot->cost = nullptr; }
                slot = nullptr; ntiles = 0;
            } else slot->cap = ntiles;
        }
        if (slot) {
            if (!slot->valid) BIHRT_CUDA(c, cudaMemsetAsync(slot->cost, 0, (size_t)ntiles * 4, c->stream));
            a.tile_cost = slot->cost;
            a.tile_order = slot->valid ? slot->order : nullptr;
        }
    }
    a.status_map = c->d_status_map;
    int rc = c->built_quality ? launch_mode<true>(c, a, mode, counted) : launch_mode<false>(c, a, mode, counted);
    if (rc == BIHRT_OK && slot) {
        if ((rc = bihrt_tile_order_launch(c, slot->cost, slot->order, ntiles, rays < c->opt_tile_sort_below)) == BIHRT_OK) slot->valid = true;
    }
    return rc;
}
