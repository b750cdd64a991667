// Internal declarations shared by build.cu, trace.cu and api.cu.  sm_100a only.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include "../../include/bihrt.h"

// -------------------------------------------------------------------------------------------
// HBM layout of a built BIH (DESIGN.md "Data layout")
// -------------------------------------------------------------------------------------------
// Node, 64 B (one 64-byte-aligned record = two sectors, 4 x LDG.128 per visit).  Index = the reference's (Karras) node
// index, so node i here is TreeInternalNode i of R/src/Tree.cuh:16-24.
//   first 16 bytes = the BIH proper, bit-exact with the reference: the two clip planes and the two child references.
//   A child reference packs
//     bit 31     : child is a leaf
//     bits 30..2 : internal child -> node index; leaf child -> first slot of the leaf in tris[]
//                  (so (ref & ~3) * 16 is the node's byte offset and (ref & 0x7FFFFFFC) * 12 the triangle's)
//     bits 1..0  : split axis OF THE CHILD (internal children; 0 for leaves) -- the traversal knows the
//                  axis of a node before it fetches it, so the ray constants for that axis are loaded
//                  in parallel with the node instead of after it.  The root's axis is in the header.
//   last 48 bytes = the bounding boxes of the two children (lo.xyz, hi.xyz each): exact min / max of the vertex
//                  coordinates below each child, from the same heaps the clip planes are range queries of
//                  (clip0 = lbox hi[axis], clip1 = rbox lo[axis]).  A BIH plane pair bounds ONE axis per level, so the
//                  reference walks into every subtree whose slab the ray crosses -- 39 nodes and 13 triangle tests per
//                  primary ray on the 1 M-triangle scene, most of them for rays that miss the mesh altogether.  With the
//                  children's boxes in the parent, a child the ray misses is never fetched: 14 nodes and 1.1 triangle
//                  tests per ray, same hits (the visited leaves are a subset of the reference's, in the reference's order).
struct __align__(16) BihNode {
    float    clip0;   // max over the left subtree of hi[axis]   (t_clipPlanes[0])
    float    clip1;   // min over the right subtree of lo[axis]  (t_clipPlanes[1])
    uint32_t ref_l;
    uint32_t ref_r;
    float    lbox[6]; // left child: lo.xyz, hi.xyz
    float    rbox[6]; // right child
};
static_assert(sizeof(BihNode) == 64, "node is one 64-byte record");
#define BIH_REF_LEAF  0x80000000u
#define BIH_REF_NODE(idx, axis) (((uint32_t)(idx) << 2) | (uint32_t)(axis))
#define BIH_REF_LEAFREF(slot)   (BIH_REF_LEAF | ((uint32_t)(slot) << 2))
#define BIH_REF_INDEX(ref)      (((ref) & 0x7FFFFFFFu) >> 2)
#define BIH_REF_AXIS(ref)       ((ref) & 3u)
#define BIH_MAX_TRIS  (1ll << 29)

// Leaf-ordered triangle, 48 B = 3 x LDG.128: v0, e1 = v1 - v0, e2 = v2 - v0 (the two edges
// RayTriangleIntersection recomputes per test, R/src/CUDAKernels.cu:18-19), the input triangle index
// (m_trisIndexes[slot]), an end-of-leaf flag and the slot number itself.  Slot order = Morton-sorted order, so a leaf is a
// contiguous run and the reference's triangleIdxs[] / firstIdxs[] / duplicatesCnts[] indirections
// (R/src/CUDAKernels.cu:215-217) are gone from the traversal.
struct __align__(16) BihTri {
    float    v0x, v0y, v0z, e1x;
    float    e1y, e1z, e2x, e2y;
    float    e2z;
    uint32_t prim;
    uint32_t last;     // 1 on the last triangle of its leaf
    uint32_t slot;     // this record's own index (= the reference's HitRecord::triangleIdx)
};

// Device-resident header of a built BIH; lives at the start of the blob that is broadcast.
struct BihHeader {
    uint32_t n;          // triangles
    uint32_t nu;         // leaves
    float    lo[3];      // scene box
    float    hi[3];
    uint32_t status;     // 0 ok, !=0 device watchdog
    uint32_t root_axis;  // split axis of node 0
    uint32_t quality;    // 0: the reference's tree (parity layout, nu - 1 nodes); 1: quality-mode tree (node slots up to n - 1, deeper)
    uint32_t pad[5];
};
static_assert(sizeof(BihHeader) == 64, "header is one 64-byte line");

// -------------------------------------------------------------------------------------------
// context
// -------------------------------------------------------------------------------------------
#define BIHRT_PROF_EVENTS 16
struct bihrt_group;       // csrc/multi.cu: the contexts of one bihrt_create_multi call + their NCCL communicators
struct bihrt_ctx {
    bihrt_group* group = nullptr; int group_rank = 0;
    int          device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    std::string  err;
    int          sm_count = 148;

    // scene (input order)
    float*   d_tri_in = nullptr;     // n x 9 floats (reference Triangle layout, 36 B)
    int64_t  n = 0, cap_n = 0;
    bool     have_scene = false, built = false;
    bool     topology_valid = false;   // a full build on this context produced keys / order / leaves for the current n

    // BIH blob: [BihHeader | nodes (nu-1, padded) | tris (n)]  -- one allocation, one broadcast
    uint8_t* d_blob = nullptr;
    size_t   blob_cap = 0;
    BihHeader* d_hdr = nullptr;
    BihNode*   d_nodes = nullptr;
    BihTri*    d_tris = nullptr;

    // build scratch (all sized by cap_n)
    uint32_t *d_keys[2] = {nullptr, nullptr}, *d_vals[2] = {nullptr, nullptr};
    uint64_t *d_keys64[2] = {nullptr, nullptr};   // quality mode: 63-bit Morton keys (allocated on first use)
    uint32_t *d_lookback_q = nullptr; size_t lookback_q_words = 0;
    uint32_t *d_umc = nullptr;        // unique codes [nu]
    uint32_t *d_first = nullptr;      // first slot of each leaf [nu+1]
    uint32_t *d_hist = nullptr;       // 4 x 256 digit histograms + tile counters + misc
    uint32_t *d_lookback = nullptr;   // onesweep / RLE decoupled look-back words
    size_t    lookback_words = 0;
    float4   *d_heaps = nullptr;      // implicit min/max heap over the slot boxes: entry e = (lo.xyz, -), (hi.xyz, -) at [2e], [2e+1]; 2P entries
    uint32_t *d_scenebox_enc = nullptr; // 6 order-preserving encoded floats

    // trace
    uint32_t* d_fb = nullptr; int fb_w = 0, fb_h = 0; size_t fb_cap = 0;
    bool      fb_exported = false;                     // a CUDA IPC handle of d_fb is out: the allocation must not move
    uint32_t* h_status = nullptr;                      // pinned + mapped host word: hdr->status of the last build (written by k_nodes)
    uint32_t* d_status_map = nullptr;                  // its device alias
    void*     d_io = nullptr; size_t io_cap = 0;      // staging for host ray lists / results
    unsigned long long* d_counters = nullptr;
    // ray sorting scratch (raysort.cu)
    uint32_t *d_rs_keys[2] = {nullptr, nullptr}, *d_rs_vals[2] = {nullptr, nullptr}, *d_rs_hist = nullptr, *d_rs_lookback = nullptr;
    BihHeader* d_rs_hdr = nullptr; size_t rs_cap = 0;
    int opt_sort_rays = 0;  // ray lists: 1 = group the rays by origin cell + direction octant before tracing (incoherent batches), 0 = trace in list order
    uint32_t* d_work = nullptr;                        // persistent-kernel work counter
    // cost-ordered tiles: the longest unit of every 32x32-pixel tile measured by the previous launch of the same frame
    // geometry, and the tile order (most expensive first) derived from it
    // (a few slots keyed by the launch geometry, so that a frame's camera pass and its shadow / bounce lists each keep theirs)
    // (a slot is reused only for a launch whose geometry matches FIELD BY FIELD: a permutation of the wrong size would skip tiles)
    struct TileKey {
        int mode = -1, w = 0, h = 0, gshift = 0, nsamp = 0, shard_index = 0, shard_count = 0, il_index = 0, il_count = 0, il_cshift = 0;
        int64_t nrays = 0; uint32_t ntiles = 0;
        bool operator==(const TileKey& o) const {
            return mode == o.mode && w == o.w && h == o.h && gshift == o.gshift && nsamp == o.nsamp && shard_index == o.shard_index &&
                   shard_count == o.shard_count && il_index == o.il_index && il_count == o.il_count && il_cshift == o.il_cshift &&
                   nrays == o.nrays && ntiles == o.ntiles;
        }
    };
    struct TileSlot { TileKey key; bool valid = false; uint32_t *cost = nullptr, *order = nullptr; size_t cap = 0; };
    TileSlot tile_slots[4]; int tile_next = 0;

    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool        build_timed = false;

    // options
    int opt_trace_blocks_per_sm = 0;   // 0 = occupancy query
    int opt_lane_groups = -1; // samples of a pixel across lanes: -1 auto (as many as divide the sample count, <= 32), else 2^k
    int opt_interleave_chunk = 8;  // multi-GPU unit interleave: consecutive units per run (power of two; reduced until it divides a tile)
    int opt_tile_order = 1; // camera modes: start the tiles that were expensive in the previous frame first (1: launches of 64 k .. 48 M rays on scenes of >= 10 k triangles, 2: always, 0: never)
    int64_t opt_tile_sort_below = 4 << 20;   // launches with fewer rays get a full sort by cost instead of the 5-class stable partition
    int opt_sm_queues = -1; // 1: per-SM work queues (tile locality in L1), 0: one global counter, -1: by launch size
    int64_t kernel_launches = 0;
    int opt_build_graph = 1;            // replay the build as a captured CUDA graph
    cudaGraphExec_t build_graph_exec = nullptr; int64_t build_graph_n = -1, build_graph_launches = 0;
    int opt_morton_bits = 30;   // 30: the reference's grid (parity path); 63: quality mode (SURVEY.md 8(f) f4, non-parity)
    int opt_leaf_cap = 4;       // quality mode: a subtree of at most this many triangles becomes one leaf
    bool built_quality = false; // the BIH in the blob is a quality-mode tree (deeper: the traversal needs the long stack, and no reference quirks)
    // winding numbers (winding.cu): far-field table, 256 B per node slot, built lazily; every place that sets `built` clears
    // wtab_valid
    float*    d_wtab = nullptr; int64_t wtab_slots = 0;
    uint32_t* d_wscratch = nullptr;                    // its build's queue, parents, leaf list and arrival counters
    bool      wtab_valid = false;
    int opt_debug_trip_watchdog = 0;   // tests: the next build reports this watchdog status (as if a sort pass had timed out)
    int opt_profile = 0;    // record an event after every build stage (bihrt_get_stat "build_stage_us_<i>")
    cudaEvent_t prof_ev[BIHRT_PROF_EVENTS] = {};
    int prof_count = 0;
};

int  bihrt_fail(bihrt_ctx* c, int code, const char* fmt, ...);
#define BIHRT_CUDA(c, call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) \
    return bihrt_fail((c), BIHRT_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)

// d_hist layout (uint32 words), shared by the build and the ray sort
#define H_HIST      0        // up to 8 x 256 digit counts (4 passes for the 30-bit keys, 8 for the 63-bit keys of the quality mode)
#define H_TILECTR   2048     // [0..7] onesweep tile counters, [8] rle tile counter
#define H_WORDS     2064
#define SORT_TILE   4096     // keys per onesweep tile (32-bit keys)

// build.cu
int bihrt_sort_pairs_launch(bihrt_ctx* c, uint32_t* keys[2], uint32_t* vals[2], uint32_t n, int passes, uint32_t* hist, uint32_t* lookback, BihHeader* hdr);
int bihrt_build_launch(bihrt_ctx* c);
int bihrt_build_setup(bihrt_ctx* c);      // once per context: scene-box accumulators and grid-barrier words in their rest state
int bihrt_build_launch_q(bihrt_ctx* c);
int bihrt_refit_launch(bihrt_ctx* c);
// stack items per lane of a walk (trace.cu, closest.cu)
#define STACK_DEPTH_PARITY  32  // <= 31 items: one per Morton bit on a root-to-leaf path, plus one
#define STACK_DEPTH_QUALITY 96  // quality mode: 63 key bits + up to 29 position bits of tie-breaking
// trace.cu
struct TraceArgs {
    const BihHeader* hdr; const BihNode* nodes; const BihTri* tris;
    const bihrt_ray* rays; int64_t nrays;
    const uint32_t* perm;     // ray lists: trace ray perm[i] as the i-th item (results still go to the ray's own slot); NULL = in list order
    int any_hit; float tmax;  // ray lists: occlusion query -- some hit with 0 < t < tmax, not the closest one
    float* out_t; int32_t* out_slot; int32_t* out_prim;
    // camera mode
    bihrt_camera cam; int w, h, spp; uint64_t seed; uint32_t flags; int shard_index, shard_count;
    int s_begin, s_end;     // samples [s_begin, s_end) of every pixel are traced by this launch (of spp in total)
    int il_index, il_count; // camera modes, multi-GPU: this launch owns units il_index, il_index + il_count, ... of every tile
    int il_cshift;          // ... in runs of 2^il_cshift consecutive units (neighbouring pixels), dealt round-robin to the ranks
    const uint32_t* tile_order; // camera modes: tile processed m-th (a permutation of this launch's tiles; NULL = in order)
    uint32_t* tile_cost;        // camera modes: longest unit of every tile, in clock ticks >> 8 (NULL = not recorded)
    int gshift;             // the samples of a pixel are spread over 2^gshift consecutive lanes (camera modes)
    uint32_t* fb;
    unsigned long long* counters; uint32_t* work;
    uint32_t* status_map;   // mapped host word for device-detected errors (tree of the wrong kind for this kernel)
    int queues;             // > 1: one work queue per SM (tile t -> queue t % queues) with stealing
    // MODE 3 and 4 (bihrt_intersect): rays with intervals instead of `rays`, and the hit record's other outputs (NULL = not wanted);
    // any_hit = BIHRT_INTERSECT_ANY (tmax comes with every ray)
    const bihrt_ray_interval* rays_iv;
    float* out_u; float* out_v; float* out_ng;
    // camera modes, set by bihrt_trace_launch: tiles per row and 0xFFFFFFFF / tile_cols, so that a warp finds its unit's
    // tile row with a multiply-high (and one correction) instead of a divide
    uint32_t tile_cols, tile_cols_rcp;
};
int bihrt_trace_launch(bihrt_ctx* c, const TraceArgs& a, int mode /*0 rays,1 render fb,2 render hits,3 ray queries,4 two-sided ray queries*/, bool counted);
int bihrt_resolve_launch(bihrt_ctx* c, uint32_t* fb, int npix, int spp);
int bihrt_tile_order_launch(bihrt_ctx* c, uint32_t* cost, uint32_t* order, uint32_t ntiles, bool full_sort);
// closest.cu: bihrt_closest_point (outputs NULL = not wanted)
struct ClosestArgs {
    const BihHeader* hdr; const BihNode* nodes; const BihTri* tris;
    const bihrt_point_query* pts; int64_t n;
    float* out_d2; float* out_u; float* out_v; int32_t* out_slot; int32_t* out_prim; float* out_q; float* out_ng;
    uint32_t* work;         // persistent-kernel work counter
    uint32_t* status_map;   // mapped host word: tree of the wrong kind for this kernel
};
int bihrt_closest_launch(bihrt_ctx* c, const ClosestArgs& a);
// winding.cu: bihrt_winding_number.  Far-field table: per node slot, the order-2 expansion of each child about its box centre,
// WTAB_FLOATS floats per child (N[3], M[3][3] row-major, Q[i][jk] for jk = 00 01 02 11 12 22, 2 unused).
#define WTAB_FLOATS 32
#define WTAB_SCRATCH_WORDS(n) (4 * (size_t)(n) + 16)   // queue, parent, leaf list, arrivals + counters
struct WindingArgs {
    const BihHeader* hdr; const BihNode* nodes; const BihTri* tris;
    const float* wtab;
    const bihrt_point_query* pts; int64_t n;
    float b2;               // fl(beta * beta); +inf: exact
    float* out_w;
    uint32_t* work;         // persistent-kernel work counter
    uint32_t* status_map;   // mapped host word: tree of the wrong kind for this kernel
};
int bihrt_winding_table_launch(bihrt_ctx* c);      // fills c->d_wtab from the blob (c->d_wtab / d_wscratch sized for c->n)
int bihrt_winding_launch(bihrt_ctx* c, const WindingArgs& a);
// raysort.cu: permutation that groups a ray list by origin cell and direction octant (perm[i] = index of the i-th ray to trace)
int bihrt_ray_sort_launch(bihrt_ctx* c, const bihrt_ray* rays, int64_t n, const uint32_t** perm);
// shade.cu
int bihrt_secondary_launch(bihrt_ctx* c, const float* t, const int32_t* slot, int64_t n, uint32_t* tile_cnt, unsigned long long* total,
                           const bihrt_camera& cam, int w, int h, int spp, uint64_t seed, uint32_t flags, int kind, const float light[3],
                           bihrt_ray* out_rays, int32_t* out_sample);

// -------------------------------------------------------------------------------------------
// device helpers
// -------------------------------------------------------------------------------------------
#ifdef __CUDACC__
// order-preserving float <-> uint (sign-magnitude total order, -0 < +0): lets scene-box min/max be
// plain integer atomics (the reference's atomicMin/MaxFloat trick, R/src/CUDAKernels.cu:52-66)
__device__ __forceinline__ uint32_t enc_float(float f) {
    uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float dec_float(uint32_t u) {
    return __uint_as_float((u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u);
}

// counter-based jitter, bit-identical to oracle/bih_oracle.c:jitter01 (replaces curand XORWOW,
// R/src/CUDAKernels.cu:411-419,458)
__host__ __device__ __forceinline__ uint32_t bihrt_mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
__device__ __forceinline__ float bihrt_jitter(uint64_t seed, uint32_t pixel, uint32_t sample, uint32_t dim) {
    uint32_t h = bihrt_mix32((uint32_t)seed ^ bihrt_mix32(pixel + 0x9e3779b9u * (sample * 2u + dim + 1u)) ^ (uint32_t)(seed >> 32));
    return __fmul_rn((float)((h >> 8) + 1u), 1.0f / 16777216.0f);
}

__device__ __forceinline__ uint32_t ld_relaxed(const uint32_t* p) {
    uint32_t v; asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}
__device__ __forceinline__ void st_relaxed(uint32_t* p, uint32_t v) {
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
#endif
