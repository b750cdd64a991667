// BIH construction on sm_100a.  Replaces the first half of Renderer::Render
// (R/src/Renderer.cpp:422-503: thrust::transform(morton_functor), thrust::sequence,
// thrust::stable_sort_by_key, thrust::reduce_by_key, thrust::unique_by_key_copy, Launch_BuildTree,
// Launch_FindClipPlanes) and the host pre-pass of App::LoadModels (R/src/App.cpp:110-156).
//
// Pipeline (one stream, no host synchronisation, Nu never leaves the device):
//   k_init        reset histograms / counters / scene-box accumulators / look-back words
//   k_scene_box   scene AABB                                   36 B read per triangle
//   k_morton      AABB centre -> 30-bit Morton key, fused 4x256 digit histogram   36 R + 4 W
//   k_onesweep x4 stable LSD radix sort, 8-bit digits, decoupled look-back       16 R + 16 W per pass
//   k_rle_*       head flags per 256-slot block, scanned -> Nu and the leaf number at every block start      4 R
//   k_reorder     per slot: leaf heads -> unique codes + first slot of each leaf (the RLE write, fused);
//                 gather the triangle, write its 48-byte leaf-ordered record and its AABB as the
//                 bottom level of an implicit min/max heap of BOXES (32-byte entries, +8 levels per block)   4+36 R + 48+~35 W
//   k_heap_up     upper heap levels (8 per block, 8 more by the last block to finish: one launch up to 16 M triangles)
//   k_nodes       per node: Karras range/split search + two heap range queries = the boxes of its two children
//                 (the clip planes are two components of them); each 64-byte node written once       ~50 R + 64 W
// Results are bit-identical to the reference algorithm (oracle/bih_oracle.c): the radix tree over the
// unique sorted codes is unique, node ids follow the Karras numbering rule, clip planes are pure
// max/min of input floats.  Quality mode (63-bit keys, capped leaves; NOT a parity path) is at the end of the file.
#include "bihrt_internal.cuh"
#include <float.h>

#define FULL 0xffffffffu
#define ENC_AUX 12          // d_scenebox_enc words 0..11: the two alternating accumulators of k_front; 12..17: quality mode / refit

// ------------------------------------------------------------------------------------------
// small block-level helpers (256 threads)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t warp_incl_scan(uint32_t v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { uint32_t t = __shfl_up_sync(FULL, v, o); if (lane >= o) v += t; }
    return v;
}
// exclusive scan over blockDim.x == 256 threads; s_w needs 8 words; returns exclusive prefix, *total = block sum
__device__ __forceinline__ uint32_t block_excl_scan_256(uint32_t v, uint32_t* s_w, uint32_t* total) {
    int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t inc = warp_incl_scan(v, lane);
    if (lane == 31) s_w[w] = inc;
    __syncthreads();
    uint32_t base = 0, tot = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) { uint32_t x = s_w[i]; if (i < w) base += x; tot += x; }
    __syncthreads();
    *total = tot;
    return base + inc - v;
}

// The streaming kernels read the input 4 triangles ("quad": 36 floats = 9 x 16 B, 144 B, 16-byte aligned) per
// thread.  A warp loads its 32 quads (4608 contiguous bytes) with nine fully coalesced 128-bit loads and
// transposes them through a per-warp shared-memory buffer (lane-strided 128-bit global loads would touch 32
// different lines per instruction and run at half the DRAM rate).  `quad0` = first quad of the warp.
__device__ __forceinline__ void load_quads_warp(const float* __restrict__ tri, uint32_t quad0, uint32_t nq, float4* s_warp, int lane, float v[36]) {
    const float4* p = reinterpret_cast<const float4*>(tri) + (size_t)quad0 * 9;
    const uint32_t nvec = min(32u, nq - quad0) * 9u;                 // 16-byte vectors this warp owns
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 9; i++) {
        const uint32_t j = i * 32 + lane;
        if (j < nvec) s_warp[j] = __ldcs(p + j);
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 9; i++) {                                    // lane reads vectors 9*lane .. 9*lane+8 (odd stride: conflict-free)
        const float4 f = s_warp[9 * lane + i];
        v[4 * i] = f.x; v[4 * i + 1] = f.y; v[4 * i + 2] = f.z; v[4 * i + 3] = f.w;
    }
}

// k_morton is bound by its divisions and histogram atomics, not by the loads: plain per-thread 128-bit loads
__device__ __forceinline__ void load_quad(const float* __restrict__ tri, uint32_t q, float v[36]) {
    const float4* p = reinterpret_cast<const float4*>(tri) + (size_t)q * 9;
#pragma unroll
    for (int i = 0; i < 9; i++) {
        const float4 f = __ldcs(p + i);
        v[4 * i] = f.x; v[4 * i + 1] = f.y; v[4 * i + 2] = f.z; v[4 * i + 3] = f.w;
    }
}

// std::minmax({a,b,c}) of R/src/App.cpp:123-125: leftmost minimum, rightmost maximum under <.
__device__ __forceinline__ void minmax3(float a, float b, float c, float& mn, float& mx) {
    mn = a; mx = a;
    if (b < mn) mn = b;
    if (!(b < mx)) mx = b;
    if (c < mn) mn = c;
    if (!(c < mx)) mx = c;
}

// ------------------------------------------------------------------------------------------
// also clears the look-back words of the four sort passes (one launch instead of a kernel + a memset node)
__global__ void __launch_bounds__(256) k_init(uint32_t* hist, uint32_t* enc, BihHeader* hdr, uint32_t n, uint4* __restrict__ lookback, uint32_t lb_vec4, uint32_t status0, uint32_t quality) {
    for (uint32_t i = blockIdx.x * 256u + threadIdx.x; i < lb_vec4; i += gridDim.x * 256u) lookback[i] = make_uint4(0u, 0u, 0u, 0u);
    if (blockIdx.x != 0) return;
    for (int i = threadIdx.x; i < H_WORDS; i += blockDim.x) hist[i] = 0;
    if (threadIdx.x < 3) { enc[threadIdx.x] = 0xFFFFFFFFu; enc[3 + threadIdx.x] = 0u; }
    if (threadIdx.x == 0) { hdr->n = n; hdr->nu = 0; hdr->status = status0; hdr->root_axis = 0; hdr->quality = quality; }
}

// ------------------------------------------------------------------------------------------
// scene AABB (R/src/App.cpp:103-106,133-137).  Sign of a zero bound may differ from the host's
// std::minmax order dependence; it cannot change any Morton code or hit (DESIGN.md).
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_scene_box(const float* __restrict__ tri, uint32_t n, uint32_t* __restrict__ enc) {
    __shared__ float4 s_stage[8][288];
    float lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
    const uint32_t nq = n >> 2;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t q0 = blockIdx.x * 256u + (threadIdx.x & ~31u); q0 < nq; q0 += gridDim.x * 256u) {
        float v[36];
        load_quads_warp(tri, q0, nq, s_stage[warp], lane, v);
        if (q0 + lane < nq) {
#pragma unroll
            for (int i = 0; i < 36; i++) { lo[i % 3] = fminf(lo[i % 3], v[i]); hi[i % 3] = fmaxf(hi[i % 3], v[i]); }
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < 9u * (n & 3u)) {           // the last n % 4 triangles
        const float f = tri[(size_t)nq * 36 + threadIdx.x];
        const int k = threadIdx.x % 3;
        lo[k] = fminf(lo[k], f); hi[k] = fmaxf(hi[k], f);
    }
#pragma unroll
    for (int k = 0; k < 3; k++) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[k] = fminf(lo[k], __shfl_xor_sync(FULL, lo[k], o));
            hi[k] = fmaxf(hi[k], __shfl_xor_sync(FULL, hi[k], o));
        }
    }
    // block-level reduction first: 6 atomics per block instead of per warp (they all hit 6 words)
    __shared__ float s_red[8][6];
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 3; k++) { s_red[w][k] = lo[k]; s_red[w][3 + k] = hi[k]; }
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        float r = s_red[0][threadIdx.x];
        for (int i = 1; i < 8; i++) r = threadIdx.x < 3 ? fminf(r, s_red[i][threadIdx.x]) : fmaxf(r, s_red[i][threadIdx.x]);
        if (threadIdx.x < 3) atomicMin(&enc[threadIdx.x], enc_float(r)); else atomicMax(&enc[threadIdx.x], enc_float(r));
    }
}


// ------------------------------------------------------------------------------------------
// Morton keys (R/src/App.cpp:128-131,144-156 + R/src/Renderer.cpp:116-136) + digit histograms
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t expand_bits10(uint32_t v) {
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}
__device__ __forceinline__ float centre_of(float mn, float mx) {
    return __fmul_rn(__fadd_rn(mn, mx), 0.5f);            // == (mn + mx) / 2.0f exactly (scaling by a power of two)
}
__device__ __forceinline__ uint32_t morton_axis_c(float centre, float slo, float shi) {
    float nrm = __fdiv_rn(__fsub_rn(centre, slo), __fsub_rn(shi, slo));
    float q = fminf(fmaxf(__fmul_rn(nrm, 1024.0f), 0.0f), 1023.0f);   // fmaxf(NaN,0)=0: flat axis -> cell 0
    return expand_bits10(__float2uint_rz(q));
}
__device__ __forceinline__ uint32_t morton_axis(float mn, float mx, float slo, float shi) {
    return morton_axis_c(centre_of(mn, mx), slo, shi);
}

__device__ __forceinline__ uint32_t morton_of_tri(const float* t, const float slo[3], const float shi[3]) {
    float mn, mx;
    minmax3(t[0], t[3], t[6], mn, mx); const uint32_t xx = morton_axis(mn, mx, slo[0], shi[0]);
    minmax3(t[1], t[4], t[7], mn, mx); const uint32_t yy = morton_axis(mn, mx, slo[1], shi[1]);
    minmax3(t[2], t[5], t[8], mn, mx); const uint32_t zz = morton_axis(mn, mx, slo[2], shi[2]);
    return xx * 4 + yy * 2 + zz;
}

// histogram update: the two high digits are nearly uniform across a warp of neighbouring triangles (one
// match_any + one shared atomic per distinct value); the two low digits are spread, plain shared atomics
__device__ __forceinline__ void hist_add(uint32_t* s_hist, uint32_t code, uint32_t act, int lane) {
    atomicAdd(&s_hist[code & 255u], 1u);
    atomicAdd(&s_hist[256 + ((code >> 8) & 255u)], 1u);
#pragma unroll
    for (int p = 2; p < 4; p++) {
        const uint32_t d = (code >> (8 * p)) & 255u;
        const uint32_t peers = __match_any_sync(act, d);
        if (lane == __ffs(peers) - 1) atomicAdd(&s_hist[p * 256 + d], __popc(peers));
    }
}

__global__ void __launch_bounds__(256) k_morton(const float* __restrict__ tri, uint32_t n, const uint32_t* __restrict__ enc,
                                                uint32_t* __restrict__ keys, uint32_t* __restrict__ hist, BihHeader* hdr) {
    __shared__ uint32_t s_hist[4 * 256];
    for (int i = threadIdx.x; i < 1024; i += 256) s_hist[i] = 0;
    float slo[3], shi[3];
#pragma unroll
    for (int k = 0; k < 3; k++) { slo[k] = dec_float(enc[k]); shi[k] = dec_float(enc[3 + k]); }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < 3; k++) { hdr->lo[k] = slo[k]; hdr->hi[k] = shi[k]; }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const uint32_t nq = n >> 2;
    // warp-uniform trip count so the match_any masks are well defined
    for (uint32_t q0 = blockIdx.x * 256u + (threadIdx.x & ~31u); q0 < nq; q0 += gridDim.x * 256u) {
        const uint32_t q = q0 + lane;
        const bool valid = q < nq;
        const uint32_t act = __ballot_sync(FULL, valid);
        if (valid) {
            float v[36];
            load_quad(tri, q, v);
            uint4 c;
            c.x = morton_of_tri(v, slo, shi); c.y = morton_of_tri(v + 9, slo, shi);
            c.z = morton_of_tri(v + 18, slo, shi); c.w = morton_of_tri(v + 27, slo, shi);
            *reinterpret_cast<uint4*>(keys + (size_t)q * 4) = c;
            hist_add(s_hist, c.x, act, lane); hist_add(s_hist, c.y, act, lane);
            hist_add(s_hist, c.z, act, lane); hist_add(s_hist, c.w, act, lane);
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < 32) {                      // the last n % 4 triangles
        const bool valid = (uint32_t)lane < (n & 3u);
        const uint32_t act = __ballot_sync(FULL, valid);
        if (valid) {
            float t[9];
#pragma unroll
            for (int i = 0; i < 9; i++) t[i] = tri[((size_t)nq * 4 + lane) * 9 + i];
            const uint32_t code = morton_of_tri(t, slo, shi);
            keys[(size_t)nq * 4 + lane] = code;
            hist_add(s_hist, code, act, lane);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 1024; i += 256) { uint32_t v = s_hist[i]; if (v) atomicAdd(&hist[H_HIST + i], v); }
}

// ------------------------------------------------------------------------------------------
// k_front = k_init + k_scene_box + k_morton in ONE cooperative launch (the parity path; the quality mode and the refit keep
// the three kernels).  All CTAs are co-resident, so a grid barrier can stand where the kernel boundary was:
//   phase 0  clear the digit histograms, tile counters and look-back words of this build, reset the OTHER scene-box accumulator
//            (two accumulators alternate between builds: nothing has to be cleared before the first atomic of this one)
//   phase 1  scene box; with KEEP the centre of every triangle's AABB stays in shared memory
//   -------  grid barrier
//   phase 2  Morton keys + digit histograms, from the kept centres (the input is read ONCE, 36 B per triangle) or, for scenes
//            whose centres do not fit (n > ~1.8 M), from a second read of the input
// At 1 M triangles: 4 + 11 + 14 us of three launches -> one launch.
// ------------------------------------------------------------------------------------------
#define H_BAR    3000      // d_hist words [H_BAR] = arrivals, [H_BAR + 1] = generation of the grid barrier (self-resetting)
#define H_EPOCH  3002      // builds started on this context: selects the scene-box accumulator enc[(epoch & 1) * 6 ..]
#define FRONT_THREADS 256
#define FRONT_STAGE_BYTES (8 * 288 * 16)              // load_quads_warp staging, one 4608-byte buffer per warp
#define FRONT_KEEP_BYTES_PER_ITER (FRONT_THREADS * 48) // 4 triangles x 3 centre floats per thread and iteration
#define FRONT_MAX_KEEP_ITERS 6

__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
    uint32_t v; asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v;
}
// Barrier over all CTAs of a cooperative launch.  bar[0] counts arrivals and is back at 0 when the barrier opens, bar[1] is the
// generation the waiting CTAs spin on, so the words never need a reset between launches.
__device__ __forceinline__ void grid_barrier(uint32_t* bar, uint32_t G) {
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t gen = ld_relaxed(bar + 1);
        uint32_t old;
        asm volatile("atom.add.release.gpu.global.u32 %0, [%1], 1;" : "=r"(old) : "l"(bar) : "memory");
        if (old == G - 1) {
            st_relaxed(bar, 0u);
            asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(bar + 1), "r"(gen + 1u) : "memory");
        } else {
            while (ld_acquire_u32(bar + 1) == gen) { }
        }
    }
    __syncthreads();
}

template <bool KEEP>
__global__ void __launch_bounds__(FRONT_THREADS, KEEP ? 2 : 3) k_front(const float* __restrict__ tri, uint32_t n, uint32_t* __restrict__ enc2,
                                                            uint32_t* __restrict__ keys, uint32_t* __restrict__ hist, BihHeader* hdr,
                                                            uint4* __restrict__ lookback, uint32_t lb_vec4, uint32_t status0) {
    extern __shared__ float4 s_dyn[];
    float4 (*s_stage)[288] = reinterpret_cast<float4 (*)[288]>(s_dyn);
    float* s_centre = reinterpret_cast<float*>(s_dyn) + FRONT_STAGE_BYTES / 4;      // [iter][12][FRONT_THREADS]
    __shared__ uint32_t s_hist[4 * 256];
    __shared__ float s_red[8][6];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t G = gridDim.x;
    const uint32_t epoch = ld_relaxed(hist + H_EPOCH);          // read before this CTA arrives at the barrier; bumped after it
    uint32_t* enc = enc2 + (epoch & 1u) * 6u;
    // ---- phase 0
    for (uint32_t i = blockIdx.x * FRONT_THREADS + tid; i < lb_vec4; i += G * FRONT_THREADS) lookback[i] = make_uint4(0u, 0u, 0u, 0u);
    for (int i = tid; i < 1024; i += FRONT_THREADS) s_hist[i] = 0;
    if (blockIdx.x == 0) {
        for (int i = tid; i < H_WORDS; i += FRONT_THREADS) hist[i] = 0;
        uint32_t* other = enc2 + ((epoch & 1u) ^ 1u) * 6u;
        if (tid < 3) { other[tid] = 0xFFFFFFFFu; other[3 + tid] = 0u; }
        if (tid == 0) { hdr->n = n; hdr->nu = 0; hdr->status = status0; hdr->root_axis = 0; hdr->quality = 0u; }
    }
    // ---- phase 1: scene AABB (R/src/App.cpp:103-106,133-137) and, with KEEP, the centre of every triangle's AABB (:128-131)
    float lo[3] = { INFINITY, INFINITY, INFINITY }, hi[3] = { -INFINITY, -INFINITY, -INFINITY };
    const uint32_t nq = n >> 2;
    {
        int it = 0;
        for (uint32_t q0 = blockIdx.x * FRONT_THREADS + (tid & ~31u); q0 < nq; q0 += G * FRONT_THREADS, it++) {
            float v[36];
            load_quads_warp(tri, q0, nq, s_stage[warp], lane, v);
            if (q0 + lane < nq) {
#pragma unroll
                for (int t = 0; t < 4; t++) {
#pragma unroll
                    for (int k = 0; k < 3; k++) {
                        float mn, mx;
                        minmax3(v[9 * t + k], v[9 * t + 3 + k], v[9 * t + 6 + k], mn, mx);
                        lo[k] = fminf(lo[k], mn); hi[k] = fmaxf(hi[k], mx);
                        if (KEEP) s_centre[(it * 12 + t * 3 + k) * FRONT_THREADS + tid] = centre_of(mn, mx);
                    }
                }
            }
        }
    }
    if (blockIdx.x == 0 && tid < 9u * (n & 3u)) {                  // the last n % 4 triangles
        const float f = tri[(size_t)nq * 36 + tid];
        const int k = tid % 3;
        lo[k] = fminf(lo[k], f); hi[k] = fmaxf(hi[k], f);
    }
#pragma unroll
    for (int k = 0; k < 3; k++) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[k] = fminf(lo[k], __shfl_xor_sync(FULL, lo[k], o));
            hi[k] = fmaxf(hi[k], __shfl_xor_sync(FULL, hi[k], o));
        }
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 3; k++) { s_red[warp][k] = lo[k]; s_red[warp][3 + k] = hi[k]; }
    }
    __syncthreads();
    if (tid < 6) {
        float r = s_red[0][tid];
        for (int i = 1; i < 8; i++) r = tid < 3 ? fminf(r, s_red[i][tid]) : fmaxf(r, s_red[i][tid]);
        if (tid < 3) atomicMin(&enc[tid], enc_float(r)); else atomicMax(&enc[tid], enc_float(r));
    }
    grid_barrier(hist + H_BAR, G);
    // ---- phase 2: Morton keys (R/src/App.cpp:144-156 + R/src/Renderer.cpp:116-136) + the digit histograms of the four sort passes
    float slo[3], shi[3];
#pragma unroll
    for (int k = 0; k < 3; k++) { slo[k] = dec_float(__ldcg(enc + k)); shi[k] = dec_float(__ldcg(enc + 3 + k)); }
    if (blockIdx.x == 0 && tid == 0) {
#pragma unroll
        for (int k = 0; k < 3; k++) { hdr->lo[k] = slo[k]; hdr->hi[k] = shi[k]; }
        st_relaxed(hist + H_EPOCH, epoch + 1u);
    }
    {
        int it = 0;
        for (uint32_t q0 = blockIdx.x * FRONT_THREADS + (tid & ~31u); q0 < nq; q0 += G * FRONT_THREADS, it++) {
            const uint32_t q = q0 + lane;
            const bool valid = q < nq;
            const uint32_t act = __ballot_sync(FULL, valid);
            if (valid) {
                uint32_t code[4];
                if (KEEP) {
#pragma unroll
                    for (int t = 0; t < 4; t++) {
                        const uint32_t xx = morton_axis_c(s_centre[(it * 12 + t * 3 + 0) * FRONT_THREADS + tid], slo[0], shi[0]);
                        const uint32_t yy = morton_axis_c(s_centre[(it * 12 + t * 3 + 1) * FRONT_THREADS + tid], slo[1], shi[1]);
                        const uint32_t zz = morton_axis_c(s_centre[(it * 12 + t * 3 + 2) * FRONT_THREADS + tid], slo[2], shi[2]);
                        code[t] = xx * 4 + yy * 2 + zz;
                    }
                } else {
                    float v[36];
                    load_quad(tri, q, v);
#pragma unroll
                    for (int t = 0; t < 4; t++) code[t] = morton_of_tri(v + 9 * t, slo, shi);
                }
                *reinterpret_cast<uint4*>(keys + (size_t)q * 4) = make_uint4(code[0], code[1], code[2], code[3]);
#pragma unroll
                for (int t = 0; t < 4; t++) hist_add(s_hist, code[t], act, lane);
            }
        }
    }
    if (blockIdx.x == 0 && tid < 32) {                               // the last n % 4 triangles
        const bool valid = (uint32_t)lane < (n & 3u);
        const uint32_t act = __ballot_sync(FULL, valid);
        if (valid) {
            float t[9];
#pragma unroll
            for (int i = 0; i < 9; i++) t[i] = tri[((size_t)nq * 4 + lane) * 9 + i];
            const uint32_t code = morton_of_tri(t, slo, shi);
            keys[(size_t)nq * 4 + lane] = code;
            hist_add(s_hist, code, act, lane);
        }
    }
    __syncthreads();
    for (int i = tid; i < 1024; i += FRONT_THREADS) { uint32_t v = s_hist[i]; if (v) atomicAdd(&hist[H_HIST + i], v); }
}

// scene-box accumulators and the grid-barrier words in their rest state (once per context)
int bihrt_build_setup(bihrt_ctx* c) {
    const uint32_t enc_init[18] = { 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u, 0u, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u, 0u,
                                    0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0u, 0u, 0u };
    BIHRT_CUDA(c, cudaMemcpy(c->d_scenebox_enc, enc_init, sizeof enc_init, cudaMemcpyHostToDevice));
    BIHRT_CUDA(c, cudaMemset(c->d_hist, 0, 4096 * sizeof(uint32_t)));
    BIHRT_CUDA(c, cudaFuncSetAttribute(k_front<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, FRONT_STAGE_BYTES + FRONT_MAX_KEEP_ITERS * FRONT_KEEP_BYTES_PER_ITER));
    BIHRT_CUDA(c, cudaFuncSetAttribute(k_front<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, FRONT_STAGE_BYTES));
    return BIHRT_OK;
}

static int front_launch(bihrt_ctx* c, uint32_t n, uint4* lookback, uint32_t lb_vec4) {
    const uint32_t nq = n >> 2;
    uint32_t G = max(1u, min((uint32_t)(c->sm_count * 2), (nq + FRONT_THREADS - 1) / FRONT_THREADS));
    const uint32_t iters = (nq + G * FRONT_THREADS - 1) / (G * FRONT_THREADS);
    const bool keep = iters <= FRONT_MAX_KEEP_ITERS;
    if (!keep) G = (uint32_t)(c->sm_count * 3);       // streaming variant: three resident blocks per SM (36 KB of staging each)
    const size_t smem = FRONT_STAGE_BYTES + (keep ? (size_t)max(1u, iters) * FRONT_KEEP_BYTES_PER_ITER : 0);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(G); cfg.blockDim = dim3(FRONT_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = c->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative; attr[0].val.cooperative = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    const float* tri = c->d_tri_in; uint32_t* enc = c->d_scenebox_enc; uint32_t* keys = c->d_keys[0]; uint32_t* hist = c->d_hist; BihHeader* hdr = c->d_hdr;
    const uint32_t status0 = (uint32_t)c->opt_debug_trip_watchdog;
    if (keep) BIHRT_CUDA(c, cudaLaunchKernelEx(&cfg, k_front<true>, tri, n, enc, keys, hist, hdr, lookback, lb_vec4, status0));
    else      BIHRT_CUDA(c, cudaLaunchKernelEx(&cfg, k_front<false>, tri, n, enc, keys, hist, hdr, lookback, lb_vec4, status0));
    return BIHRT_OK;
}

// ------------------------------------------------------------------------------------------
// One pass of a stable least-significant-digit radix sort, 8-bit digit, single sweep over the data
// with chained-scan decoupled look-back across tiles (replaces thrust::sequence +
// thrust::stable_sort_by_key, R/src/Renderer.cpp:436-445).  Stability: a tile is ranked in index
// order (warp-striped items, per-warp match-any ranking), tiles are ordered by the look-back chain.
// ------------------------------------------------------------------------------------------
#ifndef OS_BALLOT
#define OS_BALLOT 1
#endif
#define OS_THREADS 256
#define OS_ITEMS   16
#define OS_TILE    (OS_THREADS * OS_ITEMS)      // 4096 keys (32-bit keys; the 64-bit keys of the quality mode use 8 items = 2048 keys)
#define OS_ITEMS64 8
#define OS_TILE64  (OS_THREADS * OS_ITEMS64)
#define LB_FLAG_AGG   0x40000000u
#define LB_FLAG_INCL  0x80000000u
#define LB_MASK       0x3FFFFFFFu
#define SPIN_LIMIT    (1u << 22)

// 4 resident blocks per SM for the 32-bit keys (64 registers, no spills; the compiler's own choice was 80 -> 3 blocks):
// 10 M keys 90 -> 84 us per pass, 1 M unchanged; 5 blocks (48 registers) spill and gain nothing
template <typename K, int ITEMS, bool FIRST, int LB_BATCH>
__global__ void __launch_bounds__(OS_THREADS, sizeof(K) == 4 ? 4 : 3) k_onesweep(const K* __restrict__ keys_in, const uint32_t* __restrict__ vals_in,
                                                         K* __restrict__ keys_out, uint32_t* __restrict__ vals_out,
                                                         uint32_t n, int pass, uint32_t* __restrict__ hist,
                                                         uint32_t* __restrict__ lookback, BihHeader* hdr) {
    constexpr int OS_ITEMS_ = ITEMS;
    constexpr uint32_t OS_TILE_ = OS_THREADS * ITEMS;
    __shared__ uint32_t s_whist[8][256];
    __shared__ K s_keys[OS_TILE_];
    __shared__ uint32_t s_vals[OS_TILE_];
    __shared__ uint32_t s_binstart[256];
    __shared__ uint32_t s_goff[256];
    __shared__ uint32_t s_w[8];
    __shared__ uint32_t s_tile;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int shift = pass * 8;
    if (tid == 0) s_tile = atomicAdd(&hist[H_TILECTR + pass], 1u);
    for (int i = tid; i < 8 * 256; i += OS_THREADS) (&s_whist[0][0])[i] = 0;
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint32_t tile_base = tile * OS_TILE_;
    const uint32_t valid = min((uint32_t)OS_TILE_, n - tile_base);

    // global base of each digit for this pass = exclusive scan of the whole-array histogram
    uint32_t tot;
    uint32_t gbase = block_excl_scan_256(hist[H_HIST + pass * 256 + tid], s_w, &tot);

    K key[OS_ITEMS_]; uint32_t rank[OS_ITEMS_];
    const uint32_t i0 = tile_base + warp * (32 * OS_ITEMS_) + lane;
#pragma unroll
    for (int i = 0; i < OS_ITEMS_; i++) {
        uint32_t gi = i0 + i * 32;
        key[i] = gi < n ? __ldcs(keys_in + gi) : ~(K)0;
    }
    const uint32_t lt = (1u << lane) - 1u;
#pragma unroll
    for (int i = 0; i < OS_ITEMS_; i++) {
        uint32_t d = (uint32_t)(key[i] >> shift) & 255u;
#if OS_BALLOT
        uint32_t peers = FULL;
#pragma unroll
        for (int b = 0; b < 8; b++) {
            const uint32_t bit = (d >> b) & 1u;
            peers &= __ballot_sync(FULL, bit) ^ (bit - 1u);
        }
#else
        uint32_t peers = __match_any_sync(FULL, d);
#endif
        int leader = __ffs(peers) - 1;
        uint32_t old = 0;
        if (lane == leader) { old = s_whist[warp][d]; s_whist[warp][d] = old + __popc(peers); }
        old = __shfl_sync(FULL, old, leader);
        rank[i] = old + __popc(peers & lt);
        __syncwarp();
    }
    __syncthreads();

    // digit `tid`: exclusive scan over the 8 warps, then over digits
    uint32_t cnt = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) { uint32_t c = s_whist[w][tid]; s_whist[w][tid] = cnt; cnt += c; }
    uint32_t binstart = block_excl_scan_256(cnt, s_w, &tot);
    s_binstart[tid] = binstart;
    // padding keys (all ones, digit 255 in every pass; a valid 63-bit key has digit <= 127 in its last pass) sit at the very end of the tile: not counted
    uint32_t cnt_real = cnt - ((tid == 255) ? ((uint32_t)OS_TILE_ - valid) : 0u);

    // decoupled look-back: exclusive count of this digit over all previous tiles
    uint32_t excl = 0;
    uint32_t* lb = lookback + (size_t)tile * 256 + tid;
    if (tile == 0) {
        st_relaxed(lb, cnt_real | LB_FLAG_INCL);
    } else {
        st_relaxed(lb, cnt_real | LB_FLAG_AGG);
        // All tiles of a launch are resident at once and publish their aggregates at about the same time, so a look-back that
        // reads ONE predecessor per L2 round trip walks ~sqrt(2 * tile) trips (22 at 1 M keys, ~6 us of a 15 us pass).  Read
        // LB_BATCH predecessors per trip instead (independent loads) and consume them in order: ~sqrt(2 * tile / LB_BATCH) trips.
        // Measured (1 M keys, per pass): batch 1 / 8 / 16 / 32 = 20.4 / 18.8 / 19.7 / 20.4 us; with several waves of tiles (10 M
        // keys) the predecessors of a tile have finished long before it starts and the wider reads only cost: 90 / 94 / 107 us.
        // The host picks 8 for launches of at most one wave, else 1.
        int t = (int)tile - 1;
        uint32_t spins = 0;
        bool done = false;
        while (!done) {
            uint32_t v[LB_BATCH];
#pragma unroll
            for (int i = 0; i < LB_BATCH; i++) v[i] = (t - i >= 0) ? ld_relaxed(lb - 256 * (size_t)(tile - (uint32_t)(t - i))) : LB_FLAG_INCL;
#pragma unroll
            for (int i = 0; i < LB_BATCH; i++) {
                if (done) break;
                const uint32_t f = v[i] & ~LB_MASK;
                if (f == 0) break;                    // not published yet: read again from here
                excl += v[i] & LB_MASK;
                t--;
                if (f == LB_FLAG_INCL) done = true;
            }
            if (!done && ++spins > SPIN_LIMIT) { atomicOr(&hdr->status, 1u); break; }
        }
        st_relaxed(lb, (excl + cnt_real) | LB_FLAG_INCL);
    }
    s_goff[tid] = gbase + excl - binstart;
    __syncthreads();

    // tile-local reorder through shared memory so the global scatter is coalesced per digit
#pragma unroll
    for (int i = 0; i < OS_ITEMS_; i++) {
        uint32_t d = (uint32_t)(key[i] >> shift) & 255u;
        uint32_t pos = s_binstart[d] + s_whist[warp][d] + rank[i];
        s_keys[pos] = key[i];
        uint32_t gi = i0 + i * 32;
        uint32_t v;
        if (FIRST) v = gi;                                   // thrust::sequence fused: value = input index
        else v = gi < n ? __ldcs(vals_in + gi) : 0u;
        s_vals[pos] = v;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < OS_ITEMS_; k++) {
        uint32_t j = tid + k * OS_THREADS;
        if (j < valid) {
            K kk = s_keys[j];
            uint32_t dst = s_goff[(uint32_t)(kk >> shift) & 255u] + j;
            keys_out[dst] = kk;
            vals_out[dst] = s_vals[j];
        }
    }
}

// The same sort for other 32-bit key / value pairs (ray sorting, csrc/raysort.cu): `passes` 8-bit passes starting at bit 0,
// hist = digit histograms of keys[0] (layout above) with zeroed tile counters, lookback = passes x tiles x 256 zeroed words.
// The sorted pairs end in buffer passes & 1.
int bihrt_sort_pairs_launch(bihrt_ctx* c, uint32_t* keys[2], uint32_t* vals[2], uint32_t n, int passes, uint32_t* hist, uint32_t* lookback, BihHeader* hdr) {
    const uint32_t os_tiles = (n + OS_TILE - 1) / OS_TILE;
    const bool one_wave = os_tiles <= (uint32_t)c->sm_count * 3u;     // all tiles resident at once: batched look-back (see k_onesweep)
    int cur = 0;
    for (int pass = 0; pass < passes; pass++) {
        uint32_t* lb = lookback + (size_t)pass * os_tiles * 256;
        if (pass == 0 && one_wave)  k_onesweep<uint32_t, OS_ITEMS, true, 8><<<os_tiles, OS_THREADS, 0, c->stream>>>(keys[cur], nullptr, keys[cur ^ 1], vals[cur ^ 1], n, pass, hist, lb, hdr);
        else if (pass == 0)         k_onesweep<uint32_t, OS_ITEMS, true, 1><<<os_tiles, OS_THREADS, 0, c->stream>>>(keys[cur], nullptr, keys[cur ^ 1], vals[cur ^ 1], n, pass, hist, lb, hdr);
        else if (one_wave)          k_onesweep<uint32_t, OS_ITEMS, false, 8><<<os_tiles, OS_THREADS, 0, c->stream>>>(keys[cur], vals[cur], keys[cur ^ 1], vals[cur ^ 1], n, pass, hist, lb, hdr);
        else                        k_onesweep<uint32_t, OS_ITEMS, false, 1><<<os_tiles, OS_THREADS, 0, c->stream>>>(keys[cur], vals[cur], keys[cur ^ 1], vals[cur ^ 1], n, pass, hist, lb, hdr);
        cur ^= 1;
    }
    c->kernel_launches += passes;
    BIHRT_CUDA(c, cudaGetLastError());
    return BIHRT_OK;
}

// ------------------------------------------------------------------------------------------
// Run-length encoding of the sorted keys: unique codes, first slot of every leaf, Nu
// (replaces thrust::reduce_by_key + thrust::unique_by_key_copy, R/src/Renderer.cpp:450-472;
// duplicatesCnts[k] = first[k+1] - first[k]).  Reduce-then-scan: count heads per tile, scan the tile
// counts in one block, write.  (A chained look-back over thousands of 8 KB tiles serialises on L2 round
// trips; the second read of the keys comes from L2.)  Nu stays on the device.
// ------------------------------------------------------------------------------------------
#define RLE_ITEMS 8
#define RLE_TILE  (256 * RLE_ITEMS)

__device__ __forceinline__ uint32_t rle_heads(const uint32_t* __restrict__ keys, uint32_t n, uint32_t g0, uint32_t key[RLE_ITEMS], uint32_t& cnt) {
    if (g0 + RLE_ITEMS <= n) {
        const uint4 a = *reinterpret_cast<const uint4*>(keys + g0), b = *reinterpret_cast<const uint4*>(keys + g0 + 4);
        key[0] = a.x; key[1] = a.y; key[2] = a.z; key[3] = a.w; key[4] = b.x; key[5] = b.y; key[6] = b.z; key[7] = b.w;
    } else {
#pragma unroll
        for (int i = 0; i < RLE_ITEMS; i++) key[i] = (g0 + i < n) ? keys[g0 + i] : 0u;
    }
    uint32_t prev = (g0 > 0 && g0 < n) ? keys[g0 - 1] : 0u;
    uint32_t heads = 0;
    cnt = 0;
#pragma unroll
    for (int i = 0; i < RLE_ITEMS; i++) {
        const uint32_t gi = g0 + i;
        const bool h = (gi < n) && (gi == 0 || key[i] != prev);
        prev = key[i];
        heads |= (h ? 1u : 0u) << i;
        cnt += h;
    }
    return heads;
}

__global__ void __launch_bounds__(256) k_rle_count(const uint32_t* __restrict__ keys, uint32_t n, uint32_t* __restrict__ tile_cnt) {
    uint32_t key[RLE_ITEMS], cnt;
    rle_heads(keys, n, blockIdx.x * RLE_TILE + threadIdx.x * RLE_ITEMS, key, cnt);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(FULL, cnt, o);
    // a warp's 32 threads x 8 keys are 256 consecutive slots = one block of k_reorder, which writes the leaves
    if ((threadIdx.x & 31) == 0) tile_cnt[blockIdx.x * 8u + (threadIdx.x >> 5)] = cnt;
}

// exclusive scan of the tile counts in place (one block), Nu and the sentinel first[Nu] = n
// (folding it into the last block of k_rle_count was measured: 13.3 -> 14.4 us at 1 M triangles, 38 -> 80 us at 10 M)
__global__ void __launch_bounds__(1024) k_rle_scan(uint32_t* __restrict__ tile_cnt, uint32_t ntiles, uint32_t n,
                                                   uint32_t* __restrict__ first, BihHeader* hdr) {
    __shared__ uint32_t s_w[32];
    __shared__ uint32_t s_carry;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < ntiles; base += 1024) {
        const uint32_t i = base + threadIdx.x;
        const uint32_t v = i < ntiles ? tile_cnt[i] : 0u;
        uint32_t inc = warp_incl_scan(v, lane);
        if (lane == 31) s_w[w] = inc;
        __syncthreads();
        if (w == 0) { uint32_t x = s_w[lane]; uint32_t xi = warp_incl_scan(x, lane); s_w[lane] = xi - x; }
        __syncthreads();
        const uint32_t excl = s_carry + s_w[w] + inc - v;
        if (i < ntiles) tile_cnt[i] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) s_carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) { const uint32_t nu = s_carry; hdr->nu = nu; first[nu] = n; }
}

#define H_HEAPCTR 3005     // d_hist word: blocks of k_heap_up that have finished (back at 0 when the kernel ends)
// ------------------------------------------------------------------------------------------
// Leaves, tree and clip planes without any inter-thread dependency:
//   k_reorder     thread per sorted slot: the triangle's AABB becomes the bottom level of six implicit binary
//                 heaps (max-heaps of hi.xyz, min-heaps of lo.xyz over the triangles in sorted order); each
//                 block also reduces its 256 slots through 8 heap levels.  A leaf (unique Morton cell) is
//                 the slot range [first[k], first[k+1]), so FindClipPlanes' per-leaf union loop
//                 (R/src/CUDAKernels.cu:511-529) is part of the range query below.
//   k_heap_up     the remaining heap levels, 8 per launch.
//   k_nodes       thread per internal node i: range [a,b] and split by the same neighbour-prefix
//                 searches as the reference's BuildTree (R/src/CUDAKernels.cu:591-710) -- so node i is
//                 TreeInternalNode i by construction -- then the two clip planes as RANGE QUERIES on the
//                 heaps: clip0 = max hi[axis] over the slots of leaves [a, split], clip1 = min lo[axis] over
//                 those of [split+1, b].  max/min of the same input floats as the reference's float atomics
//                 (:52-66,532-547), hence bit-identical, but O(log range) independent loads per node
//                 instead of O(depth) atomics per leaf that all meet at the root, and no chain of
//                 fences/atomics between threads (a bottom-up climb serialises on ~depth L2 round trips).
// ------------------------------------------------------------------------------------------
struct Box { float lo[3], hi[3]; };

// Heap entry e (1 = root; the per-slot triangle boxes sit at [P, 2P)) = two float4 at heaps[2e], heaps[2e+1]:
// (lo.x, lo.y, lo.z, -) and (hi.x, hi.y, hi.z, -): the six extrema of one subtree of slots in ONE 32-byte sector, so a
// range query fetches a whole box per step.  Entries whose subtree holds no slot below n are never read by a range
// query inside [0, n) and are left unwritten.
__device__ __forceinline__ void heap_store(float4* __restrict__ heaps, uint32_t e, const float r[6]) {
    heaps[2 * (size_t)e] = make_float4(r[3], r[4], r[5], 0.f);        // lo
    heaps[2 * (size_t)e + 1] = make_float4(r[0], r[1], r[2], 0.f);    // hi
}

// One block reduces 256 consecutive elements of the level that starts at heap index `in_base` through up to 8 further
// levels: r[] holds this thread's element on entry (3 maxima, 3 minima).  Five levels inside each warp with shuffles,
// three more over the 8 warp results: two block barriers instead of sixteen.
__device__ __forceinline__ void heap_reduce_block(float r[6], float (*s)[8], float4* __restrict__ heaps, uint32_t P, uint32_t in_base, uint32_t blk) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t level_base = in_base;
#pragma unroll
    for (int l = 1; l <= 5; l++) {
        level_base >>= 1;
        if (level_base == 0) return;                              // above the root (warp-uniform)
#pragma unroll
        for (int c = 0; c < 6; c++) {
            const float y = __shfl_xor_sync(FULL, r[c], 1 << (l - 1));
            r[c] = c < 3 ? fmaxf(r[c], y) : fminf(r[c], y);
        }
        const uint32_t i = (blk * 256u + threadIdx.x) >> l;    // element of this level
        if ((lane & ((1 << l) - 1)) == 0 && i < level_base) heap_store(heaps, level_base + i, r);
    }
    if (lane == 0) {
#pragma unroll
        for (int c = 0; c < 6; c++) s[c][w] = r[c];
    }
    __syncthreads();
    if (w == 0) {
#pragma unroll
        for (int c = 0; c < 6; c++) r[c] = lane < 8 ? s[c][lane] : (c < 3 ? -INFINITY : INFINITY);
#pragma unroll
        for (int l = 6; l <= 8; l++) {
            level_base >>= 1;
            if (level_base == 0) return;
#pragma unroll
            for (int c = 0; c < 6; c++) {
                const float y = __shfl_xor_sync(FULL, r[c], 1 << (l - 6));
                r[c] = c < 3 ? fmaxf(r[c], y) : fminf(r[c], y);
            }
            const uint32_t i = (blk * 8u + lane) >> (l - 5);
            if (lane < 8 && (lane & ((1 << (l - 5)) - 1)) == 0 && i < level_base) heap_store(heaps, level_base + i, r);
        }
    }
}

// Leaf-ordered triangle records + bottom heap levels: one thread per sorted slot gathers its input triangle
// (36 B), writes the 48-byte record (coalesced) and the triangle's AABB (std::minmax semantics of
// R/src/App.cpp:123-127) as heap level 0.  end-of-leaf = the next slot has a different Morton code.
template <bool RLE, bool QUALITY>
__global__ void __launch_bounds__(256) k_reorder(const float* __restrict__ tri_in, const uint32_t* __restrict__ idx_sorted,
                                                 const uint32_t* __restrict__ keys_sorted, uint32_t n, BihTri* __restrict__ tris,
                                                 float4* __restrict__ heaps, uint32_t P, const uint32_t* __restrict__ tile_off,
                                                 uint32_t* __restrict__ umc, uint32_t* __restrict__ first) {
    __shared__ float s[6][8];
    __shared__ uint32_t s_w[8];
    const uint32_t j = blockIdx.x * 256u + threadIdx.x;
    float mn[3] = { INFINITY, INFINITY, INFINITY }, mx[3] = { -INFINITY, -INFINITY, -INFINITY };
    uint32_t key = 0, head = 0;
    if (j < n) {
        const uint32_t p = idx_sorted[j];
        const float* t = tri_in + (size_t)p * 9;
        float v[9];
#pragma unroll
        for (int i = 0; i < 9; i++) v[i] = __ldg(t + i);
        uint32_t last = 0;                                   // quality mode: leaves are marked by k_nodes_q
        if (!QUALITY) {
            key = keys_sorted[j];
            last = (j + 1 == n || keys_sorted[j + 1] != key) ? 1u : 0u;
        }
        if (RLE) head = (j == 0 || keys_sorted[j - 1] != key) ? 1u : 0u;
        float4* dst = reinterpret_cast<float4*>(tris + j);
        __stcs(dst, make_float4(v[0], v[1], v[2], __fsub_rn(v[3], v[0])));
        __stcs(dst + 1, make_float4(__fsub_rn(v[4], v[1]), __fsub_rn(v[5], v[2]), __fsub_rn(v[6], v[0]), __fsub_rn(v[7], v[1])));
        __stcs(dst + 2, make_float4(__fsub_rn(v[8], v[2]), __uint_as_float(p), __uint_as_float(last), __uint_as_float(j)));
        minmax3(v[0], v[3], v[6], mn[0], mx[0]);
        minmax3(v[1], v[4], v[7], mn[1], mx[1]);
        minmax3(v[2], v[5], v[8], mn[2], mx[2]);
        const float r0[6] = { mx[0], mx[1], mx[2], mn[0], mn[1], mn[2] };
        heap_store(heaps, P + j, r0);
    }
    if (RLE) {
        // run-length encoding of the sorted keys (thrust::reduce_by_key + unique_by_key_copy, R/src/Renderer.cpp:450-472):
        // this slot starts leaf k = heads before it; k_rle_count / k_rle_scan supplied the heads before this block
        uint32_t total;
        const uint32_t k = tile_off[blockIdx.x] + block_excl_scan_256(head, s_w, &total);
        if (head) { umc[k] = key; first[k] = j; }
    }
    float r[6] = { mx[0], mx[1], mx[2], mn[0], mn[1], mn[2] };
    heap_reduce_block(r, s, heaps, P, P, blockIdx.x);
}

// 8 more levels above the level of `in_count` used elements that starts at heap index `in_base`; the last block to finish goes on
// with the <= 256 elements the launch produced (8 further levels: one launch covers 16 levels, i.e. everything above k_reorder's
// for up to 16 M triangles)
__global__ void __launch_bounds__(256) k_heap_up(float4* __restrict__ heaps, uint32_t P, uint32_t in_base, uint32_t in_count, uint32_t* __restrict__ done_ctr) {
    __shared__ float s[6][8];
    __shared__ uint32_t s_last;
    const uint32_t i = blockIdx.x * 256u + threadIdx.x;
    float r[6] = { -INFINITY, -INFINITY, -INFINITY, INFINITY, INFINITY, INFINITY };
    if (i < in_count) {
        const float4 lo = heaps[2 * (size_t)(in_base + i)], hi = heaps[2 * (size_t)(in_base + i) + 1];
        r[0] = hi.x; r[1] = hi.y; r[2] = hi.z; r[3] = lo.x; r[4] = lo.y; r[5] = lo.z;
    }
    heap_reduce_block(r, s, heaps, P, in_base, blockIdx.x);
    if (gridDim.x > 256 || (in_base >> 8) <= 1) return;          // the host launches the next step itself / nothing above
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(done_ctr, 1u) == gridDim.x - 1 ? 1u : 0u;
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    if (threadIdx.x == 0) *done_ctr = 0u;
    const uint32_t base2 = in_base >> 8;
#pragma unroll
    for (int c = 0; c < 3; c++) { r[c] = -INFINITY; r[3 + c] = INFINITY; }
    if (threadIdx.x < gridDim.x) {
        const float4 lo = __ldcg(heaps + 2 * (size_t)(base2 + threadIdx.x)), hi = __ldcg(heaps + 2 * (size_t)(base2 + threadIdx.x) + 1);
        r[0] = hi.x; r[1] = hi.y; r[2] = hi.z; r[3] = lo.x; r[4] = lo.y; r[5] = lo.z;
    }
    __syncthreads();
    heap_reduce_block(r, s, heaps, P, base2, 0u);
}

// The heap levels above the 8 that k_reorder builds, for n slots in heaps padded to P: returns the number of k_heap_up launches
static int heap_levels_launch(bihrt_ctx* c, uint32_t n, uint32_t P) {
    int launches = 0;
    for (uint32_t lvl = P >> 8, used = (n + 255) / 256; lvl > 1; lvl >>= 8, used = (used + 255) / 256) {   // level with `lvl` elements
        const uint32_t hb = (used + 255) / 256;
        k_heap_up<<<hb, 256, 0, c->stream>>>(c->d_heaps, P, lvl, used, c->d_hist + H_HEAPCTR);
        if (hb <= 256 && (lvl >> 8) > 1) { lvl >>= 8; used = hb; }       // its last block has done the next 8 levels as well
        launches++;
    }
    return launches;
}

// Boxes of the slot ranges [l0, r0) and [l1, r1) (heap indices at the bottom level), both walked in one loop so that up to
// eight independent 128-bit loads are in flight; box = lo.xyz, hi.xyz.
__device__ __forceinline__ void heap_merge(const float4* __restrict__ heaps, uint32_t e, float b[6]) {
    const float4 lo = __ldg(heaps + 2 * (size_t)e), hi = __ldg(heaps + 2 * (size_t)e + 1);
    b[0] = fminf(b[0], lo.x); b[1] = fminf(b[1], lo.y); b[2] = fminf(b[2], lo.z);
    b[3] = fmaxf(b[3], hi.x); b[4] = fmaxf(b[4], hi.y); b[5] = fmaxf(b[5], hi.z);
}
__device__ __forceinline__ void heap_range_boxes(const float4* __restrict__ heaps, uint32_t l0, uint32_t r0, uint32_t l1, uint32_t r1,
                                                 float bl[6], float br[6]) {
#pragma unroll
    for (int k = 0; k < 3; k++) { bl[k] = br[k] = INFINITY; bl[3 + k] = br[3 + k] = -INFINITY; }
    while (l0 < r0 || l1 < r1) {
        if (l0 < r0) { if (l0 & 1u) heap_merge(heaps, l0++, bl); if (r0 & 1u) heap_merge(heaps, --r0, bl); l0 >>= 1; r0 >>= 1; }
        if (l1 < r1) { if (l1 & 1u) heap_merge(heaps, l1++, br); if (r1 & 1u) heap_merge(heaps, --r1, br); l1 >>= 1; r1 >>= 1; }
    }
}
__device__ __forceinline__ void node_store(BihNode* __restrict__ nd, int axis, uint32_t ref_l, uint32_t ref_r, const float bl[6], const float br[6]) {
    float4* p = reinterpret_cast<float4*>(nd);
    // clip planes = the children's extents on the split axis: max of hi[axis] over the left subtree, min of lo[axis] over the
    // right one -- the same maxima / minima of the same input floats as the reference's float atomics (:52-66,532-547)
    const float c0 = axis == 0 ? bl[3] : (axis == 1 ? bl[4] : bl[5]), c1 = axis == 0 ? br[0] : (axis == 1 ? br[1] : br[2]);
    p[0] = make_float4(c0, c1, __uint_as_float(ref_l), __uint_as_float(ref_r));
    p[1] = make_float4(bl[0], bl[1], bl[2], bl[3]);
    p[2] = make_float4(bl[4], bl[5], br[0], br[1]);
    p[3] = make_float4(br[2], br[3], br[4], br[5]);
}

#ifndef NODES_BLOCK
#define NODES_BLOCK 128
#endif
#ifndef NODES_MINB
#define NODES_MINB 1
#endif
__global__ void __launch_bounds__(NODES_BLOCK, NODES_MINB) k_nodes(const uint32_t* __restrict__ umc, const uint32_t* __restrict__ first,
                                               BihHeader* hdr, const float4* __restrict__ heaps, uint32_t P,
                                               BihNode* __restrict__ nodes, uint32_t* __restrict__ status_map) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int nu = (int)hdr->nu;
    if (idx == 0) *status_map = hdr->status;      // last kernel of the build: the watchdog word, mirrored into mapped host memory
    if (idx > nu - 2) return;
    const uint32_t cur = __ldg(umc + idx);
    // common-prefix length with leaf j, -1 outside the array (R/src/CUDAKernels.cu:600-614,628-631)
    auto lcp = [&](int j) -> int { return (j < 0 || j > nu - 1) ? -1 : __clz(cur ^ __ldg(umc + j)); };
    const int d = lcp(idx + 1) > lcp(idx - 1) ? 1 : -1;          // :616 (never equal for distinct sorted keys)
    const int lcp_min = lcp(idx - d);                            // :620
    int l_max = 1;
    do { l_max *= 2; } while (lcp(idx + l_max * d) > lcp_min);   // :624-633
    int l = 0;
    for (int t = l_max / 2; t >= 1; t /= 2)                      // :638-650
        if (lcp(idx + (l + t) * d) > lcp_min) l += t;
    const int other_end = idx + l * d;                           // :651
    const int lcp_ends = lcp(other_end);                         // :652
    int s = 0;
    for (int t = l;;) {                                          // :658-675
        t = (t + 1) >> 1;
        if (lcp(idx + (s + t) * d) > lcp_ends) s += t;
        if (t == 1) break;
    }
    const int split = idx + s * d + min(d, 0);                   // :677
    const int a = min(idx, other_end), b = max(idx, other_end);
    const uint32_t ms = __ldg(umc + split), ms1 = __ldg(umc + split + 1);
    const int axis = (__clz(ms ^ ms1) + 1) % 3;                  // :702-706
    // a node over leaves [l,r] splits on the first bit in which umc[l] and umc[r] differ, so a child's axis
    // follows from its range ends; it is stored in the parent's reference (see bihrt_internal.cuh)
    const uint32_t ref_l = (a == split) ? BIH_REF_LEAFREF(__ldg(first + split))
                                        : BIH_REF_NODE(split, (__clz(__ldg(umc + a) ^ ms) + 1) % 3);
    const uint32_t ref_r = (split + 1 == b) ? BIH_REF_LEAFREF(__ldg(first + split + 1))
                                            : BIH_REF_NODE(split + 1, (__clz(ms1 ^ __ldg(umc + b)) + 1) % 3);
    // leaves [a, split] are slots [first[a], first[split+1]); leaves [split+1, b] are [first[split+1], first[b+1])
    const uint32_t sa = __ldg(first + a), sm = __ldg(first + split + 1), sb = __ldg(first + b + 1);
    float bl[6], br[6];
    heap_range_boxes(heaps, sa + P, sm + P, sm + P, sb + P, bl, br);
    node_store(nodes + idx, axis, ref_l, ref_r, bl, br);
    if (idx == 0) hdr->root_axis = (uint32_t)axis;
}

// ==========================================================================================
// QUALITY MODE (SURVEY.md 8(f) f4; NOT a parity path, reported separately).  The reference quantises the triangle
// centres to a 10-bit grid per axis (R/src/Renderer.cpp:116-136) and makes every occupied grid cell a leaf
// (R/src/CUDAKernels.cu:206-224): at 10 M triangles a ray tests 24 triangles and the leaves hold up to hundreds.  Here:
//   * 21 bits per axis -> 63-bit Morton keys, 8 x 8-bit passes of the same onesweep sort;
//   * ties broken by the sorted position (Karras 2012, section 4), so the radix tree is built over all n triangles;
//   * a subtree of at most `leaf_cap` triangles becomes ONE leaf (a contiguous slot range, as in the parity layout);
//   * clip planes by the same heap range queries, so every plane bounds its subtree and the traversal kernel is the same.
// Node i is still the Karras node i; nodes inside a collapsed subtree are simply never written or referenced.
// ==========================================================================================
__device__ __forceinline__ uint64_t expand_bits21(uint32_t v) {
    uint64_t x = v & 0x1fffffu;
    x = (x | x << 32) & 0x001f00000000ffffull;
    x = (x | x << 16) & 0x001f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}
__device__ __forceinline__ uint64_t morton_axis21(float mn, float mx, float slo, float shi) {
    const float centre = __fmul_rn(__fadd_rn(mn, mx), 0.5f);
    const float nrm = __fdiv_rn(__fsub_rn(centre, slo), __fsub_rn(shi, slo));
    const float q = fminf(fmaxf(__fmul_rn(nrm, 2097152.0f), 0.0f), 2097151.0f);
    return expand_bits21(__float2uint_rz(q));
}
__device__ __forceinline__ uint64_t morton63_of_tri(const float* t, const float slo[3], const float shi[3]) {
    float mn, mx;
    minmax3(t[0], t[3], t[6], mn, mx); const uint64_t xx = morton_axis21(mn, mx, slo[0], shi[0]);
    minmax3(t[1], t[4], t[7], mn, mx); const uint64_t yy = morton_axis21(mn, mx, slo[1], shi[1]);
    minmax3(t[2], t[5], t[8], mn, mx); const uint64_t zz = morton_axis21(mn, mx, slo[2], shi[2]);
    return (xx << 2) | (yy << 1) | zz;
}

__global__ void __launch_bounds__(256) k_morton_q(const float* __restrict__ tri, uint32_t n, const uint32_t* __restrict__ enc,
                                                  uint64_t* __restrict__ keys, uint32_t* __restrict__ hist, BihHeader* hdr) {
    __shared__ uint32_t s_hist[8 * 256];
    for (int i = threadIdx.x; i < 2048; i += 256) s_hist[i] = 0;
    float slo[3], shi[3];
#pragma unroll
    for (int k = 0; k < 3; k++) { slo[k] = dec_float(enc[k]); shi[k] = dec_float(enc[3 + k]); }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
#pragma unroll
        for (int k = 0; k < 3; k++) { hdr->lo[k] = slo[k]; hdr->hi[k] = shi[k]; }
    }
    __syncthreads();
    for (uint32_t i = blockIdx.x * 256u + threadIdx.x; i < n; i += gridDim.x * 256u) {
        float t[9];
#pragma unroll
        for (int k = 0; k < 9; k++) t[k] = __ldcs(tri + (size_t)i * 9 + k);
        const uint64_t code = morton63_of_tri(t, slo, shi);
        keys[i] = code;
#pragma unroll
        for (int p = 0; p < 8; p++) atomicAdd(&s_hist[p * 256 + ((uint32_t)(code >> (8 * p)) & 255u)], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2048; i += 256) { const uint32_t v = s_hist[i]; if (v) atomicAdd(&hist[H_HIST + i], v); }
}

// length of the common prefix of the (key, position) pairs i and j: 64 key bits, then 32 position bits
__device__ __forceinline__ int delta_q(const uint64_t* __restrict__ keys, int n, uint64_t ki, int i, int j) {
    if (j < 0 || j > n - 1) return -1;
    const uint64_t x = ki ^ __ldg(keys + j);
    return x ? __clzll((long long)x) : 64 + __clz(i ^ j);
}
// split axis of the bit at prefix length p: key bit 62 (p = 1) is x's top bit; position bits keep cycling
__device__ __forceinline__ uint32_t axis_of_prefix(int p) { return (uint32_t)((p + 2) % 3); }

__global__ void __launch_bounds__(128) k_nodes_q(const uint64_t* __restrict__ keys, uint32_t n_, uint32_t cap, BihHeader* hdr,
                                                 const float4* __restrict__ heaps, uint32_t P, BihNode* __restrict__ nodes,
                                                 BihTri* __restrict__ tris, uint32_t* __restrict__ status_map) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = (int)n_;
    if (idx == 0) *status_map = hdr->status;
    if (n_ <= cap) {                                       // the whole scene is one leaf
        if (idx == 0) { hdr->nu = 1; hdr->root_axis = 0; tris[n - 1].last = 1u; }
        return;
    }
    uint32_t made = 0;                                     // leaves this thread creates
    if (idx <= n - 2) {
        const uint64_t cur = __ldg(keys + idx);
        auto lcp = [&](int j) -> int { return delta_q(keys, n, cur, idx, j); };
        const int d = lcp(idx + 1) > lcp(idx - 1) ? 1 : -1;
        const int lcp_min = lcp(idx - d);
        int l_max = 1;
        do { l_max *= 2; } while (lcp(idx + l_max * d) > lcp_min);
        int l = 0;
        for (int t = l_max / 2; t >= 1; t /= 2)
            if (lcp(idx + (l + t) * d) > lcp_min) l += t;
        const int other_end = idx + l * d;
        const int a = min(idx, other_end), b = max(idx, other_end);
        // nodes inside a collapsed subtree are never referenced: nothing to do (the root always has more than cap triangles)
        if ((uint32_t)(b - a + 1) > cap || idx == 0) {
            const int lcp_ends = lcp(other_end);
            int s = 0;
            for (int t = l;;) {
                t = (t + 1) >> 1;
                if (lcp(idx + (s + t) * d) > lcp_ends) s += t;
                if (t == 1) break;
            }
            const int split = idx + s * d + min(d, 0);
            const uint64_t ka = __ldg(keys + a), ks = __ldg(keys + split), ks1 = __ldg(keys + split + 1), kb = __ldg(keys + b);
            auto pre = [&](uint64_t x, uint64_t y, int i, int j) -> int { const uint64_t z = x ^ y; return z ? __clzll((long long)z) : 64 + __clz(i ^ j); };
            const uint32_t axis = axis_of_prefix(pre(ks, ks1, split, split + 1));
            const bool leaf_l = (uint32_t)(split - a + 1) <= cap, leaf_r = (uint32_t)(b - split) <= cap;
            const uint32_t ref_l = leaf_l ? BIH_REF_LEAFREF(a) : BIH_REF_NODE(split, axis_of_prefix(pre(ka, ks, a, split)));
            const uint32_t ref_r = leaf_r ? BIH_REF_LEAFREF(split + 1) : BIH_REF_NODE(split + 1, axis_of_prefix(pre(ks1, kb, split + 1, b)));
            if (leaf_l) { tris[split].last = 1u; made++; }
            if (leaf_r) { tris[b].last = 1u; made++; }
            float bl[6], br[6];
            heap_range_boxes(heaps, a + P, split + 1 + P, split + 1 + P, b + 1 + P, bl, br);
            node_store(nodes + idx, (int)axis, ref_l, ref_r, bl, br);
            if (idx == 0) hdr->root_axis = axis;
        }
    }
    made = __reduce_add_sync(FULL, made);
    if ((threadIdx.x & 31) == 0 && made) atomicAdd(&hdr->nu, made);      // leaves (k_init zeroed it)
}

int bihrt_build_launch_q(bihrt_ctx* c) {
    const uint32_t n = (uint32_t)c->n;
    cudaStream_t st = c->stream;
    const uint32_t os_tiles = (n + OS_TILE64 - 1) / OS_TILE64;
    const size_t lb_words = (size_t)8 * os_tiles * 256;
    if (lb_words > c->lookback_q_words || !c->d_keys64[0]) return bihrt_fail(c, BIHRT_ERR_INTERNAL, "quality-mode scratch not allocated");
    const uint32_t lb_vec4 = (uint32_t)((lb_words + 3) / 4);
    k_init<<<(int)max(1u, min((uint32_t)c->sm_count, (lb_vec4 + 1023u) / 1024u)), 256, 0, st>>>(c->d_hist, c->d_scenebox_enc + ENC_AUX, c->d_hdr, n,
                                                                                      reinterpret_cast<uint4*>(c->d_lookback_q), lb_vec4, (uint32_t)c->opt_debug_trip_watchdog, 1u);
    const int stream_grid = (int)max(1u, min((uint32_t)(c->sm_count * 3), ((n >> 2) + 255) / 256));
    k_scene_box<<<stream_grid, 256, 0, st>>>(c->d_tri_in, n, c->d_scenebox_enc + ENC_AUX);
    k_morton_q<<<(int)max(1u, min((uint32_t)(c->sm_count * 4), (n + 255) / 256)), 256, 0, st>>>(c->d_tri_in, n, c->d_scenebox_enc + ENC_AUX, c->d_keys64[0], c->d_hist, c->d_hdr);
    int cur = 0;
    for (int pass = 0; pass < 8; pass++) {
        uint32_t* lb = c->d_lookback_q + (size_t)pass * os_tiles * 256;
        if (pass == 0)
            k_onesweep<uint64_t, OS_ITEMS64, true, 1><<<os_tiles, OS_THREADS, 0, st>>>(c->d_keys64[cur], nullptr, c->d_keys64[cur ^ 1], c->d_vals[cur ^ 1], n, pass, c->d_hist, lb, c->d_hdr);
        else
            k_onesweep<uint64_t, OS_ITEMS64, false, 1><<<os_tiles, OS_THREADS, 0, st>>>(c->d_keys64[cur], c->d_vals[cur], c->d_keys64[cur ^ 1], c->d_vals[cur ^ 1], n, pass, c->d_hist, lb, c->d_hdr);
        cur ^= 1;
    }
    uint32_t P = 256;
    while (P < n) P <<= 1;
    k_reorder<false, true><<<(n + 255) / 256, 256, 0, st>>>(c->d_tri_in, c->d_vals[cur], nullptr, n, c->d_tris, c->d_heaps, P, nullptr, nullptr, nullptr);
    const int launches = heap_levels_launch(c, n, P);
    k_nodes_q<<<(n + 127) / 128, 128, 0, st>>>(c->d_keys64[cur], n, (uint32_t)c->opt_leaf_cap, c->d_hdr, c->d_heaps, P, c->d_nodes, c->d_tris, c->d_status_map);
    c->kernel_launches += 13 + launches;
    BIHRT_CUDA(c, cudaGetLastError());
    return BIHRT_OK;
}

// ------------------------------------------------------------------------------------------
int bihrt_build_launch(bihrt_ctx* c) {
    const uint32_t n = (uint32_t)c->n;
    cudaStream_t st = c->stream;
    const uint32_t os_tiles = (n + OS_TILE - 1) / OS_TILE;
    const uint32_t rle_tiles = (n + RLE_TILE - 1) / RLE_TILE;
    const uint32_t rle_blocks = rle_tiles * 8;                     // 256-slot blocks (k_reorder's), rounded up to whole RLE tiles
    const size_t lb_words = (size_t)4 * os_tiles * 256 + rle_blocks;
    if (lb_words > c->lookback_words) return bihrt_fail(c, BIHRT_ERR_INTERNAL, "look-back buffer too small");

    int pe = 0;
#define PROF_MARK() do { if (c->opt_profile && pe < BIHRT_PROF_EVENTS) cudaEventRecord(c->prof_ev[pe++], st); } while (0)
    PROF_MARK();
    const uint32_t lb_vec4 = (uint32_t)((lb_words + 3) / 4);        // the buffer is allocated with 16 spare words
    PROF_MARK();   // 1
    PROF_MARK();   // 2
    { int rc = front_launch(c, n, reinterpret_cast<uint4*>(c->d_lookback), lb_vec4); if (rc) return rc; }
    PROF_MARK();   // 3: after init + scene box + morton (one cooperative launch)
    int cur = 0;
    const bool one_wave = os_tiles <= (uint32_t)c->sm_count * 3u;     // all tiles resident at once: batched look-back (see k_onesweep)
    for (int pass = 0; pass < 4; pass++) {
        uint32_t* lb = c->d_lookback + (size_t)pass * os_tiles * 256;
        if (pass == 0 && one_wave)  k_onesweep<uint32_t, OS_ITEMS, true, 8><<<os_tiles, OS_THREADS, 0, st>>>(c->d_keys[cur], nullptr, c->d_keys[cur ^ 1], c->d_vals[cur ^ 1], n, pass, c->d_hist, lb, c->d_hdr);
        else if (pass == 0)         k_onesweep<uint32_t, OS_ITEMS, true, 1><<<os_tiles, OS_THREADS, 0, st>>>(c->d_keys[cur], nullptr, c->d_keys[cur ^ 1], c->d_vals[cur ^ 1], n, pass, c->d_hist, lb, c->d_hdr);
        else if (one_wave)          k_onesweep<uint32_t, OS_ITEMS, false, 8><<<os_tiles, OS_THREADS, 0, st>>>(c->d_keys[cur], c->d_vals[cur], c->d_keys[cur ^ 1], c->d_vals[cur ^ 1], n, pass, c->d_hist, lb, c->d_hdr);
        else                        k_onesweep<uint32_t, OS_ITEMS, false, 1><<<os_tiles, OS_THREADS, 0, st>>>(c->d_keys[cur], c->d_vals[cur], c->d_keys[cur ^ 1], c->d_vals[cur ^ 1], n, pass, c->d_hist, lb, c->d_hdr);
        cur ^= 1;
        PROF_MARK();   // 4..7: after each sort pass
    }
    // 4 passes: sorted data is back in buffer 0
    uint32_t* tile_cnt = c->d_lookback + (size_t)4 * os_tiles * 256;
    k_rle_count<<<rle_tiles, 256, 0, st>>>(c->d_keys[cur], n, tile_cnt);
    k_rle_scan<<<1, 1024, 0, st>>>(tile_cnt, rle_blocks, n, c->d_first, c->d_hdr);
    PROF_MARK();   // 8: after rle
    // heaps are padded to a power of two >= n (Nu <= n is only known on the device)
    uint32_t P = 256;
    while (P < n) P <<= 1;
    k_reorder<true, false><<<(n + 255) / 256, 256, 0, st>>>(c->d_tri_in, c->d_vals[cur], c->d_keys[cur], n, c->d_tris, c->d_heaps, P, tile_cnt, c->d_umc, c->d_first);
    PROF_MARK();   // 9: after reorder + slot boxes + leaves
    const int launches = heap_levels_launch(c, n, P);
    PROF_MARK();   // 10: after upper heap levels
    k_nodes<<<(n + NODES_BLOCK - 1) / NODES_BLOCK, NODES_BLOCK, 0, st>>>(c->d_umc, c->d_first, c->d_hdr, c->d_heaps, P, c->d_nodes, c->d_status_map);
    PROF_MARK();   // 11: after nodes
    PROF_MARK();   // 12: after reorder
    c->prof_count = pe;
    c->kernel_launches += 9 + launches;    // k_front, 4 x k_onesweep, k_rle_count, k_rle_scan, k_reorder, k_heap_up.., k_nodes
    BIHRT_CUDA(c, cudaGetLastError());
    return BIHRT_OK;
}

// ------------------------------------------------------------------------------------------
// Refit (SURVEY.md 8(f) f3, NOT a parity path): after bihrt_scene_update_vertices, keep the Morton order,
// the leaves and the tree topology of the last full build and recompute only what depends on vertex
// positions: scene box, leaf-ordered triangle records, AABB heaps, clip planes.  The result is a valid BIH
// (every plane still bounds its subtree) but not the tree the reference would build for the moved vertices;
// it is the cheap path for small deformations between full rebuilds (4 kernels instead of 12).
// ------------------------------------------------------------------------------------------
__global__ void k_refit_box(const uint32_t* __restrict__ enc, BihHeader* hdr) {
    if (threadIdx.x < 3) { hdr->lo[threadIdx.x] = dec_float(enc[threadIdx.x]); hdr->hi[threadIdx.x] = dec_float(enc[3 + threadIdx.x]); }
}
__global__ void k_refit_init(uint32_t* enc) {
    if (threadIdx.x < 3) { enc[threadIdx.x] = 0xFFFFFFFFu; enc[3 + threadIdx.x] = 0u; }
}

int bihrt_refit_launch(bihrt_ctx* c) {
    const uint32_t n = (uint32_t)c->n;
    cudaStream_t st = c->stream;
    uint32_t P = 256;
    while (P < n) P <<= 1;
    const int stream_grid = (int)max(1u, min((uint32_t)(c->sm_count * 3), ((n >> 2) + 255) / 256));
    k_refit_init<<<1, 32, 0, st>>>(c->d_scenebox_enc + ENC_AUX);
    k_scene_box<<<stream_grid, 256, 0, st>>>(c->d_tri_in, n, c->d_scenebox_enc + ENC_AUX);
    k_refit_box<<<1, 32, 0, st>>>(c->d_scenebox_enc + ENC_AUX, c->d_hdr);
    k_reorder<false, false><<<(n + 255) / 256, 256, 0, st>>>(c->d_tri_in, c->d_vals[0], c->d_keys[0], n, c->d_tris, c->d_heaps, P, nullptr, nullptr, nullptr);
    const int launches = heap_levels_launch(c, n, P);
    k_nodes<<<(n + NODES_BLOCK - 1) / NODES_BLOCK, NODES_BLOCK, 0, st>>>(c->d_umc, c->d_first, c->d_hdr, c->d_heaps, P, c->d_nodes, c->d_status_map);
    c->kernel_launches += 5 + launches;
    BIHRT_CUDA(c, cudaGetLastError());
    return BIHRT_OK;
}
