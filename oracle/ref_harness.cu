// ref_harness.cu -- runs the REFERENCE'S OWN kernels, unmodified, on this GPU.  TEST INFRASTRUCTURE ONLY.
//
// This translation unit #include's R/src/CUDAKernels.cu straight from the read-only reference tree
// (nothing is copied into this repository) and links R/src/Camera.cu + R/src/Ray.cu (-rdc=true, as the
// reference project does, R/BIH_Raytracer.vcxproj:681,720).  It launches the reference's
//   __global__ BuildTree        R/src/CUDAKernels.cu:591-710
//   __global__ FindClipPlanes   R/src/CUDAKernels.cu:497-549
//   __device__ TraverseTree     R/src/CUDAKernels.cu:227-368   (through a 10-line wrapper kernel)
// and restates only the five thrust calls of Renderer::Render (R/src/Renderer.cpp:422-472) and the
// sentinel initialisation of GPUArrayManager::AllocateBIHTree (R/src/GPUArrayManager.cpp:58-91), which
// live in translation units that need a GL context.  Built by `make -C oracle ref REF=<reference src dir>`
// into oracle/_ref/ (git-ignored); bench.py reports it as the "reference kernels on B200" baseline.
#define STR2(x) #x
#define STR(x) STR2(x)
#include STR(REF_SRC_DIR/CUDAKernels.cu)

#include <thrust/device_vector.h>
#include <thrust/execution_policy.h>
#include <thrust/iterator/constant_iterator.h>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/reduce.h>
#include <thrust/sequence.h>
#include <thrust/sort.h>
#include <thrust/transform.h>
#include <thrust/unique.h>
#include <limits>
#include <vector>

// Out-of-line members the included TU references but that live in GL-dependent files of the reference.
// (Renderer::Launch_* are defined in CUDAKernels.cu itself; they are never called here.)

namespace {

// 30-bit Morton code of a point in the unit cube: the published formula (T. Karras, "Thinking Parallel,
// Part III", 2012) that R/src/Renderer.cpp:116-136 also uses; written here, not copied.
struct morton_of_norm_centre {
    __device__ static unsigned spread(unsigned v) {
        v = (v * 0x00010001u) & 0xFF0000FFu; v = (v * 0x00000101u) & 0x0F00F00Fu;
        v = (v * 0x00000011u) & 0xC30C30C3u; v = (v * 0x00000005u) & 0x49249249u; return v;
    }
    __device__ uint32_t operator()(float3 c) const {
        float x = fminf(fmaxf(c.x * 1024.0f, 0.0f), 1023.0f), y = fminf(fmaxf(c.y * 1024.0f, 0.0f), 1023.0f),
              z = fminf(fmaxf(c.z * 1024.0f, 0.0f), 1023.0f);
        return spread((unsigned)x) * 4 + spread((unsigned)y) * 2 + spread((unsigned)z);
    }
};

struct Scene {
    int n = 0, nu = 0;
    thrust::device_vector<Triangle> tris;
    thrust::device_vector<float3> lo, hi, cnorm;
    thrust::device_vector<uint32_t> codes, idx, umc, cnt;
    thrust::device_vector<int> first, leafParents;
    thrust::device_vector<TreeInternalNode> nodes;
    float3 sceneLo, sceneHi;
    float last_build_ms = 0;
};

__global__ void ref_trace_kernel(const float* rays6, int nrays, TreeInternalNode* tree, int* firstIdxs, uint32_t* cnts,
                                 Triangle* tris, uint32_t* trisIdx, float3 lo, float3 hi, int nu, float* out_t, int* out_slot) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nrays) return;
    Ray r(glm::vec3(rays6[6 * i], rays6[6 * i + 1], rays6[6 * i + 2]), glm::vec3(rays6[6 * i + 3], rays6[6 * i + 4], rays6[6 * i + 5]));
    HitRecord rec;                      // Color(), R/src/CUDAKernels.cu:380-382
    rec.triangleIdx = -1;
    rec.t = FLT_MAX;
    if (nu >= 2) TraverseTree(r, tree, firstIdxs, cnts, tris, trisIdx, lo, hi, rec);
    out_t[i] = (float)rec.t;
    out_slot[i] = rec.triangleIdx;
}

}  // namespace

extern "C" {

__attribute__((visibility("default"))) void* refh_create() { return new Scene(); }
__attribute__((visibility("default"))) void refh_destroy(void* p) { delete (Scene*)p; }

// host arrays exactly as App::LoadModels uploads them (R/src/App.cpp:158-164)
__attribute__((visibility("default"))) int refh_load(void* p, const float* tri9, const float* lo3, const float* hi3, const float* cnorm3,
                                                      const float* scene_lo, const float* scene_hi, int n) {
    Scene& s = *(Scene*)p;
    s.n = n;
    std::vector<Triangle> ht(n);
    std::vector<float3> hl(n), hh(n), hc(n);
    for (int i = 0; i < n; i++) {
        ht[i].v0 = glm::vec3(tri9[9 * i], tri9[9 * i + 1], tri9[9 * i + 2]);
        ht[i].v1 = glm::vec3(tri9[9 * i + 3], tri9[9 * i + 4], tri9[9 * i + 5]);
        ht[i].v2 = glm::vec3(tri9[9 * i + 6], tri9[9 * i + 7], tri9[9 * i + 8]);
        hl[i] = make_float3(lo3[3 * i], lo3[3 * i + 1], lo3[3 * i + 2]);
        hh[i] = make_float3(hi3[3 * i], hi3[3 * i + 1], hi3[3 * i + 2]);
        hc[i] = make_float3(cnorm3[3 * i], cnorm3[3 * i + 1], cnorm3[3 * i + 2]);
    }
    s.tris = ht; s.lo = hl; s.hi = hh; s.cnorm = hc;
    s.sceneLo = make_float3(scene_lo[0], scene_lo[1], scene_lo[2]);
    s.sceneHi = make_float3(scene_hi[0], scene_hi[1], scene_hi[2]);
    s.codes.resize(n); s.idx.resize(n); s.umc.resize(n); s.cnt.resize(n); s.first.resize(n);
    s.leafParents.resize(n + 1); s.nodes.resize(n > 1 ? n - 1 : 1);
    return cudaDeviceSynchronize() == cudaSuccess ? 0 : -1;
}

// One frame's build = R/src/Renderer.cpp:422-503 (with the reference's synchronisation after every step)
__attribute__((visibility("default"))) int refh_build(void* p) {
    Scene& s = *(Scene*)p;
    const int n = s.n;
    // GPUArrayManager::AllocateBIHTree sentinels (R/src/GPUArrayManager.cpp:58-91); the reference does this once
    // at load and never resets clip planes (SURVEY.md 0.9) -- done per build here so rebuilds are independent.
    {
        TreeInternalNode init;
        init.parent = -1; init.children[0] = init.children[1] = -1; init.t_axis = -1;
        init.t_clipPlanes[0] = std::numeric_limits<float>::lowest(); init.t_clipPlanes[1] = std::numeric_limits<float>::max();
        init.isLeaf[0] = init.isLeaf[1] = false; init.ID = -1; init.traversed = false;
        thrust::fill(s.nodes.begin(), s.nodes.end(), init);
        thrust::fill(s.leafParents.begin(), s.leafParents.end(), -1);
    }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaDeviceSynchronize();
    cudaEventRecord(e0);
    thrust::transform(thrust::device, s.cnorm.begin(), s.cnorm.begin() + n, s.codes.begin(), morton_of_norm_centre());   // :422-426
    cudaDeviceSynchronize();
    thrust::sequence(thrust::device, s.idx.begin(), s.idx.begin() + n);                                                    // :436
    cudaDeviceSynchronize();
    thrust::stable_sort_by_key(thrust::device, s.codes.begin(), s.codes.begin() + n, s.idx.begin());                        // :441-445
    cudaDeviceSynchronize();
    auto end = thrust::reduce_by_key(thrust::device, s.codes.begin(), s.codes.begin() + n, thrust::make_constant_iterator(1),
                                     s.umc.begin(), s.cnt.begin());                                                         // :450-459
    cudaDeviceSynchronize();
    s.nu = (int)(end.first - s.umc.begin());
    thrust::unique_by_key_copy(thrust::device, s.codes.begin(), s.codes.begin() + n, thrust::make_counting_iterator(0),
                               s.umc.begin(), s.first.begin());                                                             // :466-472
    cudaDeviceSynchronize();
    if (s.nu >= 2) {
        const int nu = s.nu;
        BuildTree<<<nu / 64 + 1, 64>>>(thrust::raw_pointer_cast(s.umc.data()), thrust::raw_pointer_cast(s.nodes.data()),
                                       thrust::raw_pointer_cast(s.leafParents.data()), nu);                                  // launcher :712-723
        cudaDeviceSynchronize();
        FindClipPlanes<<<nu / 256 + 1, 256>>>(thrust::raw_pointer_cast(s.nodes.data()), thrust::raw_pointer_cast(s.lo.data()),
                                              thrust::raw_pointer_cast(s.hi.data()), thrust::raw_pointer_cast(s.idx.data()),
                                              thrust::raw_pointer_cast(s.leafParents.data()), thrust::raw_pointer_cast(s.cnt.data()),
                                              thrust::raw_pointer_cast(s.first.data()), nu);                                 // launcher :551-565
        cudaDeviceSynchronize();
    }
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    cudaEventElapsedTime(&s.last_build_ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return cudaGetLastError() == cudaSuccess ? s.nu : -1;
}

__attribute__((visibility("default"))) float refh_last_build_ms(void* p) { return ((Scene*)p)->last_build_ms; }

// copy the reference's arrays back (SoA, trimmed by the caller)
__attribute__((visibility("default"))) int refh_export(void* p, uint32_t* codes, uint32_t* idx, uint32_t* umc, uint32_t* cnt, int* first,
                                                        float* clip2, int* axis, unsigned char* is_leaf2, int* children2, int* parent,
                                                        int* leaf_parents) {
    Scene& s = *(Scene*)p;
    const int n = s.n, nu = s.nu, ni = nu > 1 ? nu - 1 : 0;
    thrust::copy(s.codes.begin(), s.codes.begin() + n, codes);
    thrust::copy(s.idx.begin(), s.idx.begin() + n, idx);
    thrust::copy(s.umc.begin(), s.umc.begin() + nu, umc);
    thrust::copy(s.cnt.begin(), s.cnt.begin() + nu, cnt);
    thrust::copy(s.first.begin(), s.first.begin() + nu, first);
    thrust::copy(s.leafParents.begin(), s.leafParents.begin() + nu, leaf_parents);
    std::vector<TreeInternalNode> h(ni);
    if (ni) cudaMemcpy(h.data(), thrust::raw_pointer_cast(s.nodes.data()), sizeof(TreeInternalNode) * ni, cudaMemcpyDeviceToHost);
    for (int i = 0; i < ni; i++) {
        clip2[2 * i] = h[i].t_clipPlanes[0]; clip2[2 * i + 1] = h[i].t_clipPlanes[1];
        axis[i] = h[i].t_axis; is_leaf2[2 * i] = h[i].isLeaf[0]; is_leaf2[2 * i + 1] = h[i].isLeaf[1];
        children2[2 * i] = h[i].children[0]; children2[2 * i + 1] = h[i].children[1]; parent[i] = h[i].parent;
    }
    return nu;
}

// traces host rays with the reference's TraverseTree; returns kernel ms (CUDA events), outputs on the host
__attribute__((visibility("default"))) float refh_trace(void* p, const float* rays6, int nrays, float* out_t, int* out_slot, int reps) {
    Scene& s = *(Scene*)p;
    thrust::device_vector<float> d_rays(rays6, rays6 + (size_t)nrays * 6), d_t(nrays);
    thrust::device_vector<int> d_slot(nrays);
    // the reference's 64-entry StackElement array + spills need more than the default local-memory stack
    cudaDeviceSetLimit(cudaLimitStackSize, 4096);
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    float best = 1e30f;
    for (int r = 0; r < (reps < 1 ? 1 : reps); r++) {
        cudaEventRecord(e0);
        ref_trace_kernel<<<(nrays + 63) / 64, 64>>>(thrust::raw_pointer_cast(d_rays.data()), nrays, thrust::raw_pointer_cast(s.nodes.data()),
                                                    thrust::raw_pointer_cast(s.first.data()), thrust::raw_pointer_cast(s.cnt.data()),
                                                    thrust::raw_pointer_cast(s.tris.data()), thrust::raw_pointer_cast(s.idx.data()),
                                                    s.sceneLo, s.sceneHi, s.nu, thrust::raw_pointer_cast(d_t.data()),
                                                    thrust::raw_pointer_cast(d_slot.data()));
        cudaEventRecord(e1);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        if (ms < best) best = ms;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (cudaGetLastError() != cudaSuccess) return -1.0f;
    thrust::copy(d_t.begin(), d_t.end(), out_t);
    thrust::copy(d_slot.begin(), d_slot.end(), out_slot);
    return best;
}

}  // extern "C"
