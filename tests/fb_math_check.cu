// Checks the framebuffer-render arithmetic of the trace kernel (bih-gpu-raytracer_b200/csrc/fb_math.cuh) on the GPU;
// tests/test_gpu_fb_math.py builds and runs it.
//
//   fb_math_check TABLES.bin
//
// 1. camera_div(x, -w, camera_rcp(w)) == __fdiv_rn(x, w), bit for bit, for every w in [1, 65535] and, for every integer i in
//    [0, 65536], x = i, i + 2^-24, i + 0.5, i + (1 - 2^-24) (each sum rounded as the kernel rounds px + ru) and the floats
//    next to i on either side.  Prints "div <mismatches> <w> <x>" (w and x of the first mismatch found, 0 0 when none).
// 2. The colour tables as the kernel fills them, for n = 1 .. COLOUR_TABLE_MAX samples per pixel: entry h of table n is
//    written to TABLES.bin at offset (n * (n + 1) / 2 - 1 + h) * 4, for the test to compare with the oracle's packing.
#include <cstdio>
#include <cstdint>
#include <cstring>
#include <vector>
#include "../bih-gpu-raytracer_b200/csrc/fb_math.cuh"

#define CHECK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e_)); return 2; } } while (0)

__global__ void k_div(unsigned long long* bad, unsigned long long* first) {
    const float w = (float)(blockIdx.x + 1);
    const float r = camera_rcp(w), neg_w = -w;
    for (uint32_t i = threadIdx.x; i <= 65536u; i += blockDim.x) {
        const float fi = (float)i;
        const float xs[6] = { fi, __fadd_rn(fi, 0x1p-24f), __fadd_rn(fi, 0.5f), __fadd_rn(fi, 1.f - 0x1p-24f),
                              nextafterf(fi, 0.f), nextafterf(fi, 131072.f) };
#pragma unroll
        for (int k = 0; k < 6; k++) {
            const float x = xs[k];
            if (__float_as_uint(camera_div(x, neg_w, r)) != __float_as_uint(__fdiv_rn(x, w))) {
                atomicAdd(bad, 1ull);
                atomicCAS(first, 0ull, ((unsigned long long)(blockIdx.x + 1) << 32) | __float_as_uint(x));
            }
        }
    }
}

__global__ void k_colour(uint32_t* out) {
    __shared__ uint32_t table[COLOUR_TABLE_MAX + 1];
    const int n = blockIdx.x + 1;
    fill_colour_table(table, n, threadIdx.x, blockDim.x);
    __syncthreads();
    for (int h = threadIdx.x; h <= n; h += blockDim.x) out[n * (n + 1) / 2 - 1 + h] = table[h];
}

int main(int argc, char** argv) {
    if (argc != 2) { fprintf(stderr, "usage: %s TABLES.bin\n", argv[0]); return 2; }
    unsigned long long* d;
    CHECK(cudaMalloc(&d, 16));
    CHECK(cudaMemset(d, 0, 16));
    k_div<<<65535, 256>>>(d, d + 1);
    CHECK(cudaGetLastError());
    unsigned long long h[2];
    CHECK(cudaMemcpy(h, d, 16, cudaMemcpyDeviceToHost));
    uint32_t xbits = (uint32_t)h[1];
    float x;
    memcpy(&x, &xbits, 4);
    printf("div %llu %u %.9g\n", h[0], (unsigned)(h[1] >> 32), x);

    const int entries = (COLOUR_TABLE_MAX + 1) * (COLOUR_TABLE_MAX + 2) / 2 - 1;
    uint32_t* t;
    CHECK(cudaMalloc(&t, entries * 4));
    k_colour<<<COLOUR_TABLE_MAX, 128>>>(t);
    CHECK(cudaGetLastError());
    std::vector<uint32_t> tab(entries);
    CHECK(cudaMemcpy(tab.data(), t, entries * 4, cudaMemcpyDeviceToHost));
    FILE* f = fopen(argv[1], "wb");
    if (!f || fwrite(tab.data(), 4, entries, f) != (size_t)entries || fclose(f)) { fprintf(stderr, "cannot write %s\n", argv[1]); return 2; }
    printf("colour %d\n", COLOUR_TABLE_MAX);
    return 0;
}
