// C ABI of libbihrt.so (include/bihrt.h): context, scene load, build, export, trace, framebuffer.
// Host side of the path: replaces App::LoadModels (R/src/App.cpp:65-167), GPUArrayManager
// (R/src/GPUArrayManager.cpp) and the launch half of Renderer (R/src/Renderer.cpp:415-503,638-640).
#include "bihrt_internal.cuh"
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

int bihrt_fail(bihrt_ctx* c, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (c) c->err = buf;
    return code;
}

#define ENTER(c) do { if (!(c)) return BIHRT_ERR_INVALID; BIHRT_CUDA((c), cudaSetDevice((c)->device)); } while (0)

static bool is_device_ptr(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}

template <typename T>
static int dev_alloc(bihrt_ctx* c, T** p, size_t count) {
    if (*p) { cudaFree(*p); *p = nullptr; }
    if (count == 0) count = 1;
    cudaError_t e = cudaMalloc((void**)p, count * sizeof(T));
    if (e != cudaSuccess) { *p = nullptr; cudaGetLastError(); return bihrt_fail(c, BIHRT_ERR_NOMEM, "cudaMalloc(%zu bytes) failed: %s", count * sizeof(T), cudaGetErrorString(e)); }
    return BIHRT_OK;
}
template <typename T>
static void dev_free(T** p) { if (*p) { cudaFree(*p); *p = nullptr; } }

template <typename T>
static int fetch(bihrt_ctx* c, std::vector<T>& dst, const T* src, size_t count) {
    dst.resize(count);
    if (count) BIHRT_CUDA(c, cudaMemcpyAsync(dst.data(), src, count * sizeof(T), cudaMemcpyDeviceToHost, c->stream));
    return BIHRT_OK;
}

static size_t lookback_words_for(int64_t n) {
    // must match build.cu: 4 onesweep passes x tiles(4096) x 256 + 8 words per rle tile(2048)
    size_t os_tiles = (size_t)((n + 4095) / 4096), rle_tiles = (size_t)((n + 2047) / 2048);
    return 4 * os_tiles * 256 + rle_tiles * 8 + 16;
}

static size_t blob_capacity(int64_t n) { return 64 + (size_t)n * sizeof(BihNode) + (size_t)n * 48 + 64; }

static void bind_blob(bihrt_ctx* c, int64_t cap) {
    c->d_hdr = reinterpret_cast<BihHeader*>(c->d_blob);
    c->d_nodes = reinterpret_cast<BihNode*>(c->d_blob + 64);
    c->d_tris = reinterpret_cast<BihTri*>(c->d_blob + 64 + (size_t)cap * sizeof(BihNode));
}

// GPUArrayManager::AllocateTris / AllocateMortonCodes / AllocateBIHTree (R/src/GPUArrayManager.cpp:7-91)
static int ensure_capacity(bihrt_ctx* c, int64_t n, bool with_build_scratch) {
    int rc;
    if (n > c->cap_n || !c->d_blob) {
        int64_t cap = std::max<int64_t>(n, 1);
        if ((rc = dev_alloc(c, &c->d_blob, blob_capacity(cap)))) return rc;
        c->blob_cap = blob_capacity(cap);
        dev_free(&c->d_tri_in);
        for (int i = 0; i < 2; i++) { dev_free(&c->d_keys[i]); dev_free(&c->d_vals[i]); }
        dev_free(&c->d_umc); dev_free(&c->d_first); dev_free(&c->d_lookback); dev_free(&c->d_heaps);
        dev_free(&c->d_keys64[0]); dev_free(&c->d_keys64[1]); dev_free(&c->d_lookback_q); c->lookback_q_words = 0;
        c->cap_n = cap;
        c->have_scene = false; c->built = false;
        if (c->build_graph_exec) { cudaGraphExecDestroy(c->build_graph_exec); c->build_graph_exec = nullptr; }
        bind_blob(c, cap);
    }
    if (with_build_scratch && !c->d_keys[0]) {
        int64_t cap = c->cap_n;
        if ((rc = dev_alloc(c, &c->d_tri_in, (size_t)cap * 9 + 4))) return rc;
        for (int i = 0; i < 2; i++) {
            if ((rc = dev_alloc(c, &c->d_keys[i], (size_t)cap + 8))) return rc;
            if ((rc = dev_alloc(c, &c->d_vals[i], (size_t)cap + 8))) return rc;
        }
        if ((rc = dev_alloc(c, &c->d_umc, (size_t)cap + 8))) return rc;
        if ((rc = dev_alloc(c, &c->d_first, (size_t)cap + 8))) return rc;
        c->lookback_words = lookback_words_for(cap);
        if ((rc = dev_alloc(c, &c->d_lookback, c->lookback_words))) return rc;
        size_t P = 256;
        while (P < (size_t)cap) P <<= 1;
        if ((rc = dev_alloc(c, &c->d_heaps, 4 * P))) return rc;      // 2P entries x 2 float4
    }
    return BIHRT_OK;
}

extern "C" {

int bihrt_version(void) { return BIHRT_VERSION; }

int bihrt_create(bihrt_ctx** out, const bihrt_config* cfg) {
    if (!out) return BIHRT_ERR_INVALID;
    *out = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { cudaGetLastError(); return BIHRT_ERR_CUDA; }   // no CPU fallback
    bihrt_ctx* c = new (std::nothrow) bihrt_ctx();
    if (!c) return BIHRT_ERR_NOMEM;
    c->device = cfg ? cfg->device : 0;
    if (c->device < 0 || c->device >= ndev) { delete c; return BIHRT_ERR_INVALID; }
    cudaDeviceProp prop;
    if (cudaSetDevice(c->device) != cudaSuccess || cudaGetDeviceProperties(&prop, c->device) != cudaSuccess) { delete c; return BIHRT_ERR_CUDA; }
    if (prop.major < 10) { delete c; return BIHRT_ERR_CUDA; }   // sm_100a code only
    c->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return BIHRT_ERR_CUDA; }
    c->stream = c->own_stream;
    cudaEventCreate(&c->ev0); cudaEventCreate(&c->ev1);
    int rc = 0;
    rc |= dev_alloc(c, &c->d_hist, 4096);
    rc |= dev_alloc(c, &c->d_scenebox_enc, 24);
    rc |= dev_alloc(c, &c->d_counters, 8);
    rc |= dev_alloc(c, &c->d_work, 1024);
    // hdr->status of the last build, mirrored by the build's last kernel into mapped host memory: the host can look at it
    // without a copy or a synchronisation of its own
    if (cudaHostAlloc((void**)&c->h_status, 64, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess ||
        cudaHostGetDevicePointer((void**)&c->d_status_map, c->h_status, 0) != cudaSuccess) { cudaGetLastError(); rc |= 1; }
    else *c->h_status = 0;
    if (rc) { bihrt_destroy(c); return BIHRT_ERR_NOMEM; }
    if (bihrt_build_setup(c) != BIHRT_OK) { bihrt_destroy(c); return BIHRT_ERR_CUDA; }
    *out = c;
    return BIHRT_OK;
}

void bihrt_destroy(bihrt_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    dev_free(&c->d_tri_in); dev_free(&c->d_blob);
    for (int i = 0; i < 2; i++) { dev_free(&c->d_keys[i]); dev_free(&c->d_vals[i]); }
    dev_free(&c->d_umc); dev_free(&c->d_first); dev_free(&c->d_hist); dev_free(&c->d_lookback);
    dev_free(&c->d_heaps); dev_free(&c->d_scenebox_enc);
    dev_free(&c->d_keys64[0]); dev_free(&c->d_keys64[1]); dev_free(&c->d_lookback_q);
    dev_free(&c->d_fb); dev_free(&c->d_counters); dev_free(&c->d_work);
    for (auto& ts : c->tile_slots) { dev_free(&ts.cost); dev_free(&ts.order); }
    if (c->d_io) { cudaFree(c->d_io); c->d_io = nullptr; }
    for (int i = 0; i < 2; i++) { dev_free(&c->d_rs_keys[i]); dev_free(&c->d_rs_vals[i]); }
    dev_free(&c->d_rs_hist); dev_free(&c->d_rs_lookback); dev_free(&c->d_rs_hdr);
    if (c->h_status) { cudaFreeHost(c->h_status); c->h_status = nullptr; }
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    if (c->build_graph_exec) cudaGraphExecDestroy(c->build_graph_exec);
    for (int i = 0; i < BIHRT_PROF_EVENTS; i++) if (c->prof_ev[i]) cudaEventDestroy(c->prof_ev[i]);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
}

const char* bihrt_last_error(const bihrt_ctx* c) { return c ? c->err.c_str() : "null context"; }

// The handle means what it means to every CUDA call: 0 is the legacy default stream (what
// torch.cuda.current_stream().cuda_stream is when torch runs on its default stream), BIHRT_STREAM_OWN the context's
// private non-blocking stream.
int bihrt_set_stream(bihrt_ctx* c, void* s) {
    ENTER(c);
    BIHRT_CUDA(c, cudaStreamSynchronize(c->stream));
    c->stream = (s == BIHRT_STREAM_OWN) ? c->own_stream : (cudaStream_t)s;
    return BIHRT_OK;
}

int bihrt_get_stream(bihrt_ctx* c, void** s) {
    if (!c || !s) return BIHRT_ERR_INVALID;
    *s = (void*)c->stream;
    return BIHRT_OK;
}

// the device watchdog of the last build that has COMPLETED (never blocks)
static int check_status(bihrt_ctx* c) {
    const uint32_t st = c->h_status ? *(volatile uint32_t*)c->h_status : 0u;
    if (st & 0x100u) return bihrt_fail(c, BIHRT_ERR_STATE, "the BIH in this context is a %s tree but the context traces %s trees: set the option morton_bits "
                                       "to the builder's value before adopting a replicated BIH", c->built_quality ? "parity" : "quality-mode", c->built_quality ? "quality-mode" : "parity");
    if (st) return bihrt_fail(c, BIHRT_ERR_INTERNAL, "device watchdog tripped during build (status %u): the BIH is invalid, rebuild", st);
    return BIHRT_OK;
}

int bihrt_sync(bihrt_ctx* c) {
    ENTER(c);
    BIHRT_CUDA(c, cudaStreamSynchronize(c->stream));
    return check_status(c);
}

int bihrt_set_option(bihrt_ctx* c, const char* name, int64_t v) {
    if (!c || !name) return BIHRT_ERR_INVALID;
    if (!strcmp(name, "trace_blocks_per_sm")) c->opt_trace_blocks_per_sm = (int)v;
    else if (!strcmp(name, "trace_refill_threshold")) c->opt_refill_threshold = (int)std::max<int64_t>(1, std::min<int64_t>(32, v));
    else if (!strcmp(name, "build_graph")) c->opt_build_graph = (int)v;
    else if (!strcmp(name, "morton_bits")) {
        // 30: the reference's 10-bit grid (parity path).  63: quality mode (non-parity): 21 bits per axis, ties broken by position,
        // subtrees of at most leaf_cap triangles collapsed into leaves.  Takes effect at the next bihrt_build / bihrt_bih_adopt.
        if (v != 30 && v != 63) return bihrt_fail(c, BIHRT_ERR_INVALID, "morton_bits must be 30 (reference grid) or 63 (quality mode)");
        c->opt_morton_bits = (int)v;
        if (c->build_graph_exec) { cudaGraphExecDestroy(c->build_graph_exec); c->build_graph_exec = nullptr; }
    }
    else if (!strcmp(name, "leaf_cap")) {
        if (v < 1 || v > 64) return bihrt_fail(c, BIHRT_ERR_INVALID, "leaf_cap must be 1..64");
        c->opt_leaf_cap = (int)v;
        if (c->build_graph_exec) { cudaGraphExecDestroy(c->build_graph_exec); c->build_graph_exec = nullptr; }
    }
    else if (!strcmp(name, "debug_trip_watchdog")) {
        c->opt_debug_trip_watchdog = (int)v;
        if (c->build_graph_exec) { cudaGraphExecDestroy(c->build_graph_exec); c->build_graph_exec = nullptr; }    // the value is a kernel argument
    }
    else if (!strcmp(name, "profile")) {
        BIHRT_CUDA(c, cudaSetDevice(c->device));          // the events belong to this context's device
        c->opt_profile = (int)v;
        if (v) for (int i = 0; i < BIHRT_PROF_EVENTS; i++) if (!c->prof_ev[i]) cudaEventCreate(&c->prof_ev[i]);
    }
    else if (!strcmp(name, "trace_lane_groups")) c->opt_lane_groups = (int)v;
    else if (!strcmp(name, "trace_sort_rays")) c->opt_sort_rays = (int)v;
    else if (!strcmp(name, "trace_sm_queues")) c->opt_sm_queues = (int)v;
    else if (!strcmp(name, "trace_tile_sort_below")) c->opt_tile_sort_below = v;
    else if (!strcmp(name, "trace_tile_order")) { c->opt_tile_order = (int)v; for (auto& ts : c->tile_slots) ts.valid = false; }
    else if (!strcmp(name, "interleave_chunk")) c->opt_interleave_chunk = (int)std::max<int64_t>(1, std::min<int64_t>(1024, v));
    else if (!strcmp(name, "trace_vote_wait")) c->opt_vote_wait = (int)v;
    else if (!strcmp(name, "trace_vote_walk")) c->opt_vote_walk = (int)v;
    else if (!strcmp(name, "trace_refill_incoherent")) c->opt_refill_incoherent = (int)std::max<int64_t>(1, std::min<int64_t>(32, v));
    else if (!strcmp(name, "trace_chunk_items")) c->opt_chunk_items = (int)std::max<int64_t>(32, (v + 31) / 32 * 32);
    else return bihrt_fail(c, BIHRT_ERR_INVALID, "unknown option '%s'", name);
    return BIHRT_OK;
}

int bihrt_get_stat(bihrt_ctx* c, const char* name, int64_t* v) {
    if (!c || !name || !v) return BIHRT_ERR_INVALID;
    if (!strcmp(name, "kernel_launches")) *v = c->kernel_launches;
    else if (!strcmp(name, "sm_count")) *v = c->sm_count;
    else if (!strcmp(name, "trace_warp_node_steps") || !strcmp(name, "trace_warp_leaf_steps")) {
        // of the last instrumented launch (bihrt_trace_counted / bihrt_render_counted): how often a WARP executed the node
        // step / the triangle test; lane-level counts (counters[0], [1]) / 32 / these = SIMD efficiency of the two phases
        unsigned long long h[2];
        BIHRT_CUDA(c, cudaSetDevice(c->device));
        BIHRT_CUDA(c, cudaMemcpyAsync(h, c->d_counters + 4, 16, cudaMemcpyDeviceToHost, c->stream));
        BIHRT_CUDA(c, cudaStreamSynchronize(c->stream));
        *v = (int64_t)h[name[11] == 'n' ? 0 : 1];
    }
    else if (!strncmp(name, "build_stage_ns_", 15)) {
        // stages: 0 init+memsets, 1 scene_box, 2 morton, 3-6 sort passes, 7 rle, 8 reorder + slot boxes, 9 upper heap levels, 10 nodes
        const int i = atoi(name + 15);
        if (!c->opt_profile || i < 0 || i + 1 >= c->prof_count) return bihrt_fail(c, BIHRT_ERR_STATE, "no profile for stage %d (set option profile=1 and build)", i);
        BIHRT_CUDA(c, cudaEventSynchronize(c->prof_ev[i + 1]));
        float ms = 0;
        BIHRT_CUDA(c, cudaEventElapsedTime(&ms, c->prof_ev[i], c->prof_ev[i + 1]));
        *v = (int64_t)(ms * 1e6f);
    }
    else return bihrt_fail(c, BIHRT_ERR_INVALID, "unknown stat '%s'", name);
    return BIHRT_OK;
}

// ---- scene load ------------------------------------------------------------------------------
static int upload_triangles(bihrt_ctx* c, const float* xyz9, int64_t n) {
    if (n > 0) {
        cudaMemcpyKind kind = is_device_ptr(xyz9) ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        BIHRT_CUDA(c, cudaMemcpyAsync(c->d_tri_in, xyz9, (size_t)n * 36, kind, c->stream));
    }
    return BIHRT_OK;
}

int bihrt_scene_load_triangles(bihrt_ctx* c, const float* xyz9, int64_t n) {
    ENTER(c);
    if (n < 0 || (n > 0 && !xyz9)) return bihrt_fail(c, BIHRT_ERR_INVALID, "bad triangle array");
    if (n >= BIH_MAX_TRIS) return bihrt_fail(c, BIHRT_ERR_INVALID, "at most 2^29-1 triangles (29-bit child references)");
    int rc = ensure_capacity(c, n, true);
    if (rc) return rc;
    if (n != c->n) {                       // the blob is laid out for n: [header | n node slots | n triangle records]
        bind_blob(c, std::max<int64_t>(n, 1));
        if (c->build_graph_exec) { cudaGraphExecDestroy(c->build_graph_exec); c->build_graph_exec = nullptr; }
    }
    c->n = n; c->have_scene = true; c->built = false; c->topology_valid = false;
    return upload_triangles(c, xyz9, n);
}

int bihrt_scene_update_vertices(bihrt_ctx* c, const float* xyz9, int64_t n) {
    ENTER(c);
    if (!c->have_scene || !c->d_tri_in) return bihrt_fail(c, BIHRT_ERR_STATE, "no scene loaded");
    if (n != c->n) return bihrt_fail(c, BIHRT_ERR_INVALID, "update must keep the triangle count (%lld != %lld)", (long long)n, (long long)c->n);
    c->built = false;
    return upload_triangles(c, xyz9, n);
}

// Minimal Wavefront OBJ reader: `v x y z` and `f a b c ...` (a, a/b, a/b/c, a//c; negative = relative),
// polygons fan-triangulated in face order.  Replaces Model(path) -> Assimp (R/src/Model.cpp:10-29);
// Assimp's own triangulation order is not reproducible here (binary-only dependency; parity unpinned).
int bihrt_scene_load_obj(bihrt_ctx* c, const char* path) {
    ENTER(c);
    if (!path) return BIHRT_ERR_INVALID;
    FILE* f = fopen(path, "r");
    if (!f) return bihrt_fail(c, BIHRT_ERR_IO, "cannot open '%s'", path);
    std::vector<float> verts, tris;
    std::vector<long> poly;
    char line[4096];
    int rc = BIHRT_OK;
    while (fgets(line, sizeof line, f)) {
        if (line[0] == 'v' && (line[1] == ' ' || line[1] == '\t')) {
            float x, y, z;
            if (sscanf(line + 2, "%f %f %f", &x, &y, &z) != 3) { rc = bihrt_fail(c, BIHRT_ERR_IO, "bad vertex line in '%s'", path); break; }
            verts.push_back(x); verts.push_back(y); verts.push_back(z);
        } else if (line[0] == 'f' && (line[1] == ' ' || line[1] == '\t')) {
            poly.clear();
            char* p = line + 2;
            for (;;) {
                while (*p == ' ' || *p == '\t') p++;
                if (*p == 0 || *p == '\n' || *p == '\r' || *p == '#') break;
                char* end;
                long idx = strtol(p, &end, 10);
                if (end == p) { rc = bihrt_fail(c, BIHRT_ERR_IO, "bad face line in '%s'", path); break; }
                long nv = (long)(verts.size() / 3);
                idx = idx < 0 ? nv + idx : idx - 1;
                if (idx < 0 || idx >= nv) { rc = bihrt_fail(c, BIHRT_ERR_IO, "face index out of range in '%s'", path); break; }
                poly.push_back(idx);
                p = end;
                while (*p && *p != ' ' && *p != '\t' && *p != '\n' && *p != '\r') p++;   // skip /vt/vn
            }
            if (rc) break;
            for (size_t k = 1; k + 1 < poly.size(); k++) {
                const long id[3] = { poly[0], poly[k], poly[k + 1] };
                for (int v = 0; v < 3; v++) for (int a = 0; a < 3; a++) tris.push_back(verts[3 * id[v] + a]);
            }
        }
    }
    fclose(f);
    if (rc) return rc;
    return bihrt_scene_load_triangles(c, tris.data(), (int64_t)(tris.size() / 9));
}

// ---- build -------------------------------------------------------------------------------------
// quality mode: 63-bit keys (two buffers) and the look-back words of 8 sort passes over 2048-key tiles, allocated on first use
static int ensure_quality_scratch(bihrt_ctx* c) {
    int rc;
    const size_t cap = (size_t)c->cap_n;
    for (int i = 0; i < 2; i++) if (!c->d_keys64[i] && (rc = dev_alloc(c, &c->d_keys64[i], cap + 8))) return rc;
    const size_t need = 8 * ((cap + 2047) / 2048) * 256 + 16;
    if (need > c->lookback_q_words) {
        if ((rc = dev_alloc(c, &c->d_lookback_q, need))) { c->lookback_q_words = 0; return rc; }
        c->lookback_q_words = need;
    }
    return BIHRT_OK;
}

int bihrt_build(bihrt_ctx* c) {
    ENTER(c);
    if (!c->have_scene || !c->d_tri_in) return bihrt_fail(c, BIHRT_ERR_STATE, "no scene loaded");
    const bool quality = c->opt_morton_bits == 63;
    if (quality) { int rq = ensure_quality_scratch(c); if (rq) return rq; }
    auto build_launch = [&]() { return quality ? bihrt_build_launch_q(c) : bihrt_build_launch(c); };
    BIHRT_CUDA(c, cudaEventRecord(c->ev0, c->stream));
    if (c->n == 0) {
        BIHRT_CUDA(c, cudaMemsetAsync(c->d_hdr, 0, sizeof(BihHeader), c->stream));
        BIHRT_CUDA(c, cudaStreamSynchronize(c->stream));
        *c->h_status = 0;
    } else if (c->opt_build_graph && !c->opt_profile && c->stream != nullptr && c->stream != cudaStreamLegacy) {    // (the legacy stream cannot be captured)
        // The build is ~16 short launches with fixed arguments for a given triangle count: capture them once
        // into a CUDA graph and replay it (the reference rebuilds every frame, R/src/Renderer.cpp:415-503).
        if (!c->build_graph_exec || c->build_graph_n != c->n) {
            if (c->build_graph_exec) { cudaGraphExecDestroy(c->build_graph_exec); c->build_graph_exec = nullptr; }
            cudaGraph_t g = nullptr;
            BIHRT_CUDA(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
            const int64_t launches_before = c->kernel_launches;
            int rc = build_launch();
            cudaError_t e = cudaStreamEndCapture(c->stream, &g);
            if (rc) { if (g) cudaGraphDestroy(g); return rc; }
            if (e != cudaSuccess) return bihrt_fail(c, BIHRT_ERR_CUDA, "graph capture of the build failed: %s", cudaGetErrorString(e));
            e = cudaGraphInstantiate(&c->build_graph_exec, g, 0);
            cudaGraphDestroy(g);
            if (e != cudaSuccess) { c->build_graph_exec = nullptr; return bihrt_fail(c, BIHRT_ERR_CUDA, "cudaGraphInstantiate failed: %s", cudaGetErrorString(e)); }
            c->build_graph_n = c->n;
            c->build_graph_launches = c->kernel_launches - launches_before;
            c->kernel_launches = launches_before;             // nothing ran during capture
        }
        BIHRT_CUDA(c, cudaGraphLaunch(c->build_graph_exec, c->stream));
        c->kernel_launches += c->build_graph_launches;
    } else {
        int rc = build_launch();
        if (rc) return rc;
    }
    BIHRT_CUDA(c, cudaEventRecord(c->ev1, c->stream));
    c->built = true; c->build_timed = true; c->topology_valid = c->n > 0 && !quality; c->built_quality = quality && c->n > 0;
    return BIHRT_OK;
}

int bihrt_refit(bihrt_ctx* c) {
    ENTER(c);
    if (!c->have_scene || !c->d_tri_in) return bihrt_fail(c, BIHRT_ERR_STATE, "no scene loaded");
    if (c->built_quality || c->opt_morton_bits == 63) return bihrt_fail(c, BIHRT_ERR_STATE, "bihrt_refit is not available in quality mode (morton_bits = 63)");
    if (!c->topology_valid) return bihrt_fail(c, BIHRT_ERR_STATE, "refit needs a full bihrt_build of the same triangle count first");
    BIHRT_CUDA(c, cudaEventRecord(c->ev0, c->stream));
    int rc = bihrt_refit_launch(c);
    if (rc) return rc;
    BIHRT_CUDA(c, cudaEventRecord(c->ev1, c->stream));
    c->built = true; c->build_timed = true;
    return BIHRT_OK;
}

static int fetch_header(bihrt_ctx* c, BihHeader* h) {
    BIHRT_CUDA(c, cudaMemcpyAsync(h, c->d_hdr, sizeof(BihHeader), cudaMemcpyDeviceToHost, c->stream));
    BIHRT_CUDA(c, cudaStreamSynchronize(c->stream));
    if (h->status) return bihrt_fail(c, BIHRT_ERR_INTERNAL, "device watchdog tripped during build (status %u)", h->status);
    return BIHRT_OK;
}

int bihrt_get_build_info(bihrt_ctx* c, bihrt_build_info* out) {
    ENTER(c);
    if (!out) return BIHRT_ERR_INVALID;
    if (!c->built) return bihrt_fail(c, BIHRT_ERR_STATE, "BIH not built");
    BihHeader h;
    int rc = fetch_header(c, &h);
    if (rc) return rc;
    memset(out, 0, sizeof *out);
    out->n = h.n; out->nu = h.nu;
    out->node_bytes = (h.quality ? (h.n > 1 ? (int64_t)(h.n - 1) : 0) : (h.nu > 1 ? (int64_t)(h.nu - 1) : 0)) * (int64_t)sizeof(BihNode);
    out->tri_bytes = (int64_t)h.n * 48;
    out->sort_passes = h.quality ? 8 : 4;
    if (c->build_timed) { float ms = 0; if (cudaEventElapsedTime(&ms, c->ev0, c->ev1) == cudaSuccess) out->last_build_ms = ms; else cudaGetLastError(); }
    return BIHRT_OK;
}

int bihrt_export_reference_view(bihrt_ctx* c, bihrt_refview* v) {
    ENTER(c);
    if (!v) return BIHRT_ERR_INVALID;
    if (!c->built || !c->d_keys[0]) return bihrt_fail(c, BIHRT_ERR_STATE, "reference view needs a BIH built on this context");
    if (c->built_quality) return bihrt_fail(c, BIHRT_ERR_STATE, "the reference view is defined for the reference's tree only (morton_bits = 30), not for a quality-mode build");
    BihHeader h;
    int rc = fetch_header(c, &h);
    if (rc) return rc;
    const size_t n = h.n, nu = h.nu, ni = nu > 1 ? nu - 1 : 0;
    v->n = (int64_t)n; v->nu = (int64_t)nu;
    for (int k = 0; k < 3; k++) { v->scene_lo[k] = h.lo[k]; v->scene_hi[k] = h.hi[k]; }
    if (n == 0) return BIHRT_OK;
    std::vector<uint32_t> first, umc;
    std::vector<BihNode> nodes;
    if ((rc = fetch(c, first, c->d_first, nu + 1))) return rc;
    if ((rc = fetch(c, nodes, c->d_nodes, ni))) return rc;
    if (v->morton_codes) BIHRT_CUDA(c, cudaMemcpyAsync(v->morton_codes, c->d_keys[0], n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (v->tris_indexes) BIHRT_CUDA(c, cudaMemcpyAsync(v->tris_indexes, c->d_vals[0], n * 4, cudaMemcpyDeviceToHost, c->stream));
    if (v->unique_morton_codes) BIHRT_CUDA(c, cudaMemcpyAsync(v->unique_morton_codes, c->d_umc, nu * 4, cudaMemcpyDeviceToHost, c->stream));
    BIHRT_CUDA(c, cudaStreamSynchronize(c->stream));
    for (size_t k = 0; k < nu; k++) {
        if (v->first_idxs) v->first_idxs[k] = (int32_t)first[k];
        if (v->duplicates_cnts) v->duplicates_cnts[k] = first[k + 1] - first[k];
        if (v->leaf_parents) v->leaf_parents[k] = -1;
    }
    for (size_t i = 0; i < ni; i++) if (v->parent) v->parent[i] = -1;
    if (v->axis && ni) v->axis[0] = (int32_t)h.root_axis;
    for (size_t i = 0; i < ni; i++) {
        const BihNode& nd = nodes[i];
        const bool ll = nd.ref_l & BIH_REF_LEAF, rl = nd.ref_r & BIH_REF_LEAF;
        const uint32_t il = BIH_REF_INDEX(nd.ref_l), ir = BIH_REF_INDEX(nd.ref_r);
        uint32_t split;
        if (!ll) split = il;
        else if (!rl) split = ir - 1;
        else split = (uint32_t)(std::lower_bound(first.begin(), first.begin() + nu, il) - first.begin());   // leaf whose first slot is il
        if (v->clip_planes) { v->clip_planes[2 * i] = nd.clip0; v->clip_planes[2 * i + 1] = nd.clip1; }
        if (v->axis) {      // a node's axis is stored in its parent's reference to it
            if (!ll) v->axis[split] = (int32_t)BIH_REF_AXIS(nd.ref_l);
            if (!rl) v->axis[split + 1] = (int32_t)BIH_REF_AXIS(nd.ref_r);
        }
        if (v->is_leaf) { v->is_leaf[2 * i] = ll; v->is_leaf[2 * i + 1] = rl; }
        if (v->children) { v->children[2 * i] = (int32_t)split; v->children[2 * i + 1] = (int32_t)split + 1; }
        if (ll) { if (v->leaf_parents) v->leaf_parents[split] = (int32_t)i; } else if (v->parent) v->parent[split] = (int32_t)i;
        if (rl) { if (v->leaf_parents) v->leaf_parents[split + 1] = (int32_t)i; } else if (v->parent) v->parent[split + 1] = (int32_t)i;
    }
    return BIHRT_OK;
}

// ---- trace -------------------------------------------------------------------------------------
static int ensure_io(bihrt_ctx* c, size_t bytes) {
    if (bytes <= c->io_cap) return BIHRT_OK;
    if (c->d_io) { cudaFree(c->d_io); c->d_io = nullptr; c->io_cap = 0; }
    cudaError_t e = cudaMalloc(&c->d_io, bytes);
    if (e != cudaSuccess) { cudaGetLastError(); return bihrt_fail(c, BIHRT_ERR_NOMEM, "cudaMalloc(%zu) for ray staging failed", bytes); }
    c->io_cap = bytes;
    return BIHRT_OK;
}

static void base_args(bihrt_ctx* c, TraceArgs& a) {
    memset(&a, 0, sizeof a);
    a.hdr = c->d_hdr; a.nodes = c->d_nodes; a.tris = c->d_tris;
    a.counters = c->d_counters; a.work = c->d_work;
    a.shard_index = 0; a.shard_count = 1; a.il_index = 0; a.il_count = 1;
    a.refill_threshold = c->opt_refill_threshold; a.chunk_items = c->opt_chunk_items;
    a.refill_incoherent = c->opt_refill_incoherent;
    a.vote_wait = c->opt_vote_wait; a.vote_walk = c->opt_vote_walk;
    a.queues = c->opt_sm_queues;      // resolved per launch in bihrt_trace_launch (-1 = by ray count)
}

// outputs may individually be host or device; host ones are staged through d_io.  t, slot, prim (4 bytes per ray) for every
// trace; u, v (4 bytes) and ng (12 bytes) for bihrt_intersect's hit records.  dev[k] is what the kernel writes (the caller's
// device array, a staging block, or NULL), host[k] the caller's host array it is copied back to (NULL: none).
enum { OUT_T, OUT_SLOT, OUT_PRIM, OUT_U, OUT_V, OUT_NG, OUT_COUNT };
static const size_t out_bytes_per_ray[OUT_COUNT] = { 4, 4, 4, 4, 4, 12 };
struct OutStage {
    void* dev[OUT_COUNT]; void* host[OUT_COUNT];
    float* t() const { return (float*)dev[OUT_T]; }
    int32_t* slot() const { return (int32_t*)dev[OUT_SLOT]; }
    int32_t* prim() const { return (int32_t*)dev[OUT_PRIM]; }
};

static int stage_outputs(bihrt_ctx* c, int64_t n, size_t front_bytes, float* t, int32_t* slot, int32_t* prim, OutStage& o, uint8_t** front,
                         float* u = nullptr, float* v = nullptr, float* ng = nullptr) {
    void* const want[OUT_COUNT] = { t, slot, prim, u, v, ng };
    bool staged[OUT_COUNT];
    size_t need = front_bytes + 256;
    for (int k = 0; k < OUT_COUNT; k++) {
        staged[k] = want[k] && !is_device_ptr(want[k]);
        if (staged[k]) need += (size_t)n * out_bytes_per_ray[k] + 16;    // (+16: every staged array starts 16-byte aligned)
    }
    int rc = ensure_io(c, need);
    if (rc) return rc;
    uint8_t* p = (uint8_t*)c->d_io;
    *front = p;
    p += (front_bytes + 255) / 256 * 256;
    for (int k = 0; k < OUT_COUNT; k++) {
        o.dev[k] = want[k]; o.host[k] = nullptr;
        if (staged[k]) { o.host[k] = want[k]; o.dev[k] = p; p += ((size_t)n * out_bytes_per_ray[k] + 15) / 16 * 16; }
    }
    return BIHRT_OK;
}

static int unstage_outputs(bihrt_ctx* c, int64_t n, const OutStage& o) {
    bool any = false;
    for (int k = 0; k < OUT_COUNT; k++) any |= o.host[k] != nullptr;
    if (!any) return BIHRT_OK;
    // host outputs: the call is synchronous anyway -- learn first whether the BIH that was traced is valid (a tripped
    // build watchdog makes the kernel trace nothing), and leave the caller's arrays untouched if it is not
    BIHRT_CUDA(c, cudaStreamSynchronize(c->stream));
    int rc = check_status(c);
    if (rc) return rc;
    for (int k = 0; k < OUT_COUNT; k++)
        if (o.host[k]) BIHRT_CUDA(c, cudaMemcpyAsync(o.host[k], o.dev[k], (size_t)n * out_bytes_per_ray[k], cudaMemcpyDeviceToHost, c->stream));
    BIHRT_CUDA(c, cudaStreamSynchronize(c->stream));
    return BIHRT_OK;
}

static int trace_impl(bihrt_ctx* c, const bihrt_ray* rays, int64_t n, float* t, int32_t* slot, int32_t* prim, uint64_t* counters,
                      bool any_hit = false, float tmax = 0.f) {
    ENTER(c);
    if (!c->built) return bihrt_fail(c, BIHRT_ERR_STATE, "BIH not built");
    { int st = check_status(c); if (st) return st; }
    if (n < 0 || (n > 0 && !rays)) return bihrt_fail(c, BIHRT_ERR_INVALID, "bad ray array");
    if (n >= (1ll << 32) - (1ll << 24)) return bihrt_fail(c, BIHRT_ERR_INVALID, "too many rays in one call (32-bit work counter)");
    if (counters) BIHRT_CUDA(c, cudaMemsetAsync(c->d_counters, 0, 64, c->stream));
    if (n > 0) {
        const bool rays_dev = is_device_ptr(rays);
        OutStage o; uint8_t* front;
        int rc = stage_outputs(c, n, rays_dev ? 0 : (size_t)n * sizeof(bihrt_ray), t, slot, prim, o, &front);
        if (rc) return rc;
        TraceArgs a; base_args(c, a);
        if (rays_dev) a.rays = rays;
        else { BIHRT_CUDA(c, cudaMemcpyAsync(front, rays, (size_t)n * sizeof(bihrt_ray), cudaMemcpyHostToDevice, c->stream)); a.rays = (const bihrt_ray*)front; }
        a.nrays = n; a.out_t = o.t(); a.out_slot = o.slot(); a.out_prim = o.prim();
        a.any_hit = any_hit ? 1 : 0; a.tmax = tmax;
        // incoherent batches (option trace_sort_rays): trace through a permutation that groups the rays by origin cell and
        // direction octant; results still land in list order
        if (c->opt_sort_rays && n >= 4096 && n < (1ll << 31)) { if ((rc = bihrt_ray_sort_launch(c, a.rays, n, &a.perm))) return rc; }
        if ((rc = bihrt_trace_launch(c, a, 0, counters != nullptr))) return rc;
        if ((rc = unstage_outputs(c, n, o))) return rc;
    }
    if (counters) {
        unsigned long long h[4];
        BIHRT_CUDA(c, cudaMemcpyAsync(h, c->d_counters, 32, cudaMemcpyDeviceToHost, c->stream));
        BIHRT_CUDA(c, cudaStreamSynchronize(c->stream));
        counters[0] = h[0]; counters[1] = h[1]; counters[2] = h[2]; counters[3] = (uint64_t)n;
    }
    return BIHRT_OK;
}

int bihrt_trace(bihrt_ctx* c, const bihrt_ray* rays, int64_t n, float* t, int32_t* slot, int32_t* prim) {
    return trace_impl(c, rays, n, t, slot, prim, nullptr);
}
int bihrt_trace_counted(bihrt_ctx* c, const bihrt_ray* rays, int64_t n, float* t, int32_t* slot, int32_t* prim, uint64_t counters[4]) {
    if (!counters) return BIHRT_ERR_INVALID;
    return trace_impl(c, rays, n, t, slot, prim, counters);
}

// Occlusion query for shadow rays: blocker[i] = slot of SOME triangle the ray hits with 0 < t < tmax, or -1.  The
// traversal is pruned at tmax and stops at the first such hit, so blocker[i] >= 0 exactly when the closest hit of
// bihrt_trace has t < tmax; which blocker is reported is unspecified.
int bihrt_trace_any(bihrt_ctx* c, const bihrt_ray* rays, int64_t n, float tmax, int32_t* blocker) {
    if (!c) return BIHRT_ERR_INVALID;
    if (!(tmax > 0.f)) return bihrt_fail(c, BIHRT_ERR_INVALID, "tmax must be positive");
    return trace_impl(c, rays, n, nullptr, blocker, nullptr, nullptr, true, tmax);
}

// Ray queries with per-ray intervals and hit records (include/bihrt.h): k_trace MODE 3.
int bihrt_intersect(bihrt_ctx* c, const bihrt_ray_interval* rays, int64_t n, uint32_t flags, const bihrt_hits* out) {
    ENTER(c);
    if (flags & ~BIHRT_INTERSECT_ANY) return bihrt_fail(c, BIHRT_ERR_INVALID, "unknown flags 0x%x", flags & ~BIHRT_INTERSECT_ANY);
    if (!out) return bihrt_fail(c, BIHRT_ERR_INVALID, "no output record");
    if (n < 0 || (n > 0 && !rays)) return bihrt_fail(c, BIHRT_ERR_INVALID, "bad ray array");
    if (n >= (1ll << 32) - (1ll << 24)) return bihrt_fail(c, BIHRT_ERR_INVALID, "too many rays in one call (32-bit work counter)");
    if (!c->built) return bihrt_fail(c, BIHRT_ERR_STATE, "BIH not built");
    { int st = check_status(c); if (st) return st; }
    if (n == 0) return BIHRT_OK;
    const bool rays_dev = is_device_ptr(rays);
    if (rays_dev && ((uintptr_t)rays & 15u)) return bihrt_fail(c, BIHRT_ERR_INVALID, "device rays must be 16-byte aligned (two 128-bit loads per ray)");
    OutStage o; uint8_t* front;
    int rc = stage_outputs(c, n, rays_dev ? 0 : (size_t)n * sizeof(bihrt_ray_interval), out->t, out->slot, out->prim, o, &front,
                           out->u, out->v, out->ng);
    if (rc) return rc;
    TraceArgs a; base_args(c, a);
    if (rays_dev) a.rays_iv = rays;
    else {
        BIHRT_CUDA(c, cudaMemcpyAsync(front, rays, (size_t)n * sizeof(bihrt_ray_interval), cudaMemcpyHostToDevice, c->stream));
        a.rays_iv = (const bihrt_ray_interval*)front;
    }
    a.nrays = n; a.any_hit = (flags & BIHRT_INTERSECT_ANY) ? 1 : 0;
    a.out_t = o.t(); a.out_slot = o.slot(); a.out_prim = o.prim();
    a.out_u = (float*)o.dev[OUT_U]; a.out_v = (float*)o.dev[OUT_V]; a.out_ng = (float*)o.dev[OUT_NG];
    if ((rc = bihrt_trace_launch(c, a, 3, false))) return rc;
    return unstage_outputs(c, n, o);
}

static int render_check(bihrt_ctx* c, const bihrt_camera* cam, int w, int h, int spp, int si, int sc) {
    if (!c->built) return bihrt_fail(c, BIHRT_ERR_STATE, "BIH not built");
    { int st = check_status(c); if (st) return st; }
    if (!cam || w <= 0 || h <= 0 || spp <= 0 || w > 65535 || h > 65535 || (int64_t)w * h >= (1ll << 31) - (1ll << 24))
        return bihrt_fail(c, BIHRT_ERR_INVALID, "bad render arguments");
    if (sc < 1 || si < 0 || si >= sc) return bihrt_fail(c, BIHRT_ERR_INVALID, "bad shard %d of %d", si, sc);
    return BIHRT_OK;
}

// CreateCUDABuffers, R/src/Renderer.cpp:762-768.  While a CUDA IPC handle of the framebuffer is out (peers hold a mapping
// of this very allocation and store into it) it must not be reallocated.
static int ensure_fb(bihrt_ctx* c, size_t px) {
    if (px <= c->fb_cap) return BIHRT_OK;
    if (c->fb_exported)
        return bihrt_fail(c, BIHRT_ERR_STATE, "framebuffer of %zu pixels is exported through CUDA IPC and cannot grow to %zu: "
                          "bihrt_framebuffer_ipc_unexport first (after the peers have closed their mappings)", c->fb_cap, px);
    int rc = dev_alloc(c, &c->d_fb, px);
    if (rc) { c->fb_cap = 0; return rc; }
    c->fb_cap = px;
    return BIHRT_OK;
}

// lane groups are limited by the 32-bit work counter: padded items = tiles x 1024 pixels x groups
static int fit_gshift(int w, int h, int shard_count, int g) {
    const uint64_t tiles = ((uint64_t)(w + 31) / 32) * ((uint64_t)(h + 31) / 32) / (uint64_t)(shard_count > 0 ? shard_count : 1) + 1;
    while (g > 0 && ((tiles * 1024u) << g) >= (1ull << 32) - (1ull << 24)) g--;
    return g;
}

// samples of one pixel laid along consecutive lanes: the largest power of two that divides the sample count (<= 32)
static int pick_gshift(bihrt_ctx* c, int nsamples) {
    int g = 0;
    while (g < 5 && nsamples > 0 && (nsamples & ((2 << g) - 1)) == 0) g++;
    if (c->opt_lane_groups >= 0) { int want = 0; while ((2 << want) <= c->opt_lane_groups) want++; g = std::min(g, want); }
    return g;
}

// `target` != nullptr: the pixels this launch owns are written there (w*h packed colours, possibly on another GPU)
// and nothing else is touched: no clearing of the other ranks' pixels, no counts, no resolve.
static int render_impl(bihrt_ctx* c, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp, uint64_t seed, uint32_t flags,
                       int32_t shard_index, int32_t shard_count, uint64_t* counters, int32_t s_begin = 0, int32_t s_end = -1,
                       int32_t il_index = 0, int32_t il_count = 1, uint32_t* target = nullptr) {
    ENTER(c);
    if (s_end < 0) s_end = spp;
    if (s_begin < 0 || s_begin > s_end || s_end > spp) return bihrt_fail(c, BIHRT_ERR_INVALID, "bad sample range [%d,%d) of %d", s_begin, s_end, spp);
    int rc = render_check(c, cam, w, h, spp, shard_index, shard_count);
    if (rc) return rc;
    const size_t px = (size_t)w * h;
    if ((rc = ensure_fb(c, px))) return rc;
    c->fb_w = w; c->fb_h = h;
    if (shard_count > 1) BIHRT_CUDA(c, cudaMemsetAsync(c->d_fb, 0, px * 4, c->stream));
    TraceArgs a; base_args(c, a);
    a.cam = *cam; a.w = w; a.h = h; a.spp = spp; a.seed = seed; a.flags = flags;
    a.shard_index = shard_index; a.shard_count = shard_count; a.fb = target ? target : c->d_fb;
    a.s_begin = s_begin; a.s_end = s_end;
    a.gshift = (shard_count > 1) ? 0 : fit_gshift(w, h, 1, pick_gshift(c, s_end - s_begin));       // tile shards keep "other pixels are 0"
    a.il_index = il_index; a.il_count = il_count;
    if (il_count > 1) {
        if (il_index < 0 || il_index >= il_count || ((32 << a.gshift) % il_count) != 0)
            return bihrt_fail(c, BIHRT_ERR_INVALID, "interleave %d of %d does not divide the %d units of a tile", il_index, il_count, 32 << a.gshift);
        // runs of neighbouring units per rank: the largest power of two <= the option that still deals whole runs per tile
        // (a function of spp and count only, so every rank derives the same pixel ownership)
        int cs = 0;
        while ((2 << cs) <= c->opt_interleave_chunk && ((32 << a.gshift) % ((2 << cs) * il_count)) == 0) cs++;
        a.il_cshift = cs;
    }
    // Every pixel is written exactly once (colours, or counts when a lane holds all of a pixel's samples) except:
    // hit counts accumulated with atomics by several lanes, and interleaved launches into the rank's own
    // framebuffer, where the pixels of the other ranks must read 0 for the reduce.
    const bool atomics = a.gshift > 0 && (flags & BIHRT_RENDER_COUNTS);
    if (!target && (atomics || il_count > 1 || s_begin == s_end)) BIHRT_CUDA(c, cudaMemsetAsync(c->d_fb, 0, px * 4, c->stream));
    if (s_begin == s_end) return BIHRT_OK;            // nothing to trace on this rank: all counts are 0
    if (!counters) return bihrt_trace_launch(c, a, 1, false);
    BIHRT_CUDA(c, cudaMemsetAsync(c->d_counters, 0, 64, c->stream));
    if ((rc = bihrt_trace_launch(c, a, 1, true))) return rc;
    unsigned long long hc[4];
    BIHRT_CUDA(c, cudaMemcpyAsync(hc, c->d_counters, 32, cudaMemcpyDeviceToHost, c->stream));
    BIHRT_CUDA(c, cudaStreamSynchronize(c->stream));
    counters[0] = hc[0]; counters[1] = hc[1]; counters[2] = hc[2]; counters[3] = (uint64_t)w * h * spp;
    return BIHRT_OK;
}

int bihrt_render_shard(bihrt_ctx* c, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp, uint64_t seed, uint32_t flags,
                       int32_t shard_index, int32_t shard_count) {
    return render_impl(c, cam, w, h, spp, seed, flags, shard_index, shard_count, nullptr);
}

int bihrt_render_samples(bihrt_ctx* c, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp, uint64_t seed, uint32_t flags,
                         int32_t sample_begin, int32_t sample_end) {
    return render_impl(c, cam, w, h, spp, seed, flags | BIHRT_RENDER_COUNTS, 0, 1, nullptr, sample_begin, sample_end);
}

int bihrt_render_interleaved(bihrt_ctx* c, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp, uint64_t seed, uint32_t flags,
                             int32_t index, int32_t count) {
    return render_impl(c, cam, w, h, spp, seed, flags | BIHRT_RENDER_COUNTS, 0, 1, nullptr, 0, -1, index, count);
}

// Interleaved render whose owned pixels go, as final colours, straight into `target_fb` (NULL = this context's own
// framebuffer).  A target on another device of this process gets peer access enabled on first use.
int bihrt_render_interleaved_to(bihrt_ctx* c, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp, uint64_t seed, uint32_t flags,
                                int32_t index, int32_t count, uint32_t* target_fb) {
    ENTER(c);                                 // allocations below must land on this context's device
    if (flags & BIHRT_RENDER_COUNTS) return bihrt_fail(c, BIHRT_ERR_INVALID, "bihrt_render_interleaved_to writes colours, not counts");
    if (target_fb) {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, target_fb) != cudaSuccess || at.type != cudaMemoryTypeDevice) {
            cudaGetLastError();
            return bihrt_fail(c, BIHRT_ERR_INVALID, "target framebuffer is not device memory");
        }
        if (at.device != c->device) {
            cudaSetDevice(c->device);
            int can = 0;
            cudaDeviceCanAccessPeer(&can, c->device, at.device);
            if (!can) return bihrt_fail(c, BIHRT_ERR_CUDA, "device %d cannot address the framebuffer on device %d", c->device, at.device);
            cudaError_t e = cudaDeviceEnablePeerAccess(at.device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return bihrt_fail(c, BIHRT_ERR_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
            cudaGetLastError();
        }
    } else {
        const size_t px = (size_t)(w > 0 ? w : 0) * (size_t)(h > 0 ? h : 0);
        int rc = ensure_fb(c, px);
        if (rc) return rc;
    }
    return render_impl(c, cam, w, h, spp, seed, flags, 0, 1, nullptr, 0, -1, index, count, target_fb ? target_fb : c->d_fb);
}

// ---- framebuffer sharing between processes (one process per GPU): CUDA IPC ----------------------------
int bihrt_framebuffer_ipc_export(bihrt_ctx* c, int32_t w, int32_t h, void* handle64) {
    ENTER(c);
    if (!handle64 || w <= 0 || h <= 0) return BIHRT_ERR_INVALID;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle is 64 bytes");
    const size_t px = (size_t)w * h;
    int rc = ensure_fb(c, px);
    if (rc) return rc;
    c->fb_w = w; c->fb_h = h;
    cudaIpcMemHandle_t hnd;
    BIHRT_CUDA(c, cudaIpcGetMemHandle(&hnd, c->d_fb));
    memcpy(handle64, &hnd, 64);
    c->fb_exported = true;
    return BIHRT_OK;
}

// The peers have closed their mappings: the framebuffer may be reallocated again.
int bihrt_framebuffer_ipc_unexport(bihrt_ctx* c) {
    if (!c) return BIHRT_ERR_INVALID;
    c->fb_exported = false;
    return BIHRT_OK;
}

int bihrt_framebuffer_ipc_open(bihrt_ctx* c, const void* handle64, uint32_t** peer_fb) {
    ENTER(c);
    if (!handle64 || !peer_fb) return BIHRT_ERR_INVALID;
    cudaIpcMemHandle_t hnd;
    memcpy(&hnd, handle64, 64);
    void* p = nullptr;
    BIHRT_CUDA(c, cudaIpcOpenMemHandle(&p, hnd, cudaIpcMemLazyEnablePeerAccess));
    *peer_fb = (uint32_t*)p;
    return BIHRT_OK;
}

int bihrt_framebuffer_ipc_close(bihrt_ctx* c, uint32_t* peer_fb) {
    ENTER(c);
    if (!peer_fb) return BIHRT_OK;
    BIHRT_CUDA(c, cudaStreamSynchronize(c->stream));
    BIHRT_CUDA(c, cudaIpcCloseMemHandle(peer_fb));
    return BIHRT_OK;
}

int bihrt_framebuffer_resolve(bihrt_ctx* c, int32_t spp) {
    ENTER(c);
    if (!c->d_fb) return bihrt_fail(c, BIHRT_ERR_STATE, "nothing rendered yet");
    if (spp <= 0) return BIHRT_ERR_INVALID;
    return bihrt_resolve_launch(c, c->d_fb, c->fb_w * c->fb_h, spp);
}

int bihrt_render_counted(bihrt_ctx* c, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp, uint64_t seed, uint32_t flags,
                         uint64_t counters[4]) {
    if (!counters) return BIHRT_ERR_INVALID;
    return render_impl(c, cam, w, h, spp, seed, flags, 0, 1, counters);
}

int bihrt_render(bihrt_ctx* c, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp, uint64_t seed, uint32_t flags) {
    return bihrt_render_shard(c, cam, w, h, spp, seed, flags, 0, 1);
}

int bihrt_render_hits(bihrt_ctx* c, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp, uint64_t seed, uint32_t flags,
                      float* t, int32_t* slot, int32_t* prim) {
    ENTER(c);
    int rc = render_check(c, cam, w, h, spp, 0, 1);
    if (rc) return rc;
    const int64_t n = (int64_t)w * h * spp;
    OutStage o; uint8_t* front;
    if ((rc = stage_outputs(c, n, 0, t, slot, prim, o, &front))) return rc;
    TraceArgs a; base_args(c, a);
    a.cam = *cam; a.w = w; a.h = h; a.spp = spp; a.seed = seed; a.flags = flags;
    a.s_begin = 0; a.s_end = spp; a.gshift = fit_gshift(w, h, 1, pick_gshift(c, spp));
    a.out_t = o.t(); a.out_slot = o.slot(); a.out_prim = o.prim();
    if ((rc = bihrt_trace_launch(c, a, 2, false))) return rc;
    return unstage_outputs(c, n, o);
}

// ---- secondary rays ------------------------------------------------------------------------------
int bihrt_secondary_rays(bihrt_ctx* c, const bihrt_camera* cam, int32_t w, int32_t h, int32_t spp, uint64_t seed, uint32_t flags,
                         int32_t kind, const float light[3], bihrt_ray* out_rays, int32_t* out_sample, int64_t* count) {
    ENTER(c);
    int rc = render_check(c, cam, w, h, spp, 0, 1);
    if (rc) return rc;
    if (!out_rays || !count || !is_device_ptr(out_rays) || (out_sample && !is_device_ptr(out_sample)))
        return bihrt_fail(c, BIHRT_ERR_INVALID, "out_rays / out_sample must be device buffers, count a host pointer");
    if (kind != BIHRT_SECONDARY_SHADOW && kind != BIHRT_SECONDARY_DIFFUSE) return bihrt_fail(c, BIHRT_ERR_INVALID, "bad kind %d", kind);
    static const float zero3[3] = { 0.f, 0.f, 0.f };
    if (!light) light = zero3;
    const int64_t n = (int64_t)w * h * spp;
    const size_t ntiles = (size_t)((n + 255) / 256);
    // staging: t[n] | slot[n] | tile counts
    if ((rc = ensure_io(c, (size_t)n * 8 + ntiles * 4 + 512))) return rc;
    float* d_t = (float*)c->d_io;
    int32_t* d_slot = (int32_t*)((uint8_t*)c->d_io + (size_t)n * 4);
    uint32_t* d_cnt = (uint32_t*)((uint8_t*)c->d_io + (size_t)n * 8);
    TraceArgs a; base_args(c, a);
    a.cam = *cam; a.w = w; a.h = h; a.spp = spp; a.seed = seed; a.flags = flags;
    a.s_begin = 0; a.s_end = spp; a.gshift = fit_gshift(w, h, 1, pick_gshift(c, spp));
    a.out_t = d_t; a.out_slot = d_slot; a.out_prim = nullptr;
    if ((rc = bihrt_trace_launch(c, a, 2, false))) return rc;
    if ((rc = bihrt_secondary_launch(c, d_t, d_slot, n, d_cnt, c->d_counters + 3, *cam, w, h, spp, seed, flags, kind, light, out_rays, out_sample))) return rc;
    unsigned long long total = 0;
    BIHRT_CUDA(c, cudaMemcpyAsync(&total, c->d_counters + 3, 8, cudaMemcpyDeviceToHost, c->stream));
    BIHRT_CUDA(c, cudaStreamSynchronize(c->stream));
    *count = (int64_t)total;
    return BIHRT_OK;
}

// ---- framebuffer -------------------------------------------------------------------------------
int bihrt_framebuffer(bihrt_ctx* c, uint32_t** dev_ptr, int32_t* w, int32_t* h) {
    if (!c) return BIHRT_ERR_INVALID;
    if (!c->d_fb) return bihrt_fail(c, BIHRT_ERR_STATE, "nothing rendered yet");
    if (dev_ptr) *dev_ptr = c->d_fb;
    if (w) *w = c->fb_w;
    if (h) *h = c->fb_h;
    return BIHRT_OK;
}

int bihrt_framebuffer_read(bihrt_ctx* c, uint32_t* host_dst) {
    ENTER(c);
    if (!c->d_fb) return bihrt_fail(c, BIHRT_ERR_STATE, "nothing rendered yet");
    if (!host_dst) return BIHRT_ERR_INVALID;
    BIHRT_CUDA(c, cudaMemcpyAsync(host_dst, c->d_fb, (size_t)c->fb_w * c->fb_h * 4, cudaMemcpyDeviceToHost, c->stream));
    BIHRT_CUDA(c, cudaStreamSynchronize(c->stream));
    return check_status(c);
}

// ---- BIH replication ----------------------------------------------------------------------------
// blob = [BihHeader 64 B][nodes (nu-1) x 16 B][triangles n x 48 B]
int bihrt_bih_blob_bytes(bihrt_ctx* c, uint64_t* bytes) {
    ENTER(c);
    if (!bytes) return BIHRT_ERR_INVALID;
    if (!c->built) return bihrt_fail(c, BIHRT_ERR_STATE, "BIH not built");
    BihHeader h;
    int rc = fetch_header(c, &h);
    if (rc) return rc;
    *bytes = 64 + (uint64_t)(h.quality ? (h.n > 1 ? h.n - 1 : 0) : (h.nu > 1 ? h.nu - 1 : 0)) * sizeof(BihNode) + (uint64_t)h.n * 48;
    return BIHRT_OK;
}

int bihrt_bih_export(bihrt_ctx* c, void* dev_dst, uint64_t bytes) {
    ENTER(c);
    uint64_t need;
    int rc = bihrt_bih_blob_bytes(c, &need);
    if (rc) return rc;
    if (!dev_dst || bytes < need) return bihrt_fail(c, BIHRT_ERR_INVALID, "blob buffer too small (%llu < %llu)", (unsigned long long)bytes, (unsigned long long)need);
    BihHeader h;
    if ((rc = fetch_header(c, &h))) return rc;
    const size_t nb = (size_t)(h.quality ? (h.n > 1 ? h.n - 1 : 0) : (h.nu > 1 ? h.nu - 1 : 0)) * sizeof(BihNode), tb = (size_t)h.n * 48;
    uint8_t* d = (uint8_t*)dev_dst;
    BIHRT_CUDA(c, cudaMemcpyAsync(d, c->d_hdr, 64, cudaMemcpyDeviceToDevice, c->stream));
    if (nb) BIHRT_CUDA(c, cudaMemcpyAsync(d + 64, c->d_nodes, nb, cudaMemcpyDeviceToDevice, c->stream));
    if (tb) BIHRT_CUDA(c, cudaMemcpyAsync(d + 64 + nb, c->d_tris, tb, cudaMemcpyDeviceToDevice, c->stream));
    return BIHRT_OK;
}

int bihrt_bih_import(bihrt_ctx* c, const void* dev_src, uint64_t bytes) {
    ENTER(c);
    if (!dev_src || bytes < 64) return bihrt_fail(c, BIHRT_ERR_INVALID, "bad blob");
    BihHeader h;
    BIHRT_CUDA(c, cudaMemcpyAsync(&h, dev_src, 64, cudaMemcpyDeviceToHost, c->stream));
    BIHRT_CUDA(c, cudaStreamSynchronize(c->stream));
    const size_t nb = (size_t)(h.quality ? (h.n > 1 ? h.n - 1 : 0) : (h.nu > 1 ? h.nu - 1 : 0)) * sizeof(BihNode), tb = (size_t)h.n * 48;
    if (h.nu > h.n || bytes < 64 + nb + tb) return bihrt_fail(c, BIHRT_ERR_INVALID, "blob truncated or corrupt");
    int rc = ensure_capacity(c, h.n, false);
    if (rc) return rc;
    if ((int64_t)h.n != c->n) {
        bind_blob(c, std::max<int64_t>(h.n, 1));
        if (c->build_graph_exec) { cudaGraphExecDestroy(c->build_graph_exec); c->build_graph_exec = nullptr; }
        c->have_scene = false;
    }
    const uint8_t* s = (const uint8_t*)dev_src;
    BIHRT_CUDA(c, cudaMemcpyAsync(c->d_hdr, s, 64, cudaMemcpyDeviceToDevice, c->stream));
    if (nb) BIHRT_CUDA(c, cudaMemcpyAsync(c->d_nodes, s + 64, nb, cudaMemcpyDeviceToDevice, c->stream));
    if (tb) BIHRT_CUDA(c, cudaMemcpyAsync(c->d_tris, s + 64 + nb, tb, cudaMemcpyDeviceToDevice, c->stream));
    c->n = h.n; c->built = true; c->build_timed = false; c->topology_valid = false; c->built_quality = h.quality != 0;
    return BIHRT_OK;
}

// In-place replication: the whole blob of an n-triangle scene, [header 64 B | n node slots | n triangle records], is one
// contiguous region whose size follows from n alone, so it can be the buffer of a broadcast on every rank: no export /
// import copies and no host read of Nu.  bihrt_bih_region lays the context's blob out for n triangles (allocating if
// needed) and returns the region; on the building rank (same n, already built) it changes nothing.  After the
// broadcast the receivers call bihrt_bih_adopt.
int bihrt_bih_region(bihrt_ctx* c, int64_t n, void** dev_ptr, uint64_t* bytes) {
    ENTER(c);
    if (n < 0 || n >= BIH_MAX_TRIS || !dev_ptr || !bytes) return BIHRT_ERR_INVALID;
    int rc = ensure_capacity(c, n, false);
    if (rc) return rc;
    if (n != c->n) {
        bind_blob(c, std::max<int64_t>(n, 1));
        if (c->build_graph_exec) { cudaGraphExecDestroy(c->build_graph_exec); c->build_graph_exec = nullptr; }
        c->n = n; c->have_scene = false; c->built = false; c->topology_valid = false;
    }
    *dev_ptr = c->d_blob;
    *bytes = 64 + (uint64_t)std::max<int64_t>(n, 1) * sizeof(BihNode) + (uint64_t)n * 48;
    return BIHRT_OK;
}

int bihrt_bih_adopt(bihrt_ctx* c, int64_t n);

// Same replication inside ONE process (a C host driving several GPUs without NCCL): a peer copy of the region over
// NVLink, ordered after everything enqueued so far on the source context's stream and before whatever the destination
// context does next.
int bihrt_bih_copy(bihrt_ctx* dst, bihrt_ctx* src) {
    if (!dst || !src) return BIHRT_ERR_INVALID;
    if (dst == src) return BIHRT_OK;
    if (!src->built) return bihrt_fail(dst, BIHRT_ERR_STATE, "source BIH not built");
    void* p = nullptr; uint64_t bytes = 0;
    int rc = bihrt_bih_region(dst, src->n, &p, &bytes);          // sets the destination device
    if (rc) return rc;
    if (dst->device != src->device) {
        int can = 0;
        cudaDeviceCanAccessPeer(&can, dst->device, src->device);
        if (can) { cudaError_t e = cudaDeviceEnablePeerAccess(src->device, 0); if (e != cudaSuccess) cudaGetLastError(); }
    }
    cudaEvent_t ev = nullptr;
    BIHRT_CUDA(dst, cudaSetDevice(src->device));
    BIHRT_CUDA(dst, cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    BIHRT_CUDA(dst, cudaEventRecord(ev, src->stream));
    BIHRT_CUDA(dst, cudaSetDevice(dst->device));
    BIHRT_CUDA(dst, cudaStreamWaitEvent(dst->stream, ev, 0));
    BIHRT_CUDA(dst, cudaMemcpyPeerAsync(dst->d_blob, dst->device, src->d_blob, src->device, (size_t)bytes, dst->stream));
    cudaEventDestroy(ev);                                        // released once the recorded work has completed
    // ... and the source's next build must not overwrite the blob while the copy is still reading it
    cudaEvent_t done = nullptr;
    BIHRT_CUDA(dst, cudaEventCreateWithFlags(&done, cudaEventDisableTiming));
    BIHRT_CUDA(dst, cudaEventRecord(done, dst->stream));
    BIHRT_CUDA(dst, cudaSetDevice(src->device));
    BIHRT_CUDA(dst, cudaStreamWaitEvent(src->stream, done, 0));
    BIHRT_CUDA(dst, cudaSetDevice(dst->device));
    cudaEventDestroy(done);
    dst->opt_morton_bits = src->built_quality ? 63 : 30;         // the replica is a tree of the builder's kind
    return bihrt_bih_adopt(dst, src->n);
}

int bihrt_bih_adopt(bihrt_ctx* c, int64_t n) {
    ENTER(c);
    if (n != c->n || !c->d_blob) return bihrt_fail(c, BIHRT_ERR_STATE, "bihrt_bih_adopt(%lld) without a matching bihrt_bih_region", (long long)n);
    c->built = true; c->build_timed = false; c->topology_valid = false;
    c->built_quality = c->opt_morton_bits == 63;                 // (the kernel refuses a tree of the other kind: see check_status)
    if (c->h_status) *c->h_status = 0;
    return BIHRT_OK;
}

}  // extern "C"
