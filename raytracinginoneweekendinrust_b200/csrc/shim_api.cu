// shim_api.cu — the C ABI (include/shimmer_b200.h): commit/upload, the wavefront driver, the
// multi-device render and the gate-1 batch query.  No CPU fallback: every device entry point
// fails with SHIM_ERR_CUDA when no CUDA device is usable.
#include <cuda_runtime.h>
#include <chrono>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include "shim_internal.h"
#include "shim_kernels.cuh"

using namespace shim;

#define CU(call)                                                                                        \
    do {                                                                                                \
        cudaError_t e_ = (call);                                                                        \
        if (e_ != cudaSuccess)                                                                          \
            return set_err(SHIM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));          \
    } while (0)

namespace {

template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    cudaError_t upload(const std::vector<T>& v) {
        release();
        n = v.size();
        // never hand out a null pointer: empty arrays still get a valid allocation
        cudaError_t e = cudaMalloc(&p, (n ? n : 1) * sizeof(T));
        if (e != cudaSuccess) return e;
        if (n) e = cudaMemcpy(p, v.data(), n * sizeof(T), cudaMemcpyHostToDevice);
        return e;
    }
    cudaError_t alloc(size_t count) {
        release();
        n = count;
        cudaError_t e = cudaMalloc(&p, (n ? n : 1) * sizeof(T));
        if (e != cudaSuccess) { p = nullptr; n = 0; }
        return e;
    }
    cudaError_t reserve(size_t count) { return count <= n && p ? cudaSuccess : alloc(count); }   // grow only
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
    size_t bytes() const { return p ? (n ? n : 1) * sizeof(T) : 0; }
};

// restores the calling thread's current device
struct DeviceGuard {
    int prev = -1;
    bool changed = false;
    cudaError_t enter(int device) {
        cudaError_t e = cudaGetDevice(&prev);
        if (e != cudaSuccess) return e;
        if (prev != device) { e = cudaSetDevice(device); changed = e == cudaSuccess; }
        return e;
    }
    ~DeviceGuard() { if (changed) cudaSetDevice(prev); }
};

// Host image of a committed scene: the arrays packed back to back (256-byte aligned), uploaded with ONE copy per
// device.  It is kept after commit so that shim_render_multi can replicate the scene on further devices.
struct SceneBlob {
    std::vector<unsigned char> bytes;
    size_t o_nodes = 0, o_snodes = 0, o_qnodes = 0, o_sph = 0, o_sph_s = 0, o_sph_mat = 0, o_msph = 0, o_rect = 0, o_tri = 0, o_cube = 0, o_obj = 0, o_mat = 0, o_tex = 0,
           o_img = 0, o_perlin = 0;
    size_t o_handle[5] = {0}, o_rank[5] = {0}, o_leaf[5] = {0}, o_sib[5] = {0};
    int n_objects = 0, n_nodes = 0, n_qnodes = 0, q_object = -1;
};

// one device's copy of a committed scene
struct DeviceScene {
    int device = -1;
    int sm_count = 0;
    unsigned char* base = nullptr;
    SceneView view;
    HrppSlot* hrpp_slots = nullptr;            // n_predictors x slots
    size_t hrpp_slots_total = 0;
    bool hrpp_cleared = false;                 // the tables hold what earlier renders learnt (SHIM_RENDER_KEEP_PREDICTORS)
    void release() {
        if (!base && !hrpp_slots) return;
        DeviceGuard g;
        if (g.enter(device) != cudaSuccess) return;
        if (base) cudaFree(base);
        if (hrpp_slots) cudaFree(hrpp_slots);
        base = nullptr; hrpp_slots = nullptr; hrpp_slots_total = 0;
    }
};

// The wavefront pool of one device (queues, counters, framebuffer sums, graphs): per device, not per scene — scenes
// come and go (one per render call in the e2e path) while the pool is reused.  It grows to the largest render seen
// and is released by shim_shutdown().
struct Wavefront {
    std::mutex render_mutex;                       // one render in flight per device (constant-memory parameters, shared pool)
    bool ready = false;
    int device = -1, sm_count = 0, max_smem = 0;
    DevBuf<f4> ray_o[2], ray_d[2], thr[2];         // ray queues: wavefront pipeline only
    DevBuf<f4> mq_o, mq_d, mq_thr, mq_hit;          // material queues (sets x regions x pool entries)
    DevBuf<i4> bvh1_hit;                            // one-Bvh worlds: hit record per queued ray
    DevBuf<uint32_t> bvh1_queue;                    // ... and the rays that can reach the tree
    DevBuf<uint32_t> cnt;
    DevBuf<float> accum, d_out, d_peer;
    float* h_out = nullptr;  // pinned staging for a pageable host framebuffer
    size_t h_out_n = 0;
    DevBuf<uint32_t> pix_table;
    int pt_key[6] = {0, 0, 0, 0, 0, 0};
    uint32_t npix = 0;
    uint32_t* h_flags = nullptr;  // pinned: done flag / counter readbacks
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_chunk[2] = {nullptr, nullptr};
    int grid_extend_gmem = 0, grid_bvh1_walk = 0, grid_stream = 0, grid_shade = 0, grid_generate = 0, grid_tail = 0;
    cudaStream_t capture_stream = nullptr;         // graphs are captured here (the caller's stream may be the legacy default stream)
    cudaStream_t work_stream = nullptr;            // shim_render_multi renders on it
    struct LoopGraph { cudaGraphExec_t exec; unsigned long long handle; };
    typedef std::tuple<uint32_t, int, int, int, int, int, int, int, int, int, int, int, uint32_t> GraphKey;
    std::map<GraphKey, LoopGraph> graphs;          // the whole wavefront loop as one graph (WHILE node), per kernel-variant key
    std::vector<cudaEvent_t> prof;                 // event pairs around the launches of an iteration (SHIM_RENDER_PROFILE)
    std::vector<cudaEvent_t> ev_d2h;
    size_t pool_bytes() const {
        size_t b = bvh1_hit.bytes() + bvh1_queue.bytes() + mq_o.bytes() + mq_d.bytes() + mq_thr.bytes() + mq_hit.bytes() + cnt.bytes() + accum.bytes() + d_out.bytes() + d_peer.bytes() +
                   pix_table.bytes();
        for (int i = 0; i < 2; ++i) b += ray_o[i].bytes() + ray_d[i].bytes() + thr[i].bytes();
        return b;
    }
    void release() {   // with the device current
        for (int i = 0; i < 2; ++i) { ray_o[i].release(); ray_d[i].release(); thr[i].release(); }
        mq_o.release(); mq_d.release(); mq_thr.release(); mq_hit.release(); bvh1_hit.release(); bvh1_queue.release(); cnt.release(); accum.release(); pix_table.release();
        d_out.release(); d_peer.release();
        if (h_flags) cudaFreeHost(h_flags);
        if (h_out) cudaFreeHost(h_out);
        h_out = nullptr; h_out_n = 0; h_flags = nullptr;
        for (cudaEvent_t* e : {&ev0, &ev1, &ev_chunk[0], &ev_chunk[1]}) { if (*e) cudaEventDestroy(*e); *e = nullptr; }
        for (auto& e : prof) cudaEventDestroy(e);
        prof.clear();
        for (auto& e : ev_d2h) cudaEventDestroy(e);
        ev_d2h.clear();
        for (auto& g : graphs) cudaGraphExecDestroy(g.second.exec);
        graphs.clear();
        if (capture_stream) cudaStreamDestroy(capture_stream);
        if (work_stream) cudaStreamDestroy(work_stream);
        capture_stream = work_stream = nullptr;
        memset(pt_key, 0, sizeof pt_key);
        npix = 0;
        ready = false;
    }
};

enum { SHIM_MAX_DEVICES = 64 };
Wavefront g_wf[SHIM_MAX_DEVICES];

}  // namespace

// what a committed scene owns on the device side: the host blob and one DeviceScene per device it has been used on
struct shim::DeviceState {
    SceneBlob blob;
    SmemLayout smem;                   // shared-memory image with the plain 64-byte nodes (total 0: does not fit)
    SmemLayout smem_signed;            // ... with SNodes, for the one-Bvh kernels (total 0: not built)
    int n_predictors = 0, hrpp_log2 = 21;
    int primary = -1;                  // the device shim_commit uploaded to
    uint32_t kinds_mask = 0;           // shading classes the scene holds (bit k = MatKind k, bit 5 = MQ_SLOW_LAMBERTIAN)
    std::mutex m;                      // guards `on`
    std::map<int, std::unique_ptr<DeviceScene>> on;
    ~DeviceState() { for (auto& kv : on) kv.second->release(); }
};
void shim::device_state_release(DeviceState* d) { delete d; }

// ------------------------------------------------------------------------------------------ commit
static int device_count_or_error() {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return set_err(SHIM_ERR_CUDA, std::string("no usable CUDA device (this backend has no CPU fallback): ") +
                                          (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0"));
    return n;
}

// uploads the blob to the CURRENT device (which must be `device`) and registers the copy
static int upload_scene(shim::DeviceState* st, int device, DeviceScene** out) {
    std::lock_guard<std::mutex> lock(st->m);
    auto it = st->on.find(device);
    if (it != st->on.end()) { *out = it->second.get(); return SHIM_OK; }
    std::unique_ptr<DeviceScene> d(new DeviceScene());
    d->device = device;
    CU(cudaDeviceGetAttribute(&d->sm_count, cudaDevAttrMultiProcessorCount, device));
    const SceneBlob& b = st->blob;
    CU(cudaMalloc(&d->base, b.bytes.size()));
    cudaError_t e = cudaMemcpy(d->base, b.bytes.data(), b.bytes.size(), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(d->base); d->base = nullptr; return set_err(SHIM_ERR_CUDA, std::string("scene upload: ") + cudaGetErrorString(e)); }
    SceneView& v = d->view;
    memset(&v, 0, sizeof v);
    unsigned char* base = d->base;
    v.nodes = (const DevNode*)(base + b.o_nodes); v.snodes = st->smem_signed.total ? (const SNode*)(base + b.o_snodes) : nullptr; v.sph = (const double*)(base + b.o_sph); v.sph_s = (const f4*)(base + b.o_sph_s);
    v.sph_mat = (const int*)(base + b.o_sph_mat); v.msph = (const f4*)(base + b.o_msph); v.rect = (const f4*)(base + b.o_rect);
    v.tri = (const f4*)(base + b.o_tri); v.cube = (const f4*)(base + b.o_cube); v.objects = (const DevObject*)(base + b.o_obj);
    v.materials = (const f4*)(base + b.o_mat); v.textures = (const f4*)(base + b.o_tex);
    v.images = base + b.o_img; v.perlin = base + b.o_perlin;
    for (int i = 0; i < 5; ++i) {
        v.handle[i] = (const int*)(base + b.o_handle[i]); v.rank[i] = (const int*)(base + b.o_rank[i]); v.leaf[i] = (const int*)(base + b.o_leaf[i]);
        v.sibling[i] = (const int*)(base + b.o_sib[i]);
    }
    v.n_objects = b.n_objects; v.n_nodes = b.n_nodes;
    v.qnodes = b.n_qnodes ? (const QNode*)(base + b.o_qnodes) : nullptr; v.n_qnodes = b.n_qnodes; v.q_object = b.q_object;
    if (st->n_predictors > 0) {  // one open-addressing table per predictor (cleared at the start of every render that uses them)
        const int log2 = st->hrpp_log2;
        d->hrpp_slots_total = ((size_t)1 << log2) * (size_t)st->n_predictors;
        cudaError_t e2 = cudaMalloc(&d->hrpp_slots, d->hrpp_slots_total * sizeof(HrppSlot));
        if (e2 != cudaSuccess) { d->release(); return set_err(SHIM_ERR_CUDA, std::string("predictor tables: ") + cudaGetErrorString(e2)); }
        v.hrpp_slots = d->hrpp_slots; v.hrpp_mask = (uint32_t)(((size_t)1 << log2) - 1); v.hrpp_log2 = log2;
    }
    *out = d.get();
    st->on[device] = std::move(d);
    return SHIM_OK;
}

// index of the Bvh object of a world that is ONE Bvh among at least one plain object, or -1
static int single_bvh_object(const FlatScene& f) {
    int n_bvh = 0, idx = -1;
    for (size_t i = 0; i < f.objects.size(); ++i) if (f.objects[i].kind == OBJ_BVH) { ++n_bvh; idx = (int)i; }
    return n_bvh == 1 && f.objects.size() > 1 ? idx : -1;
}
// ... and every primitive inside that Bvh is a triangle (the plain objects are rects, no rect sits inside the tree)
static bool bvh1_triangles_only(const FlatScene& f, int idx) {
    if (idx < 0 || !f.sph_s.empty() || !f.msph.empty() || !f.cube.empty() || f.tri.empty()) return false;
    size_t top_rects = 0;
    for (size_t i = 0; i < f.objects.size(); ++i) {
        if ((int)i == idx) continue;
        if (f.objects[i].kind != OBJ_PRIM || prim_type((uint32_t)f.objects[i].ref) != PT_RECT) return false;
        ++top_rects;
    }
    return top_rects * 2 == f.rect.size();
}

SHIM_API int shim_commit(shim_scene* s) {
    MUTABLE(s);
    const bool trace_commit = getenv("SHIM_TRACE_COMMIT") != nullptr;
    auto t_start = std::chrono::steady_clock::now();
    auto lap = [&](const char* what) {
        if (!trace_commit) return;
        auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "shim-commit %s %.1f us\n", what, std::chrono::duration<double, std::micro>(now - t_start).count());
        t_start = now;
    };
    int rc = s->sb.flatten(s->flat);
    if (rc < 0) return set_err(rc, s->sb.err);
    lap("flatten");
    if (s->flat.objects.size() > 65535) return set_err(SHIM_ERR_UNSUPPORTED, "more than 65535 top-level objects");
    rc = device_count_or_error();
    if (rc < 0) return rc;
    int device = -1;
    CU(cudaGetDevice(&device));
    if (device < 0 || device >= SHIM_MAX_DEVICES) return set_err(SHIM_ERR_UNSUPPORTED, "device ordinal out of range");
    if (s->dev) { device_state_release(s->dev); s->dev = nullptr; }
    std::unique_ptr<shim::DeviceState> st(new shim::DeviceState());
    auto layout = [&](SmemLayout& L, const FlatScene& f, bool signed_nodes) {
        // shared-memory image of what the closest-hit kernels walk; total = 0 when it cannot fit any sm_100a block
        memset(&L, 0, sizeof L);
        const size_t node_bytes = f.nodes.size() * (signed_nodes ? sizeof(SNode) : sizeof(DevNode));
        uint32_t off = 0;
        auto place = [&](uint32_t& o, uint32_t& by, size_t bytes) { o = off; by = (uint32_t)bytes; off += (uint32_t)((bytes + 127) & ~(size_t)127); };
        size_t tot = node_bytes + f.sph.size() * 8 + (f.msph.size() + f.rect.size() + f.tri.size() + f.cube.size()) * 16 +
                     f.objects.size() * sizeof(DevObject) + f.sph_mat.size() * 4 + 16;
        if (tot > 220 * 1024) return;
        place(L.off_nodes, L.bytes_nodes, node_bytes);
        place(L.off_sph, L.bytes_sph, f.sph.size() * 8);
        place(L.off_msph, L.bytes_msph, f.msph.size() * 16);
        place(L.off_rect, L.bytes_rect, f.rect.size() * 16);
        place(L.off_tri, L.bytes_tri, f.tri.size() * 16);
        place(L.off_cube, L.bytes_cube, f.cube.size() * 16);
        place(L.off_objects, L.bytes_objects, f.objects.size() * sizeof(DevObject));
        place(L.off_sph_mat, L.bytes_sph_mat, (f.sph_mat.size() * 4 + 15) & ~(size_t)15);   // bulk copies move 16-byte units (the blob pads every array)
        L.total = off;
        L.signed_nodes = signed_nodes ? 1u : 0u;
    };
    layout(st->smem, s->flat, false);
    // one plain Bvh and nothing else: the one-Bvh kernels walk the signed node layout (shim_types.h) in shared memory
    if (s->flat.objects.size() == 1 && s->flat.objects[0].kind == OBJ_BVH && (s->flat.objects[0].flags & ~OBJ_PREDICTOR) == 0) {
        layout(st->smem_signed, s->flat, true);
        if (st->smem_signed.total) s->flat.build_signed_nodes();
    }
    // a triangle mesh among plain rects (main.rs:791-829): the dense mesh walk reads quantised 32-byte nodes
    s->flat.qnodes.clear(); s->flat.q_object = -1;
    {
        bool media = false;
        for (const DevObject& o : s->flat.objects) if (o.flags & OBJ_MEDIUM) media = true;
        const int idx = single_bvh_object(s->flat);
        if (!media && bvh1_triangles_only(s->flat, idx)) s->flat.build_quantized_nodes(idx);
    }
    lap("quantised nodes");
    const FlatScene& f = s->flat;
    SceneBlob& b = st->blob;
    b.bytes.reserve((size_t)f.bytes() + 64 * 256);   // one allocation (growing a 40 MB vector array by array was a third of a large commit)
    auto put = [&](const void* src, size_t bytes) -> size_t {
        size_t off = (b.bytes.size() + 255) & ~(size_t)255;
        b.bytes.resize(off + (bytes ? bytes : 16));
        if (bytes) memcpy(b.bytes.data() + off, src, bytes);
        return off;
    };
    b.o_nodes = put(f.nodes.data(), f.nodes.size() * sizeof(DevNode));
    b.o_snodes = put(f.snodes.data(), f.snodes.size() * sizeof(SNode));
    b.o_qnodes = put(f.qnodes.data(), f.qnodes.size() * sizeof(QNode));
    b.n_qnodes = (int)f.qnodes.size(); b.q_object = f.q_object;
    b.o_sph = put(f.sph.data(), f.sph.size() * 8); b.o_sph_s = put(f.sph_s.data(), f.sph_s.size() * 16);
    b.o_sph_mat = put(f.sph_mat.data(), f.sph_mat.size() * 4);
    b.o_msph = put(f.msph.data(), f.msph.size() * 16); b.o_rect = put(f.rect.data(), f.rect.size() * 16);
    b.o_tri = put(f.tri.data(), f.tri.size() * 16); b.o_cube = put(f.cube.data(), f.cube.size() * 16);
    b.o_obj = put(f.objects.data(), f.objects.size() * sizeof(DevObject));
    b.o_mat = put(f.materials.data(), f.materials.size() * 16); b.o_tex = put(f.textures.data(), f.textures.size() * 16);
    b.o_img = put(f.images.data(), f.images.size()); b.o_perlin = put(f.perlin.data(), f.perlin.size());
    for (int i = 0; i < 5; ++i) {
        b.o_handle[i] = put(f.handle[i].data(), f.handle[i].size() * 4);
        b.o_rank[i] = put(f.rank[i].data(), f.rank[i].size() * 4);
        b.o_leaf[i] = put(f.leaf[i].data(), f.leaf[i].size() * 4);
        b.o_sib[i] = put(f.sibling[i].data(), f.sibling[i].size() * 4);
    }
    b.n_objects = (int)f.objects.size(); b.n_nodes = (int)f.nodes.size();
    lap("blob");
    st->n_predictors = (int)f.predictor_bvh.size();
    if (const char* e = getenv("SHIM_HRPP_LOG2")) { int x = atoi(e); if (x >= 8 && x <= 26) st->hrpp_log2 = x; }
    for (size_t i = 0; i + 1 < f.materials.size(); i += 2) {   // shading classes the scene can queue hits for
        const int kind = f2i(f.materials[i].x);
        if (kind >= 0 && kind < MAT_KINDS) st->kinds_mask |= 1u << kind;
    }
    if (f.slow_lambertians) st->kinds_mask |= 1u << MQ_SLOW_LAMBERTIAN;
    st->primary = device;
    DeviceScene* ds = nullptr;
    rc = upload_scene(st.get(), device, &ds);
    if (rc < 0) return rc;
    lap("upload");
    s->dev = st.release();
    s->has_media = false;
    for (const DevObject& o : f.objects) if (o.flags & OBJ_MEDIUM) s->has_media = true;
    s->committed = true;
    return SHIM_OK;
}

// ------------------------------------------------------------------------------------------ per-device set-up
template <class K>
static cudaError_t opt_in_smem(K kernel, int bytes) { return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); }

// one-time set-up of a device's pool (with the device current and its render_mutex held)
static int wf_init(Wavefront& w, int device) {
    if (w.ready) return SHIM_OK;
    w.device = device;
    CU(cudaDeviceGetAttribute(&w.sm_count, cudaDevAttrMultiProcessorCount, device));
    CU(cudaDeviceGetAttribute(&w.max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    CU(w.cnt.alloc(CNT_WORDS));
    CU(cudaMallocHost(&w.h_flags, 128 * sizeof(uint32_t)));
    CU(cudaEventCreate(&w.ev0)); CU(cudaEventCreate(&w.ev1)); CU(cudaEventCreate(&w.ev_chunk[0])); CU(cudaEventCreate(&w.ev_chunk[1]));
    const int dyn = w.max_smem - 1024;
    CU(opt_in_smem(wf_extend<true, false, false, false>, dyn)); CU(opt_in_smem(wf_extend<true, false, true, false>, dyn));
    CU(opt_in_smem(wf_extend<true, true, false, false>, dyn));  CU(opt_in_smem(wf_extend<true, true, true, false>, dyn));
    CU(opt_in_smem(wf_extend<true, false, false, true>, dyn));  CU(opt_in_smem(wf_extend<true, false, true, true>, dyn));
    CU(opt_in_smem(wf_bvh1_walk<true, false>, dyn));  CU(opt_in_smem(wf_bvh1_walk<true, true>, dyn));
    CU(opt_in_smem(wf_bvh1_walk<true, false, SHIM_BVH1_TRI_THREADS, PT_TRI>, dyn));
    CU(opt_in_smem(wf_bvh1_walk<false, false, SHIM_BVH1_TRI_THREADS, PT_TRI, 1>, dyn));
    CU(opt_in_smem(wf_extend_list<false, SHIM_LIST_THREADS>, dyn)); CU(opt_in_smem(wf_extend_list<true, SHIM_LIST_THREADS>, dyn));
    CU(opt_in_smem(wf_extend_list<false, SHIM_LIST_THREADS, true>, dyn)); CU(opt_in_smem(wf_extend_list<true, SHIM_LIST_THREADS, true>, dyn));
    CU(opt_in_smem(wf_extend_solo<false, SHIM_SOLO_SPHERE_THREADS, PT_SPHERE, false>, dyn));
    CU(opt_in_smem(wf_extend_solo<false, SHIM_SOLO_SPHERE_THREADS, PT_SPHERE, true>, dyn));
    CU(opt_in_smem(wf_extend_solo<false, SHIM_SOLO_ANY_THREADS, -1, false>, dyn));
    CU(opt_in_smem(wf_extend_solo<false, SHIM_SOLO_ANY_THREADS, -1, true>, dyn));
    CU(opt_in_smem(wf_trace_solo<SHIM_SOLO_SPHERE_THREADS, PT_SPHERE>, dyn));
    CU(opt_in_smem(wf_trace_solo<SHIM_SOLO_ANY_THREADS, -1>, dyn));
    int per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wf_extend<false, false, false, false>, SHIM_EXTEND_THREADS, 0));
    w.grid_extend_gmem = w.sm_count * (per_sm > 0 ? per_sm : 1);
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wf_bvh1_walk<false, false, SHIM_BVH1_TRI_THREADS, PT_TRI>, SHIM_BVH1_TRI_THREADS, 0));
    w.grid_bvh1_walk = w.sm_count * (per_sm > 0 ? per_sm : 1);
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wf_bvh1_finish, 256, 0));
    w.grid_stream = w.sm_count * (per_sm > 0 ? per_sm : 1);
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wf_shade, 256, 0));
    w.grid_shade = w.sm_count * (per_sm > 0 ? per_sm : 1);
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, wf_generate, 256, 0));
    w.grid_generate = w.sm_count * (per_sm > 0 ? per_sm : 1);
    w.grid_tail = w.sm_count * 4;   // 128-thread blocks, one path per thread: covers the 65536-path trigger in one wave
    w.ready = true;
    return SHIM_OK;
}

// environment switches (read per render: the tests and the probes under tools/ force kernel variants with them)
struct Switches {
    bool no_trace, no_fuse, no_bvh1, no_smem, no_graph, solo_any, no_solo, no_list, no_bvh1_tri, trace, no_qnodes;
    int tail;   // < 0: default
    long q_smem_kb;   // < 0: default (SHIM_BVH1_Q_SMEM_KB)
    long pool;  // <= 0: default
    static bool on(const char* name) { return getenv(name) != nullptr; }
    static bool zero(const char* name) { const char* e = getenv(name); return e && atoi(e) == 0; }
    Switches() {
        no_trace = on("SHIM_NO_TRACE"); no_fuse = on("SHIM_NO_FUSE"); no_bvh1 = on("SHIM_NO_BVH1"); no_smem = on("SHIM_NO_SMEM");
        no_graph = on("SHIM_NO_GRAPH"); solo_any = on("SHIM_SOLO_ANY"); no_solo = zero("SHIM_SOLO"); no_list = zero("SHIM_LIST");
        no_bvh1_tri = zero("SHIM_BVH1_TRI"); trace = on("SHIM_TRACE");
        no_qnodes = zero("SHIM_QNODES");
        const char* q = getenv("SHIM_Q_SMEM_KB"); q_smem_kb = q ? atol(q) : -1;
        const char* t = getenv("SHIM_TAIL"); tail = t ? atoi(t) : -1;
        const char* p = getenv("SHIM_POOL_PATHS"); pool = p ? atol(p) : 0;
    }
};

// which kernels a render of this scene uses (DESIGN.md §4)
static void choose_variant(const shim_scene* s, const shim::DeviceState* st, const Wavefront& w, const Switches& sw, WfParams& k, bool* use_smem_out) {
    const FlatScene& f = s->flat;
    k.bvh1_index = -1;
    {   // worlds with exactly one BVH among at least one plain object, no medium, no predictor -> wf_bvh1_list / _walk / _finish
        const int idx = single_bvh_object(f);
        if (idx >= 0 && !s->has_media && !k.use_hrpp && !sw.no_bvh1) k.bvh1_index = idx;
    }
    k.smem = st->smem;
    const bool use_smem = k.smem.total != 0 && (int)k.smem.total <= w.max_smem - 1024 && !sw.no_smem;
    if (!use_smem) k.smem.total = 0;
    *use_smem_out = use_smem;
    k.solo = 0; k.solo_only = -1; k.fused_generate = 0; k.trace_pipeline = 0;
    const bool signed_fits = st->smem_signed.total != 0 && (int)st->smem_signed.total <= w.max_smem - 1024 && !sw.no_smem;
    if (signed_fits && !k.count_nodes && !k.use_hrpp && !s->has_media && f.objects.size() == 1 && f.objects[0].kind == OBJ_BVH &&
        (f.objects[0].flags & ~OBJ_PREDICTOR) == 0 && !sw.no_solo) {
        const bool spheres_only = f.msph.empty() && f.rect.empty() && f.tri.empty() && f.cube.empty() && !sw.solo_any;
        k.solo_only = spheres_only ? (int)PT_SPHERE : -1;
        k.solo = spheres_only ? SHIM_SOLO_SPHERE_THREADS : SHIM_SOLO_ANY_THREADS;   // 72 / 80 registers, no spills
        k.fused_generate = sw.no_fuse ? 0 : 1;
        if (!sw.no_trace) { k.trace_pipeline = k.solo; k.fused_generate = 1; }   // wf_generate is not part of this pipeline
        k.smem = st->smem_signed;   // the one-Bvh kernels walk SNodes
        *use_smem_out = true;
    }
    k.bvh1_tri_threads = 0;
    k.bvh1_list_rects = 0;
    if (k.bvh1_index >= 0 && f.objects.size() - 1 <= SHIM_BVH1_LIST_RECTS) {
        bool plain_rects = true;
        for (size_t i = 0; i < f.objects.size(); ++i)
            if ((int)i != k.bvh1_index && (f.objects[i].kind != OBJ_PRIM || f.objects[i].flags != 0 || prim_type((uint32_t)f.objects[i].ref) != PT_RECT)) plain_rects = false;
        k.bvh1_list_rects = plain_rects ? 1 : 0;
    }
    if (k.bvh1_index >= 0 && !sw.no_bvh1_tri && bvh1_triangles_only(f, k.bvh1_index)) k.bvh1_tri_threads = SHIM_BVH1_TRI_THREADS;
    // quantised nodes (built at commit for exactly these worlds): staged in shared memory when the whole tree fits
    k.bvh1_q = 0; k.bvh1_q_smem = 0;
    if (k.bvh1_tri_threads && !k.count_nodes && !f.qnodes.empty() && f.q_object == k.bvh1_index && !sw.no_qnodes) {
        k.bvh1_q = 1;
        const long cap_kb = sw.q_smem_kb >= 0 ? sw.q_smem_kb : SHIM_BVH1_Q_SMEM_KB;
        long cap = cap_kb * 1024L;
        if (cap > w.max_smem - 2048) cap = w.max_smem - 2048;
        const size_t fit = cap > 0 ? (size_t)cap / sizeof(QNode) : 0;
        // all of the tree or none of it: a staged top of a larger tree was measured slower than leaving the whole
        // shared-memory carve-out to L1 (igea, 267 k triangles: 92.0 ms with the top 160 KB staged, 90.0 ms without)
        k.bvh1_q_smem = f.qnodes.size() <= fit ? (uint32_t)f.qnodes.size() : 0u;
    }
    k.list_threads = 0;
    if (use_smem && !k.count_nodes && !k.use_hrpp && f.nodes.empty() && !k.solo && !sw.no_list) {
        k.list_threads = SHIM_LIST_THREADS;
        k.fused_generate = sw.no_fuse ? 0 : 1;   // camera rays of new samples are made inside wf_extend_list
    }
    k.tail_threshold = sw.tail >= 0 ? (uint32_t)sw.tail : 65536u;   // measured on Book-1: 32 k 3.40 ms, 48 k 3.38, 64 k 3.35, 96 k 3.48
}

// Sizes the pool for this render and lays the material queues out.  The pool is the number of paths in flight:
// every sample of the render when that fits (fewest iterations), never more than 2^24.
static int wf_reserve(Wavefront& w, const shim::DeviceState* st, const shim_render_params& p, const Switches& sw, WfParams& k) {
    uint64_t want = p.pool_paths > 0 ? (uint64_t)p.pool_paths : (sw.pool > 0 ? (uint64_t)sw.pool : k.total_samples);
    if (want > (1ull << 24)) want = 1ull << 24;
    if (want < 1024) want = 1024;
    const uint32_t pool = (uint32_t)((want + 31ull) & ~31ull);
    k.pool = pool;
    // material queues: only the kinds the scene has, two kinds per pool-sized region (one up, one down)
    int n_kinds = 0;
    for (int kind = 0; kind < MQ_CLASSES; ++kind) {
        k.mq_first[kind] = 0; k.mq_dir[kind] = 1;
        if (!(st->kinds_mask & (1u << kind))) continue;
        const long long region = n_kinds / 2;
        if (n_kinds % 2 == 0) { k.mq_first[kind] = region * (long long)pool; k.mq_dir[kind] = 1; }
        else { k.mq_first[kind] = region * (long long)pool + (long long)pool - 1; k.mq_dir[kind] = -1; }
        ++n_kinds;
    }
    const size_t regions = (size_t)((n_kinds + 1) / 2 > 0 ? (n_kinds + 1) / 2 : 1);
    k.mq_set_stride = (long long)(regions * pool);
    const size_t sets = k.trace_pipeline ? 2 : 1;   // the trace pipeline goes from one set to the other
    const size_t mq_entries = sets * regions * pool;
    CU(w.mq_o.reserve(mq_entries)); CU(w.mq_d.reserve(mq_entries)); CU(w.mq_thr.reserve(mq_entries)); CU(w.mq_hit.reserve(mq_entries));
    if (!k.trace_pipeline)   // ray queues belong to the wavefront pipeline
        for (int i = 0; i < 2; ++i) { CU(w.ray_o[i].reserve(pool)); CU(w.ray_d[i].reserve(pool)); CU(w.thr[i].reserve(pool)); }
    if (k.bvh1_index >= 0) { CU(w.bvh1_hit.reserve(pool)); CU(w.bvh1_queue.reserve(pool)); }
    k.bvh1_hit = w.bvh1_hit.p; k.bvh1_queue = w.bvh1_queue.p;
    for (int i = 0; i < 2; ++i) { k.ray_o[i] = w.ray_o[i].p; k.ray_d[i] = w.ray_d[i].p; k.thr[i] = w.thr[i].p; }
    k.mq_o = w.mq_o.p; k.mq_d = w.mq_d.p; k.mq_thr = w.mq_thr.p; k.mq_hit = w.mq_hit.p;
    return SHIM_OK;
}

static void launch_extend(const Wavefront& w, const WfParams& k, bool use_smem, cudaStream_t st) {
    const int grid = use_smem ? w.sm_count : w.grid_extend_gmem;   // one persistent block per SM owns the shared-memory copy of the scene
    const uint32_t smem = use_smem ? k.smem.total : 0;
    const bool S = use_smem, C = k.count_nodes != 0, M = k.has_media != 0, H = k.use_hrpp != 0;
    if (k.bvh1_index >= 0) {  // one BVH among plain objects, no medium, no predictor: list pass, dense tree walk, finish pass
        if (C) wf_bvh1_list<true><<<w.grid_stream, 256, 0, st>>>();
        else if (k.bvh1_list_rects) wf_bvh1_list<false, true><<<w.grid_stream, 256, 0, st>>>();
        else wf_bvh1_list<false><<<w.grid_stream, 256, 0, st>>>();
        const int wgrid = S ? w.sm_count : w.grid_bvh1_walk;
        if (k.bvh1_q) {   // triangle-only tree on quantised nodes, one block per SM owns the shared-memory top of the tree
            if (k.bvh1_q_smem) wf_bvh1_walk<false, false, SHIM_BVH1_TRI_THREADS, PT_TRI, 1><<<w.sm_count, SHIM_BVH1_TRI_THREADS, k.bvh1_q_smem * (uint32_t)sizeof(QNode), st>>>();
            else wf_bvh1_walk<false, false, SHIM_BVH1_TRI_THREADS, PT_TRI, 2><<<w.sm_count, SHIM_BVH1_TRI_THREADS, 0, st>>>();
        } else if (k.bvh1_tri_threads && !C) {   // triangle-only tree: no primitive dispatch, more warps
            if (S) wf_bvh1_walk<true, false, SHIM_BVH1_TRI_THREADS, PT_TRI><<<wgrid, SHIM_BVH1_TRI_THREADS, smem, st>>>();
            else wf_bvh1_walk<false, false, SHIM_BVH1_TRI_THREADS, PT_TRI><<<wgrid, SHIM_BVH1_TRI_THREADS, 0, st>>>();
        } else if (S) {
            if (C) wf_bvh1_walk<true, true><<<wgrid, SHIM_EXTEND_THREADS, smem, st>>>(); else wf_bvh1_walk<true, false><<<wgrid, SHIM_EXTEND_THREADS, smem, st>>>();
        } else {
            if (C) wf_bvh1_walk<false, true><<<wgrid, SHIM_EXTEND_THREADS, 0, st>>>(); else wf_bvh1_walk<false, false><<<wgrid, SHIM_EXTEND_THREADS, 0, st>>>();
        }
        wf_bvh1_finish<<<w.grid_stream, 256, 0, st>>>();
        return;
    }
    if (k.list_threads) {   // no Bvh in the world, scene image in shared memory
        if (k.fused_generate) {
            if (M) wf_extend_list<true, SHIM_LIST_THREADS, true><<<grid, SHIM_LIST_THREADS, smem, st>>>();
            else wf_extend_list<false, SHIM_LIST_THREADS, true><<<grid, SHIM_LIST_THREADS, smem, st>>>();
        } else if (M) wf_extend_list<true, SHIM_LIST_THREADS><<<grid, SHIM_LIST_THREADS, smem, st>>>();
        else wf_extend_list<false, SHIM_LIST_THREADS><<<grid, SHIM_LIST_THREADS, smem, st>>>();
        return;
    }
    if (k.solo) {   // one plain Bvh, scene image in shared memory
        if (k.solo_only == PT_SPHERE) {
            if (k.fused_generate) wf_extend_solo<false, SHIM_SOLO_SPHERE_THREADS, PT_SPHERE, true><<<grid, SHIM_SOLO_SPHERE_THREADS, smem, st>>>();
            else wf_extend_solo<false, SHIM_SOLO_SPHERE_THREADS, PT_SPHERE, false><<<grid, SHIM_SOLO_SPHERE_THREADS, smem, st>>>();
        } else {
            if (k.fused_generate) wf_extend_solo<false, SHIM_SOLO_ANY_THREADS, -1, true><<<grid, SHIM_SOLO_ANY_THREADS, smem, st>>>();
            else wf_extend_solo<false, SHIM_SOLO_ANY_THREADS, -1, false><<<grid, SHIM_SOLO_ANY_THREADS, smem, st>>>();
        }
        return;
    }
#define SHIM_LAUNCH(SS, CC, MM, HH) wf_extend<SS, CC, MM, HH><<<grid, SHIM_EXTEND_THREADS, smem, st>>>()
#define SHIM_LAUNCH_M(SS, CC, HH) do { if (M) SHIM_LAUNCH(SS, CC, true, HH); else SHIM_LAUNCH(SS, CC, false, HH); } while (0)
#define SHIM_LAUNCH_S(CC, HH) do { if (S) SHIM_LAUNCH_M(true, CC, HH); else SHIM_LAUNCH_M(false, CC, HH); } while (0)
    if (H) SHIM_LAUNCH_S(false, true);       // node counting is not combined with the predictor
    else if (C) SHIM_LAUNCH_S(true, false);
    else SHIM_LAUNCH_S(false, false);
#undef SHIM_LAUNCH_S
#undef SHIM_LAUNCH_M
#undef SHIM_LAUNCH
}

static void launch_tail(const Wavefront& w, const WfParams& k, cudaStream_t st) {
    if (k.solo) {
        if (k.solo_only == PT_SPHERE) wf_tail<false, true, PT_SPHERE><<<w.grid_tail, 128, 0, st>>>(); else wf_tail<false, true, -1><<<w.grid_tail, 128, 0, st>>>();
        return;
    }
    if (k.count_nodes) wf_tail<false, false, -1, true><<<w.grid_tail, 128, 0, st>>>();   // never with k.solo or k.use_hrpp
    else if (k.use_hrpp) wf_tail<true><<<w.grid_tail, 128, 0, st>>>(); else wf_tail<false><<<w.grid_tail, 128, 0, st>>>();
}
static void launch_trace(const Wavefront& w, const WfParams& k, cudaStream_t st) {
    if (k.solo_only == PT_SPHERE) wf_trace_solo<SHIM_SOLO_SPHERE_THREADS, PT_SPHERE><<<w.sm_count, SHIM_SOLO_SPHERE_THREADS, k.smem.total, st>>>();
    else wf_trace_solo<SHIM_SOLO_ANY_THREADS, -1><<<w.sm_count, SHIM_SOLO_ANY_THREADS, k.smem.total, st>>>();
}
static void launch_tail_mq(const Wavefront& w, const WfParams& k, cudaStream_t st) {
    const int grid = w.sm_count * SHIM_TAIL_MQ_BLOCKS;
    if (k.solo_only == PT_SPHERE) wf_tail_mq<PT_SPHERE><<<grid, 128, 0, st>>>(); else wf_tail_mq<-1><<<grid, 128, 0, st>>>();
}
// one wavefront iteration on `st` (the parameters are already in constant memory, the queue index in the counters)
static void launch_iteration(const Wavefront& w, const WfParams& k, bool use_smem, cudaStream_t st) {
    if (k.trace_pipeline) {   // shade -> closest hit, then endgame / loop condition / counters of the next iteration
        launch_trace(w, k, st);
        launch_tail_mq(w, k, st);
        return;
    }
    wf_generate<<<w.grid_generate, 256, 0, st>>>();
    launch_extend(w, k, use_smem, st);
    wf_shade<<<w.grid_shade, 256, 0, st>>>();
    launch_tail(w, k, st);   // also the loop's condition: done flag / WHILE-node condition
}

// The whole loop as one CUDA graph: a WHILE conditional node whose body is one iteration; wf_tail sets the condition
// on the device, so a render is one graph launch and the host never polls.  Built once per kernel-variant key on an
// internal stream.
enum { SHIM_CHUNK = 4 };  // iterations per done-flag readback of the host-driven loop

// Nsight Compute cannot profile kernel nodes of a graph that contains conditional nodes ("not supported for profiling"),
// and other CUPTI-injection tools may not list them either: when the process runs under such a tool the very same
// kernels are launched by the host-driven loop instead, so that every launch stays visible.
static bool under_profiler() {
    static const char* const marks[] = {"NV_COMPUTE_PROFILER_PERFWORKS_DIR", "CUDA_INJECTION64_PATH", "NV_TPS_LAUNCH_TOKEN",
                                        "NVIDIA_PROCESS_INJECTION_CRASH_REPORTING", "NSYS_PROFILING_SESSION_ID"};
    for (const char* m : marks) if (getenv(m)) return true;
    return false;
}

static int loop_graph(Wavefront& w, const WfParams& k, bool use_smem, Wavefront::LoopGraph* out) {
    // everything launch_iteration branches on (the launches themselves take no arguments)
    const Wavefront::GraphKey key(use_smem ? k.smem.total : 0u, use_smem ? 1 : 0, k.count_nodes != 0, k.has_media != 0, k.use_hrpp != 0,
                                  k.bvh1_index >= 0 ? 1 + k.bvh1_list_rects : 0, k.bvh1_tri_threads, k.list_threads, k.solo, k.solo_only, k.fused_generate, k.trace_pipeline,
                                  k.bvh1_q ? 1u + k.bvh1_q_smem : 0u);
    auto it = w.graphs.find(key);
    if (it != w.graphs.end()) { *out = it->second; return SHIM_OK; }
    if (!w.capture_stream) CU(cudaStreamCreateWithFlags(&w.capture_stream, cudaStreamNonBlocking));
    cudaGraph_t graph = nullptr;
    CU(cudaGraphCreate(&graph, 0));
    cudaGraphConditionalHandle handle;
    CU(cudaGraphConditionalHandleCreate(&handle, graph, 1, cudaGraphCondAssignDefault));
    cudaGraphNodeParams np = {};
    np.type = cudaGraphNodeTypeConditional;
    np.conditional.handle = handle;
    np.conditional.type = cudaGraphCondTypeWhile;
    np.conditional.size = 1;
    cudaGraphNode_t node;
    CU(cudaGraphAddNode(&node, graph, nullptr, 0, &np));
    cudaGraph_t body = np.conditional.phGraph_out[0];
    CU(cudaStreamBeginCaptureToGraph(w.capture_stream, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal));
    launch_iteration(w, k, use_smem, w.capture_stream);
    CU(cudaStreamEndCapture(w.capture_stream, nullptr));
    cudaGraphExec_t exec = nullptr;
    CU(cudaGraphInstantiate(&exec, graph, 0));
    CU(cudaGraphDestroy(graph));
    Wavefront::LoopGraph lg{exec, (unsigned long long)handle};
    w.graphs[key] = lg;
    *out = lg;
    return SHIM_OK;
}

static int check_render_params(const shim_scene* s, const shim_camera* cam, const shim_render_params* pp, const void* out) {
    if (!s->committed) return set_err(SHIM_ERR_STATE, "shim_render: scene not committed");
    if (!cam || !pp || !out) return set_err(SHIM_ERR_INVALID, "shim_render: null argument");
    const shim_render_params& p = *pp;
    if (p.width < 2 || p.height < 2 || p.samples_per_pixel < 1 || p.tile_width < 1 || p.tile_height < 1 || p.max_depth < 0 ||
        p.sample_count < -1 || p.sample_begin < 0 || (p.tile_world > 1 && (p.tile_rank < 0 || p.tile_rank >= p.tile_world)))
        return set_err(SHIM_ERR_INVALID, "shim_render: bad render params");
    if ((uint64_t)p.width * (uint64_t)p.height > 0x7fffffffull) return set_err(SHIM_ERR_INVALID, "shim_render: image too large");
    if (p.max_depth > 255) return set_err(SHIM_ERR_UNSUPPORTED, "shim_render: max_depth above 255 (the bounce is carried in 8 bits of the ray record)");
    if ((int64_t)p.sample_begin + (p.sample_count > 0 ? p.sample_count : p.samples_per_pixel) > (1 << 24))
        return set_err(SHIM_ERR_UNSUPPORTED, "shim_render: absolute sample index above 2^24 (carried in 24 bits of the ray record)");
    if ((p.flags & SHIM_RENDER_COUNT_NODES) && (p.flags & SHIM_RENDER_PREDICTORS) && s->dev->n_predictors > 0)
        return set_err(SHIM_ERR_INVALID, "shim_render: SHIM_RENDER_COUNT_NODES cannot be combined with SHIM_RENDER_PREDICTORS");
    return SHIM_OK;
}

// The render proper: device `w.device` is current, w.render_mutex is held, `ds` is the scene's copy on that device.
// Enqueues everything on `st`, waits for it, fills `stats`.
static int render_locked(shim_scene* s, DeviceScene& ds, Wavefront& w, const shim_camera* cam, const shim_render_params& p, float* d_out,
                         shim_stats* stats, cudaStream_t st) {
    int rc = wf_init(w, ds.device);
    if (rc < 0) return rc;
    const Switches sw;
    const size_t fb = (size_t)p.width * p.height * 3;
    CU(w.accum.reserve(fb));
    const int world = p.tile_world > 1 ? p.tile_world : 1;
    const int key[6] = {p.width, p.height, p.tile_width, p.tile_height, world > 1 ? p.tile_rank : 0, world};
    if (memcmp(key, w.pt_key, sizeof key) != 0) {
        std::vector<uint32_t> order = tile_pixel_order(p.width, p.height, p.tile_width, p.tile_height, key[4], world);
        memset(w.pt_key, 0, sizeof w.pt_key);
        CU(w.pix_table.upload(order));
        w.npix = (uint32_t)order.size();
        memcpy(w.pt_key, key, sizeof key);
    }

    WfParams k;
    memset(&k, 0, sizeof k);
    k.sv = ds.view;
    camera_new(cam->look_from, cam->look_at, cam->view_up, cam->vertical_fov, cam->aspect_ratio, cam->aperture, cam->focus_dist,
               cam->time_start, cam->time_end, k.cam);
    k.cnt = w.cnt.p; k.accum = w.accum.p; k.pix_table = w.pix_table.p;
    k.npix = w.npix;
    // sample_count: 0 = every sample of the image, -1 = none (a shard that owns no samples), n = that many from sample_begin
    const int count = p.sample_count > 0 ? p.sample_count : (p.sample_count < 0 ? 0 : p.samples_per_pixel);
    k.total_samples = (uint64_t)w.npix * (uint64_t)count;
    k.width = p.width; k.height = p.height; k.max_depth = p.max_depth; k.sample_begin = p.sample_begin;
    k.bg[0] = p.background[0]; k.bg[1] = p.background[1]; k.bg[2] = p.background[2];
    k.seed = p.seed; k.has_media = s->has_media ? 1 : 0; k.count_nodes = (p.flags & SHIM_RENDER_COUNT_NODES) ? 1 : 0;
    k.use_hrpp = ((p.flags & SHIM_RENDER_PREDICTORS) && s->dev->n_predictors > 0) ? 1 : 0;
    if (k.use_hrpp && !((p.flags & SHIM_RENDER_KEEP_PREDICTORS) && ds.hrpp_cleared)) {
        // a fresh Predictor per render (bvh.rs:69-81 builds them with the scene) unless the caller keeps them
        CU(cudaMemsetAsync(ds.hrpp_slots, 0xFF, ds.hrpp_slots_total * sizeof(HrppSlot), st));
        ds.hrpp_cleared = true;
    }
    bool use_smem = false;
    choose_variant(s, s->dev, w, sw, k, &use_smem);
    rc = wf_reserve(w, s->dev, p, sw, k);
    if (rc < 0) return rc;

    CU(cudaMemsetAsync(w.cnt.p, 0, CNT_WORDS * sizeof(uint32_t), st));
    CU(cudaMemsetAsync(w.accum.p, 0, fb * sizeof(float), st));
    CU(cudaEventRecord(w.ev0, st));

    const bool profile = (p.flags & SHIM_RENDER_PROFILE) != 0;
    size_t prof_used = 0;
    const size_t prof_cap = 4 * 1024;
    if (profile && w.prof.size() < prof_cap) {
        size_t have = w.prof.size();
        w.prof.resize(prof_cap);
        for (size_t i = have; i < prof_cap; ++i) CU(cudaEventCreate(&w.prof[i]));
    }
    k.max_iterations = 1u << 30;
    const bool run = k.total_samples > 0 && p.max_depth > 0;
    // Without per-kernel events the loop is ONE graph launch (WHILE node, condition set by wf_tail on the device).
    const bool use_graph = run && !profile && !sw.no_graph && !under_profiler();
    Wavefront::LoopGraph lg{nullptr, 0ull};
    if (use_graph) { int grc = loop_graph(w, k, use_smem, &lg); if (grc < 0) return grc; }
    k.loop_handle = lg.handle;
    CU(cudaMemcpyToSymbolAsync(g_p, &k, sizeof k, 0, cudaMemcpyHostToDevice, st));
    if (run && k.trace_pipeline) wf_trace_first<<<1, 32, 0, st>>>();   // counters of iteration 0 (later ones: wf_tail_mq)
    if (use_graph) {
        CU(cudaGraphLaunch(lg.exec, st));
    } else if (run) {
        // host-driven loop (profiling pass: CUDA events around every kernel): iterations are enqueued in chunks and the
        // done flag of chunk c is read back while chunk c+1 runs
        int pending = -1;
        bool done = false;
        for (int c = 0; !done; ++c) {
            for (int it = 0; it < SHIM_CHUNK; ++it) {
                const bool rec = profile && prof_used + 4 <= prof_cap;
                if (rec) CU(cudaEventRecord(w.prof[prof_used], st));
                if (!k.trace_pipeline) wf_generate<<<w.grid_generate, 256, 0, st>>>();
                if (rec) CU(cudaEventRecord(w.prof[prof_used + 1], st));
                if (k.trace_pipeline) launch_trace(w, k, st);
                else launch_extend(w, k, use_smem, st);
                if (rec) CU(cudaEventRecord(w.prof[prof_used + 2], st));
                if (k.trace_pipeline) launch_tail_mq(w, k, st);
                else { wf_shade<<<w.grid_shade, 256, 0, st>>>(); launch_tail(w, k, st); }
                if (rec) { CU(cudaEventRecord(w.prof[prof_used + 3], st)); prof_used += 4; }
            }
            int slot = c & 1;
            CU(cudaMemcpyAsync(w.h_flags + 16 * slot, w.cnt.p + CNT_DONE, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
            CU(cudaEventRecord(w.ev_chunk[slot], st));
            if (pending >= 0) {
                CU(cudaEventSynchronize(w.ev_chunk[pending]));
                if (w.h_flags[16 * pending]) done = true;
            }
            pending = slot;
            if (c > (1 << 24)) return set_err(SHIM_ERR_CUDA, "wavefront did not terminate");
        }
    }
    wf_finalize<<<w.sm_count * 4, 256, 0, st>>>(w.accum.p, d_out, fb, (float)p.samples_per_pixel, (p.flags & SHIM_RENDER_RAW_SUM) ? 1 : 0);
    CU(cudaEventRecord(w.ev1, st));
    CU(cudaMemcpyAsync(w.h_flags + 32, w.cnt.p, CNT_WORDS * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    if (stats) {
        memset(stats, 0, sizeof *stats);
        const uint64_t* c64 = reinterpret_cast<const uint64_t*>(w.h_flags + 32 + CNT_U64_BASE);
        stats->rays = c64[C64_RAYS];
        stats->samples = k.total_samples;
        stats->node_visits = c64[C64_NODES];
        stats->prim_tests = c64[C64_PRIMS];
        stats->hrpp_true_positive = c64[C64_HRPP_TP];
        stats->hrpp_false_positive = c64[C64_HRPP_FP];
        stats->hrpp_no_prediction = c64[C64_HRPP_NONE];
        stats->iterations = w.h_flags[32 + CNT_ITER];
        stats->extend_variant = k.trace_pipeline ? 4u : k.solo ? 2u : (k.list_threads ? 3u : (k.bvh1_index >= 0 ? 1u : 0u));
        // trace pipeline: wf_trace_first + two kernels per iteration body + wf_finalize; wavefront: four per body + wf_finalize
        // (the last body may find the queue already empty)
        stats->kernel_launches = !run ? 1ull : (k.trace_pipeline ? 2ull * w.h_flags[32 + CNT_BODIES] + 2ull
                                                                 : (k.bvh1_index >= 0 ? 6ull : 4ull) * w.h_flags[32 + CNT_BODIES] + 1ull);
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, w.ev0, w.ev1));
        stats->device_ms = ms;
        stats->pool_paths = k.pool;
        stats->pool_bytes = w.pool_bytes();
        stats->devices = 1;
        // per-launch durations of the closest-hit kernel while it had work: launches past the done flag are skipped
        uint64_t it_done = stats->iterations;
        for (size_t i = 0; i + 3 < prof_used && i / 4 < it_done; i += 4) {
            float g = 0, e = 0, sh = 0;
            CU(cudaEventElapsedTime(&g, w.prof[i], w.prof[i + 1]));
            CU(cudaEventElapsedTime(&e, w.prof[i + 1], w.prof[i + 2]));
            CU(cudaEventElapsedTime(&sh, w.prof[i + 2], w.prof[i + 3]));
            stats->generate_ms += g;
            stats->extend_ms += e;
            stats->shade_ms += sh;
            stats->extend_launches += 1;
            if (sw.trace) fprintf(stderr, "shim-trace iter %3zu generate %.4f extend %.4f shade %.4f ms\n", i / 4, g, e, sh);
        }
    }
    return SHIM_OK;
}

// the scene's copy on `device` (the current device), uploaded on first use
static int scene_on_device(shim_scene* s, int device, DeviceScene** out) {
    if (device < 0 || device >= SHIM_MAX_DEVICES) return set_err(SHIM_ERR_UNSUPPORTED, "device ordinal out of range");
    return upload_scene(s->dev, device, out);
}

SHIM_API int shim_render_device(shim_scene* s, const shim_camera* cam, const shim_render_params* pp, float* d_out, shim_stats* stats,
                                void* cuda_stream) {
    NEED(s);
    int rc = check_render_params(s, cam, pp, d_out);
    if (rc < 0) return rc;
    // the output buffer and the stream belong to the caller's current device: it has to be the one the scene lives on
    int cur_dev = -1;
    CU(cudaGetDevice(&cur_dev));
    if (cur_dev != s->dev->primary)
        return set_err(SHIM_ERR_STATE, "shim_render: the scene was committed on CUDA device " + std::to_string(s->dev->primary) +
                                           " but the current device is " + std::to_string(cur_dev));
    DeviceScene* ds = nullptr;
    rc = scene_on_device(s, cur_dev, &ds);
    if (rc < 0) return rc;
    Wavefront& w = g_wf[cur_dev];
    std::lock_guard<std::mutex> render_lock(w.render_mutex);   // before anything touches the shared pool
    return render_locked(s, *ds, w, cam, *pp, d_out, stats, (cudaStream_t)cuda_stream);
}

// device framebuffer -> caller's host buffer (with w.render_mutex held: the staging buffers are shared)
static int copy_out(Wavefront& w, const float* d_src, float* out, size_t fb, cudaStream_t st) {
    // a page-locked destination (shim_host_alloc, or memory the caller registered) takes the D2H directly
    bool pinned_out = false;
    {
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, out) == cudaSuccess) pinned_out = at.type == cudaMemoryTypeHost;
        else cudaGetLastError();
    }
    if (pinned_out) {
        CU(cudaMemcpyAsync(out, d_src, fb * sizeof(float), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        return SHIM_OK;
    }
    // otherwise: persistent pinned staging, no allocation on the per-call path
    if (w.h_out_n < fb) {
        if (w.h_out) cudaFreeHost(w.h_out);
        w.h_out = nullptr; w.h_out_n = 0;
        CU(cudaMallocHost(&w.h_out, fb * sizeof(float)));
        w.h_out_n = fb;
    }
    // D2H in chunks through the pinned staging buffer; the copy of chunk k into the caller's (pageable) buffer
    // overlaps the D2H of the chunks behind it
    const int chunks = 8;
    if (w.ev_d2h.empty()) { w.ev_d2h.resize(chunks); for (auto& e : w.ev_d2h) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming)); }
    const size_t per = (fb + chunks - 1) / chunks;
    for (int c = 0; c < chunks; ++c) {
        size_t off = (size_t)c * per, cnt = off < fb ? (fb - off < per ? fb - off : per) : 0;
        if (cnt) CU(cudaMemcpyAsync(w.h_out + off, d_src + off, cnt * sizeof(float), cudaMemcpyDeviceToHost, st));
        CU(cudaEventRecord(w.ev_d2h[c], st));
    }
    // two host threads copy alternate chunks out of the staging buffer as they land (a single memcpy of a 1200x800
    // framebuffer costs about as much as a quarter of the Book-1 render)
    cudaError_t err0 = cudaSuccess, err1 = cudaSuccess;
    auto drain = [&](int first, cudaError_t* err) {
        for (int c = first; c < chunks; c += 2) {
            size_t off = (size_t)c * per, cnt = off < fb ? (fb - off < per ? fb - off : per) : 0;
            cudaError_t e = cudaEventSynchronize(w.ev_d2h[c]);
            if (e != cudaSuccess) { *err = e; return; }
            if (cnt) memcpy(out + off, w.h_out + off, cnt * sizeof(float));
        }
    };
    {
        std::thread helper(drain, 1, &err1);
        drain(0, &err0);
        helper.join();
    }
    if (err0 != cudaSuccess || err1 != cudaSuccess)
        return set_err(SHIM_ERR_CUDA, std::string("framebuffer copy: ") + cudaGetErrorString(err0 != cudaSuccess ? err0 : err1));
    return SHIM_OK;
}

SHIM_API int shim_render(shim_scene* s, const shim_camera* cam, const shim_render_params* p, float* out, shim_stats* stats) {
    NEED(s);
    int rc = check_render_params(s, cam, p, out);
    if (rc < 0) return rc;
    const size_t fb = (size_t)p->width * p->height * 3;
    // host buffers in, host buffers out: the call runs on the scene's device whatever the caller's current device is
    DeviceGuard guard;
    CU(guard.enter(s->dev->primary));
    DeviceScene* ds = nullptr;
    rc = scene_on_device(s, s->dev->primary, &ds);
    if (rc < 0) return rc;
    Wavefront& w = g_wf[s->dev->primary];
    std::lock_guard<std::mutex> render_lock(w.render_mutex);   // held across the render AND the copy out of the shared d_out / staging
    CU(w.d_out.reserve(fb));
    const auto t0 = std::chrono::steady_clock::now();
    rc = render_locked(s, *ds, w, cam, *p, w.d_out.p, stats, nullptr);
    if (rc != SHIM_OK) return rc;
    rc = copy_out(w, w.d_out.p, out, fb, nullptr);
    if (stats) stats->wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    return rc;
}

// ------------------------------------------------------------------------------------------ one image on several devices
__global__ void wf_add_inplace(float* acc, const float* part, size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) acc[i] += part[i];
}
__global__ void wf_mean_inplace(float* acc, size_t n, float spp) {   // renderer.rs:147, the same division as wf_finalize
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) acc[i] = acc[i] / spp;
}

// Renderer::render's tile fan-out (renderer.rs:63-95) across devices instead of threads: the scene is replicated,
// device i renders its shard (a range of sample indices, or the tiles with index % n == i) with private accumulation
// on one host thread and one stream per device, and the raw sums are combined ONCE at the end on the first device
// (peer copies over NVLink + an add kernel) before the mean is taken and copied to the caller's host buffer.
SHIM_API int shim_render_multi(shim_scene* s, const shim_camera* cam, const shim_render_params* pp, int n_devices, const int* devices,
                               int mode, float* out, shim_stats* stats) {
    NEED(s);
    int rc = check_render_params(s, cam, pp, out);
    if (rc < 0) return rc;
    if (mode != SHIM_SHARD_SAMPLES && mode != SHIM_SHARD_TILES) return set_err(SHIM_ERR_INVALID, "shim_render_multi: mode must be SHIM_SHARD_SAMPLES or SHIM_SHARD_TILES");
    if (pp->tile_world > 1) return set_err(SHIM_ERR_INVALID, "shim_render_multi: the call shards the image itself (tile_world must be 0 or 1)");
    rc = device_count_or_error();
    if (rc < 0) return rc;
    const int have = rc;
    if (n_devices <= 0) n_devices = have;
    if (n_devices > have || n_devices > SHIM_MAX_DEVICES) return set_err(SHIM_ERR_INVALID, "shim_render_multi: more devices requested than present");
    std::vector<int> dev(n_devices);
    for (int i = 0; i < n_devices; ++i) {
        dev[i] = devices ? devices[i] : i;
        if (dev[i] < 0 || dev[i] >= have) return set_err(SHIM_ERR_INVALID, "shim_render_multi: bad device ordinal");
        for (int j = 0; j < i; ++j) if (dev[j] == dev[i]) return set_err(SHIM_ERR_INVALID, "shim_render_multi: device listed twice");
    }
    const shim_render_params& p = *pp;
    const size_t fb = (size_t)p.width * p.height * 3;
    const int total = p.sample_count > 0 ? p.sample_count : (p.sample_count < 0 ? 0 : p.samples_per_pixel);

    // one multi-device render at a time: each holds several devices' pools until its combine, and two of them taking
    // the same pools in different orders would wait for each other forever
    static std::mutex multi_mutex;
    std::lock_guard<std::mutex> multi_lock(multi_mutex);
    struct Part { int rc = SHIM_OK; std::string err; shim_stats st; bool rendered = false; };
    std::vector<Part> part(n_devices);
    // every device's pool stays locked from its render until the combine has read its sums
    std::vector<std::unique_lock<std::mutex>> locks(n_devices);
    auto t0 = std::chrono::steady_clock::now();
    auto work = [&](int i) {
        Part& me = part[i];
        memset(&me.st, 0, sizeof me.st);
        auto fail = [&](int code) { me.rc = code; me.err = shim_last_error(); };
        if (cudaSetDevice(dev[i]) != cudaSuccess) { me.rc = set_err(SHIM_ERR_CUDA, "cudaSetDevice failed"); me.err = shim_last_error(); return; }
        shim_render_params q = p;
        q.flags |= SHIM_RENDER_RAW_SUM;
        if (mode == SHIM_SHARD_SAMPLES) {   // contiguous ranges of absolute sample indices, the remainder to the first devices
            const int base = total / n_devices, rem = total % n_devices;
            const int cnt = base + (i < rem ? 1 : 0);
            q.sample_begin = p.sample_begin + i * base + (i < rem ? i : rem);
            q.sample_count = cnt > 0 ? cnt : -1;
        } else {
            q.tile_rank = i; q.tile_world = n_devices;
            q.sample_count = total > 0 ? total : -1;
        }
        DeviceScene* ds = nullptr;
        int r = scene_on_device(s, dev[i], &ds);
        if (r < 0) return fail(r);
        Wavefront& w = g_wf[dev[i]];
        locks[i] = std::unique_lock<std::mutex>(w.render_mutex);
        if (!w.work_stream && cudaStreamCreateWithFlags(&w.work_stream, cudaStreamNonBlocking) != cudaSuccess) {
            me.rc = set_err(SHIM_ERR_CUDA, "cudaStreamCreate failed"); me.err = shim_last_error(); return;
        }
        if (w.d_out.reserve(fb) != cudaSuccess) { me.rc = set_err(SHIM_ERR_CUDA, "framebuffer allocation failed"); me.err = shim_last_error(); return; }
        if (i == 0 && n_devices > 1 && w.d_peer.reserve(fb) != cudaSuccess) { me.rc = set_err(SHIM_ERR_CUDA, "peer buffer allocation failed"); me.err = shim_last_error(); return; }
        r = render_locked(s, *ds, w, cam, q, w.d_out.p, &me.st, w.work_stream);
        if (r < 0) return fail(r);
        me.rendered = true;
    };
    {
        std::vector<std::thread> th;
        for (int i = 1; i < n_devices; ++i) th.emplace_back(work, i);
        DeviceGuard guard;   // the calling thread renders on the first device and gets its own device back afterwards
        cudaError_t ge = guard.enter(dev[0]);
        if (ge == cudaSuccess) work(0); else { part[0].rc = set_err(SHIM_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(ge)); part[0].err = shim_last_error(); }
        for (auto& t : th) t.join();
        for (int i = 0; i < n_devices; ++i) if (part[i].rc < 0) { locks.clear(); return set_err(part[i].rc, "device " + std::to_string(dev[i]) + ": " + part[i].err); }
        // ---- the one combine: peer copy of every other device's sums onto the first device, add, mean, copy out
        Wavefront& w0 = g_wf[dev[0]];
        cudaStream_t st0 = w0.work_stream;
        for (int i = 1; i < n_devices; ++i) {
            Wavefront& wi = g_wf[dev[i]];
            int can = 0;   // direct NVLink copies where the devices can reach each other (the copy is staged through the host otherwise)
            if (cudaDeviceCanAccessPeer(&can, dev[0], dev[i]) == cudaSuccess && can) {
                cudaError_t pe = cudaDeviceEnablePeerAccess(dev[i], 0);
                if (pe != cudaSuccess) cudaGetLastError();   // already enabled
            }
            CU(cudaMemcpyPeerAsync(w0.d_peer.p, dev[0], wi.d_out.p, dev[i], fb * sizeof(float), st0));
            wf_add_inplace<<<w0.sm_count * 4, 256, 0, st0>>>(w0.d_out.p, w0.d_peer.p, fb);
        }
        if (!(p.flags & SHIM_RENDER_RAW_SUM)) wf_mean_inplace<<<w0.sm_count * 4, 256, 0, st0>>>(w0.d_out.p, fb, (float)p.samples_per_pixel);
        CU(cudaGetLastError());
        rc = copy_out(w0, w0.d_out.p, out, fb, st0);
        locks.clear();
        if (rc < 0) return rc;
    }
    if (stats) {
        memset(stats, 0, sizeof *stats);
        for (int i = 0; i < n_devices; ++i) {
            const shim_stats& a = part[i].st;
            stats->rays += a.rays; stats->samples += a.samples; stats->node_visits += a.node_visits; stats->prim_tests += a.prim_tests;
            stats->hrpp_true_positive += a.hrpp_true_positive; stats->hrpp_false_positive += a.hrpp_false_positive;
            stats->hrpp_no_prediction += a.hrpp_no_prediction; stats->kernel_launches += a.kernel_launches;
            if (a.iterations > stats->iterations) stats->iterations = a.iterations;
            if (a.device_ms > stats->device_ms) stats->device_ms = a.device_ms;   // the slowest device's loop
            stats->pool_bytes += a.pool_bytes;
            if (a.pool_paths > stats->pool_paths) stats->pool_paths = a.pool_paths;
            stats->extend_variant = a.extend_variant;
        }
        stats->kernel_launches += (uint64_t)(n_devices - 1) + ((p.flags & SHIM_RENDER_RAW_SUM) ? 0u : 1u);
        stats->devices = (uint64_t)n_devices;
        stats->wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
    return SHIM_OK;
}

// frees every device's pool, graphs, events and staging buffers (scenes keep their own arrays until shim_scene_destroy).
// No render may be in flight.
SHIM_API int shim_shutdown(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return SHIM_OK; }
    for (int d = 0; d < n && d < SHIM_MAX_DEVICES; ++d) {
        Wavefront& w = g_wf[d];
        std::lock_guard<std::mutex> lock(w.render_mutex);
        if (!w.ready && !w.d_out.p && !w.h_out) continue;
        DeviceGuard g;
        if (g.enter(d) != cudaSuccess) continue;
        cudaDeviceSynchronize();
        w.release();
    }
    return SHIM_OK;
}

SHIM_API uint64_t shim_pool_bytes(int device) {
    if (device < 0 || device >= SHIM_MAX_DEVICES) return 0;
    Wavefront& w = g_wf[device];
    std::lock_guard<std::mutex> lock(w.render_mutex);
    return (uint64_t)w.pool_bytes();
}

SHIM_API float* shim_host_alloc(size_t floats) {
    float* p = nullptr;
    if (cudaMallocHost(&p, (floats ? floats : 1) * sizeof(float)) != cudaSuccess) {
        set_err(SHIM_ERR_CUDA, std::string("shim_host_alloc: ") + cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    return p;
}
SHIM_API void shim_host_free(float* p) { if (p) cudaFreeHost(p); }

// ------------------------------------------------------------------------------------------ gate 1
// Blocks of `threads` for n rays, at most sm_count * 8 blocks' worth of 256 threads; the kernels' grid-stride loops
// take the rest.
static int trace_grid(const DeviceScene& ds, int64_t n, int threads) {
    int64_t grid = (n + threads - 1) / threads;
    int64_t cap = (int64_t)ds.sm_count * 8 * 256 / threads;
    return (int)(grid > cap ? cap : grid);
}

// The checks every batch query makes first, in this order: a scene, committed, n >= 0 and, for n > 0, its arrays.
static int trace_check(shim_scene* s, const char* fn, int64_t n, bool have_arrays) {
    NEED(s);
    if (!s->committed) return set_err(SHIM_ERR_STATE, std::string(fn) + ": scene not committed");
    if (n < 0 || (n > 0 && !have_arrays)) return set_err(SHIM_ERR_INVALID, std::string(fn) + ": bad arguments");
    return SHIM_OK;
}

// The device variants: the caller's arrays and stream on the scene's device, which must be current; no counters.
// launch(ds) enqueues the kernel.
template <class Launch>
static int trace_device(shim_scene* s, const char* fn, int64_t n, Launch launch) {
    if (n == 0) return SHIM_OK;
    int cur_dev = -1;
    CU(cudaGetDevice(&cur_dev));
    if (cur_dev != s->dev->primary) return set_err(SHIM_ERR_STATE, std::string(fn) + ": the scene lives on another CUDA device");
    DeviceScene* ds = nullptr;
    int rc = scene_on_device(s, cur_dev, &ds);
    if (rc < 0) return rc;
    launch(*ds);
    CU(cudaGetLastError());
    return SHIM_OK;
}

// The host variants: the rays staged on the scene's device in one allocation with the outputs and the counters, the
// kernel run on the legacy default stream, then each output array and the counters copied back.
// launch(ds, d_rays, d_out, d_cnt) enqueues the kernel; d_out[k] holds n * out[k].bytes bytes, 16-byte aligned.
struct HostOut { void* p; size_t bytes; };   // one output array and its bytes per ray
template <int K, class Launch>
static int trace_host(shim_scene* s, const float* rays, int64_t n, const HostOut (&out)[K], uint64_t* counters, Launch launch) {
    if (n == 0) { if (counters) counters[0] = counters[1] = counters[2] = 0; return SHIM_OK; }
    DeviceGuard guard;
    CU(guard.enter(s->dev->primary));
    DeviceScene* ds = nullptr;
    int rc = scene_on_device(s, s->dev->primary, &ds);
    if (rc < 0) return rc;
    // the counters, each output array, the rays
    size_t off[K + 1], total = 4 * sizeof(unsigned long long);
    for (int k = 0; k < K; ++k) { off[k] = total; total += ((size_t)n * out[k].bytes + 15) & ~(size_t)15; }
    off[K] = total; total += (size_t)n * 7 * sizeof(float);
    char* base = nullptr;
    CU(cudaMalloc(&base, total));
    std::unique_ptr<char, cudaError_t (*)(void*)> staging(base, cudaFree);
    unsigned long long* d_cnt = (unsigned long long*)base;
    float* d_rays = (float*)(base + off[K]);
    void* d_out[K];
    for (int k = 0; k < K; ++k) d_out[k] = base + off[k];
    CU(cudaMemset(d_cnt, 0, 3 * sizeof(unsigned long long)));
    CU(cudaMemcpy(d_rays, rays, (size_t)n * 7 * sizeof(float), cudaMemcpyHostToDevice));
    launch(*ds, d_rays, d_out, counters ? d_cnt : nullptr);
    CU(cudaGetLastError());
    for (int k = 0; k < K; ++k) CU(cudaMemcpy(out[k].p, d_out[k], (size_t)n * out[k].bytes, cudaMemcpyDeviceToHost));
    if (counters) {
        unsigned long long h[3];
        CU(cudaMemcpy(h, d_cnt, sizeof h, cudaMemcpyDeviceToHost));
        counters[0] = (uint64_t)n; counters[1] = h[1]; counters[2] = h[2];
    }
    return SHIM_OK;
}

SHIM_API int shim_trace_closest_device(shim_scene* s, const float* d_rays, int64_t n, float t_min, float t_max, uint64_t seed,
                                       int32_t* d_prim, float* d_t, void* cuda_stream) {
    int rc = trace_check(s, "shim_trace_closest", n, d_rays && d_prim && d_t);
    if (rc < 0) return rc;
    return trace_device(s, "shim_trace_closest", n, [&](const DeviceScene& ds) {
        trace_closest_kernel<<<trace_grid(ds, n, 256), 256, 0, (cudaStream_t)cuda_stream>>>(ds.view, d_rays, (long long)n, t_min, t_max, seed,
                                                                                             d_prim, d_t, nullptr);
    });
}

SHIM_API int shim_trace_closest(shim_scene* s, const float* rays, int64_t n, float t_min, float t_max, uint64_t seed, int32_t* prim,
                                float* t, uint64_t* counters) {
    int rc = trace_check(s, "shim_trace_closest", n, rays && prim && t);
    if (rc < 0) return rc;
    return trace_host(s, rays, n, {{prim, sizeof *prim}, {t, sizeof *t}}, counters,
                      [&](const DeviceScene& ds, const float* d_rays, void* const* d_out, unsigned long long* d_cnt) {
        trace_closest_kernel<<<trace_grid(ds, n, 256), 256>>>(ds.view, d_rays, (long long)n, t_min, t_max, seed, (int32_t*)d_out[0],
                                                              (float*)d_out[1], d_cnt);
    });
}

static_assert(sizeof(shim_hit_record) == 3 * sizeof(f4), "shim_hit_record is three 16-byte words");

SHIM_API int shim_trace_hit_device(shim_scene* s, const float* d_rays, int64_t n, float t_min, float t_max, uint64_t seed,
                                   shim_hit_record* d_out, void* cuda_stream) {
    int rc = trace_check(s, "shim_trace_hit", n, d_rays && d_out);
    if (rc < 0) return rc;
    if (((uintptr_t)d_out & 15) != 0) return set_err(SHIM_ERR_INVALID, "shim_trace_hit: d_out is not 16-byte aligned");
    return trace_device(s, "shim_trace_hit", n, [&](const DeviceScene& ds) {
        trace_hit_kernel<<<trace_grid(ds, n, SHIM_TRACE_HIT_THREADS), SHIM_TRACE_HIT_THREADS, 0, (cudaStream_t)cuda_stream>>>(
            ds.view, d_rays, (long long)n, t_min, t_max, seed, (f4*)d_out, nullptr);
    });
}

SHIM_API int shim_trace_hit(shim_scene* s, const float* rays, int64_t n, float t_min, float t_max, uint64_t seed, shim_hit_record* out,
                            uint64_t* counters) {
    int rc = trace_check(s, "shim_trace_hit", n, rays && out);
    if (rc < 0) return rc;
    return trace_host(s, rays, n, {{out, sizeof *out}}, counters,
                      [&](const DeviceScene& ds, const float* d_rays, void* const* d_out, unsigned long long* d_cnt) {
        trace_hit_kernel<<<trace_grid(ds, n, SHIM_TRACE_HIT_THREADS), SHIM_TRACE_HIT_THREADS>>>(ds.view, d_rays, (long long)n, t_min, t_max,
                                                                                                 seed, (f4*)d_out[0], d_cnt);
    });
}

SHIM_API int shim_trace_occluded_device(shim_scene* s, const float* d_rays, int64_t n, float t_min, float t_max, uint64_t seed,
                                        uint8_t* d_occluded, void* cuda_stream) {
    int rc = trace_check(s, "shim_trace_occluded", n, d_rays && d_occluded);
    if (rc < 0) return rc;
    return trace_device(s, "shim_trace_occluded", n, [&](const DeviceScene& ds) {
        trace_occluded_kernel<<<trace_grid(ds, n, SHIM_TRACE_OCCLUDED_THREADS), SHIM_TRACE_OCCLUDED_THREADS, 0, (cudaStream_t)cuda_stream>>>(
            ds.view, d_rays, (long long)n, t_min, t_max, seed, d_occluded, nullptr);
    });
}

SHIM_API int shim_trace_occluded(shim_scene* s, const float* rays, int64_t n, float t_min, float t_max, uint64_t seed, uint8_t* occluded,
                                 uint64_t* counters) {
    int rc = trace_check(s, "shim_trace_occluded", n, rays && occluded);
    if (rc < 0) return rc;
    return trace_host(s, rays, n, {{occluded, sizeof *occluded}}, counters,
                      [&](const DeviceScene& ds, const float* d_rays, void* const* d_out, unsigned long long* d_cnt) {
        trace_occluded_kernel<<<trace_grid(ds, n, SHIM_TRACE_OCCLUDED_THREADS), SHIM_TRACE_OCCLUDED_THREADS>>>(
            ds.view, d_rays, (long long)n, t_min, t_max, seed, (uint8_t*)d_out[0], d_cnt);
    });
}
