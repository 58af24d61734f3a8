// shim_kernels.cuh — sm_100a wavefront kernels.
//
// One iteration of the wavefront (replaces the per-tile loop of renderer.rs:63-85 and the
// recursion of ray.rs:32-62) is four launches:
//
//   wf_generate  tops the current ray queue up with camera rays for new samples
//                (renderer.rs:141-143, camera.rs:96-106); the last block to finish advances the
//                device-side counters for the iteration
//   wf_extend    closest hit for every queued ray (hittable.rs:100-118).  The BVH nodes and
//                primitive arrays are staged into shared memory by TMA bulk copies
//                (cp.async.bulk + mbarrier) when they fit, so the walk's 16-byte node fetches
//                are LDS; misses add the background on the spot; a hit appends the ray and its
//                hit record to the queue of its material kind (warp match.any: one atomic per
//                group of lanes that hit the same kind)
//   wf_shade     material-sorted shading, one launch covering the five material queues: each
//                256-ray chunk of a queue is streamed (coalesced) through code specialised for
//                that material: rebuild the HitRecord, emit, scatter, and append the continuing
//                ray to the next ray queue (warp-ballot compaction, one atomic per warp)
//                (wf_extend_solo / wf_extend_list: the same walk with what a
//                scene cannot need compiled out - fewer registers, more resident warps;
//                wf_trace_solo: shade + walk in one kernel, material queue to material queue)
//   wf_tail      once no samples are left to start and at most 65536 paths are alive, one
//                launch finishes them (extend + shade in a loop per thread) instead of ~35
//                near-empty iterations; it also decides whether the loop goes on
//
// Ray queues are SoA float4 streams in HBM, double buffered; all counts, the queue index and
// the termination test live on the device: the iteration is the body of a CUDA-graph WHILE
// node, so the host launches one graph per render and never polls.
#pragma once
#include <cuda_runtime.h>
#include "shim_device.h"

namespace shim {

enum { CNT_NRAYS0 = 0, CNT_NRAYS1 = 1, CNT_MQ = 2 /* ..7: one per shading class */, CNT_CUR = 8, CNT_TICKET = 9, CNT_NEXT_CUR = 10, CNT_DONE = 11, CNT_ITER = 12,
       CNT_BODIES = 13 /* iteration bodies executed */, CNT_GEN_BASE = 14 /* fused generation: queue slot of the first new sample */,
       CNT_GEN_N = 15 /* new samples of this iteration */, CNT_U64_BASE = 16 /* u64 slots from here, as pairs: ..31 */,
       CNT_TREEQ = 32 /* one-Bvh worlds: rays queued for the tree walk */, CNT_TREEQ_NEXT = 33 /* ... handed out */,
       CNT_MQ1 = 34 /* ..39: second material-queue counter set (wf_trace pipeline) */ };
enum { C64_NEXT_SAMPLE = 0, C64_RAYS = 1, C64_NODES = 2, C64_PRIMS = 3, C64_HRPP_TP = 4, C64_HRPP_FP = 5, C64_HRPP_NONE = 6, C64_GEN_FIRST = 7, C64_COUNT = 8 };
enum { CNT_WORDS = 40 };
static_assert(CNT_MQ + MQ_CLASSES <= CNT_CUR && CNT_U64_BASE + 2 * C64_COUNT <= CNT_TREEQ && CNT_MQ1 + MQ_CLASSES <= CNT_WORDS, "counter layout");

// shared-memory image of the scene arrays wf_extend walks (byte offsets, all multiples of 16)
struct SmemLayout {
    uint32_t off_nodes, off_sph, off_msph, off_rect, off_tri, off_cube, off_objects, off_sph_mat;
    uint32_t bytes_nodes, bytes_sph, bytes_msph, bytes_rect, bytes_tri, bytes_cube, bytes_objects, bytes_sph_mat;
    uint32_t total;  // 0 = scene does not fit: walk it in global memory (L2)
    uint32_t signed_nodes;  // the node region holds SNodes (sv.snodes): layout of the one-Bvh kernels
};

struct WfParams {
    SceneView sv;
    CameraPod cam;
    // ray queues (double buffered)
    f4* ray_o[2];   // origin.xyz, time
    f4* ray_d[2];   // direction.xyz, bounce | sample << 8 (int bits)
    f4* thr[2];     // throughput.rgb, pixel index (int bits)
    // material queues carry the payload.  A set is mq_set_stride entries; two material kinds share one pool-sized
    // region of it, one growing up from the region's first entry and one down from its last (their counts sum to
    // at most `pool`), and only the kinds the scene has get a region: entry j of kind k is mq_first[k] + mq_dir[k] * j
    f4* mq_o; f4* mq_d; f4* mq_thr;
    f4* mq_hit;     // t, obj | face << 16, prim_ref, material
    long long mq_first[MQ_CLASSES];
    int mq_dir[MQ_CLASSES];
    long long mq_set_stride;
    uint32_t* cnt;
    float* accum;   // W*H*3 radiance sums
    const uint32_t* pix_table;
    uint32_t npix;            // pixels rendered by this call (tile shard)
    uint64_t total_samples;   // npix * sample_count
    uint32_t pool;
    uint32_t tail_threshold;
    int width, height, max_depth, sample_begin;
    float bg[3];
    uint64_t seed;
    int has_media, count_nodes, use_hrpp;
    int bvh1_list_rects;    // the plain objects next to the one Bvh are untransformed rects, at most SHIM_BVH1_LIST_RECTS of them
    int bvh1_tri_threads;   // > 0: the one Bvh holds only triangles: wf_bvh1_walk<.., THREADS, PT_TRI>
    int list_threads; // > 0: the world has no Bvh: wf_extend_list with this many threads per block
    int trace_pipeline;   // the iteration is wf_trace (shade -> closest hit) + wf_tail_mq (endgame, loop condition, next counters); no ray queues
    int fused_generate;   // wf_generate only publishes the counters; wf_extend_solo makes the camera rays itself
    int solo_only;    // wf_extend_solo: the one primitive type of the Bvh (PT_*), or -1 when mixed
    int solo;         // > 0: the world is exactly one plain Bvh: wf_extend_solo with this many threads per block
    int bvh1_index;   // >= 0: the world is one BVH object (this one) among plain primitives, no medium: the wf_bvh1_* kernels apply
    uint32_t bvh1_q_smem;  // wf_bvh1_walk on quantised nodes (sv.qnodes): how many of them (the top of the tree) sit in shared memory; 0 with bvh1_q = 0
    int bvh1_q;            // the mesh walk uses the QNode layout
    i4* bvh1_hit;          // one-Bvh worlds: closest-hit record per queued ray (wf_bvh1_list / _walk / _finish)
    uint32_t* bvh1_queue;  // ... rays that can reach the tree
    SmemLayout smem;
    unsigned long long loop_handle;   // conditional handle of the CUDA-graph WHILE node the iteration runs in (0: host-driven loop)
    uint32_t max_iterations;          // safety stop of the device-side loop
};

// The parameters of the render in flight live in constant memory (one render per device at a time) and the index of
// the current ray queue lives in the counters (wf_generate's last block flips it), so the wavefront kernels take no
// arguments: one iteration is the body of a CUDA-graph WHILE node whose condition wf_tail sets on the device.
__constant__ WfParams g_p;

__device__ __forceinline__ unsigned long long* cnt64(uint32_t* cnt, int slot) {
    return reinterpret_cast<unsigned long long*>(cnt + CNT_U64_BASE) + slot;
}

// wf_trace pipeline: two material-queue sets (set s: counters mq_counts(p, s), entry j of kind k at mq_slot(p, s, k, j))
__device__ __forceinline__ uint32_t* mq_counts(const WfParams& p, int set) { return p.cnt + (set ? CNT_MQ1 : CNT_MQ); }
__device__ __forceinline__ size_t mq_slot(const WfParams& p, int set, int kind, uint32_t j) {
    return (size_t)((long long)set * p.mq_set_stride + p.mq_first[kind] + (long long)p.mq_dir[kind] * (long long)j);
}

// position for this lane in a queue, one atomic per warp; all 32 lanes must call it
__device__ __forceinline__ uint32_t warp_append(uint32_t* counter, bool pred) {
    unsigned mask = __ballot_sync(0xffffffffu, pred);
    if (mask == 0) return 0;
    int lane = threadIdx.x & 31;
    int leader = __ffs(mask) - 1;
    uint32_t base = 0;
    if (lane == leader) base = atomicAdd(counter, (uint32_t)__popc(mask));
    base = __shfl_sync(0xffffffffu, base, leader);
    return base + (uint32_t)__popc(mask & ((1u << lane) - 1u));
}

// Block-wide appends for the streaming kernels (256-thread blocks, several per SM).  One atomic per warp and queue on
// a handful of global counters was what these kernels waited for (ncu: 57 % of wf_bvh1_list's and 45 % of
// wf_bvh1_finish's stall samples sat on the shuffle that distributes the atomic's result - the counters saw one
// request every 2-3 cycles); here the warps add up in shared memory and one thread per queue asks for the block's slots.
// Every thread of the block must call (two barriers).  s_cnt must be zero on entry and is zero again on return.
enum { APPEND_TREEQ = MQ_CLASSES, APPEND_SLOTS = MQ_CLASSES + 1, APPEND_NONE = APPEND_SLOTS };
// slot: a material class (append to its queue of set 0), APPEND_TREEQ (the mesh walk's ray queue) or APPEND_NONE
__device__ __forceinline__ uint32_t block_append_slots(const WfParams& p, int slot, uint32_t* s_cnt, uint32_t* s_base) {
    const uint32_t lane = threadIdx.x & 31u;
    const unsigned grp = __match_any_sync(0xffffffffu, slot);
    const int leader = __ffs(grp) - 1;
    uint32_t woff = 0;
    if (slot < APPEND_SLOTS && (int)lane == leader) woff = atomicAdd(s_cnt + slot, (uint32_t)__popc(grp));
    __syncthreads();
    if (threadIdx.x < APPEND_SLOTS) {
        const uint32_t c = s_cnt[threadIdx.x];
        s_base[threadIdx.x] = c ? atomicAdd(threadIdx.x == APPEND_TREEQ ? p.cnt + CNT_TREEQ : p.cnt + CNT_MQ + threadIdx.x, c) : 0u;
        s_cnt[threadIdx.x] = 0;
    }
    __syncthreads();
    if (slot >= APPEND_SLOTS) return 0;
    woff = __shfl_sync(grp, woff, leader);
    return s_base[slot] + woff + (uint32_t)__popc(grp & ((1u << lane) - 1u));
}
// ---------------------------------------------------------------------------- TMA bulk copy helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// the ray record of global sample index g (renderer.rs:140-146): pixel from the tile-ordered table, Philox stage 0
__device__ __forceinline__ void camera_ray_record(const WfParams& p, unsigned long long g, f4& o, f4& d, f4& t) {
    uint32_t s, pi;
    if (p.total_samples <= 0xffffffffull) { s = (uint32_t)g / p.npix; pi = (uint32_t)g - s * p.npix; }   // 32-bit divide when it fits
    else { s = (uint32_t)(g / p.npix); pi = (uint32_t)(g - (unsigned long long)s * p.npix); }
    const uint32_t pixel = p.pix_table[pi];
    const int x = (int)(pixel % (uint32_t)p.width), y = (int)(pixel / (uint32_t)p.width);
    const uint32_t sample = (uint32_t)p.sample_begin + s;
    Rng rng;
    rng_init(rng, pixel, sample, p.seed);
    rng_key(rng, 0, STAGE_CAMERA);
    const Ray r = camera_sample(p.cam, x, y, p.width, p.height, rng);
    o.x = r.o.x; o.y = r.o.y; o.z = r.o.z; o.w = r.time;
    d.x = r.d.x; d.y = r.d.y; d.z = r.d.z; d.w = i2f((int)(sample << 8));
    t.x = 1.0f; t.y = 1.0f; t.z = 1.0f; t.w = i2f((int)pixel);
}

// ---------------------------------------------------------------------------- generate
// All blocks read the pre-iteration counters, write their camera rays, and the last block to
// finish (ticket) publishes the counters the rest of the iteration uses.
__global__ void __launch_bounds__(256) wf_generate() {
    const WfParams& p = g_p;
    uint32_t* c = p.cnt;
    const int cur = (int)c[CNT_NEXT_CUR];
    const uint32_t n_cur = c[cur];
    const unsigned long long first = *cnt64(c, C64_NEXT_SAMPLE);
    const unsigned long long remaining = p.total_samples - first;
    const unsigned long long room = (unsigned long long)(p.pool - n_cur);
    const uint32_t n = (uint32_t)(remaining < room ? remaining : room);
    if (!p.fused_generate) {
        for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) {
            f4 o, d, t;
            camera_ray_record(p, first + j, o, d, t);
            const uint32_t slot = n_cur + j;
            p.ray_o[cur][slot] = o;
            p.ray_d[cur][slot] = d;
            p.thr[cur][slot] = t;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        uint32_t ticket = atomicAdd(c + CNT_TICKET, 1u);
        if (ticket == gridDim.x - 1) {  // every block has read the old counters: publish the new ones
            c[CNT_TICKET] = 0;
            c[CNT_CUR] = (uint32_t)cur;            // the queue the rest of this iteration works on
            c[CNT_NEXT_CUR] = (uint32_t)(1 - cur);
            *cnt64(c, C64_NEXT_SAMPLE) = first + n;
            c[CNT_GEN_BASE] = n_cur;               // fused generation: queue slots n_cur .. n_cur + n - 1 are samples first ..
            *cnt64(c, C64_GEN_FIRST) = first;
            c[cur] = n_cur + n;
            c[1 - cur] = 0;
#pragma unroll
            for (int k = 0; k < MQ_CLASSES; ++k) c[CNT_MQ + k] = 0;
            c[CNT_TREEQ] = 0; c[CNT_TREEQ_NEXT] = 0;
            *cnt64(c, C64_RAYS) += (unsigned long long)(n_cur + n);
            c[CNT_ITER] += (n_cur + n == 0) ? 0u : 1u;
            c[CNT_BODIES] += 1u;
            __threadfence();
        }
    }
}

// ---------------------------------------------------------------------------- extend
template <bool COUNT, bool MEDIA, bool HRPP, bool SOLO = false, int ONLY = -1, bool HASBVH = true, bool FUSE = false>
__device__ __forceinline__ void extend_rays(const WfParams& p, const SceneView& sv, int cur, uint32_t n) {
    const uint32_t n_round = (n + 31u) & ~31u;
    // FUSE: queue slots from gen_base on are new samples whose camera rays are made here instead of being written by
    // wf_generate and read back (96 B of HBM traffic per sample)
    const uint32_t gen_base = FUSE ? p.cnt[CNT_GEN_BASE] : 0xffffffffu;
    const unsigned long long gen_first = FUSE ? *cnt64(p.cnt, C64_GEN_FIRST) : 0ull;
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t nodes = 0, prims = 0, h_tp = 0, h_fp = 0, h_none = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += gridDim.x * blockDim.x) {
        int kind = 7;
        f4 o, d, t, hv;
        if (i < n) {
            if (FUSE && i >= gen_base) camera_ray_record(p, gen_first + (i - gen_base), o, d, t);
            else { o = p.ray_o[cur][i]; d = p.ray_d[cur][i]; t = p.thr[cur][i]; }
            Ray r; r.o = mk3(o.x, o.y, o.z); r.d = mk3(d.x, d.y, d.z); r.time = o.w;
            // A ray with a NaN component (born as t = 0/0 in a rect test, rectangle.rs:44, when a ray starts on the
            // rect's plane with an exactly zero direction component) fails no comparison: in the reference it "hits"
            // the last object of the world list with t = NaN on every bounce until the depth limit and contributes
            // nothing, while passing every bounding box on the way.  It is dropped here instead of walking the
            // whole tree 50 times.
            const bool poisoned = ray_has_nan(r);
            Rng rng;
            if (MEDIA) {
                uint32_t bs = (uint32_t)f2i(d.w);
                rng_init(rng, (uint32_t)f2i(t.w), bs >> 8, p.seed);
                rng_key(rng, bs & 255u, STAGE_INTERSECT);
            } else {
                rng_init(rng, 0, 0, 0);
            }
            TraceCounters tc; tc.nodes = 0; tc.prims = 0; tc.hrpp_tp = 0; tc.hrpp_fp = 0; tc.hrpp_none = 0;
            Hit h; h.obj = -1; h.t = 0; h.prim = 0; h.face = 0;
            if (!poisoned) h = SOLO ? closest_hit_solo<COUNT, ONLY, true>(sv, r, 0.001f, SHIM_INF, &tc) : closest_hit<COUNT, HRPP, HASBVH>(sv, r, 0.001f, SHIM_INF, rng, &tc);
            nodes += tc.nodes; prims += tc.prims; h_tp += tc.hrpp_tp; h_fp += tc.hrpp_fp; h_none += tc.hrpp_none;
            if (poisoned) {
                // path ends without a contribution
            } else if (h.obj < 0) {  // ray.rs:60: miss returns the background
                if (p.bg[0] != 0.0f || p.bg[1] != 0.0f || p.bg[2] != 0.0f) {
                    float* a = p.accum + 3 * (size_t)(uint32_t)f2i(t.w);
                    atomicAdd(a + 0, t.x * p.bg[0]);
                    atomicAdd(a + 1, t.y * p.bg[1]);
                    atomicAdd(a + 2, t.z * p.bg[2]);
                }
            } else {
                const int mw = (SOLO && ONLY == PT_SPHERE) ? sv.sph_mat[prim_index(h.prim)] : hit_material_word(sv, h);
                const int mat = mat_word_index(mw);
                kind = mat_word_kind(mw);
                hv.x = h.t; hv.y = i2f(h.obj | (h.face << 16)); hv.z = i2f((int)h.prim); hv.w = i2f(mat);
            }
        }
        // append to the material queue: lanes that hit the same kind share one atomic
        unsigned grp = __match_any_sync(0xffffffffu, kind);
        if (kind < MQ_CLASSES) {
            int leader = __ffs(grp) - 1;
            uint32_t base = 0;
            if ((int)lane == leader) base = atomicAdd(p.cnt + CNT_MQ + kind, (uint32_t)__popc(grp));
            base = __shfl_sync(grp, base, leader);
            size_t pos = mq_slot(p, 0, kind, base + (uint32_t)__popc(grp & ((1u << lane) - 1u)));
            p.mq_o[pos] = o; p.mq_d[pos] = d; p.mq_thr[pos] = t; p.mq_hit[pos] = hv;
        }
    }
    if (COUNT) {
        atomicAdd(cnt64(p.cnt, C64_NODES), (unsigned long long)nodes);
        atomicAdd(cnt64(p.cnt, C64_PRIMS), (unsigned long long)prims);
    }
    if (HRPP) {  // hrpp.rs:85-130 statistics: one atomic per warp and counter
        for (int off = 16; off > 0; off >>= 1) {
            h_tp += __shfl_down_sync(0xffffffffu, h_tp, off);
            h_fp += __shfl_down_sync(0xffffffffu, h_fp, off);
            h_none += __shfl_down_sync(0xffffffffu, h_none, off);
        }
        if (lane == 0) {
            if (h_tp) atomicAdd(cnt64(p.cnt, C64_HRPP_TP), (unsigned long long)h_tp);
            if (h_fp) atomicAdd(cnt64(p.cnt, C64_HRPP_FP), (unsigned long long)h_fp);
            if (h_none) atomicAdd(cnt64(p.cnt, C64_HRPP_NONE), (unsigned long long)h_none);
        }
    }
}

// TMA-stages the arrays the walk reads into the block's shared memory (scene images up to ~220 KB)
// SIGNED: the node region holds SNodes (p.smem.signed_nodes; the one-Bvh kernels) - a template parameter so that the
// compiler knows which of the two node pointers is a shared-memory address (LDS instead of generic loads)
template <bool SIGNED = false>
__device__ __forceinline__ SceneView stage_scene(const WfParams& p, unsigned char* smem, uint64_t* bar) {
    SceneView sv = p.sv;
    if (threadIdx.x == 0) mbar_init(bar, 1);
    __syncthreads();
    if (threadIdx.x == 0) {
        const SmemLayout& L = p.smem;
        mbar_expect_tx(bar, L.bytes_nodes + L.bytes_sph + L.bytes_msph + L.bytes_rect + L.bytes_tri + L.bytes_cube + L.bytes_objects + L.bytes_sph_mat);
        if (L.bytes_nodes) bulk_g2s(smem + L.off_nodes, SIGNED ? (const void*)p.sv.snodes : (const void*)p.sv.nodes, L.bytes_nodes, bar);
        if (L.bytes_sph) bulk_g2s(smem + L.off_sph, p.sv.sph, L.bytes_sph, bar);
        if (L.bytes_msph) bulk_g2s(smem + L.off_msph, p.sv.msph, L.bytes_msph, bar);
        if (L.bytes_rect) bulk_g2s(smem + L.off_rect, p.sv.rect, L.bytes_rect, bar);
        if (L.bytes_tri) bulk_g2s(smem + L.off_tri, p.sv.tri, L.bytes_tri, bar);
        if (L.bytes_cube) bulk_g2s(smem + L.off_cube, p.sv.cube, L.bytes_cube, bar);
        if (L.bytes_objects) bulk_g2s(smem + L.off_objects, p.sv.objects, L.bytes_objects, bar);
        if (L.bytes_sph_mat) bulk_g2s(smem + L.off_sph_mat, p.sv.sph_mat, L.bytes_sph_mat, bar);
    }
    if (SIGNED) sv.snodes = reinterpret_cast<const SNode*>(smem + p.smem.off_nodes);
    else sv.nodes = reinterpret_cast<const DevNode*>(smem + p.smem.off_nodes);
    sv.sph = reinterpret_cast<const double*>(smem + p.smem.off_sph);
    sv.msph = reinterpret_cast<const f4*>(smem + p.smem.off_msph);
    sv.rect = reinterpret_cast<const f4*>(smem + p.smem.off_rect);
    sv.tri = reinterpret_cast<const f4*>(smem + p.smem.off_tri);
    sv.cube = reinterpret_cast<const f4*>(smem + p.smem.off_cube);
    sv.objects = reinterpret_cast<const DevObject*>(smem + p.smem.off_objects);
    sv.sph_mat = reinterpret_cast<const int*>(smem + p.smem.off_sph_mat);
    mbar_wait(bar, 0);
    return sv;
}

#ifndef SHIM_EXTEND_THREADS
#define SHIM_EXTEND_THREADS 640
#endif
// threads per block of the specialised kernels (one persistent block per SM; measured in round 1, DESIGN.md §4)
#ifndef SHIM_SOLO_SPHERE_THREADS
#define SHIM_SOLO_SPHERE_THREADS 896   // sphere-only Bvh worlds: 72 registers
#endif
#define SHIM_SOLO_ANY_THREADS 768      // one plain Bvh of mixed primitives: 80 registers
#define SHIM_LIST_THREADS 1024         // worlds without a Bvh: 64 registers
#ifndef SHIM_BVH1_TRI_THREADS
#define SHIM_BVH1_TRI_THREADS 1024     // one triangle-only Bvh among rects (56-63 registers)
#endif
template <bool SMEM, bool COUNT, bool MEDIA, bool HRPP>
__global__ void __launch_bounds__(SHIM_EXTEND_THREADS, 1) wf_extend() {
    const WfParams& p = g_p;
    const int cur = (int)p.cnt[CNT_CUR];
    const uint32_t n = p.cnt[cur];
    if (blockIdx.x * blockDim.x >= n) return;  // nothing for this block: do not even stage the scene
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bar;
    const SceneView sv = SMEM ? stage_scene(p, smem, &bar) : p.sv;
    extend_rays<COUNT, MEDIA, HRPP>(p, sv, cur, n);
}

// The same kernel for worlds that are one plain Bvh and nothing else (Book-1): closest_hit_solo needs fewer registers,
// so more warps are resident to cover the walk's dependent latencies.
template <bool COUNT, int THREADS, int ONLY, bool FUSE = false>
__global__ void __launch_bounds__(THREADS, 1) wf_extend_solo() {
    const WfParams& p = g_p;
    const int cur = (int)p.cnt[CNT_CUR];
    const uint32_t n = p.cnt[cur];
    if (blockIdx.x * blockDim.x >= n) return;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bar;
    SceneView sv = stage_scene<true>(p, smem, &bar);
    extend_rays<COUNT, false, false, true, ONLY, true, FUSE>(p, sv, cur, n);
}

// wf_extend for worlds without any Bvh (flat lists like the Cornell scenes, main.rs:477-557): the tree walk and its
// stack are compiled out, which frees registers for more resident warps.
template <bool MEDIA, int THREADS, bool FUSE = false>
__global__ void __launch_bounds__(THREADS, 1) wf_extend_list() {
    const WfParams& p = g_p;
    const int cur = (int)p.cnt[CNT_CUR];
    const uint32_t n = p.cnt[cur];
    if (blockIdx.x * blockDim.x >= n) return;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bar;
    SceneView sv = stage_scene(p, smem, &bar);
    extend_rays<false, MEDIA, false, false, -1, false, FUSE>(p, sv, cur, n);
}

// ---------------------------------------------------------------------------- extend, one-BVH worlds
// Worlds like the reference's mesh scenes (main.rs:791-829): six Cornell rects + Translate(Bvh(triangles)).  Most
// rays never enter the mesh's bounds, so in the plain kernel a warp idles on the few lanes that walk the tree
// (measured 9 of 32 lanes active on the bunny config; 7 of 32 in the node loop with per-warp lists of 128 rays).
// The closest hit of such a world is three launches:
//   wf_bvh1_list    every ray against the list objects and the BVH's root boxes (full warps, streaming); the result
//                   goes to a 16-byte record per ray, rays that can reach the tree are appended to a device-wide queue
//   wf_bvh1_walk    persistent warps pull queue entries and walk them; a lane whose walk ends writes its result to
//                   the ray's record and, once SHIM_BVH1_REFILL_IDLE lanes of the warp are idle, the idle lanes take
//                   the next entries of the queue - no barrier anywhere, the warps stay dense until the queue of the
//                   whole iteration is drained
//   wf_bvh1_finish  every ray's record -> background / material queue (full warps, one atomic per group of lanes
//                   with the same material kind)
// List order is kept (hittable.rs:100-118): a later object wins an equal t.
#ifndef SHIM_BVH1_REFILL_IDLE
#define SHIM_BVH1_REFILL_IDLE 12
#endif
#ifndef SHIM_BVH1_Q_SMEM_KB
#define SHIM_BVH1_Q_SMEM_KB 200   // a quantised tree up to this size (6400 nodes) is staged in shared memory whole
#endif
enum { BVH1_NONE = 0xffff, BVH1_DROP = 0xfffe };   // obj field of a record: no hit / path ends without a contribution
// record: x = t bits, y = obj | face << 16 | post << 24 (post: the list hit comes after the Bvh in list order), z = prim_ref

// writes ray i + its hit record as entry j of the queue of material class `kind`
__device__ __forceinline__ void bvh1_write_entry(const WfParams& p, int cur, uint32_t i, int kind, uint32_t j, const f4& hv) {
    const size_t pos = mq_slot(p, 0, kind, j);
    p.mq_o[pos] = p.ray_o[cur][i]; p.mq_d[pos] = p.ray_d[cur][i]; p.mq_thr[pos] = p.thr[cur][i]; p.mq_hit[pos] = hv;
}
// a ray's final record -> background (ray.rs:60) or the material kind + hit record to append
__device__ __forceinline__ int bvh1_resolve(const WfParams& p, const SceneView& sv, int cur, uint32_t i, const i4& rec, f4& hv) {
    const int obj = rec.y & 0xffff;
    if (obj == BVH1_DROP) return 7;
    if (obj == BVH1_NONE) {
        if (p.bg[0] != 0.0f || p.bg[1] != 0.0f || p.bg[2] != 0.0f) {
            const f4 t = p.thr[cur][i];
            float* a = p.accum + 3 * (size_t)(uint32_t)f2i(t.w);
            atomicAdd(a + 0, t.x * p.bg[0]);
            atomicAdd(a + 1, t.y * p.bg[1]);
            atomicAdd(a + 2, t.z * p.bg[2]);
        }
        return 7;
    }
    Hit h; h.t = i2f(rec.x); h.obj = obj; h.prim = (uint32_t)rec.z; h.face = (rec.y >> 16) & 0xff;
    const int mw = hit_material_word(sv, h);
    hv.x = h.t; hv.y = i2f(h.obj | (h.face << 16)); hv.z = i2f((int)h.prim); hv.w = i2f(mat_word_index(mw));
    return mat_word_kind(mw);
}

// RECTS: every list object is a plain rect (the Cornell walls of the mesh scenes) and there are at most
// SHIM_BVH1_LIST_RECTS of them: their records are copied to shared memory once per block and tested without the
// per-object transform and primitive dispatch (818 -> ~400 thread instructions per ray on the bunny config)
#define SHIM_BVH1_LIST_RECTS 16
template <bool COUNT, bool RECTS = false>
__global__ void __launch_bounds__(256) wf_bvh1_list() {
    const WfParams& p = g_p;
    const SceneView& sv = p.sv;
    const int cur = (int)p.cnt[CNT_CUR];
    const uint32_t n = p.cnt[cur];
    const int bo = p.bvh1_index;
    uint32_t prims = 0;
    __shared__ f4 s_rect[2 * SHIM_BVH1_LIST_RECTS];
    __shared__ int s_obj[SHIM_BVH1_LIST_RECTS], s_ref[SHIM_BVH1_LIST_RECTS];
    __shared__ uint32_t s_cnt[APPEND_SLOTS], s_base[APPEND_SLOTS];
    if (threadIdx.x < APPEND_SLOTS) s_cnt[threadIdx.x] = 0;
    if (!RECTS) __syncthreads();
    if (RECTS) {
        if ((int)threadIdx.x < sv.n_objects && (int)threadIdx.x != bo) {
            const int m = (int)threadIdx.x - ((int)threadIdx.x > bo ? 1 : 0);   // list order is kept
            const int ref = sv.objects[threadIdx.x].ref;
            s_obj[m] = (int)threadIdx.x; s_ref[m] = ref;
            s_rect[2 * m] = sv.rect[2 * (size_t)prim_index((uint32_t)ref)];
            s_rect[2 * m + 1] = sv.rect[2 * (size_t)prim_index((uint32_t)ref) + 1];
        }
        __syncthreads();
    }
    for (uint32_t base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {   // block-uniform trip count (barriers inside)
        const uint32_t i = base + threadIdx.x;
        bool need = false;
        int kind = APPEND_NONE;
        f4 hv;
        if (i < n) {
            f4 o = p.ray_o[cur][i], d = p.ray_d[cur][i];
            Ray r; r.o = mk3(o.x, o.y, o.z); r.d = mk3(d.x, d.y, d.z); r.time = o.w;
            i4 rec; rec.x = f2i(SHIM_INF); rec.y = BVH1_DROP; rec.z = 0; rec.w = 0;
            if (!ray_has_nan(r)) {   // see extend_rays: a NaN ray ends its path without a contribution
                float closest = SHIM_INF;
                int obj = BVH1_NONE, face_hit = 0; uint32_t prim = 0; bool post = false;
                if (RECTS) {
                    for (int m = 0; m < sv.n_objects - 1; ++m) {
                        float t;
                        if (hit_rect(s_rect + 2 * m, r, 0.001f, closest, t)) { closest = t; obj = s_obj[m]; prim = (uint32_t)s_ref[m]; post = obj > bo; }
                    }
                } else {
                    for (int oi = 0; oi < sv.n_objects; ++oi) {
                        if (oi == bo) continue;
                        const DevObject& ob = sv.objects[oi];
                        RayCtx pc;
                        pc.r = object_ray(ob, r);
                        float t; int face = 0;
                        if (COUNT) prims++;
                        if (hit_prim(sv, (uint32_t)ob.ref, pc, 0.001f, closest, t, face)) {
                            closest = t; obj = oi; prim = (uint32_t)ob.ref; face_hit = face; post = oi > bo;
                        }
                    }
                }
                // can the ray reach the tree at all?  (the root's two child boxes, against the closest list hit)
                const DevObject& bob = sv.objects[bo];
                RayCtx c;
                make_ctx(c, object_ray(bob, r));
                const DevNode& rn = sv.nodes[bob.ref];
                f4 na = rn.a, nb = rn.b, nc = rn.c;
                float tl, tr;
                need = slab(na.x, na.y, na.z, na.w, nb.x, nb.y, c, 0.001f, closest, tl) ||
                       (rn.d.y != CHILD_NONE && slab(nb.z, nb.w, nc.x, nc.y, nc.z, nc.w, c, 0.001f, closest, tr));
                rec.x = f2i(closest); rec.y = obj | (face_hit << 16) | ((post ? 1 : 0) << 24); rec.z = (int)prim;
            }
            if (need) p.bvh1_hit[i] = rec;                      // the walk may replace it, wf_bvh1_finish writes it out
            else kind = bvh1_resolve(p, sv, cur, i, rec, hv);   // final already
        }
        const uint32_t at = block_append_slots(p, need ? (int)APPEND_TREEQ : kind, s_cnt, s_base);
        if (need) p.bvh1_queue[at] = i;
        else if (kind < MQ_CLASSES) bvh1_write_entry(p, cur, i, kind, at, hv);
    }
    if (COUNT) atomicAdd(cnt64(p.cnt, C64_PRIMS), (unsigned long long)prims);
}

#ifndef SHIM_BVH1_PRIM_BATCH
#define SHIM_BVH1_PRIM_BATCH 8
#endif
#ifndef SHIM_BVH1_STEPS_PER_VOTE
#define SHIM_BVH1_STEPS_PER_VOTE 2
#endif
// QN: the tree is walked on its quantised 32-byte nodes (QNode, breadth-first order).  1: all of them are staged in
// shared memory by bulk copies (p.bvh1_q_smem = their number); 2: they are fetched from global memory with one 32-byte
// load per node.  (SMEM and QN exclude each other.)
template <bool SMEM, bool COUNT, int THREADS = SHIM_EXTEND_THREADS, int ONLY = -1, int QN = 0>
__global__ void __launch_bounds__(THREADS, 1) wf_bvh1_walk() {
    const WfParams& p = g_p;
    const int cur_q = (int)p.cnt[CNT_CUR];
    const uint32_t count = p.cnt[CNT_TREEQ];
    if (blockIdx.x * blockDim.x >= count) return;   // fewer entries than one per thread up to this block: the others take them
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bar;
    const SceneView sv = SMEM ? stage_scene(p, smem, &bar) : p.sv;
    if (QN == 1) {
        const uint32_t q_smem = p.bvh1_q_smem;
        if (threadIdx.x == 0) mbar_init(&bar, 1);
        __syncthreads();
        if (threadIdx.x == 0) {
            const uint32_t bytes = q_smem * (uint32_t)sizeof(QNode);
            mbar_expect_tx(&bar, bytes);
            for (uint32_t off = 0; off < bytes; off += 32768u)
                bulk_g2s(smem + off, reinterpret_cast<const unsigned char*>(p.sv.qnodes) + off, bytes - off < 32768u ? bytes - off : 32768u, &bar);
        }
        mbar_wait(&bar, 0);
    }
    const uint32_t q_base = smem_u32(smem);
    const uint32_t lane = threadIdx.x & 31u, lt_mask = (1u << lane) - 1u;
    const int bo = p.bvh1_index;
    const DevObject& bob = sv.objects[bo];
    uint32_t nodes = 0, prims = 0;
    int stack[SHIM_BVH_STACK];
    // Every lane owns one walk (the state of bvh_closest, resumable).  The warp alternates between rounds of node steps
    // and rounds of primitive tests: a lane that has reached a primitive waits until SHIM_BVH1_PRIM_BATCH lanes have
    // one (or no lane is left at an inner node), so that both kinds of rounds run with fuller warps than a loop in
    // which every lane tests its primitive as soon as it gets there.
    bool active = false, more = true;
    uint32_t ray = 0;
    float list_t = SHIM_INF;
    bool list_hit = false, post = false;
    RayCtx c;
    BvhBest best; best.t = 0; best.prim = 0; best.face = 0; best.any = false;
    float t_cull = 0;
    int cur = SHIM_STACK_END, sp = 0;
    while (more || __any_sync(0xffffffffu, active)) {
        const unsigned idle = __ballot_sync(0xffffffffu, !active);
        if (more && idle) {
            const uint32_t n_idle = (uint32_t)__popc(idle);
            uint32_t got = 0;
            if (lane == (uint32_t)(__ffs(idle) - 1)) got = atomicAdd(p.cnt + CNT_TREEQ_NEXT, n_idle);
            got = __shfl_sync(0xffffffffu, got, __ffs(idle) - 1);
            const uint32_t my = got + (uint32_t)__popc(idle & lt_mask);
            if (!active && my < count) {
                ray = p.bvh1_queue[my];
                const i4 rec = p.bvh1_hit[ray];
                list_t = i2f(rec.x);
                list_hit = (rec.y & 0xffff) != BVH1_NONE;
                post = ((rec.y >> 24) & 1) != 0;
                f4 o = p.ray_o[cur_q][ray], d = p.ray_d[cur_q][ray];
                Ray r; r.o = mk3(o.x, o.y, o.z); r.d = mk3(d.x, d.y, d.z); r.time = o.w;
                make_ctx(c, object_ray(bob, r));
                best.t = list_t; best.prim = 0; best.face = 0; best.any = false;
                t_cull = list_t; sp = 0; cur = QN ? 0 : bob.ref;
                active = true;
            }
            if (got + n_idle >= count) more = false;
        }
        if (!__any_sync(0xffffffffu, active)) continue;   // (`more` is false by now: the loop ends)
        for (;;) {
            // ---- node rounds.  The votes that steer a round are a sixth of its instructions, so the quantised walk takes
            // SHIM_BVH1_STEPS_PER_VOTE node steps per vote (a lane that reaches a primitive early waits for the batch anyway).
            auto node_step = [&]() {
                i4 ch;
                float tl, tr;
                bool hl, hr;
                if (COUNT) nodes++;
                if (QN) {
                    uint32_t w[8];
                    if (QN == 1) {
                        const uint32_t a = q_base + (uint32_t)cur * (uint32_t)sizeof(QNode);
                        asm("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]) : "r"(a));
                        asm("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4+16];" : "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]) : "r"(a));
                    } else {
                        asm("ld.global.nc.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                            : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]) : "l"(sv.qnodes + cur));
                    }
                    slab_pair_q(w, c, 0.001f, t_cull, tl, tr, hl, hr);
                    ch.x = (int)w[6]; ch.y = (int)w[7];
                } else {
                    f4 na, nb, nc;
                    load_node(sv.nodes, cur, na, nb, nc, ch);
                    hl = slab(na.x, na.y, na.z, na.w, nb.x, nb.y, c, 0.001f, t_cull, tl);
                    hr = slab(nb.z, nb.w, nc.x, nc.y, nc.z, nc.w, c, 0.001f, t_cull, tr);
                }
                hr = hr && ch.y != CHILD_NONE;
                if (hl && hr) {
                    bool swap = tr < tl;
                    cur = swap ? ch.y : ch.x;
                    if (sp < SHIM_BVH_STACK) stack[sp++] = swap ? ch.x : ch.y;
                } else if (hl) {
                    cur = ch.x;
                } else if (hr) {
                    cur = ch.y;
                } else {
                    cur = sp > 0 ? stack[--sp] : SHIM_STACK_END;
                }
            };
            for (;;) {
                // (an idle lane has cur == SHIM_STACK_END: cur alone tells the three states apart)
                const bool at_node = (uint32_t)cur < (uint32_t)SHIM_STACK_END;
                const unsigned nm = __ballot_sync(0xffffffffu, at_node);
                if (nm == 0u) break;
                const unsigned pm = __ballot_sync(0xffffffffu, cur < 0);
                if (__popc(pm) >= SHIM_BVH1_PRIM_BATCH) break;
                if (at_node) node_step();
#pragma unroll
                for (int extra = 1; extra < (QN ? SHIM_BVH1_STEPS_PER_VOTE : 1); ++extra)
                    if ((uint32_t)cur < (uint32_t)SHIM_STACK_END) node_step();
            }
            // ---- one round of primitive tests (same rules as bvh_closest: closer wins, an exact tie goes to the later leaf)
            if (active && cur < 0) {
                const uint32_t ref = ~(uint32_t)cur;
                float t; int face = 0;
                if (COUNT) prims++;
                if (hit_prim<ONLY>(sv, ref, c, 0.001f, t_cull, t, face) && !(t > best.t)) {
                    bool take = !best.any || t < best.t;
                    if (!take) take = tie_goes_to_candidate<ONLY>(sv, c, 0.001f, ref, best.prim, t);
                    if (take) { best.t = t; best.prim = ref; best.face = face; best.any = true; t_cull = t + fabsf(t) * 3.8146973e-06f; }
                }
                cur = sp > 0 ? stack[--sp] : SHIM_STACK_END;
            }
            // ---- retire finished walks
            if (active && cur == SHIM_STACK_END) {
                active = false;
                // an equal t goes to the later list object (hittable.rs:100-118)
                if (best.any && (!list_hit || best.t < list_t || !post)) {
                    i4 rec; rec.x = f2i(best.t); rec.y = bo | (best.face << 16); rec.z = (int)best.prim; rec.w = 0;
                    p.bvh1_hit[ray] = rec;
                }
            }
            const unsigned act = __ballot_sync(0xffffffffu, active);
            if (act == 0u) break;
            if (more && __popc(act) <= 32 - SHIM_BVH1_REFILL_IDLE) break;
        }
    }
    if (COUNT) {
        atomicAdd(cnt64(p.cnt, C64_NODES), (unsigned long long)nodes);
        atomicAdd(cnt64(p.cnt, C64_PRIMS), (unsigned long long)prims);
    }
}

// the rays that went through the tree walk: record -> background / material queue (full warps)
__global__ void __launch_bounds__(256) wf_bvh1_finish() {
    const WfParams& p = g_p;
    const SceneView& sv = p.sv;
    const int cur = (int)p.cnt[CNT_CUR];
    const uint32_t n = p.cnt[CNT_TREEQ];
    __shared__ uint32_t s_cnt[APPEND_SLOTS], s_base[APPEND_SLOTS];
    if (threadIdx.x < APPEND_SLOTS) s_cnt[threadIdx.x] = 0;
    __syncthreads();
    for (uint32_t base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {
        const uint32_t j = base + threadIdx.x;
        int kind = APPEND_NONE;
        f4 hv;
        uint32_t i = 0;
        if (j < n) {
            i = p.bvh1_queue[j];
            kind = bvh1_resolve(p, sv, cur, i, p.bvh1_hit[i], hv);
            if (kind >= MQ_CLASSES) kind = APPEND_NONE;
        }
        const uint32_t at = block_append_slots(p, kind, s_cnt, s_base);
        if (kind < MQ_CLASSES) bvh1_write_entry(p, cur, i, kind, at, hv);
    }
}

// ---------------------------------------------------------------------------- shade
struct ShadeOut { bool cont; Ray ray; f3 thr; };

// ray.rs:44-58 for one hit of material kind KIND; adds emission to the framebuffer
template <int KIND>
__device__ __forceinline__ void shade_one(const WfParams& p, const SceneView& sv, const Ray& r, const Hit& h, int mat, f3 thr, int bounce,
                                          uint32_t pixel, uint32_t sample, ShadeOut& out) {
    HitRec rec;
    reconstruct_hit(sv, r, h, mat_needs_uv(sv, mat), rec);
    out.cont = false;
    if (KIND == MAT_DIFFUSE_LIGHT) {  // ray.rs:46-48, 57: emitted, no scatter
        f3 e = mat_emit(sv, mat, rec);
        float* a = p.accum + 3 * (size_t)pixel;
        atomicAdd(a + 0, thr.x * e.x);
        atomicAdd(a + 1, thr.y * e.y);
        atomicAdd(a + 2, thr.z * e.z);
    } else {
        Rng rng;
        rng_init(rng, pixel, sample, p.seed);
        rng_key(rng, (uint32_t)bounce, STAGE_SCATTER);
        f3 att;
        if (mat_scatter(sv, KIND, mat, r, rec, rng, att, out.ray)) {
            out.thr = thr * att;
            out.cont = bounce + 1 < p.max_depth;  // ray.rs:39-42: depth exhausted -> black
        }
    }
}

template <int KIND, int QUEUE = KIND>
__device__ __forceinline__ void shade_chunk(const WfParams& p, int cur, uint32_t j, uint32_t n) {
    const int nxt = 1 - cur;
    ShadeOut so;
    so.cont = false; so.ray.o = mk3(0, 0, 0); so.ray.d = mk3(0, 0, 0); so.ray.time = 0; so.thr = mk3(0, 0, 0);
    uint32_t bs = 0, pixel = 0;
    if (j < n) {
        size_t q = mq_slot(p, 0, QUEUE, j);
        f4 o = p.mq_o[q], d = p.mq_d[q], t = p.mq_thr[q], hv = p.mq_hit[q];
        Ray r; r.o = mk3(o.x, o.y, o.z); r.d = mk3(d.x, d.y, d.z); r.time = o.w;
        bs = (uint32_t)f2i(d.w); pixel = (uint32_t)f2i(t.w);
        Hit h; h.t = hv.x; h.obj = f2i(hv.y) & 0xffff; h.face = f2i(hv.y) >> 16; h.prim = (uint32_t)f2i(hv.z);
        shade_one<KIND>(p, p.sv, r, h, f2i(hv.w), mk3(t.x, t.y, t.z), (int)(bs & 255u), pixel, bs >> 8, so);
    }
    if (KIND != MAT_DIFFUSE_LIGHT) {
        uint32_t pos = warp_append(p.cnt + nxt, so.cont);   // (a block-wide append measured 1 % slower here: one counter, long chunks)
        if (so.cont) {
            f4 o; o.x = so.ray.o.x; o.y = so.ray.o.y; o.z = so.ray.o.z; o.w = so.ray.time;
            f4 d; d.x = so.ray.d.x; d.y = so.ray.d.y; d.z = so.ray.d.z; d.w = i2f((int)(bs + 1u));
            f4 t; t.x = so.thr.x; t.y = so.thr.y; t.z = so.thr.z; t.w = i2f((int)pixel);
            p.ray_o[nxt][pos] = o;
            p.ray_d[nxt][pos] = d;
            p.thr[nxt][pos] = t;
        }
    }
}

// One launch for all material queues: the queues are cut into 256-ray chunks, chunks are dealt
// round-robin to the persistent blocks, and each chunk runs the code specialised for its material.
__global__ void __launch_bounds__(256) wf_shade() {   // 72 registers, 3 blocks per SM (forcing 4 or 5: 1-7 % slower)
    const WfParams& p = g_p;
    const int cur = (int)p.cnt[CNT_CUR];
    uint32_t n[MQ_CLASSES], first[MQ_CLASSES + 1];
    first[0] = 0;
#pragma unroll
    for (int k = 0; k < MQ_CLASSES; ++k) {
        n[k] = p.cnt[CNT_MQ + k];
        first[k + 1] = first[k] + (n[k] + 255u) / 256u;
    }
    for (uint32_t w = blockIdx.x; w < first[MQ_CLASSES]; w += gridDim.x) {
        if (w < first[1]) shade_chunk<MAT_LAMBERTIAN>(p, cur, (w - first[0]) * 256u + threadIdx.x, n[0]);
        else if (w < first[2]) shade_chunk<MAT_METAL>(p, cur, (w - first[1]) * 256u + threadIdx.x, n[1]);
        else if (w < first[3]) shade_chunk<MAT_DIELECTRIC>(p, cur, (w - first[2]) * 256u + threadIdx.x, n[2]);
        else if (w < first[4]) shade_chunk<MAT_DIFFUSE_LIGHT>(p, cur, (w - first[3]) * 256u + threadIdx.x, n[3]);
        else if (w < first[5]) shade_chunk<MAT_ISOTROPIC>(p, cur, (w - first[4]) * 256u + threadIdx.x, n[4]);
        else shade_chunk<MAT_LAMBERTIAN, MQ_SLOW_LAMBERTIAN>(p, cur, (w - first[5]) * 256u + threadIdx.x, n[5]);   // expensive textures, dense
    }
}

// ---------------------------------------------------------------------------- tail
// Runs after wf_shade.  When every sample has been started and at most tail_threshold paths are
// alive, each thread takes one of them and follows it to its end; the queue is then empty.
// It is also where the loop ends: the render is done when the next queue is empty and every sample has been started;
// that sets the done flag and, when the iteration runs inside a CUDA-graph WHILE node, the node's condition.
__device__ __forceinline__ void loop_publish(const WfParams& p, bool done) {
    if (p.cnt[CNT_ITER] >= p.max_iterations) done = true;
    p.cnt[CNT_DONE] = done ? 1u : 0u;
    if (p.loop_handle) cudaGraphSetConditional((cudaGraphConditionalHandle)p.loop_handle, done ? 0u : 1u);
}
// Trace pipeline: what wf_generate's last block publishes for the next iteration (it writes no rays there), done by
// the one thread that ends the previous iteration in wf_tail_mq - the iteration is then two launches, not three.
__device__ __forceinline__ void trace_prepare_iteration(const WfParams& p) {
    uint32_t* c = p.cnt;
    const int cur = (int)c[CNT_NEXT_CUR];
    uint32_t n_cur = 0;
    for (int k = 0; k < MAT_KINDS; ++k) n_cur += mq_counts(p, cur)[k];
    const unsigned long long first = *cnt64(c, C64_NEXT_SAMPLE);
    const unsigned long long remaining = p.total_samples - first;
    const unsigned long long room = (unsigned long long)(p.pool - n_cur);
    const uint32_t n = (uint32_t)(remaining < room ? remaining : room);
    c[CNT_CUR] = (uint32_t)cur;
    c[CNT_NEXT_CUR] = (uint32_t)(1 - cur);
    *cnt64(c, C64_NEXT_SAMPLE) = first + n;
    *cnt64(c, C64_GEN_FIRST) = first;
    c[CNT_GEN_N] = n;
    for (int k = 0; k < MAT_KINDS; ++k) mq_counts(p, 1 - cur)[k] = 0;   // wf_trace fills the other set
    c[CNT_ITER] += (n_cur + n == 0) ? 0u : 1u;
    c[CNT_BODIES] += 1u;
}
// after the last iteration: leave nothing for a further wf_trace launch to pick up (the host-driven loop enqueues a few)
__device__ __forceinline__ void trace_finish(const WfParams& p) {
    for (int k = 0; k < MAT_KINDS; ++k) { mq_counts(p, 0)[k] = 0; mq_counts(p, 1)[k] = 0; }
    p.cnt[CNT_GEN_N] = 0;
}
__global__ void wf_trace_first() {   // before the loop: the counters of iteration 0
    if (blockIdx.x == 0 && threadIdx.x == 0) { trace_prepare_iteration(g_p); __threadfence(); }
}
// COUNT: node visits and primitive tests of the endgame's walks go to C64_NODES / C64_PRIMS like wf_extend's (a counted
// render: SHIM_RENDER_COUNT_NODES)
template <bool HRPP, bool SOLO = false, int ONLY = -1, bool COUNT = false>
__global__ void __launch_bounds__(128) wf_tail() {
    const WfParams& p = g_p;
    const int cur = (int)p.cnt[CNT_CUR];
    const int nxt = 1 - cur;
    const uint32_t n = p.cnt[nxt];
    const bool all_started = *cnt64(p.cnt, C64_NEXT_SAMPLE) >= p.total_samples;
    if (n == 0 || n > p.tail_threshold || !all_started) {
        if (blockIdx.x == 0 && threadIdx.x == 0) loop_publish(p, n == 0 && all_started);
        return;
    }
    uint32_t traced = 0;
    TraceCounters tc; tc.nodes = 0; tc.prims = 0; tc.hrpp_tp = 0; tc.hrpp_fp = 0; tc.hrpp_none = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        f4 o = p.ray_o[nxt][i], d = p.ray_d[nxt][i], t = p.thr[nxt][i];
        uint32_t sample = (uint32_t)f2i(d.w) >> 8, pixel = (uint32_t)f2i(t.w);
        Ray r; r.o = mk3(o.x, o.y, o.z); r.d = mk3(d.x, d.y, d.z); r.time = o.w;
        f3 thr = mk3(t.x, t.y, t.z);
        for (int bounce = f2i(d.w) & 255; bounce < p.max_depth; ++bounce) {
            Rng rng;
            rng_init(rng, pixel, sample, p.seed);
            rng_key(rng, (uint32_t)bounce, STAGE_INTERSECT);
            ++traced;
            if (ray_has_nan(r)) break;  // see extend_rays
            Hit h;
            if constexpr (COUNT) h = closest_hit<true, false>(p.sv, r, 0.001f, SHIM_INF, rng, &tc);
            else h = SOLO ? closest_hit_solo<false, ONLY>(p.sv, r, 0.001f, SHIM_INF, &tc) : closest_hit<false, HRPP>(p.sv, r, 0.001f, SHIM_INF, rng, &tc);
            if (h.obj < 0) {
                float* a = p.accum + 3 * (size_t)pixel;
                atomicAdd(a + 0, thr.x * p.bg[0]);
                atomicAdd(a + 1, thr.y * p.bg[1]);
                atomicAdd(a + 2, thr.z * p.bg[2]);
                break;
            }
            const int mw = hit_material_word(p.sv, h);
            const int mat = mat_word_index(mw);
            ShadeOut so;
            so.cont = false;
            switch (mat_word_kind(mw)) {
            case MQ_SLOW_LAMBERTIAN:
            case MAT_LAMBERTIAN: shade_one<MAT_LAMBERTIAN>(p, p.sv, r, h, mat, thr, bounce, pixel, sample, so); break;
            case MAT_METAL: shade_one<MAT_METAL>(p, p.sv, r, h, mat, thr, bounce, pixel, sample, so); break;
            case MAT_DIELECTRIC: shade_one<MAT_DIELECTRIC>(p, p.sv, r, h, mat, thr, bounce, pixel, sample, so); break;
            case MAT_DIFFUSE_LIGHT: shade_one<MAT_DIFFUSE_LIGHT>(p, p.sv, r, h, mat, thr, bounce, pixel, sample, so); break;
            default: shade_one<MAT_ISOTROPIC>(p, p.sv, r, h, mat, thr, bounce, pixel, sample, so); break;
            }
            if (!so.cont) break;
            r = so.ray;
            thr = so.thr;
        }
    }
    // queue `nxt` has not been counted yet (wf_generate counts a queue when its iteration starts)
    unsigned long long extra = traced;
    for (int off = 16; off > 0; off >>= 1) extra += __shfl_down_sync(0xffffffffu, extra, off);
    if ((threadIdx.x & 31) == 0 && extra) atomicAdd(cnt64(p.cnt, C64_RAYS), extra);
    if constexpr (COUNT) {
        atomicAdd(cnt64(p.cnt, C64_NODES), (unsigned long long)tc.nodes);
        atomicAdd(cnt64(p.cnt, C64_PRIMS), (unsigned long long)tc.prims);
    }
    if (HRPP) {
        if (tc.hrpp_tp) atomicAdd(cnt64(p.cnt, C64_HRPP_TP), (unsigned long long)tc.hrpp_tp);
        if (tc.hrpp_fp) atomicAdd(cnt64(p.cnt, C64_HRPP_FP), (unsigned long long)tc.hrpp_fp);
        if (tc.hrpp_none) atomicAdd(cnt64(p.cnt, C64_HRPP_NONE), (unsigned long long)tc.hrpp_none);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        uint32_t ticket = atomicAdd(p.cnt + CNT_TICKET, 1u);
        if (ticket == gridDim.x - 1) { p.cnt[CNT_TICKET] = 0; p.cnt[nxt] = 0; loop_publish(p, true); __threadfence(); }
    }
}

// ---------------------------------------------------------------------------- trace pipeline (one-Bvh worlds)
// Nearly every shaded hit continues (absorption is rare), so compacting the scattered rays into a ray queue only to
// read them back buys nothing.  wf_trace goes from material queue to material queue: an entry of set `cur` is shaded by
// the code of its material, the scattered ray is walked through the tree right away and the new hit is appended to its
// material's queue in the other set; new samples enter as camera rays made on the spot.  Per ray and bounce that is one
// 64-byte read and one 64-byte write instead of 224 bytes through two queues, and two launches less per iteration.
template <int KIND>
__device__ __noinline__ bool trace_shade_entry(const WfParams& p, int set, uint32_t j, f4& o, f4& d, f4& t) {
    const size_t q = mq_slot(p, set, KIND, j);
    const f4 eo = p.mq_o[q], ed = p.mq_d[q], et = p.mq_thr[q], hv = p.mq_hit[q];
    Ray r; r.o = mk3(eo.x, eo.y, eo.z); r.d = mk3(ed.x, ed.y, ed.z); r.time = eo.w;
    const uint32_t bs = (uint32_t)f2i(ed.w), pixel = (uint32_t)f2i(et.w);
    Hit h; h.t = hv.x; h.obj = f2i(hv.y) & 0xffff; h.face = f2i(hv.y) >> 16; h.prim = (uint32_t)f2i(hv.z);
    ShadeOut so;
    so.cont = false; so.ray.o = mk3(0, 0, 0); so.ray.d = mk3(0, 0, 0); so.ray.time = 0; so.thr = mk3(0, 0, 0);
    shade_one<KIND>(p, p.sv, r, h, f2i(hv.w), mk3(et.x, et.y, et.z), (int)(bs & 255u), pixel, bs >> 8, so);
    if (!so.cont) return false;
    o.x = so.ray.o.x; o.y = so.ray.o.y; o.z = so.ray.o.z; o.w = so.ray.time;
    d.x = so.ray.d.x; d.y = so.ray.d.y; d.z = so.ray.d.z; d.w = i2f((int)(bs + 1u));
    t.x = so.thr.x; t.y = so.thr.y; t.z = so.thr.z; t.w = i2f((int)pixel);
    return true;
}

template <int THREADS, int ONLY>
__global__ void __launch_bounds__(THREADS, 1) wf_trace_solo() {
    const WfParams& p = g_p;
    const int cur = (int)p.cnt[CNT_CUR];
    // work items: the new samples, then the entries of the five queues of set `cur`, every segment padded to whole warps
    uint32_t seg_n[MAT_KINDS + 1], seg_start[MAT_KINDS + 2];
    seg_n[0] = p.cnt[CNT_GEN_N];
#pragma unroll
    for (int k = 0; k < MAT_KINDS; ++k) seg_n[k + 1] = mq_counts(p, cur)[k];
    seg_start[0] = 0;
#pragma unroll
    for (int k = 0; k <= MAT_KINDS; ++k) seg_start[k + 1] = seg_start[k] + ((seg_n[k] + 31u) & ~31u);
    const uint32_t total = seg_start[MAT_KINDS + 1];
    if (blockIdx.x * blockDim.x >= total) return;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ uint64_t bar;
    const SceneView sv = stage_scene<true>(p, smem, &bar);
    const unsigned long long gen_first = *cnt64(p.cnt, C64_GEN_FIRST);
    const uint32_t lane = threadIdx.x & 31u;
    uint32_t* out_cnt = mq_counts(p, 1 - cur);
    uint32_t traced = 0;
    for (uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x; slot < total; slot += gridDim.x * blockDim.x) {
        f4 o, d, t;
        bool have = false;
        // which segment (the same for the whole warp)
        if (slot < seg_start[1]) { const uint32_t j = slot; if (j < seg_n[0]) { camera_ray_record(p, gen_first + j, o, d, t); have = true; } }
        else if (slot < seg_start[2]) { const uint32_t j = slot - seg_start[1]; if (j < seg_n[1]) have = trace_shade_entry<MAT_LAMBERTIAN>(p, cur, j, o, d, t); }
        else if (slot < seg_start[3]) { const uint32_t j = slot - seg_start[2]; if (j < seg_n[2]) have = trace_shade_entry<MAT_METAL>(p, cur, j, o, d, t); }
        else if (slot < seg_start[4]) { const uint32_t j = slot - seg_start[3]; if (j < seg_n[3]) have = trace_shade_entry<MAT_DIELECTRIC>(p, cur, j, o, d, t); }
        else if (slot < seg_start[5]) { const uint32_t j = slot - seg_start[4]; if (j < seg_n[4]) have = trace_shade_entry<MAT_DIFFUSE_LIGHT>(p, cur, j, o, d, t); }
        else { const uint32_t j = slot - seg_start[5]; if (j < seg_n[5]) have = trace_shade_entry<MAT_ISOTROPIC>(p, cur, j, o, d, t); }
        int kind = 7;
        f4 hv;
        if (have) {
            ++traced;
            Ray r; r.o = mk3(o.x, o.y, o.z); r.d = mk3(d.x, d.y, d.z); r.time = o.w;
            if (!ray_has_nan(r)) {   // see extend_rays
                TraceCounters tc; tc.nodes = 0; tc.prims = 0; tc.hrpp_tp = 0; tc.hrpp_fp = 0; tc.hrpp_none = 0;
                const Hit h = closest_hit_solo<false, ONLY, true>(sv, r, 0.001f, SHIM_INF, &tc);   // SNodes in shared memory
                if (h.obj < 0) {  // ray.rs:60
                    if (p.bg[0] != 0.0f || p.bg[1] != 0.0f || p.bg[2] != 0.0f) {
                        float* a = p.accum + 3 * (size_t)(uint32_t)f2i(t.w);
                        atomicAdd(a + 0, t.x * p.bg[0]);
                        atomicAdd(a + 1, t.y * p.bg[1]);
                        atomicAdd(a + 2, t.z * p.bg[2]);
                    }
                } else {
                    const int mw = ONLY == PT_SPHERE ? sv.sph_mat[prim_index(h.prim)] : hit_material_word(sv, h);
                    kind = mat_word_kind(mw);
                    hv.x = h.t; hv.y = i2f(h.obj | (h.face << 16)); hv.z = i2f((int)h.prim); hv.w = i2f(mat_word_index(mw));
                }
            }
        }
        const unsigned grp = __match_any_sync(0xffffffffu, kind);
        if (kind < MAT_KINDS) {
            const int leader = __ffs(grp) - 1;
            uint32_t base = 0;
            if ((int)lane == leader) base = atomicAdd(out_cnt + kind, (uint32_t)__popc(grp));
            base = __shfl_sync(grp, base, leader);
            const size_t pos = mq_slot(p, 1 - cur, kind, base + (uint32_t)__popc(grp & ((1u << lane) - 1u)));
            p.mq_o[pos] = o; p.mq_d[pos] = d; p.mq_thr[pos] = t; p.mq_hit[pos] = hv;
        }
    }
    for (int off = 16; off > 0; off >>= 1) traced += __shfl_down_sync(0xffffffffu, traced, off);
    if (lane == 0 && traced) atomicAdd(cnt64(p.cnt, C64_RAYS), (unsigned long long)traced);
}

// wf_tail for the trace pipeline: the survivors are material-queue entries (hits waiting to be shaded)
#ifndef SHIM_TAIL_MQ_BLOCKS
#define SHIM_TAIL_MQ_BLOCKS 4   // blocks of 128 threads per SM (one path per thread)
#endif
template <int ONLY>
__global__ void __launch_bounds__(128, SHIM_TAIL_MQ_BLOCKS) wf_tail_mq() {
    const WfParams& p = g_p;
    // Thread 0 reads the counters once and the block branches on that copy: the last block to take a ticket rewrites
    // them (next iteration), so no thread may look at global memory again after its block's ticket is taken.
    __shared__ uint32_t s_seg[MAT_KINDS + 2];
    if (threadIdx.x == 0) {
        const int nx = 1 - (int)p.cnt[CNT_CUR];
#pragma unroll
        for (int k = 0; k < MAT_KINDS; ++k) s_seg[k] = mq_counts(p, nx)[k];
        s_seg[MAT_KINDS] = (*cnt64(p.cnt, C64_NEXT_SAMPLE) >= p.total_samples) ? 1u : 0u;
        s_seg[MAT_KINDS + 1] = (uint32_t)nx;
    }
    __syncthreads();
    const int nxt = (int)s_seg[MAT_KINDS + 1];
    uint32_t seg_n[MAT_KINDS], n = 0;
#pragma unroll
    for (int k = 0; k < MAT_KINDS; ++k) { seg_n[k] = s_seg[k]; n += seg_n[k]; }
    const bool all_started = s_seg[MAT_KINDS] != 0u;
    if (n == 0 || n > p.tail_threshold || !all_started) {
        if (threadIdx.x == 0) {
            const uint32_t ticket = atomicAdd(p.cnt + CNT_TICKET, 1u);
            if (ticket == gridDim.x - 1) {
                p.cnt[CNT_TICKET] = 0;
                const bool done = n == 0 && all_started;
                loop_publish(p, done);
                if (done) trace_finish(p); else trace_prepare_iteration(p);
                __threadfence();
            }
        }
        return;
    }
    uint32_t traced = 0;
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        int kind = 0;
        uint32_t j = i;
        while (j >= seg_n[kind]) { j -= seg_n[kind]; ++kind; }
        const size_t q = mq_slot(p, nxt, kind, j);
        const f4 eo = p.mq_o[q], ed = p.mq_d[q], et = p.mq_thr[q], hv = p.mq_hit[q];
        Ray r; r.o = mk3(eo.x, eo.y, eo.z); r.d = mk3(ed.x, ed.y, ed.z); r.time = eo.w;
        const uint32_t sample = (uint32_t)f2i(ed.w) >> 8, pixel = (uint32_t)f2i(et.w);
        int bounce = f2i(ed.w) & 255;
        f3 thr = mk3(et.x, et.y, et.z);
        Hit h; h.t = hv.x; h.obj = f2i(hv.y) & 0xffff; h.face = f2i(hv.y) >> 16; h.prim = (uint32_t)f2i(hv.z);
        int mat = f2i(hv.w);
        for (;;) {
            ShadeOut so;
            so.cont = false;
            switch (kind) {
            case MAT_LAMBERTIAN: shade_one<MAT_LAMBERTIAN>(p, p.sv, r, h, mat, thr, bounce, pixel, sample, so); break;
            case MAT_METAL: shade_one<MAT_METAL>(p, p.sv, r, h, mat, thr, bounce, pixel, sample, so); break;
            case MAT_DIELECTRIC: shade_one<MAT_DIELECTRIC>(p, p.sv, r, h, mat, thr, bounce, pixel, sample, so); break;
            case MAT_DIFFUSE_LIGHT: shade_one<MAT_DIFFUSE_LIGHT>(p, p.sv, r, h, mat, thr, bounce, pixel, sample, so); break;
            default: shade_one<MAT_ISOTROPIC>(p, p.sv, r, h, mat, thr, bounce, pixel, sample, so); break;
            }
            if (!so.cont) break;
            r = so.ray; thr = so.thr; ++bounce;
            ++traced;
            if (ray_has_nan(r)) break;
            TraceCounters tc; tc.nodes = 0; tc.prims = 0; tc.hrpp_tp = 0; tc.hrpp_fp = 0; tc.hrpp_none = 0;
            h = closest_hit_solo<false, ONLY>(p.sv, r, 0.001f, SHIM_INF, &tc);
            if (h.obj < 0) {
                float* a = p.accum + 3 * (size_t)pixel;
                atomicAdd(a + 0, thr.x * p.bg[0]);
                atomicAdd(a + 1, thr.y * p.bg[1]);
                atomicAdd(a + 2, thr.z * p.bg[2]);
                break;
            }
            const int mw = hit_material_word(p.sv, h);
            mat = mat_word_index(mw);
            kind = mat_word_kind(mw);
        }
    }
    unsigned long long extra = traced;
    for (int off = 16; off > 0; off >>= 1) extra += __shfl_down_sync(0xffffffffu, extra, off);
    if ((threadIdx.x & 31) == 0 && extra) atomicAdd(cnt64(p.cnt, C64_RAYS), extra);
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        uint32_t ticket = atomicAdd(p.cnt + CNT_TICKET, 1u);
        if (ticket == gridDim.x - 1) {
            p.cnt[CNT_TICKET] = 0;
            trace_finish(p);
            loop_publish(p, true);
            __threadfence();
        }
    }
}

// out = accum / spp (renderer.rs:147) or the raw sums
__global__ void wf_finalize(const float* accum, float* out, size_t n, float spp, int raw) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = raw ? accum[i] : accum[i] / spp;
}

// gate 1: the grid-stride loop of the three ray-batch queries.  ANY: the occlusion walk, which ends at the first
// accepted hit (closest_hit<..., ANY = true>).  `store` (StoreClosest / StoreRecord / StoreOccluded) writes ray i's answer.
template <bool ANY, class Store>
__device__ __forceinline__ void trace_batch(const SceneView& sv, const float* rays, long long n, float t_min, float t_max, uint64_t seed,
                                            unsigned long long* counters, Store store) {
    uint32_t nodes = 0, prims = 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        Ray r; Rng rng;
        batch_ray(rays, i, seed, r, rng);
        TraceCounters tc; tc.nodes = 0; tc.prims = 0; tc.hrpp_tp = 0; tc.hrpp_fp = 0; tc.hrpp_none = 0;
        // a scene with quantised nodes is queried on them (what its renders walk), unless node visits are being counted
        Hit h = counters ? closest_hit<true, false, true, false, ANY>(sv, r, t_min, t_max, rng, &tc)
                         : (sv.qnodes ? closest_hit<false, false, true, true, ANY>(sv, r, t_min, t_max, rng, &tc)
                                      : closest_hit<false, false, true, false, ANY>(sv, r, t_min, t_max, rng, &tc));
        nodes += tc.nodes; prims += tc.prims;
        store(sv, i, r, h);
    }
    if (counters) {
        atomicAdd(counters + 1, (unsigned long long)nodes);
        atomicAdd(counters + 2, (unsigned long long)prims);
    }
}

// closest hit for a batch of rays
__global__ void __launch_bounds__(256) trace_closest_kernel(SceneView sv, const float* rays, long long n, float t_min, float t_max,
                                                            uint64_t seed, int* prim_id, float* t_out, unsigned long long* counters) {
    trace_batch<false>(sv, rays, n, t_min, t_max, seed, counters, StoreClosest{prim_id, t_out});
}

// Hittable::hit with the whole record for a batch of rays: the walk of trace_closest_kernel, then the HitRecord rebuilt
// in registers.  128-thread blocks, three per SM: 158 registers and no spills (at the 128 registers of two 256-thread
// blocks the walk plus the record spill 88 bytes).
#define SHIM_TRACE_HIT_THREADS 128
__global__ void __launch_bounds__(SHIM_TRACE_HIT_THREADS, 3) trace_hit_kernel(SceneView sv, const float* rays, long long n, float t_min, float t_max,
                                                        uint64_t seed, f4* out, unsigned long long* counters) {
    trace_batch<false>(sv, rays, n, t_min, t_max, seed, counters, StoreRecord{out});
}

// Occlusion (any hit) for a batch of rays: occluded[i] = 1 exactly where trace_closest_kernel reports prim_id >= 0.
// 256-thread blocks, two per SM: 128 registers and no spills (with __launch_bounds__(256) alone ptxas also settles on
// 128 registers but spills 16 bytes, as trace_closest_kernel does).
#define SHIM_TRACE_OCCLUDED_THREADS 256
__global__ void __launch_bounds__(SHIM_TRACE_OCCLUDED_THREADS, 2) trace_occluded_kernel(SceneView sv, const float* rays, long long n, float t_min,
                                                                                     float t_max, uint64_t seed, uint8_t* occluded,
                                                                                     unsigned long long* counters) {
    trace_batch<true>(sv, rays, n, t_min, t_max, seed, counters, StoreOccluded{occluded});
}

}  // namespace shim
