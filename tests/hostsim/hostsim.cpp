// hostsim.cpp — TEST HARNESS ONLY.  Compiles the product's __host__ __device__ arithmetic
// (csrc/shim_device.h) and its flattener for the CPU, so that the device math can be checked
// against the oracle in this GPU-less container before spending GPU time.  It is not part
// of the package, is never loaded by it, and exists only under tests/.
//
// It links the product's CUDA-free builder entry points (shim_builder.cpp, shim_scene.cpp),
// so scenes are recorded through the very same shim_* calls; only commit / trace / radiance
// are replaced by serial loops over the shared inline functions.
#include <cstring>
#include <vector>

#include "../../raytracinginoneweekendinrust_b200/csrc/shim_device.h"
#include "../../raytracinginoneweekendinrust_b200/csrc/shim_internal.h"

using namespace shim;

void shim::device_state_release(DeviceState*) {}

// HRPP tables of the harness (the product keeps them in device memory)
#include <map>
namespace {
struct HrppHost { std::vector<HrppSlot> slots; int log2 = 0; bool on = false; uint64_t tp = 0, fp = 0, none = 0; };
std::map<shim_scene*, HrppHost> g_hrpp;
SceneView view_of(shim_scene* s) {
    SceneView sv = s->flat.view();
    auto it = g_hrpp.find(s);
    if (it != g_hrpp.end() && it->second.on) {
        sv.hrpp_slots = it->second.slots.data();
        sv.hrpp_log2 = it->second.log2; sv.hrpp_mask = (uint32_t)(((size_t)1 << it->second.log2) - 1);
    }
    return sv;
}
bool hrpp_on(shim_scene* s) { auto it = g_hrpp.find(s); return it != g_hrpp.end() && it->second.on; }
void hrpp_count(shim_scene* s, const TraceCounters& tc) {
    auto it = g_hrpp.find(s);
    if (it != g_hrpp.end()) { it->second.tp += tc.hrpp_tp; it->second.fp += tc.hrpp_fp; it->second.none += tc.hrpp_none; }
}
}  // namespace

// fresh predictor tables for every BVH recorded with a predictor (2^log2 slots each)
extern "C" __attribute__((visibility("default"))) int hs_enable_predictors(shim_scene* s, int log2) {
    HrppHost& h = g_hrpp[s];
    size_t n = s->flat.predictor_bvh.size();
    h.log2 = log2; h.on = n > 0; h.tp = h.fp = h.none = 0;
    HrppSlot empty;
    memset(&empty, 0xFF, sizeof empty);
    h.slots.assign(((size_t)1 << log2) * n, empty);
    return (int)n;
}
extern "C" __attribute__((visibility("default"))) void hs_predictor_stats(shim_scene* s, uint64_t* out3) {
    HrppHost& h = g_hrpp[s];
    out3[0] = h.tp; out3[1] = h.fp; out3[2] = h.none;
}

extern "C" __attribute__((visibility("default"))) int hs_commit(shim_scene* s);
// the harness library answers shim_commit with the CPU-side flatten only (no device)
extern "C" __attribute__((visibility("default"))) int shim_commit(shim_scene* s) { return hs_commit(s); }
extern "C" __attribute__((visibility("default"))) int hs_commit(shim_scene* s) {
    int rc = s->sb.flatten(s->flat);
    if (rc < 0) return set_err(rc, s->sb.err);
    s->has_media = false;
    for (const DevObject& o : s->flat.objects) if (o.flags & OBJ_MEDIUM) s->has_media = true;
    s->committed = true;
    return 0;
}

namespace {
// The batch kernels' loop (trace_batch in shim_kernels.cuh) run ray by ray: the same rays, Philox keying and store
// functors, the walk chosen by the template flags and always counted.  counters: rays, node visits, primitive tests.
template <bool HRPP, bool QN, bool ANY, class Store>
void trace_batch(shim_scene* s, const float* rays, int64_t n, float t_min, float t_max, uint64_t seed, Store store, uint64_t* counters) {
    SceneView sv = view_of(s);
    uint64_t nodes = 0, prims = 0;
    for (int64_t i = 0; i < n; ++i) {
        Ray r; Rng rng;
        batch_ray(rays, i, seed, r, rng);
        TraceCounters tc; tc.nodes = 0; tc.prims = 0; tc.hrpp_tp = 0; tc.hrpp_fp = 0; tc.hrpp_none = 0;
        Hit h = closest_hit<true, HRPP, true, QN, ANY>(sv, r, t_min, t_max, rng, &tc);
        if (HRPP) hrpp_count(s, tc);
        nodes += tc.nodes; prims += tc.prims;
        store(sv, i, r, h);
    }
    if (counters) { counters[0] = (uint64_t)n; counters[1] = nodes; counters[2] = prims; }
}

// quantised nodes for the one Bvh object of a world (what the batch kernels walk for a scene that has them); false if
// the world has no single Bvh object or its boxes cannot be quantised
bool quantise(shim_scene* s) {
    int idx = -1, n_bvh = 0;
    for (size_t i = 0; i < s->flat.objects.size(); ++i) if (s->flat.objects[i].kind == OBJ_BVH) { ++n_bvh; idx = (int)i; }
    if (n_bvh != 1) return false;
    return s->flat.q_object == idx || s->flat.build_quantized_nodes(idx);
}
}  // namespace

// trace_closest_kernel's walk on the exact nodes, or with the predictors hs_enable_predictors set up
extern "C" __attribute__((visibility("default"))) int hs_trace_closest(shim_scene* s, const float* rays, int64_t n, float t_min,
                                                                      float t_max, uint64_t seed, int32_t* prim, float* t,
                                                                      uint64_t* counters) {
    if (hrpp_on(s)) trace_batch<true, false, false>(s, rays, n, t_min, t_max, seed, StoreClosest{prim, t}, counters);
    else trace_batch<false, false, false>(s, rays, n, t_min, t_max, seed, StoreClosest{prim, t}, counters);
    return 0;
}

// closest hit of a one-Bvh world with closest_hit_solo, on the plain node layout or the signed one (SNode):
// the two must agree bit for bit, counters included
extern "C" __attribute__((visibility("default"))) int hs_trace_closest_solo(shim_scene* s, const float* rays, int64_t n, float t_min,
                                                                           float t_max, int signed_nodes, int32_t* prim, float* t,
                                                                           uint64_t* counters) {
    if (s->flat.objects.size() != 1 || s->flat.objects[0].kind != OBJ_BVH || s->flat.objects[0].flags != 0) return -1;
    if (signed_nodes && s->flat.snodes.empty()) s->flat.build_signed_nodes();
    SceneView sv = view_of(s);
    uint64_t nodes = 0, prims = 0;
    for (int64_t i = 0; i < n; ++i) {
        const float* q = rays + i * 7;
        Ray r; r.o = mk3(q[0], q[1], q[2]); r.d = mk3(q[3], q[4], q[5]); r.time = q[6];
        TraceCounters tc; tc.nodes = 0; tc.prims = 0; tc.hrpp_tp = 0; tc.hrpp_fp = 0; tc.hrpp_none = 0;
        Hit h = signed_nodes ? closest_hit_solo<true, -1, true>(sv, r, t_min, t_max, &tc) : closest_hit_solo<true, -1, false>(sv, r, t_min, t_max, &tc);
        nodes += tc.nodes; prims += tc.prims;
        prim[i] = hit_handle(sv, h);
        t[i] = h.obj < 0 ? INFINITY : h.t;
    }
    if (counters) { counters[0] = (uint64_t)n; counters[1] = nodes; counters[2] = prims; }
    return 0;
}

// closest hit of a world with ONE Bvh object among plain objects, the Bvh walked on its quantised nodes (QNode, what
// wf_bvh1_walk reads): must equal the walk over the exact boxes in id and t; returns the number of QNodes or -1
extern "C" __attribute__((visibility("default"))) int hs_trace_closest_q(shim_scene* s, const float* rays, int64_t n, float t_min,
                                                                        float t_max, int32_t* prim, float* t, uint64_t* counters) {
    if (!quantise(s)) return -1;
    trace_batch<false, true, false>(s, rays, n, t_min, t_max, 0, StoreClosest{prim, t}, counters);
    return (int)s->flat.qnodes.size();
}

// trace_hit_kernel's walk and record words (out: 3 f4 per ray, shim_hit_record).  quantised = 1 walks the one Bvh
// object on its quantised nodes (-1 if the scene cannot have them), 0 the exact nodes.
extern "C" __attribute__((visibility("default"))) int hs_trace_hit(shim_scene* s, const float* rays, int64_t n, float t_min, float t_max,
                                                                  uint64_t seed, int quantised, f4* out, uint64_t* counters) {
    if (quantised && !quantise(s)) return -1;
    if (quantised) trace_batch<false, true, false>(s, rays, n, t_min, t_max, seed, StoreRecord{out}, counters);
    else trace_batch<false, false, false>(s, rays, n, t_min, t_max, seed, StoreRecord{out}, counters);
    return 0;
}

// trace_occluded_kernel's any-hit walk: out[i] = 1 where the walk accepts a hit.  quantised as in hs_trace_hit.
extern "C" __attribute__((visibility("default"))) int hs_trace_occluded(shim_scene* s, const float* rays, int64_t n, float t_min,
                                                                       float t_max, uint64_t seed, int quantised, uint8_t* out,
                                                                       uint64_t* counters) {
    if (quantised && !quantise(s)) return -1;
    if (quantised) trace_batch<false, true, true>(s, rays, n, t_min, t_max, seed, StoreOccluded{out}, counters);
    else trace_batch<false, false, true>(s, rays, n, t_min, t_max, seed, StoreOccluded{out}, counters);
    return 0;
}
// the QNode array (8 words per node) for inspection
extern "C" __attribute__((visibility("default"))) int hs_qnodes(shim_scene* s, uint32_t* out, int max_nodes) {
    int n = (int)s->flat.qnodes.size();
    if (out) memcpy(out, s->flat.qnodes.data(), sizeof(QNode) * (size_t)(n < max_nodes ? n : max_nodes));
    return n;
}

// the wavefront's per-path arithmetic, executed path by path (same order of operations as
// wf_generate / wf_extend / wf_shade)
extern "C" __attribute__((visibility("default"))) int hs_sample_radiance(shim_scene* s, const shim_camera* cam,
                                                                        const shim_render_params* p, const int32_t* xys, int64_t n,
                                                                        float* out_rgb, uint64_t* rays_out) {
    SceneView sv = view_of(s);
    CameraPod c;
    camera_new(cam->look_from, cam->look_at, cam->view_up, cam->vertical_fov, cam->aspect_ratio, cam->aperture, cam->focus_dist,
               cam->time_start, cam->time_end, c);
    uint64_t rays = 0;
    for (int64_t i = 0; i < n; ++i) {
        int x = xys[i * 3], y = xys[i * 3 + 1];
        uint32_t sample = (uint32_t)xys[i * 3 + 2], pixel = (uint32_t)(y * p->width + x);
        Rng rng;
        rng_init(rng, pixel, sample, p->seed);
        rng_key(rng, 0, STAGE_CAMERA);
        Ray r = camera_sample(c, x, y, p->width, p->height, rng);
        f3 thr = mk3(1, 1, 1), L = mk3(0, 0, 0);
        for (int bounce = 0; bounce < p->max_depth; ++bounce) {
            rng_init(rng, pixel, sample, p->seed);
            rng_key(rng, (uint32_t)bounce, STAGE_INTERSECT);
            ++rays;
            if (ray_has_nan(r)) break;  // as wf_extend: a NaN ray ends the path
            TraceCounters tc; tc.nodes = 0; tc.prims = 0; tc.hrpp_tp = 0; tc.hrpp_fp = 0; tc.hrpp_none = 0;
            Hit h = hrpp_on(s) ? closest_hit<false, true>(sv, r, 0.001f, INFINITY, rng, &tc) : closest_hit<false, false>(sv, r, 0.001f, INFINITY, rng, &tc);
            hrpp_count(s, tc);
            if (h.obj < 0) { L = L + mk3(thr.x * p->background[0], thr.y * p->background[1], thr.z * p->background[2]); break; }
            int mat = hit_material(sv, h);
            int kind = mat_kind(sv, mat);
            HitRec rec;
            reconstruct_hit(sv, r, h, mat_needs_uv(sv, mat), rec);
            if (kind == MAT_DIFFUSE_LIGHT) { L = L + thr * mat_emit(sv, mat, rec); break; }
            rng_init(rng, pixel, sample, p->seed);
            rng_key(rng, (uint32_t)bounce, STAGE_SCATTER);
            f3 att; Ray out;
            if (!mat_scatter(sv, kind, mat, r, rec, rng, att, out)) break;
            thr = thr * att;
            r = out;
        }
        out_rgb[i * 3] = L.x; out_rgb[i * 3 + 1] = L.y; out_rgb[i * 3 + 2] = L.z;
    }
    if (rays_out) *rays_out = rays;
    return 0;
}

namespace {
// the render's choice of the mesh pipeline (shim_api.cu: single_bvh_object, no medium): the index of the one Bvh object
// among plain objects, or -1
int split_object(const shim_scene* s) {
    if (s->has_media) return -1;
    int n_bvh = 0, idx = -1;
    for (size_t i = 0; i < s->flat.objects.size(); ++i) if (s->flat.objects[i].kind == OBJ_BVH) { ++n_bvh; idx = (int)i; }
    return n_bvh == 1 && s->flat.objects.size() > 1 ? idx : -1;
}

// one ray counted as wf_bvh1_list<COUNT = true> + wf_bvh1_walk<S, COUNT = true> count it: one primitive test per list
// object; the root's two child boxes against the closest list hit as the gate (not a node visit); if a box passes, the
// walk from the root bounded by that t.  The walk is bvh_closest's: same stack order, t_cull widening and tie rule.
void count_split(const SceneView& sv, int bo, const Ray& r, TraceCounters& tc) {
    float closest = INFINITY;
    for (int oi = 0; oi < sv.n_objects; ++oi) {
        if (oi == bo) continue;
        const DevObject& ob = sv.objects[oi];
        RayCtx pc;
        pc.r = object_ray(ob, r);
        float t; int face = 0;
        tc.prims++;
        if (hit_prim(sv, (uint32_t)ob.ref, pc, 0.001f, closest, t, face)) closest = t;
    }
    const DevObject& bob = sv.objects[bo];
    RayCtx c;
    make_ctx(c, object_ray(bob, r));
    const DevNode& rn = sv.nodes[bob.ref];
    float tl, tr;
    const bool need = slab(rn.a.x, rn.a.y, rn.a.z, rn.a.w, rn.b.x, rn.b.y, c, 0.001f, closest, tl) ||
                      (rn.d.y != CHILD_NONE && slab(rn.b.z, rn.b.w, rn.c.x, rn.c.y, rn.c.z, rn.c.w, c, 0.001f, closest, tr));
    if (!need) return;
    BvhBest best;
    bvh_closest<true>(sv, bob.ref, c, 0.001f, closest, best, &tc);
}
}  // namespace

// The paths of hs_sample_radiance (same samples, Philox keying and order of operations), counted as a counted render
// with a pool that holds every sample counts them.  Iteration j of such a render traces exactly the bounce-j rays, and
// the endgame (wf_tail) takes over from the first bounce b >= 1 that at most tail_threshold paths reach; its rays are
// counted as closest_hit counts them.  Rays of the iterations before are counted as the render's closest-hit kernels
// count them: the mesh pipeline's (count_split) for a world with one Bvh among plain objects and no medium, closest_hit's
// for every other world.  generic != 0 counts every ray as closest_hit does.  out: rays, node visits, primitive tests.
extern "C" __attribute__((visibility("default"))) int hs_render_counts(shim_scene* s, const shim_camera* cam, const shim_render_params* p,
                                                                      const int32_t* xys, int64_t n, uint32_t tail_threshold, int generic,
                                                                      uint64_t* out) {
    if (p->max_depth < 0 || p->max_depth > 255) return -1;
    SceneView sv = view_of(s);
    const int bo = generic ? -1 : split_object(s);
    CameraPod c;
    camera_new(cam->look_from, cam->look_at, cam->view_up, cam->vertical_fov, cam->aspect_ratio, cam->aperture, cam->focus_dist,
               cam->time_start, cam->time_end, c);
    // per bounce: rays traced, and node visits / primitive tests as closest_hit counts them and as the render's
    // iteration kernels count them
    std::vector<uint64_t> rays(256, 0), gen_nodes(256, 0), gen_prims(256, 0), it_nodes(256, 0), it_prims(256, 0);
    for (int64_t i = 0; i < n; ++i) {
        int x = xys[i * 3], y = xys[i * 3 + 1];
        uint32_t sample = (uint32_t)xys[i * 3 + 2], pixel = (uint32_t)(y * p->width + x);
        Rng rng;
        rng_init(rng, pixel, sample, p->seed);
        rng_key(rng, 0, STAGE_CAMERA);
        Ray r = camera_sample(c, x, y, p->width, p->height, rng);
        for (int bounce = 0; bounce < p->max_depth; ++bounce) {
            rng_init(rng, pixel, sample, p->seed);
            rng_key(rng, (uint32_t)bounce, STAGE_INTERSECT);
            ++rays[bounce];
            if (ray_has_nan(r)) break;  // as wf_extend: a NaN ray ends the path, nothing is walked
            TraceCounters tc; tc.nodes = 0; tc.prims = 0; tc.hrpp_tp = 0; tc.hrpp_fp = 0; tc.hrpp_none = 0;
            Hit h = closest_hit<true, false>(sv, r, 0.001f, INFINITY, rng, &tc);
            gen_nodes[bounce] += tc.nodes; gen_prims[bounce] += tc.prims;
            if (bo >= 0) {
                TraceCounters ts; ts.nodes = 0; ts.prims = 0; ts.hrpp_tp = 0; ts.hrpp_fp = 0; ts.hrpp_none = 0;
                count_split(sv, bo, r, ts);
                it_nodes[bounce] += ts.nodes; it_prims[bounce] += ts.prims;
            } else {
                it_nodes[bounce] += tc.nodes; it_prims[bounce] += tc.prims;
            }
            if (h.obj < 0) break;
            int mat = hit_material(sv, h);
            int kind = mat_kind(sv, mat);
            if (kind == MAT_DIFFUSE_LIGHT) break;
            HitRec rec;
            reconstruct_hit(sv, r, h, mat_needs_uv(sv, mat), rec);
            rng_init(rng, pixel, sample, p->seed);
            rng_key(rng, (uint32_t)bounce, STAGE_SCATTER);
            f3 att; Ray next;
            if (!mat_scatter(sv, kind, mat, r, rec, rng, att, next)) break;
            r = next;
        }
    }
    int endgame = 1;
    while (endgame < 256 && rays[endgame] > tail_threshold) ++endgame;
    out[0] = out[1] = out[2] = 0;
    for (int b = 0; b < 256; ++b) {
        out[0] += rays[b];
        out[1] += b < endgame ? it_nodes[b] : gen_nodes[b];
        out[2] += b < endgame ? it_prims[b] : gen_prims[b];
    }
    return 0;
}

extern "C" __attribute__((visibility("default"))) void hs_texture_value(shim_scene* s, int tex, float u, float v, const float* p,
                                                                       float* out) {
    SceneView sv = s->flat.view();
    f3 c = tex_value(sv, tex, u, v, mk3(p[0], p[1], p[2]));
    out[0] = c.x; out[1] = c.y; out[2] = c.z;
}

extern "C" __attribute__((visibility("default"))) void hs_philox(const uint32_t* ctr, const uint32_t* key, uint32_t* out) {
    philox4x32_10(ctr[0], ctr[1], ctr[2], ctr[3], key[0], key[1], out[0], out[1], out[2], out[3]);
}
