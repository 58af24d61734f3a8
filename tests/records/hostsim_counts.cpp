// hostsim_counts.cpp — TEST HARNESS ONLY.  The occlusion harness (tests/records/hostsim_occluded.cpp, which includes the
// record harness and the hostsim harness whole; all unchanged) plus hs_render_counts: the rays, node visits and primitive
// tests of a counted render (SHIM_RENDER_COUNT_NODES), path by path on the CPU, for tests/test_counters.py.  Built into
// tests/records/_build/libhostsim_counts.so by tests/counters_support.py.
#include "hostsim_occluded.cpp"

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
