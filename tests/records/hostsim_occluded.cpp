// hostsim_occluded.cpp — TEST HARNESS ONLY.  The record harness (tests/records/hostsim_hit.cpp, which includes the
// hostsim harness whole; both unchanged) plus hs_trace_occluded: trace_occluded_kernel's arithmetic run ray by ray on
// the CPU, for the occlusion query's parity (tests/test_occlusion.py).  Built into
// tests/records/_build/libhostsim_occluded.so by tests/occlusion_support.py.
#include "hostsim_hit.cpp"

// closest_hit<..., ANY = true> as trace_occluded_kernel runs it: out[i] = 1 where the walk accepts a hit.  quantised as
// in hs_trace_hit (1: the one Bvh object on its quantised nodes, -1 if the scene cannot have them; 0: the exact nodes
// with node counting).
extern "C" __attribute__((visibility("default"))) int hs_trace_occluded(shim_scene* s, const float* rays, int64_t n, float t_min,
                                                                       float t_max, uint64_t seed, int quantised, uint8_t* out,
                                                                       uint64_t* counters) {
    if (quantised) {
        int idx = -1, n_bvh = 0;
        for (size_t i = 0; i < s->flat.objects.size(); ++i) if (s->flat.objects[i].kind == OBJ_BVH) { ++n_bvh; idx = (int)i; }
        if (n_bvh != 1) return -1;
        if (s->flat.q_object != idx && !s->flat.build_quantized_nodes(idx)) return -1;
    }
    SceneView sv = s->flat.view();
    uint64_t nodes = 0, prims = 0;
    for (int64_t i = 0; i < n; ++i) {
        const float* q = rays + i * 7;
        Ray r; r.o = mk3(q[0], q[1], q[2]); r.d = mk3(q[3], q[4], q[5]); r.time = q[6];
        Rng rng;
        rng_init(rng, (uint32_t)i, 0, seed);
        rng_key(rng, 0, STAGE_INTERSECT);
        TraceCounters tc; tc.nodes = 0; tc.prims = 0; tc.hrpp_tp = 0; tc.hrpp_fp = 0; tc.hrpp_none = 0;
        Hit h = quantised ? closest_hit<true, false, true, true, true>(sv, r, t_min, t_max, rng, &tc)
                          : closest_hit<true, false, true, false, true>(sv, r, t_min, t_max, rng, &tc);
        nodes += tc.nodes; prims += tc.prims;
        out[i] = h.obj >= 0 ? 1 : 0;
    }
    if (counters) { counters[0] = (uint64_t)n; counters[1] = nodes; counters[2] = prims; }
    return 0;
}
