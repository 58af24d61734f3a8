// oracle_hit.cpp — TEST HARNESS ONLY.  The CPU oracle (oracle/shimmer_oracle.cpp, included whole and unchanged) plus
// orc_trace_hit: the oracle's whole HitRecord per ray, for the record-level parity of shim_trace_hit
// (tests/test_hit_records.py).  Built with the oracle's own flags into tests/records/_build/liborc_hit.so.
#include "../../oracle/shimmer_oracle.cpp"

// world.hit for each ray, the stream keyed as in orc_trace_closest.  out: 12 words per ray in the layout of
// shim_hit_record: point[3], normal[3], t, u, v (f32), front_face, material, hittable id (i32).
// A miss: t = +inf, material = hittable = -1, everything else 0.  counters (optional, 3 x u64): rays, node visits,
// primitive tests.
ORC_API int orc_trace_hit(void* sp, const float* rays, int64_t n, float t_min, float t_max, uint64_t seed, uint32_t* out,
                          uint64_t* counters) {
    Scene* s = (Scene*)sp;
    Ctx ctx; ctx.scene = s;
    for (int64_t i = 0; i < n; ++i) {
        const float* r = rays + i * 7;
        Ray ray{v3(r[0], r[1], r[2]), v3(r[3], r[4], r[5]), r[6]};
        Rng rng; rng.keyed = true; rng.pixel = (uint32_t)i; rng.sample = 0; rng.k0 = (uint32_t)seed; rng.k1 = (uint32_t)(seed >> 32);
        rng.key(0, STAGE_INTERSECT);
        ctx.rng = &rng;
        HitRecord rec;
        ctx.cnt.rays++;
        float f[9] = {0, 0, 0, 0, 0, 0, F32_INF, 0, 0};
        int32_t w[3] = {0, -1, -1};
        if (s->world.hit(ray, t_min, t_max, ctx, rec)) {
            float g[9] = {rec.point.x, rec.point.y, rec.point.z, rec.normal.x, rec.normal.y, rec.normal.z, rec.t, rec.u, rec.v};
            memcpy(f, g, sizeof f);
            w[0] = rec.front_face ? 1 : 0; w[1] = rec.material; w[2] = rec.prim_id;
        }
        memcpy(out + i * 12, f, sizeof f);
        memcpy(out + i * 12 + 9, w, sizeof w);
    }
    if (counters) { counters[0] = ctx.cnt.rays; counters[1] = ctx.cnt.node_visits; counters[2] = ctx.cnt.prim_tests; }
    return 0;
}
