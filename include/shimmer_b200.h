/* shimmer_b200.h — C ABI of the B200 path-tracing backend for the `shimmer` crate.
 *
 * Drop-in boundary: the reference's `Renderer::render` (reference src/renderer.rs:42-52,
 * called from src/main.rs:168-179).  The reference has no FFI; its "operator API" is the
 * three traits Hittable / Material / Texture (hittable.rs:64-82, materials/material.rs:16-23,
 * textures/texture.rs:3-5) whose implementors are built through the constructors cited on
 * each entry point below.  A Rust host keeps those constructors and has each of them also
 * record its arguments through the matching call here (INTEGRATION.md shows the binding);
 * trait objects never cross the boundary.
 *
 * Conventions
 *  - every call returns an int: >= 0 success (ids count from 0 per kind, in creation order),
 *    < 0 a shim_status error; shim_last_error() returns the message for the calling thread.
 *    Nothing aborts or throws across the boundary.
 *  - the caller owns every buffer it passes in or receives results in; inputs are copied at
 *    the call; device memory belongs to the scene handle and is freed by shim_scene_destroy.
 *  - a scene handle is single-caller (not re-entrant); shim_render blocks.
 *  - there is NO CPU fallback: if no CUDA device is usable every device call fails with
 *    SHIM_ERR_CUDA.
 */
#ifndef SHIMMER_B200_H
#define SHIMMER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct shim_scene shim_scene;

typedef enum shim_status {
    SHIM_OK = 0,
    SHIM_ERR_INVALID = -1,     /* bad id / argument */
    SHIM_ERR_UNSUPPORTED = -2, /* nesting the device interpreter does not implement */
    SHIM_ERR_CUDA = -3,        /* CUDA runtime error (message has the detail) */
    SHIM_ERR_STATE = -4        /* call order (e.g. render before commit) */
} shim_status;

const char* shim_last_error(void);
int shim_version(void);

/* ---- scene lifetime ------------------------------------------------------------------ */
shim_scene* shim_scene_create(void);
void shim_scene_destroy(shim_scene* s);

/* ---- textures: textures/solid_color.rs:12-18, checker.rs:12-24, marble.rs:12-20,
 *      image_texture.rs:12-17 ------------------------------------------------------------ */
int shim_texture_solid(shim_scene* s, float r, float g, float b);
int shim_texture_checker(shim_scene* s, float scale, int even_tex, int odd_tex);
/* Marble::new draws a random Perlin seed; the caller passes it so renders are reproducible */
int shim_texture_marble(shim_scene* s, float scale, uint32_t perlin_seed);
/* ImageTexture::new(path): the host decodes the file and hands over tightly packed RGB8 */
int shim_texture_image(shim_scene* s, const uint8_t* rgb8, int width, int height);

/* ---- materials: lambertian.rs:21-31, metal.rs:16-23, dialectric.rs:19-24,
 *      diffuse_light.rs:13-23, isotropic.rs:19-29 ---------------------------------------- */
int shim_material_lambertian(shim_scene* s, int albedo_tex);
int shim_material_metal(shim_scene* s, float r, float g, float b, float fuzz);
int shim_material_dielectric(shim_scene* s, float index_of_refraction);
int shim_material_diffuse_light(shim_scene* s, int emission_tex);
int shim_material_isotropic(shim_scene* s, int albedo_tex);

/* ---- hittables (ids are the primitive ids shim_trace_closest reports) ------------------
 * Sphere::new sphere.rs:26; MovingSphere::new moving_sphere.rs:29; XyRect/XzRect/YzRect::new
 * rectangle.rs:24/86/148; Tri::new triangle.rs:21; Cube::new cube.rs:23 */
int shim_sphere(shim_scene* s, float cx, float cy, float cz, float radius, int material);
int shim_moving_sphere(shim_scene* s, float c0x, float c0y, float c0z, float c1x, float c1y, float c1z,
                       float time_start, float time_end, float radius, int material);
int shim_xy_rect(shim_scene* s, float x0, float x1, float y0, float y1, float z, int material);
int shim_xz_rect(shim_scene* s, float x0, float x1, float z0, float z1, float y, int material);
int shim_yz_rect(shim_scene* s, float y0, float y1, float z0, float z1, float x, int material);
int shim_tri(shim_scene* s, const float* p0p1p2 /* 9 floats */, int material);
int shim_cube(shim_scene* s, float minx, float miny, float minz, float maxx, float maxy, float maxz, int material);
/* HittableList::new / add, hittable.rs:89-97 */
int shim_list_create(shim_scene* s);
int shim_list_add(shim_scene* s, int list, int hittable);
/* main.rs:745-789 load_to_tris: n triangles (9 floats each) appended to `list`; returns the first id */
int shim_tris_bulk(shim_scene* s, const float* xyz, int n_tris, int material, int list);
/* Bvh::new / Bvh::with_predictor, bvh.rs:46-81.  The tree is built on the host exactly as
 * BvhNode::new_helper does (bvh.rs:249-333): per-node random axis (here: splitmix64(seed)),
 * stable sort on bounding_box(0,0).min[axis], median split, post-order node indices. */
int shim_bvh(shim_scene* s, int list, float time0, float time1, uint64_t axis_seed, int with_predictor);
/* A caller-built tree (the Rust side keeps its own Bvh): per node left/right are >= 0 for a
 * node index or ~hittable_id for a primitive child; boxes are recomputed by the library. */
int shim_bvh_from_nodes(shim_scene* s, int n_nodes, const int32_t* left, const int32_t* right, int root,
                        float time0, float time1, int with_predictor);
/* Translate::new instance.rs:23, RotateY::new instance.rs:63, ConstantMedium::new hittable.rs:151 */
int shim_translate(shim_scene* s, int hittable, float dx, float dy, float dz);
int shim_rotate_y(shim_scene* s, int hittable, float degrees);
int shim_constant_medium(shim_scene* s, int boundary, float density, int albedo_tex);
/* the `world: &HittableList` argument of render, in list order */
int shim_world_add(shim_scene* s, int hittable);
/* Scene options, set before shim_commit.  SHIM_OPT_DEVICE_BVH: which tree the kernels walk for each
 * Bvh — a binned-SAH rebuild of its primitive list (default; results do not depend on the tree) or the
 * recorded bvh.rs topology (node indices then equal the reference's, e.g. for HRPP comparisons). */
enum { SHIM_OPT_DEVICE_BVH = 1 };
enum { SHIM_DEVICE_BVH_SAH = 0, SHIM_DEVICE_BVH_REFERENCE = 1 };
int shim_scene_set_option(shim_scene* s, int option, int value);
/* flattens the world into SoA arrays and uploads them to the current CUDA device */
int shim_commit(shim_scene* s);

/* introspection (tests, stats) */
int shim_bvh_info(shim_scene* s, int bvh, int* n_nodes, int* root, int* height);
int shim_bvh_nodes(shim_scene* s, int bvh, int32_t* left, int32_t* right, int32_t* parent, float* boxes6);
uint64_t shim_scene_device_bytes(shim_scene* s);

/* ---- camera: the nine Camera::new arguments, camera.rs:44-54 -------------------------- */
typedef struct shim_camera {
    float look_from[3], look_at[3], view_up[3];
    float vertical_fov, aspect_ratio, aperture, focus_dist, time_start, time_end;
} shim_camera;

/* ---- render: Renderer::render, renderer.rs:42-105 -------------------------------------- */
enum { SHIM_RENDER_RAW_SUM = 1, SHIM_RENDER_PREDICTORS = 2, SHIM_RENDER_COUNT_NODES = 4,
       SHIM_RENDER_PROFILE = 8 /* CUDA events around every wf_extend launch -> stats.extend_ms */,
       SHIM_RENDER_KEEP_PREDICTORS = 16 /* with PREDICTORS: keep what earlier renders of this scene learnt (the reference
                                           builds fresh Predictors with every scene, bvh.rs:69-81: default = clear) */ };
typedef struct shim_render_params {
    int32_t width, height;         /* Renderer::new */
    int32_t samples_per_pixel;     /* divisor of the mean */
    int32_t max_depth;
    int32_t tile_width, tile_height; /* Tile::tile order drives the device ray queue order */
    float background[3];
    uint64_t seed;                 /* Philox key */
    int32_t sample_begin;          /* first absolute sample index rendered by this call */
    int32_t sample_count;          /* samples per pixel rendered by this call; 0 = samples_per_pixel, -1 = none
                                      (a shard that owns no samples: the framebuffer comes back zero) */
    int32_t tile_rank, tile_world; /* tile sharding: this call renders tiles with index % world == rank (world 0/1 = all) */
    int32_t flags;                 /* SHIM_RENDER_* */
    int32_t pool_paths;            /* wavefront pool size; 0 = default */
} shim_render_params;

typedef struct shim_stats {
    uint64_t rays;                 /* world.hit calls issued by the integrator, ray.rs:44 */
    uint64_t samples;              /* ray_color invocations, renderer.rs:145 */
    uint64_t node_visits, prim_tests; /* only with SHIM_RENDER_COUNT_NODES: inner BVH nodes whose two child boxes were
                                      tested, and primitive intersection tests, summed over every ray of the render
                                      (the endgame's included).  A counted render walks the exact 64-byte nodes with
                                      its own kernels, not the ones a timed render of the scene runs: the generic
                                      closest hit (the world list in order, each Bvh culled by the closest hit so far),
                                      or for a world with one Bvh among plain objects and no medium the mesh pipeline
                                      (one test per list object, the root's child boxes as an uncounted gate against the
                                      closest list hit, then the walk from the root).  The signed-node walk of the
                                      one-Bvh kernels visits the same nodes; the quantised walk of the mesh kernels
                                      visits about 4 % more. */
    uint64_t hrpp_true_positive, hrpp_false_positive, hrpp_no_prediction;
    uint64_t kernel_launches;
    uint64_t iterations;
    double device_ms;              /* CUDA events around the wavefront loop */
    double extend_ms, shade_ms, generate_ms; /* event sums per kernel class (extend only, with SHIM_RENDER_PROFILE) */
    uint64_t extend_launches;      /* wf_extend launches that had rays, covered by extend_ms */
    uint64_t extend_variant;       /* which closest-hit kernel ran: 0 wf_extend, 1 wf_bvh1_list + wf_bvh1_walk + wf_bvh1_finish, 2 wf_extend_solo, 3 wf_extend_list, 4 wf_trace_solo */
    uint64_t pool_paths;           /* paths in flight this render was given (min(samples, 2^24) unless pool_paths says otherwise) */
    uint64_t pool_bytes;           /* device memory of the wavefront pool(s) after this render (queues, counters, framebuffers) */
    uint64_t devices;              /* devices that rendered (1 except for shim_render_multi) */
    double wall_ms;                /* host wall time of the whole call incl. the framebuffer copy (shim_render, shim_render_multi) */
} shim_stats;

/* host framebuffer: width*height*3 floats, linear radiance, row-major, y = 0 is the bottom row
 * (ImageColors, renderer.rs:168-194) */
int shim_render(shim_scene* s, const shim_camera* cam, const shim_render_params* p, float* out_rgb, shim_stats* stats);
/* Page-locked host memory for the framebuffer a renderer reuses across calls (the Vec behind ImageColors,
 * renderer.rs:168-194).  shim_render copies straight into a buffer obtained here (one D2H, no staging);
 * any other host pointer works too and goes through the library's pinned staging buffer.  Needs a CUDA device. */
float* shim_host_alloc(size_t floats);
void shim_host_free(float* p);
/* same, into a device buffer of the current device on `cuda_stream` (0 = default stream) */
int shim_render_device(shim_scene* s, const shim_camera* cam, const shim_render_params* p, float* d_out_rgb,
                       shim_stats* stats, void* cuda_stream);

/* One image on several devices of this process — the tile fan-out of Renderer::render (renderer.rs:63-95) across
 * GPUs instead of threads.  The scene is replicated on first use; device i renders its shard on its own host thread
 * and stream with private accumulation (SHIM_SHARD_SAMPLES: a contiguous range of absolute sample indices;
 * SHIM_SHARD_TILES: the tiles with index % n_devices == i); the sums are combined once at the end on devices[0]
 * (peer copies + add) and the mean lands in out_rgb (host).  devices = NULL: ordinals 0 .. n_devices-1;
 * n_devices <= 0: every device.  stats: rays/samples summed, device_ms = the slowest device's loop. */
enum { SHIM_SHARD_SAMPLES = 0, SHIM_SHARD_TILES = 1 };
int shim_render_multi(shim_scene* s, const shim_camera* cam, const shim_render_params* p, int n_devices, const int* devices,
                      int mode, float* out_rgb, shim_stats* stats);
/* Releases every device's wavefront pool (queues, graphs, events, staging buffers).  Scenes stay valid; the next
 * render allocates again.  No render may be in flight.  shim_pool_bytes: what a device's pool holds right now. */
int shim_shutdown(void);
uint64_t shim_pool_bytes(int device);

/* ---- gate 1: closest hit for a batch of rays (Hittable::hit on the world, hittable.rs:100-118)
 * rays: n x 7 floats (origin, direction, time).  prim_id: hittable id or -1; t: hit parameter
 * (+inf on a miss).  Volume objects draw from the Philox stream keyed (ray index, 0, STAGE_INTERSECT). */
int shim_trace_closest(shim_scene* s, const float* rays, int64_t n, float t_min, float t_max, uint64_t seed,
                       int32_t* prim_id, float* t, uint64_t* counters3 /* optional: rays, node visits, prim tests */);
int shim_trace_closest_device(shim_scene* s, const float* d_rays, int64_t n, float t_min, float t_max, uint64_t seed,
                              int32_t* d_prim_id, float* d_t, void* cuda_stream);

/* Hittable::hit on the world (hittable.rs:100-118) with the whole HitRecord (hittable.rs:15-52).  48 bytes.
 * The same rays, walk and Philox stream as shim_trace_closest: `hittable` and `t` equal its prim_id and t bit for bit.
 * A miss is hittable = -1, material = -1, t = +inf and every other field 0.  The record is what the reference's
 * hit() chain returns: sphere / moving-sphere uv are always evaluated (sphere.rs:41-46); a RotateY hit carries the
 * normal set_face_normal gave it with the rotated ray and the front_face of the inner hit, untouched
 * (instance.rs:124-141); a Translate hit has the offset added to its point (instance.rs:40-42).  A ConstantMedium hit is
 * normal (1, 0, 0), u = v = 0, front_face = 1 (hittable.rs:216-231), and its material is the Isotropic that
 * shim_constant_medium allotted: the next material id after those created so far, taken at that call, so a
 * medium's phase material is numbered among the shim_material_* ids in call order. */
typedef struct shim_hit_record {
    float point[3], normal[3];  /* world space; normal face-forwarded as HitRecord::new / set_face_normal leave it */
    float t, u, v;
    int32_t front_face;         /* 1 / 0 */
    int32_t material;           /* material id; a ConstantMedium hit reports the Isotropic that shim_constant_medium allotted */
    int32_t hittable;           /* the id shim_trace_closest reports; -1 = miss */
} shim_hit_record;
int shim_trace_hit(shim_scene* s, const float* rays, int64_t n, float t_min, float t_max, uint64_t seed,
                   shim_hit_record* out, uint64_t* counters3 /* optional, as shim_trace_closest */);
/* same on device buffers of the scene's device (it must be current), launched on `cuda_stream` (0 = default stream);
 * d_out must be 16-byte aligned (each record is written as three 16-byte stores) */
int shim_trace_hit_device(shim_scene* s, const float* d_rays, int64_t n, float t_min, float t_max, uint64_t seed,
                          shim_hit_record* d_out, void* cuda_stream);

/* Occlusion (any hit): is anything hit on the ray with t in [t_min, t_max]?  occluded[i] = 1 / 0, one byte per ray.
 * The walk stops at the first hit it accepts instead of searching for the closest one, on the same rays, node layouts
 * and Philox stream as shim_trace_closest (a medium draws its free path from the same stream), and
 *     occluded[i] == (shim_trace_closest(s, rays, n, t_min, t_max, seed, ...).prim_id[i] >= 0)
 * for every ray, bit for bit; its node visits and primitive tests (counters3) are never more than that query's.
 * Visibility between two points a and b (shadow rays, ambient occlusion, "can the camera see p"): origin = a,
 * direction = b - a (not normalised), t in [eps, 1 - eps], e.g. eps = 1e-3; occluded = 0 means a sees b.
 * Errors as shim_trace_closest; nothing is written on error. */
int shim_trace_occluded(shim_scene* s, const float* rays, int64_t n, float t_min, float t_max, uint64_t seed,
                        uint8_t* occluded, uint64_t* counters3 /* optional: rays, node visits, prim tests */);
/* same on device buffers of the scene's device (it must be current), launched on `cuda_stream` (0 = default stream) */
int shim_trace_occluded_device(shim_scene* s, const float* d_rays, int64_t n, float t_min, float t_max, uint64_t seed,
                               uint8_t* d_occluded, void* cuda_stream);

/* ---- host helpers that mirror reference functions (no device needed) ------------------- */
/* Tile::tile, renderer.rs:242-296: writes up to cap tiles as (width, height, x0, y0); returns the count */
int shim_tile_layout(int image_width, int image_height, int tile_width, int tile_height, int32_t* out4, int cap);
/* Camera::new derived fields: origin, horizontal, vertical, lower_left_corner, u, v (18 floats), lens_radius, t0, t1 */
int shim_camera_fields(const shim_camera* cam, float* out21);
/* Aabb::hit, aabb.rs:28-41, evaluated the way the kernels do it (reciprocal direction, fused multiply-add per
 * plane, a zero direction component clamped to +-1e-30 instead of an infinite reciprocal): 1 hit, 0 miss.
 * layout 0: the 64-byte node's slab test; layout 1: the signed shared-memory node of the one-Bvh kernels. */
int shim_aabb_hit(const float* min3, const float* max3, const float* origin3, const float* direction3, float t_min, float t_max,
                  int layout);
/* hrpp::hash, hrpp.rs:174-193 */
uint64_t shim_hrpp_hash(const float* origin3, const float* direction3);
/* Renderer::write_ppm, renderer.rs:107-127: P3 text, no gamma, top row first; returns bytes written or < 0 */
int64_t shim_write_ppm(const float* rgb, int width, int height, const char* path /* NULL = stdout */);

#ifdef __cplusplus
}
#endif
#endif /* SHIMMER_B200_H */
