"""Generates rust/shimmer-patch/shimmer-b200.patch: the changes to the reference crate (a checkout of
jalberse/RayTracingInOneWeekendInRust) that route Renderer::render through libshimmer_b200.

    python rust/shimmer-patch/make_patch.py REFERENCE_CHECKOUT [OUT]     (OUT: the committed patch by default)

It copies Cargo.toml and src/ of the reference to a temporary tree, applies the edits below, adds src/backend.rs
(rust/shimmer-patch/backend.rs) and writes the unified diff (-U2, paths a/ b/: apply with `patch -p1` or `git apply`).
Every edit names the exact reference text it replaces and fails if that text is not found exactly once, so a changed
upstream is noticed here and not as a bad hunk.  No Rust toolchain exists in this image: the patch is checked to apply
(tests/test_rust_binding.py), it has not been compiled."""
import shutil
import subprocess
import sys
import tempfile
from pathlib import Path

HERE = Path(__file__).resolve().parent

REC_T = "    fn record(&self, r: &mut crate::backend::Recorder) -> shimmer_b200::Result<shimmer_b200::TextureId> {\n"
REC_M = "    fn record(&self, r: &mut crate::backend::Recorder) -> shimmer_b200::Result<shimmer_b200::MaterialId> {\n"
REC_H = "    fn record(&self, r: &mut crate::backend::Recorder) -> shimmer_b200::Result<shimmer_b200::HittableId> {\n"


def after(line, body):
    """insert `body` right after the (unique) line `line`"""
    return (line, line + body)


EDITS = {
    "Cargo.toml": [("rayon = \"1.6.1\"\n", "rayon = \"1.6.1\"\nshimmer-b200 = { path = \"../rust/shimmer-b200\" }\n")],
    "src/lib.rs": [("mod aabb;\n", "mod aabb;\npub mod backend;\n")],
    # ---------------------------------------------------------------- traits: one provided method each
    "src/textures/texture.rs": [after("    fn value(&self, u: f32, v: f32, p: &Vec3) -> Vec3;\n",
        "    /// Describes this texture to the device backend (backend.rs).  User-defined textures keep this default.\n"
        "    fn record(&self, _r: &mut crate::backend::Recorder) -> shimmer_b200::Result<shimmer_b200::TextureId> {\n"
        "        Err(crate::backend::unsupported(\"a user-defined Texture\"))\n    }\n")],
    "src/materials/material.rs": [after("    fn scatter(&self, ray: &Ray, hit_record: &HitRecord) -> Option<ScatterRecord>;\n",
        "    /// Describes this material to the device backend (backend.rs).  User-defined materials keep this default.\n"
        "    fn record(&self, _r: &mut crate::backend::Recorder) -> shimmer_b200::Result<shimmer_b200::MaterialId> {\n"
        "        Err(crate::backend::unsupported(\"a user-defined Material\"))\n    }\n")],
    "src/hittable.rs": [
        after("    fn bounding_box(&self, time_0: f32, time_1: f32) -> Option<Aabb>;\n",
              "    /// Describes this object to the device backend (backend.rs).  User-defined hittables keep this default.\n"
              "    fn record(&self, _r: &mut crate::backend::Recorder) -> shimmer_b200::Result<shimmer_b200::HittableId> {\n"
              "        Err(crate::backend::unsupported(\"a user-defined Hittable\"))\n    }\n"),
        after("impl Hittable for HittableList {\n", REC_H +
              "        let list = r.scene.list()?;\n        for o in &self.objects {\n            let h = r.hittable(o)?;\n"
              "            r.scene.list_add(list, h)?;\n        }\n        Ok(list)\n    }\n"),
        ("    phase_function: Arc<dyn Material>,\n    neg_inv_density: f32,\n}\n",
         "    phase_function: Arc<dyn Material>,\n    neg_inv_density: f32,\n    density: f32,\n    albedo: Arc<dyn Texture>,\n}\n"),
        ("            phase_function: Arc::new(Isotropic::new(texture)),\n            neg_inv_density: -1.0 / density,\n",
         "            phase_function: Arc::new(Isotropic::new(texture.clone())),\n            neg_inv_density: -1.0 / density,\n"
         "            density,\n            albedo: texture,\n"),
        ("        ConstantMedium {\n            boundary,\n            phase_function: Arc::new(Isotropic::from_color(color)),\n"
         "            neg_inv_density: -1.0 / density,\n",
         "        let albedo: Arc<dyn Texture> = Arc::new(crate::textures::solid_color::SolidColor::new(color));\n"
         "        ConstantMedium {\n            boundary,\n            phase_function: Arc::new(Isotropic::new(albedo.clone())),\n"
         "            neg_inv_density: -1.0 / density,\n            density,\n            albedo,\n"),
        after("impl Hittable for ConstantMedium {\n", REC_H +
              "        let b = r.hittable(&self.boundary)?;\n        let t = r.texture(&self.albedo)?;\n"
              "        r.scene.constant_medium(b, self.density, t)\n    }\n"),
    ],
    # ---------------------------------------------------------------- textures
    "src/textures/solid_color.rs": [after("impl Texture for SolidColor {\n", REC_T +
        "        r.scene.texture_solid(self.color.x, self.color.y, self.color.z)\n    }\n")],
    "src/textures/checker.rs": [after("impl Texture for Checker {\n", REC_T +
        "        let even = r.texture(&self.even)?;\n        let odd = r.texture(&self.odd)?;\n"
        "        r.scene.texture_checker(self.scale, even, odd)\n    }\n")],
    "src/textures/marble.rs": [
        ("    scale: f32,\n}\n", "    scale: f32,\n    /// the seed given to Perlin::new (the device rebuilds the permutation tables from it)\n    seed: u32,\n}\n"),
        ("        let perlin = Perlin::new(random::<u32>());\n", "        let seed = random::<u32>();\n        let perlin = Perlin::new(seed);\n"),
        ("        Marble { noise: turb, scale }\n", "        Marble { noise: turb, scale, seed }\n"),
        after("impl Texture for Marble {\n", REC_T + "        r.scene.texture_marble(self.scale, self.seed)\n    }\n"),
    ],
    "src/textures/image_texture.rs": [after("impl Texture for ImageTexture {\n", REC_T +
        "        r.scene.texture_image(self.image.as_raw(), self.image.width(), self.image.height())\n    }\n")],
    # ---------------------------------------------------------------- materials
    "src/materials/lambertian.rs": [after("impl Material for Lambertian {\n", REC_M +
        "        let t = r.texture(&self.albedo)?;\n        r.scene.lambertian(t)\n    }\n")],
    "src/materials/metal.rs": [after("impl Material for Metal {\n", REC_M +
        "        r.scene.metal(crate::backend::v3(self.albedo), self.fuzz)\n    }\n")],
    "src/materials/dialectric.rs": [after("impl Material for Dialectric {\n", REC_M +
        "        r.scene.dielectric(self.index_of_refraction)\n    }\n")],
    "src/materials/diffuse_light.rs": [after("impl Material for DiffuseLight {\n", REC_M +
        "        let t = r.texture(&self.emission_texture)?;\n        r.scene.diffuse_light(t)\n    }\n")],
    "src/materials/isotropic.rs": [after("impl Material for Isotropic {\n", REC_M +
        "        let t = r.texture(&self.albedo)?;\n        r.scene.isotropic(t)\n    }\n")],
    # ---------------------------------------------------------------- geometry
    "src/geometry/sphere.rs": [after("impl Hittable for Sphere {\n", REC_H +
        "        let m = r.material(&self.material)?;\n        r.scene.sphere(crate::backend::v3(self.center), self.radius, m)\n    }\n")],
    "src/geometry/moving_sphere.rs": [after("impl Hittable for MovingSphere {\n", REC_H +
        "        let m = r.material(&self.material)?;\n"
        "        r.scene.moving_sphere(crate::backend::v3(self.center_start), crate::backend::v3(self.center_end), self.time_start, self.time_end, self.radius, m)\n    }\n")],
    "src/geometry/rectangle.rs": [
        after("impl Hittable for XyRect {\n", REC_H + "        let m = r.material(&self.material)?;\n"
              "        r.scene.xy_rect(self.x0, self.x1, self.y0, self.y1, self.z, m)\n    }\n"),
        after("impl Hittable for XzRect {\n", REC_H + "        let m = r.material(&self.material)?;\n"
              "        r.scene.xz_rect(self.x0, self.x1, self.z0, self.z1, self.y, m)\n    }\n"),
        after("impl Hittable for YzRect {\n", REC_H + "        let m = r.material(&self.material)?;\n"
              "        r.scene.yz_rect(self.y0, self.y1, self.z0, self.z1, self.x, m)\n    }\n"),
    ],
    "src/geometry/triangle.rs": [after("impl Hittable for Tri {\n", REC_H +
        "        let m = r.material(&self.material)?;\n"
        "        r.scene.tri(crate::backend::v3(self.p0), crate::backend::v3(self.p1), crate::backend::v3(self.p2), m)\n    }\n")],
    "src/geometry/cube.rs": [
        ("    sides: HittableList,\n}\n", "    sides: HittableList,\n    material: Arc<dyn Material>,\n}\n"),
        ("        let mut sides = HittableList::new();\n", "        let material_kept = material.clone();\n        let mut sides = HittableList::new();\n"),
        ("            max_point,\n            sides,\n        }\n", "            max_point,\n            sides,\n            material: material_kept,\n        }\n"),
        after("impl Hittable for Cube {\n", REC_H + "        let m = r.material(&self.material)?;\n"
              "        r.scene.cube(crate::backend::v3(self.min_point), crate::backend::v3(self.max_point), m)\n    }\n"),
    ],
    "src/geometry/instance.rs": [
        after("impl Hittable for Translate {\n", REC_H + "        let h = r.hittable(&self.hittable)?;\n"
              "        r.scene.translate(h, crate::backend::v3(self.displacement))\n    }\n"),
        ("    cos_theta: f32,\n    bbox: Option<Aabb>,\n}\n", "    cos_theta: f32,\n    bbox: Option<Aabb>,\n    degrees: f32,\n}\n"),
        ("            cos_theta,\n            bbox,\n        }\n", "            cos_theta,\n            bbox,\n            degrees,\n        }\n"),
        after("impl Hittable for RotateY {\n", REC_H + "        let h = r.hittable(&self.hittable)?;\n"
              "        r.scene.rotate_y(h, self.degrees)\n    }\n"),
    ],
    # ---------------------------------------------------------------- bvh.rs: the crate keeps its own tree and uploads the topology
    "src/bvh.rs": [
        ("    nodes: Vec<BvhNode>,\n    max_depth: u32,\n}\n", "    nodes: Vec<BvhNode>,\n    max_depth: u32,\n    time_0: f32,\n    time_1: f32,\n}\n"),
        ("            nodes,\n            max_depth,\n        }\n", "            nodes,\n            max_depth,\n            time_0,\n            time_1,\n        }\n"),
        after("impl Hittable for Bvh {\n", REC_H +
              "        // node indices are the crate's own (post-order, bvh.rs:249-333), so the leaf indices HRPP stores agree\n"
              "        let mut left = Vec::with_capacity(self.nodes.len());\n        let mut right = Vec::with_capacity(self.nodes.len());\n"
              "        for node in &self.nodes {\n            for (child, out) in [(&node.left, &mut left), (&node.right, &mut right)] {\n"
              "                out.push(match child {\n                    Child::Index(i) => *i as i32,\n"
              "                    Child::Hittable(h) => !r.hittable(h)?.0, // ~id marks a primitive child\n                });\n"
              "            }\n        }\n        let with_predictor = r.predictor_bvhs.contains(&self.id);\n"
              "        r.scene.bvh_from_nodes(&left, &right, self.root_index, self.time_0, self.time_1, with_predictor)\n    }\n"),
    ],
    # ---------------------------------------------------------------- camera.rs: keep the nine arguments
    "src/camera.rs": [
        ("    /// Shutter close time\n    time_end: f32,\n}\n",
         "    /// Shutter close time\n    time_end: f32,\n    /// the arguments of `new`, kept for the device backend (which derives the same fields)\n"
         "    pod: shimmer_b200::Camera,\n}\n"),
        ("            lens_radius,\n            time_start,\n            time_end,\n        }\n    }\n",
         "            lens_radius,\n            time_start,\n            time_end,\n            pod: shimmer_b200::Camera {\n"
         "                look_from: [look_from.x, look_from.y, look_from.z],\n                look_at: [look_at.x, look_at.y, look_at.z],\n"
         "                view_up: [view_up.x, view_up.y, view_up.z],\n                vertical_fov: vertical_field_of_view,\n"
         "                aspect_ratio,\n                aperture,\n                focus_dist,\n                time_start,\n                time_end,\n"
         "            },\n        }\n    }\n\n    pub fn to_pod(&self) -> shimmer_b200::Camera {\n        self.pod\n    }\n"),
    ],
    # ---------------------------------------------------------------- renderer.rs: render goes to the device
    "src/renderer.rs": [
        ("        let stderr = io::stderr();\n        let mut stderr_buf_writer = io::BufWriter::new(stderr);\n\n        let tiles = Tile::tile(",
         "        if std::env::var_os(\"SHIMMER_CPU\").is_none() {\n            // the B200 backend: same arguments, same PPM on stdout (backend.rs)\n"
         "            return crate::backend::render_on_device(\n                self.image_width,\n                self.image_height,\n                camera,\n"
         "                world,\n                background,\n                samples_per_pixel,\n                max_depth,\n                tile_width,\n"
         "                tile_height,\n                &predictors,\n            );\n        }\n"
         "        let stderr = io::stderr();\n        let mut stderr_buf_writer = io::BufWriter::new(stderr);\n\n        let tiles = Tile::tile("),
    ],
}


def main():
    if not 2 <= len(sys.argv) <= 3:
        sys.exit(__doc__)
    REF = Path(sys.argv[1])
    OUT = Path(sys.argv[2]) if len(sys.argv) > 2 else HERE / "shimmer-b200.patch"
    tmp = Path(tempfile.mkdtemp(prefix="shimmer_patch_"))
    for side in ("a", "b"):
        (tmp / side).mkdir()
        shutil.copy(REF / "Cargo.toml", tmp / side / "Cargo.toml")
        shutil.copytree(REF / "src", tmp / side / "src")
    for rel, edits in EDITS.items():
        p = tmp / "b" / rel
        s = p.read_text()
        for old, new in edits:
            assert s.count(old) == 1, f"{rel}: expected exactly one occurrence of {old!r}, found {s.count(old)}"
            s = s.replace(old, new)
        p.write_text(s)
    shutil.copy(HERE / "backend.rs", tmp / "b" / "src" / "backend.rs")
    out = subprocess.run(["diff", "-ruN", "-U2", "a", "b"], cwd=tmp, capture_output=True, text=True).stdout
    # stable header lines (no timestamps)
    lines = []
    for ln in out.splitlines(keepends=True):
        if ln.startswith(("--- a/", "+++ b/", "--- b/", "+++ a/")):
            ln = ln.split("\t")[0].rstrip("\n") + "\n"
        lines.append(ln)
    OUT.write_text("".join(lines))
    shutil.rmtree(tmp)
    print(f"wrote {OUT}: {sum(1 for l in lines if l.startswith('+') and not l.startswith('+++'))} added lines, "
          f"{sum(1 for l in lines if l.startswith('-') and not l.startswith('---'))} removed")


if __name__ == "__main__":
    main()
