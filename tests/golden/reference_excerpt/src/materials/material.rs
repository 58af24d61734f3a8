// line 1: not recorded
// line 2: not recorded
// line 3: not recorded
// line 4: not recorded
// line 5: not recorded
// line 6: not recorded
// line 7: not recorded
// line 8: not recorded
// line 9: not recorded
// line 10: not recorded
// line 11: not recorded
// line 12: not recorded
// line 13: not recorded
// line 14: not recorded
// line 15: not recorded
pub trait Material: Send + Sync {
    /// Returns None if the ray is absorbed and not scattered
    fn scatter(&self, ray: &Ray, hit_record: &HitRecord) -> Option<ScatterRecord>;

    fn emit(&self, _u: f32, _v: f32, _point: &Vec3) -> Vec3 {
        vec3(0.0, 0.0, 0.0)
