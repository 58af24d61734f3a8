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
// line 16: not recorded
// line 17: not recorded
// line 18: not recorded
// line 19: not recorded
// line 20: not recorded
// line 21: not recorded
// line 22: not recorded
// line 23: not recorded
// line 24: not recorded
}

impl Texture for Checker {
    fn value(&self, u: f32, v: f32, p: &glam::Vec3) -> glam::Vec3 {
        let sines =
            f32::sin(self.scale * p.x) * f32::sin(self.scale * p.y) * f32::sin(self.scale * p.z);
