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
}

impl Texture for SolidColor {
    fn value(&self, _u: f32, _v: f32, _p: &Vec3) -> Vec3 {
        self.color
    }
