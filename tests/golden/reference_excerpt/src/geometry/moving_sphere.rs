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
// line 25: not recorded
// line 26: not recorded
// line 27: not recorded
// line 28: not recorded
// line 29: not recorded
// line 30: not recorded
// line 31: not recorded
// line 32: not recorded
// line 33: not recorded
// line 34: not recorded
// line 35: not recorded
// line 36: not recorded
// line 37: not recorded
// line 38: not recorded
// line 39: not recorded
// line 40: not recorded
// line 41: not recorded
// line 42: not recorded
// line 43: not recorded
// line 44: not recorded
// line 45: not recorded
// line 46: not recorded
// line 47: not recorded
// line 48: not recorded
// line 49: not recorded
// line 50: not recorded
// line 51: not recorded
}

impl Hittable for MovingSphere {
    fn hit(
        &self,
        ray: &crate::ray::Ray,
