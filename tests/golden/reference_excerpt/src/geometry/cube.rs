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
    min_point: Vec3,
    max_point: Vec3,
    sides: HittableList,
}

impl Cube {
    pub fn new(min_point: Vec3, max_point: Vec3, material: Arc<dyn Material>) -> Self {
        let mut sides = HittableList::new();
        sides.add(Arc::new(XyRect::new(
            min_point.x,
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
// line 52: not recorded
// line 53: not recorded
// line 54: not recorded
// line 55: not recorded
// line 56: not recorded
// line 57: not recorded
// line 58: not recorded
// line 59: not recorded
// line 60: not recorded
// line 61: not recorded
// line 62: not recorded
// line 63: not recorded
// line 64: not recorded
// line 65: not recorded
// line 66: not recorded
// line 67: not recorded
// line 68: not recorded
// line 69: not recorded
// line 70: not recorded
// line 71: not recorded
// line 72: not recorded
// line 73: not recorded
// line 74: not recorded
// line 75: not recorded
// line 76: not recorded
            min_point,
            max_point,
            sides,
        }
    }
}

impl Hittable for Cube {
    fn hit(
        &self,
        ray: &crate::ray::Ray,
