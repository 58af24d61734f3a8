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
}

impl Hittable for Translate {
    fn hit(
        &self,
        ray: &crate::ray::Ray,
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
    sin_theta: f32,
    cos_theta: f32,
    bbox: Option<Aabb>,
}

impl RotateY {
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
// line 77: not recorded
// line 78: not recorded
// line 79: not recorded
// line 80: not recorded
// line 81: not recorded
// line 82: not recorded
// line 83: not recorded
// line 84: not recorded
// line 85: not recorded
// line 86: not recorded
// line 87: not recorded
// line 88: not recorded
// line 89: not recorded
// line 90: not recorded
// line 91: not recorded
// line 92: not recorded
// line 93: not recorded
// line 94: not recorded
// line 95: not recorded
// line 96: not recorded
// line 97: not recorded
            sin_theta,
            cos_theta,
            bbox,
        }
    }

// line 104: not recorded
// line 105: not recorded
// line 106: not recorded
// line 107: not recorded
// line 108: not recorded
// line 109: not recorded
// line 110: not recorded
}

impl Hittable for RotateY {
    fn hit(
        &self,
        ray: &Ray,
