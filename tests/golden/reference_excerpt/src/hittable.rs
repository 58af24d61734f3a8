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
// line 77: not recorded
// line 78: not recorded
    /// full range of motion between `time_0` and `time_1`. If the object does not move,
    /// these values have no effect on the bounding box.
    fn bounding_box(&self, time_0: f32, time_1: f32) -> Option<Aabb>;
}

pub struct HittableList {
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
}

impl Hittable for HittableList {
    fn hit(
        &self,
        ray: &Ray,
// line 104: not recorded
// line 105: not recorded
// line 106: not recorded
// line 107: not recorded
// line 108: not recorded
// line 109: not recorded
// line 110: not recorded
// line 111: not recorded
// line 112: not recorded
// line 113: not recorded
// line 114: not recorded
// line 115: not recorded
// line 116: not recorded
// line 117: not recorded
// line 118: not recorded
// line 119: not recorded
// line 120: not recorded
// line 121: not recorded
// line 122: not recorded
// line 123: not recorded
// line 124: not recorded
// line 125: not recorded
// line 126: not recorded
// line 127: not recorded
// line 128: not recorded
// line 129: not recorded
// line 130: not recorded
// line 131: not recorded
// line 132: not recorded
// line 133: not recorded
// line 134: not recorded
// line 135: not recorded
// line 136: not recorded
// line 137: not recorded
// line 138: not recorded
// line 139: not recorded
// line 140: not recorded
// line 141: not recorded
// line 142: not recorded
// line 143: not recorded
// line 144: not recorded
    boundary: Arc<dyn Hittable>,
    phase_function: Arc<dyn Material>,
    neg_inv_density: f32,
}

impl ConstantMedium {
// line 151: not recorded
// line 152: not recorded
// line 153: not recorded
// line 154: not recorded
    ) -> ConstantMedium {
        ConstantMedium {
            boundary,
            phase_function: Arc::new(Isotropic::new(texture)),
            neg_inv_density: -1.0 / density,
        }
    }

// line 163: not recorded
// line 164: not recorded
        density: f32,
        color: Vec3,
    ) -> ConstantMedium {
        ConstantMedium {
            boundary,
            phase_function: Arc::new(Isotropic::from_color(color)),
            neg_inv_density: -1.0 / density,
        }
    }
}

impl Hittable for ConstantMedium {
    fn hit(
        &self,
        ray: &Ray,
