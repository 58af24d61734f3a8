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
}

impl Material for DiffuseLight {
    fn scatter(
        &self,
        _ray: &crate::ray::Ray,
