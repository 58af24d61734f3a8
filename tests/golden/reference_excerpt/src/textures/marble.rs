// line 1: not recorded
// line 2: not recorded
// line 3: not recorded
// line 4: not recorded
// line 5: not recorded
// line 6: not recorded
pub struct Marble {
    noise: Turbulence<Perlin, Perlin>,
    scale: f32,
}

impl Marble {
    pub fn new(scale: f32) -> Marble {
        let perlin = Perlin::new(random::<u32>());
        let turb: Turbulence<_, Perlin> = Turbulence::new(perlin)
            .set_frequency(1.0)
            .set_power(1.0)
            .set_roughness(6);
        Marble { noise: turb, scale }
    }
}

impl Texture for Marble {
    fn value(&self, _u: f32, _v: f32, p: &glam::Vec3) -> glam::Vec3 {
        vec3(1.0, 1.0, 1.0)
            * 0.5
