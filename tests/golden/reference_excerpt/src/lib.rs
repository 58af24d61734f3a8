mod aabb;
pub mod bvh;
pub mod camera;
pub mod geometry;
