// scene_host.hpp — host side of the scene boundary: TOML -> objects -> flattened SoA.
//
// Mirrors Scene::from_toml / SceneSpec::to_scene (reference src/scene.rs:143-150, 292-441) and
// the geometry set-up they call (Mesh::load / prism / cube and Geometry::{translate, scale,
// rotate_*}, src/geometry.rs:426-510, 753-866).  Set-up runs in f64 exactly once per scene; the
// flattened scene handed to the device is fp32.
#pragma once

#include <cstdint>
#include <string>
#include <vector>

namespace rtb {

struct D3 {
    double x = 0, y = 0, z = 0;
};

enum GeomKind : int { GEOM_SPHERE = 0, GEOM_PLANE = 1, GEOM_MESH = 2 };
enum BrdfKind : int { BRDF_DIFFUSE = 0, BRDF_SPECULAR = 1, BRDF_PHONG = 2, BRDF_DIELECTRIC = 3, BRDF_METAL = 4 };
constexpr double METAL_MIN_ROUGHNESS = 0.05;   // rough metal: roughness in [0.05, 1], GGX alpha = roughness^2

struct HostObject {
    D3 emitted;
    int brdf = BRDF_DIFFUSE;
    D3 k;                      // kd (diffuse) / ks (specular) / {ior, 0, 0} (dielectric) / {roughness, 0, 0} (metal)
    double phong_kd = 0, phong_ks = 0;
    int phong_power = 0;
    D3 color_d, color_s;       // phong colours; dielectric: color_d = transmission tint; metal: color_s = F0
    int geom = GEOM_SPHERE;
    D3 pos;                    // sphere centre / plane point
    double r = 0;
    D3 n;                      // plane normal (kept un-normalised, as the reference does)
    // mesh
    std::vector<D3> vertices;
    std::vector<uint32_t> indices;
    D3 bb_min, bb_max;         // Mesh::bounding_box incl. the scale() quirk (src/geometry.rs:503-506)
    double surface_area = 0;   // Mesh::new computes areas BEFORE the transforms and never refreshes
    std::vector<double> cumulative_area;  // WeightedIndex cumulative weights (same remark)
};

struct HostScene {
    D3 cam_pos, cam_dir;
    std::vector<HostObject> objects;
    int light = -1;  // Scene::light_source (src/scene.rs:129-137)
};

// error codes are those of include/rtb200.h
int load_scene_text(const std::string& toml_text, const std::string& assets_dir, HostScene& out, std::string& err);
int load_scene_file(const std::string& path, const std::string& assets_dir, HostScene& out, std::string& err);

// ---- flattened fp32 scene -----------------------------------------------------------------
constexpr int MAX_OBJECTS = 256;   // materials + analytic primitives live in __constant__ memory
constexpr int PRIM_PLANE = 0;
constexpr int PRIM_SPHERE = 1;

struct FlatPrim {      // analytic primitive, in object order
    float a[4];        // plane: n.xyz, dot(pos, n)        sphere: centre.xyz, r
    float b[4];        // plane: pos.xyz, -                sphere: r*r, -, -, -
    int32_t type;      // PRIM_*
    int32_t obj;       // object index (Hit.id)
    int32_t group;     // planes: index of the first coincident plane (self-intersection class)
    int32_t pad;
};

struct FlatMaterial {  // one per object
    float emitted[4];  // rgb, -
    float k[4];        // diffuse kd / specular ks rgb; phong: kd, ks, power, -; dielectric: ior, orientation sign, -; metal: alpha, -, -
    float color_d[4];  // phong colour_d; dielectric: tint
    float color_s[4];  // phong colour_s; metal: F0
    int32_t brdf;
    int32_t geom;
    int32_t first_tri;  // meshes: first global triangle index, else -1
    int32_t n_tri;
};

// one entry of the light table: an emitting sphere or mesh with weight w = lum709(max(emitted, 0)) * area > 0, all in f64
// after the transforms (a mesh's TRUE area, not Mesh::surface_area)
struct FlatLight {
    int32_t obj;
    double prob;                   // w / sum of w
    double area;
    std::vector<double> tri_cdf;   // meshes: cumulative triangle areas / area (the last entry is 1)
};

struct FlatScene {
    float cam_pos[3], cam_dir[3];
    int32_t n_objects = 0;
    int32_t light_obj = -1;
    int32_t light_geom = 0;
    std::vector<FlatPrim> prims;
    std::vector<FlatMaterial> materials;
    std::vector<float> tri_verts;     // 9 floats per triangle (a, b, c), global order
    std::vector<int32_t> tri_obj;     // owning object per triangle
    // mesh light tables (only when the light is a mesh)
    std::vector<float> light_cdf;     // cumulative areas of the UNTRANSFORMED mesh (reference quirk)
    float light_area = 0;
    int32_t n_planes = 0, n_spheres = 0, n_meshes = 0;
    std::vector<FlatLight> lights;    // RTB_EST_NEE_ALL_LIGHTS: the light table (light_rule.cuh), in object order
};

int flatten_scene(const HostScene& hs, FlatScene& out, std::string& err);

// Dielectric meshes: +1 / -1 per triangle = whether its stored normal norm((c-a) x (b-a)) points out of the solid.  The
// winding is made consistent across shared edges (vertices matched by position) within each connected piece, and each
// piece is oriented by the sign of its signed volume (f64).  An open piece gets an arbitrary side.
std::vector<int> triangle_outward(const HostObject& o);

// shared tail of every way to build a HostScene: Scene::new's light rule (src/scene.rs:126-141) + mesh tables
int finish_host_scene(HostScene& hs, std::string& err);
void init_mesh_tables(HostObject& o);   // Mesh::new: Heron areas, cumulative weights, bounding box

}  // namespace rtb
