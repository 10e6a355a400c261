// scene_host.cpp — see scene_host.hpp.  Reference citations are relative to /root/reference.
#include "scene_host.hpp"

#include <algorithm>
#include <array>
#include <cmath>
#include <cstring>
#include <fstream>
#include <limits>
#include <map>
#include <sstream>

#include "../../include/rtb200.h"
#include "toml_subset.hpp"

namespace rtb {
namespace {

using toml::Value;

struct SpecError {
    int code;
    std::string msg;
};

[[noreturn]] void bad(const std::string& m) { throw SpecError{RTB_EPARSE, m}; }

inline D3 add(D3 a, D3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
inline D3 sub(D3 a, D3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline D3 mul(D3 a, double s) { return {a.x * s, a.y * s, a.z * s}; }
inline double len(D3 a) { return std::sqrt(a.x * a.x + a.y * a.y + a.z * a.z); }

const Value& need(const Value& t, const char* key, const char* where) {
    const Value* v = t.find(key);
    if (!v) bad(std::string("missing field `") + key + "` in " + where);
    return *v;
}
double num(const Value& v, const char* what) {
    if (!v.is_number()) bad(std::string("expected a number for ") + what);
    return v.as_double();
}
D3 vec3(const Value& v, const char* what) {
    if (v.kind != Value::Array || v.elems.size() != 3) bad(std::string("expected an array of 3 numbers for ") + what);
    return {num(*v.elems[0], what), num(*v.elems[1], what), num(*v.elems[2], what)};
}
const std::string& str(const Value& v, const char* what) {
    if (v.kind != Value::String) bad(std::string("expected a string for ") + what);
    return v.str;
}

// ---- mesh helpers ---------------------------------------------------------------------------
void enclose(HostObject& o) {  // BoundingBox::enclose, src/geometry.rs:927-953
    double inf = std::numeric_limits<double>::infinity();
    o.bb_min = {inf, inf, inf};
    o.bb_max = {-inf, -inf, -inf};
    for (const D3& p : o.vertices) {
        if (p.x < o.bb_min.x) o.bb_min.x = p.x;
        if (p.x > o.bb_max.x) o.bb_max.x = p.x;
        if (p.y < o.bb_min.y) o.bb_min.y = p.y;
        if (p.y > o.bb_max.y) o.bb_max.y = p.y;
        if (p.z < o.bb_min.z) o.bb_min.z = p.z;
        if (p.z > o.bb_max.z) o.bb_max.z = p.z;
    }
}

void mesh_init(HostObject& o) {  // Mesh::new, src/geometry.rs:754-775 (Heron areas, :614-620)
    o.surface_area = 0;
    o.cumulative_area.clear();
    for (size_t i = 0; i + 2 < o.indices.size(); i += 3) {
        D3 a = o.vertices[o.indices[i]], b = o.vertices[o.indices[i + 1]], c = o.vertices[o.indices[i + 2]];
        double ab = len(sub(a, b)), bc = len(sub(b, c)), ca = len(sub(c, a));
        double s = (ab + bc + ca) / 2.;
        o.surface_area += std::sqrt(s * (s - ab) * (s - bc) * (s - ca));
        o.cumulative_area.push_back(o.surface_area);
    }
    enclose(o);
}

void make_prism(HostObject& o, D3 p, double w, double h, double d) {  // Mesh::prism, src/geometry.rs:839-862
    o.vertices = {{p.x, p.y, p.z},         {p.x, p.y, p.z + d},         {p.x, p.y + h, p.z},
                  {p.x, p.y + h, p.z + d}, {p.x + w, p.y, p.z},         {p.x + w, p.y, p.z + d},
                  {p.x + w, p.y + h, p.z}, {p.x + w, p.y + h, p.z + d}};
    o.indices = {1, 3, 7, 1, 5, 7, 0, 2, 6, 0, 4, 6, 0, 1, 3, 0, 2, 3,
                 4, 5, 7, 4, 6, 7, 2, 3, 7, 2, 6, 7, 0, 1, 5, 0, 4, 5};
    mesh_init(o);
}

bool parse_f64(const std::string& s, double& out) {
    if (s.empty()) return false;
    char* end = nullptr;
    out = std::strtod(s.c_str(), &end);
    return *end == 0;
}

void load_obj(HostObject& o, const std::string& path) {  // Mesh::load, src/geometry.rs:777-833
    std::ifstream f(path);
    if (!f) throw SpecError{RTB_EMESH, "cannot open mesh file " + path};
    std::string line;
    int lineno = 0;
    while (std::getline(f, line)) {
        ++lineno;
        std::istringstream ss(line);
        std::string cmd;
        if (!(ss >> cmd)) continue;
        if (cmd == "v" || cmd == "vn") {
            double c[3];
            for (int k = 0; k < 3; ++k) {
                std::string tok;
                if (!(ss >> tok)) throw SpecError{RTB_EMESH, path + ":" + std::to_string(lineno) + ": unexpected end of file"};
                if (!parse_f64(tok, c[k])) throw SpecError{RTB_EMESH, path + ":" + std::to_string(lineno) + ": Ill-formed float " + tok};
            }
            if (cmd == "v") o.vertices.push_back({c[0], c[1], c[2]});  // vn is validated, never used (flat shading)
        } else if (cmd == "f") {
            for (int k = 0; k < 3; ++k) {  // triangles only; extra vertices on the line are ignored like the reference
                std::string tok;
                if (!(ss >> tok)) throw SpecError{RTB_EMESH, path + ":" + std::to_string(lineno) + ": unexpected end of file"};
                std::string first = tok.substr(0, tok.find('/'));  // parse_face keeps the position index only
                char* end = nullptr;
                unsigned long long v = first.empty() ? 0 : std::strtoull(first.c_str(), &end, 10);
                if (first.empty() || first[0] == '-' || first[0] == '+' || *end != 0)
                    throw SpecError{RTB_EMESH, path + ":" + std::to_string(lineno) + ": Ill-formed integer " + first};
                if (v == 0) throw SpecError{RTB_EMESH, path + ":" + std::to_string(lineno) + ": face index 0"};
                o.indices.push_back((uint32_t)(v - 1));
            }
        }
    }
    for (uint32_t i : o.indices)
        if (i >= o.vertices.size()) throw SpecError{RTB_EMESH, path + ": face index out of range"};
    if (o.indices.empty()) throw SpecError{RTB_EMESH, path + ": mesh has no faces"};  // WeightedIndex::new fails on empty
    mesh_init(o);
}

D3 rot(int axis, D3 s, double a) {  // Vec3::rotate_{x,y,z}, src/geometry.rs:111-133
    double c = std::cos(a), sn = std::sin(a);
    if (axis == 0) return {s.x, s.y * c - s.z * sn, s.y * sn + s.z * c};
    if (axis == 1) return {s.x * c + s.z * sn, s.y, s.z * c - s.x * sn};
    return {s.x * c - s.y * sn, s.x * sn + s.y * c, s.z};
}

D3 center(const HostObject& o) { return mul(add(o.bb_min, o.bb_max), 0.5); }  // BoundingBox::center (:1063), /2

void apply_transform(HostObject& o, const Value& t) {  // src/scene.rs:411-429, src/geometry.rs:427-510
    if (t.kind != Value::Table || t.items.size() != 1) bad("a transform must be a table with exactly one key");
    const std::string& key = t.items[0].first;
    const Value& v = *t.items[0].second;
    if (key == "translate") {
        D3 d = vec3(v, "translate");
        if (o.geom == GEOM_MESH) {
            for (D3& p : o.vertices) p = add(p, d);
            o.bb_min = add(o.bb_min, d);
            o.bb_max = add(o.bb_max, d);
        } else {
            o.pos = add(o.pos, d);
        }
    } else if (key == "scale") {
        double s = num(v, "scale");
        if (o.geom == GEOM_SPHERE) o.r *= s;
        else if (o.geom == GEOM_MESH) {
            D3 c = center(o);
            for (D3& p : o.vertices) p = add(c, mul(sub(p, c), s));
            // reference quirk: min + (min - c)*s (not c + ...), src/geometry.rs:503-506.  The box stays
            // centred and enclosing; it only matters as the pivot of later transforms.
            o.bb_min = add(o.bb_min, mul(sub(o.bb_min, c), s));
            o.bb_max = add(o.bb_max, mul(sub(o.bb_max, c), s));
        }
    } else if (key == "rotate_x" || key == "rotate_y" || key == "rotate_z") {
        int axis = key == "rotate_x" ? 0 : (key == "rotate_y" ? 1 : 2);
        double a = num(v, key.c_str());
        if (o.geom == GEOM_PLANE) o.n = rot(axis, o.n, a);
        else if (o.geom == GEOM_MESH) {
            D3 c = center(o);
            for (D3& p : o.vertices) p = add(c, rot(axis, sub(p, c), a));
            enclose(o);  // fit_bounds(), src/geometry.rs:456,472,488
        }
    } else {
        bad("unknown variant `" + key + "`, expected one of `translate`, `scale`, `rotate_x`, `rotate_y`, `rotate_z`");
    }
}

void build_object(const Value& spec, const std::string& assets_dir, HostObject& o) {
    if (spec.kind != Value::Table) bad("objects entries must be tables");
    if (const Value* e = spec.find("emitted")) o.emitted = vec3(*e, "emitted");
    const Value& b = need(spec, "brdf", "object");
    if (b.kind != Value::Table) bad("brdf must be a table");
    const std::string& bt = str(need(b, "type", "brdf"), "brdf.type");
    if (bt == "diffuse") {
        o.brdf = BRDF_DIFFUSE;
        o.k = vec3(need(b, "kd", "brdf"), "kd");
    } else if (bt == "specular") {
        o.brdf = BRDF_SPECULAR;
        o.k = vec3(need(b, "ks", "brdf"), "ks");
    } else if (bt == "phong") {
        o.brdf = BRDF_PHONG;
        o.phong_kd = num(need(b, "kd", "brdf"), "kd");
        o.phong_ks = num(need(b, "ks", "brdf"), "ks");
        o.color_d = vec3(need(b, "color_d", "brdf"), "color_d");
        o.color_s = vec3(need(b, "color_s", "brdf"), "color_s");
        const Value& pw = need(b, "power", "brdf");
        if (pw.kind != Value::Integer || pw.integer < 0) bad("phong power must be a non-negative integer (usize)");
        o.phong_power = (int)pw.integer;
    } else if (bt == "dielectric") {
        o.brdf = BRDF_DIELECTRIC;
        const double ior = num(need(b, "ior", "brdf"), "ior");
        if (!std::isfinite(ior) || !(ior > 0)) bad("dielectric ior must be a finite number > 0");
        o.k = {ior, 0, 0};
        o.color_d = {1, 1, 1};
        if (const Value* t = b.find("tint")) {
            o.color_d = vec3(*t, "tint");
            for (double c : {o.color_d.x, o.color_d.y, o.color_d.z})
                if (!(c >= 0 && c <= 1)) bad("dielectric tint components must lie in [0, 1]");
        }
    } else {
        bad("unknown variant `" + bt + "`, expected one of `diffuse`, `specular`, `phong`, `dielectric`");
    }
    const Value& g = need(spec, "geometry", "object");
    if (g.kind != Value::Table) bad("geometry must be a table");
    const std::string& gt = str(need(g, "type", "geometry"), "geometry.type");
    if (gt == "sphere") {
        o.geom = GEOM_SPHERE;
        o.pos = vec3(need(g, "pos", "geometry"), "pos");
        o.r = num(need(g, "r", "geometry"), "r");
    } else if (gt == "plane") {
        o.geom = GEOM_PLANE;
        o.pos = vec3(need(g, "pos", "geometry"), "pos");
        o.n = vec3(need(g, "n", "geometry"), "n");
    } else if (gt == "cube") {
        o.geom = GEOM_MESH;
        double s = num(need(g, "size", "geometry"), "size");
        make_prism(o, vec3(need(g, "pos", "geometry"), "pos"), s, s, s);  // Mesh::cube, src/geometry.rs:864-866
    } else if (gt == "prism") {
        o.geom = GEOM_MESH;
        D3 sz = vec3(need(g, "size", "geometry"), "size");
        make_prism(o, vec3(need(g, "pos", "geometry"), "pos"), sz.x, sz.y, sz.z);
    } else if (gt == "mesh") {
        o.geom = GEOM_MESH;
        const std::string& p = str(need(g, "path", "geometry"), "path");
        load_obj(o, assets_dir.empty() ? p : assets_dir + "/" + p);
    } else {
        bad("unknown variant `" + gt + "`, expected one of `sphere`, `cube`, `prism`, `plane`, `mesh`");
    }
    if (const Value* tr = spec.find("transforms")) {
        if (tr->kind != Value::Array) bad("transforms must be an array");
        for (auto& t : tr->elems) apply_transform(o, *t);
    }
}

}  // namespace

int load_scene_text(const std::string& text, const std::string& assets_dir, HostScene& out, std::string& err) {
    try {
        toml::ValuePtr root = toml::parse(text);
        const Value& cam = need(*root, "camera", "scene");
        if (cam.kind != Value::Table) bad("camera must be a table");
        out.cam_pos = vec3(need(cam, "pos", "camera"), "camera.pos");
        out.cam_dir = vec3(need(cam, "dir", "camera"), "camera.dir");
        const Value& objs = need(*root, "objects", "scene");
        if (objs.kind != Value::Array) bad("objects must be an array of tables");
        out.objects.clear();
        for (auto& spec : objs.elems) {
            HostObject o;
            build_object(*spec, assets_dir, o);
            out.objects.push_back(std::move(o));
        }
        if (int rc = finish_host_scene(out, err)) return rc;
        return RTB_OK;
    } catch (const toml::ParseError& e) {
        err = e.what();
        return RTB_EPARSE;
    } catch (const SpecError& e) {
        err = e.msg;
        return e.code;
    }
}

void init_mesh_tables(HostObject& o) { mesh_init(o); }

int finish_host_scene(HostScene& out, std::string& err) {
    // Scene::new, src/scene.rs:126-141: first object with any |emitted component| >= 1e-5
    out.light = -1;
    for (size_t i = 0; i < out.objects.size(); ++i) {
        const D3& e = out.objects[i].emitted;
        bool zero = std::fabs(e.x) < 0.00001 && std::fabs(e.y) < 0.00001 && std::fabs(e.z) < 0.00001;
        if (!zero) { out.light = (int)i; break; }
    }
    if (out.light < 0) {
        err = "scene has no emitter (the reference hits unreachable!() at src/scene.rs:136)";
        return RTB_ENOLIGHT;
    }
    if (out.objects[out.light].geom == GEOM_PLANE) {
        err = "the light is a plane: Geometry::sample is unimplemented!() for planes (src/geometry.rs:593)";
        return RTB_EUNSUPPORTED;
    }
    return RTB_OK;
}

int load_scene_file(const std::string& path, const std::string& assets_dir, HostScene& out, std::string& err) {
    std::ifstream f(path, std::ios::binary);
    if (!f) {
        err = "cannot open " + path;
        return RTB_EIO;
    }
    std::stringstream ss;
    ss << f.rdbuf();
    std::string dir = assets_dir;
    if (dir.empty()) {  // default: <dir of the toml>/assets, the layout `raytracer <scenes dir>` expects
        size_t slash = path.find_last_of('/');
        dir = (slash == std::string::npos ? std::string(".") : path.substr(0, slash)) + "/assets";
    }
    return load_scene_text(ss.str(), dir, out, err);
}

int flatten_scene(const HostScene& hs, FlatScene& fs, std::string& err) {
    if ((int)hs.objects.size() > MAX_OBJECTS) {
        err = "too many objects (" + std::to_string(hs.objects.size()) + " > " + std::to_string(MAX_OBJECTS) + ")";
        return RTB_EUNSUPPORTED;
    }
    fs = FlatScene();
    fs.cam_pos[0] = (float)hs.cam_pos.x; fs.cam_pos[1] = (float)hs.cam_pos.y; fs.cam_pos[2] = (float)hs.cam_pos.z;
    fs.cam_dir[0] = (float)hs.cam_dir.x; fs.cam_dir[1] = (float)hs.cam_dir.y; fs.cam_dir[2] = (float)hs.cam_dir.z;
    fs.n_objects = (int)hs.objects.size();
    fs.light_obj = hs.light;
    fs.light_geom = hs.objects[hs.light].geom;
    for (int i = 0; i < fs.n_objects; ++i) {
        const HostObject& o = hs.objects[i];
        FlatMaterial m;
        std::memset(&m, 0, sizeof(m));
        m.emitted[0] = (float)o.emitted.x; m.emitted[1] = (float)o.emitted.y; m.emitted[2] = (float)o.emitted.z;
        m.brdf = o.brdf;
        m.geom = o.geom;
        m.first_tri = -1;
        if (o.brdf == BRDF_PHONG) {
            m.k[0] = (float)o.phong_kd; m.k[1] = (float)o.phong_ks; m.k[2] = (float)o.phong_power;
            m.color_d[0] = (float)o.color_d.x; m.color_d[1] = (float)o.color_d.y; m.color_d[2] = (float)o.color_d.z;
            m.color_s[0] = (float)o.color_s.x; m.color_s[1] = (float)o.color_s.y; m.color_s[2] = (float)o.color_s.z;
        } else if (o.brdf == BRDF_DIELECTRIC) {
            m.k[0] = (float)o.k.x;
            m.k[1] = 1.0f;   // spheres and planes; meshes below
            m.color_d[0] = (float)o.color_d.x; m.color_d[1] = (float)o.color_d.y; m.color_d[2] = (float)o.color_d.z;
        } else {
            m.k[0] = (float)o.k.x; m.k[1] = (float)o.k.y; m.k[2] = (float)o.k.z;
        }
        if (o.geom == GEOM_MESH) {
            m.first_tri = (int)(fs.tri_verts.size() / 9);
            m.n_tri = (int)(o.indices.size() / 3);
            // a dielectric mesh gets ONE orientation sign: the side of its first triangle.  Triangles wound the other way
            // (the built-in cube / prism alternate within each face) are stored with b and c swapped.
            std::vector<int> out;
            if (o.brdf == BRDF_DIELECTRIC) {
                out = triangle_outward(o);
                m.k[1] = (float)out[0];
            }
            for (size_t k = 0; k < o.indices.size(); ++k) {
                const size_t t = k / 3, c = k % 3;
                const bool swap = !out.empty() && out[t] != out[0] && c != 0;
                const D3& p = o.vertices[o.indices[swap ? 3 * t + 3 - c : k]];
                fs.tri_verts.push_back((float)p.x);
                fs.tri_verts.push_back((float)p.y);
                fs.tri_verts.push_back((float)p.z);
            }
            fs.tri_obj.insert(fs.tri_obj.end(), (size_t)m.n_tri, i);
            fs.n_meshes++;
        } else {
            FlatPrim p;
            std::memset(&p, 0, sizeof(p));
            p.obj = i;
            if (o.geom == GEOM_PLANE) {
                p.type = PRIM_PLANE;
                p.a[0] = (float)o.n.x; p.a[1] = (float)o.n.y; p.a[2] = (float)o.n.z;
                p.a[3] = (float)(o.pos.x * o.n.x + o.pos.y * o.n.y + o.pos.z * o.n.z);
                p.b[0] = (float)o.pos.x; p.b[1] = (float)o.pos.y; p.b[2] = (float)o.pos.z;
                p.group = (int)fs.prims.size();
                for (size_t q = 0; q < fs.prims.size(); ++q) {  // coincident planes share a self-intersection class
                    const FlatPrim& e = fs.prims[q];
                    if (e.type == PRIM_PLANE && e.a[0] == p.a[0] && e.a[1] == p.a[1] && e.a[2] == p.a[2] && e.a[3] == p.a[3]) {
                        p.group = e.group;
                        break;
                    }
                }
                fs.n_planes++;
            } else {
                p.type = PRIM_SPHERE;
                p.a[0] = (float)o.pos.x; p.a[1] = (float)o.pos.y; p.a[2] = (float)o.pos.z; p.a[3] = (float)o.r;
                p.b[0] = (float)(o.r * o.r);
                p.group = (int)fs.prims.size();
                fs.n_spheres++;
            }
            fs.prims.push_back(p);
        }
        fs.materials.push_back(m);
    }
    // analytic table order: all planes (object order), then all spheres (object order) — the device loops are
    // type-specialised.  Ties between equal-t hits keep the reference's lowest-object-index rule within each
    // kind (the duplicated wall of the reference scenes); a plane/sphere tie at bit-identical t has measure zero.
    {
        std::vector<FlatPrim> planes, spheres;
        for (const FlatPrim& q : fs.prims) (q.type == PRIM_PLANE ? planes : spheres).push_back(q);
        // A plane that coincides exactly with an earlier one (every reference scene repeats one wall as object 5,
        // scenes/*.toml) can never be reported: trace_ray keeps the lowest object index on equal t (src/scene.rs:277-284)
        // and an occlusion test is unchanged by a second copy.  It stays an object (material table) but is dropped
        // from the device primitive table.
        {
            std::vector<FlatPrim> uniq;
            for (const FlatPrim& q : planes) {
                bool dup = false;
                for (const FlatPrim& e : uniq)
                    dup |= e.a[0] == q.a[0] && e.a[1] == q.a[1] && e.a[2] == q.a[2] && e.a[3] == q.a[3];
                if (!dup) uniq.push_back(q);
            }
            planes.swap(uniq);
        }
        for (size_t k = 0; k < planes.size(); ++k) planes[k].group = (int)k;   // self-intersection class = own index
        for (size_t k = 0; k < spheres.size(); ++k) spheres[k].group = (int)(planes.size() + k);
        fs.n_planes = (int)planes.size();
        fs.prims = planes;
        fs.prims.insert(fs.prims.end(), spheres.begin(), spheres.end());
    }
    const HostObject& L = hs.objects[hs.light];
    if (L.geom == GEOM_MESH) {
        fs.light_area = (float)L.surface_area;
        for (double c : L.cumulative_area) fs.light_cdf.push_back((float)c);
    }
    // RTB_EST_NEE_ALL_LIGHTS: every emitting sphere and mesh, weighted by power (light_rule.cuh, DESIGN §3f).  Planes have no
    // sampler; they and zero-weight emitters stay out and add their emission wherever a path meets them.
    double total = 0;
    for (int i = 0; i < fs.n_objects; ++i) {
        const HostObject& o = hs.objects[i];
        if (o.geom == GEOM_PLANE) continue;
        const double lum = 0.2126 * std::max(o.emitted.x, 0.0) + 0.7152 * std::max(o.emitted.y, 0.0) + 0.0722 * std::max(o.emitted.z, 0.0);
        FlatLight l;
        l.obj = i;
        l.area = 0;
        if (o.geom == GEOM_SPHERE) {
            l.area = 4.0 * M_PI * o.r * o.r;
        } else {
            for (size_t k = 0; k + 2 < o.indices.size(); k += 3) {
                const D3 a = o.vertices[o.indices[k]], e1 = sub(o.vertices[o.indices[k + 1]], a), e2 = sub(o.vertices[o.indices[k + 2]], a);
                l.area += 0.5 * len({e1.y * e2.z - e1.z * e2.y, e1.z * e2.x - e1.x * e2.z, e1.x * e2.y - e1.y * e2.x});
                l.tri_cdf.push_back(l.area);
            }
            for (double& c : l.tri_cdf) c /= l.area;
        }
        const double w = lum * l.area;
        if (!(w > 0) || !std::isfinite(w)) continue;
        l.prob = w;
        total += w;
        fs.lights.push_back(std::move(l));
    }
    for (FlatLight& l : fs.lights) l.prob /= total;
    (void)err;
    return RTB_OK;
}

std::vector<int> triangle_outward(const HostObject& o) {
    const size_t n = o.indices.size() / 3;
    // vertex ids by position (rtb_scene_create hands every triangle its own three vertices)
    std::map<std::array<double, 3>, int> vid;
    std::vector<int> v(3 * n);
    for (size_t k = 0; k < 3 * n; ++k) {
        const D3& p = o.vertices[o.indices[k]];
        v[k] = vid.emplace(std::array<double, 3>{p.x, p.y, p.z}, (int)vid.size()).first->second;
    }
    // undirected edge -> (triangle, traversed low -> high id)
    std::map<std::pair<int, int>, std::vector<std::pair<int, bool>>> edges;
    for (size_t t = 0; t < n; ++t)
        for (int e = 0; e < 3; ++e) {
            const int a = v[3 * t + e], b = v[3 * t + (e + 1) % 3];
            if (a != b) edges[{std::min(a, b), std::max(a, b)}].push_back({(int)t, a < b});
        }
    // rel[t] = +1 / -1: wound like / against the seed of its piece (consistent neighbours traverse a shared edge in opposite
    // directions); pieces are flood-filled one after another
    std::vector<int> rel(n, 0), out(n, 1), piece;
    for (size_t seed = 0; seed < n; ++seed) {
        if (rel[seed]) continue;
        rel[seed] = 1;
        piece.assign(1, (int)seed);
        double vol = 0;
        for (size_t q = 0; q < piece.size(); ++q) {
            const int t = piece[q];
            const D3 &a = o.vertices[o.indices[3 * t]], &b = o.vertices[o.indices[3 * t + 1]], &c = o.vertices[o.indices[3 * t + 2]];
            vol += rel[t] * (a.x * (b.y * c.z - b.z * c.y) + a.y * (b.z * c.x - b.x * c.z) + a.z * (b.x * c.y - b.y * c.x));
            for (int e = 0; e < 3; ++e) {
                const int a0 = v[3 * t + e], b0 = v[3 * t + (e + 1) % 3];
                if (a0 == b0) continue;
                const bool up = a0 < b0;
                for (const auto& nb : edges[{std::min(a0, b0), std::max(a0, b0)}]) {
                    if (rel[nb.first]) continue;
                    rel[nb.first] = nb.second == up ? -rel[t] : rel[t];
                    piece.push_back(nb.first);
                }
            }
        }
        // vol > 0: the winding rel = +1 runs counter-clockwise seen from outside, so (b-a) x (c-a) points out and the stored
        // normal (c-a) x (b-a) points in
        for (int t : piece) out[t] = vol > 0 ? -rel[t] : rel[t];
    }
    return out;
}

}  // namespace rtb
