// Host-side mirror of the reference crate's interface (see ray_tracing.hpp).  Scene loading,
// transform construction and flattening happen here in FP64 with the reference's operand order
// (compile with -ffp-contract=off); all tracing is delegated to the CUDA core via the C ABI.
#include "ray_tracing.hpp"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <stdexcept>

#include "json.hpp"

namespace ray_tracing {

using algebra::Vector3d;
using algebra::transform::InversableTransform;
using algebra::transform::Transform;

// ------------------------------------------------------------------------------------------------
// algebra
// ------------------------------------------------------------------------------------------------
namespace algebra {

Vector3d Vector3d::cross(const Vector3d& o) const {
    return Vector3d(y * o.z - z * o.y, z * o.x - x * o.z, x * o.y - y * o.x);
}
double Vector3d::squared_length() const { return x * x + y * y + z * z; }
double Vector3d::length() const { return std::sqrt(squared_length()); }
Vector3d Vector3d::normalize() const {
    double l = length();
    return Vector3d(x / l, y / l, z / l);
}

namespace transform {

static const double kPi = 3.14159265358979323846264338327950288;

Transform Transform::unit() {
    Transform t;
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) t.m[i][j] = (i == j) ? 1.0 : 0.0;
    return t;
}
Transform Transform::translate(const Vector3d& v) {
    Transform t = unit();
    t.m[0][3] = v.x;
    t.m[1][3] = v.y;
    t.m[2][3] = v.z;
    return t;
}
Transform Transform::scale(const Vector3d& v) {
    Transform t = unit();
    t.m[0][0] = v.x;
    t.m[1][1] = v.y;
    t.m[2][2] = v.z;
    return t;
}
static inline double radians_of(double degrees) { return degrees * (kPi / 180.0); }
Transform Transform::rotate_roll(double degrees) {
    double r = radians_of(degrees), c = std::cos(r), s = std::sin(r);
    Transform t = unit();
    t.m[1][1] = c;  t.m[1][2] = -s;
    t.m[2][1] = s;  t.m[2][2] = c;
    return t;
}
Transform Transform::rotate_pitch(double degrees) {
    double r = radians_of(degrees), c = std::cos(r), s = std::sin(r);
    Transform t = unit();
    t.m[0][0] = c;   t.m[0][2] = s;
    t.m[2][0] = -s;  t.m[2][2] = c;
    return t;
}
Transform Transform::rotate_yaw(double degrees) {
    double r = radians_of(degrees), c = std::cos(r), s = std::sin(r);
    Transform t = unit();
    t.m[0][0] = c;  t.m[0][1] = -s;
    t.m[1][0] = s;  t.m[1][1] = c;
    return t;
}
Transform Transform::rotate(const Vector3d& d) {
    return rotate_roll(d.x) * rotate_pitch(d.y) * rotate_yaw(d.z);
}
Transform Transform::rotate_inverse(const Vector3d& d) {
    return rotate_yaw(d.z) * rotate_pitch(d.y) * rotate_roll(d.x);
}
Transform Transform::operator*(const Transform& rhs) const {
    Transform out;
    for (int i = 0; i < 4; i++)
        for (int j = 0; j < 4; j++) {
            double acc = m[i][0] * rhs.m[0][j];
            acc = acc + m[i][1] * rhs.m[1][j];
            acc = acc + m[i][2] * rhs.m[2][j];
            acc = acc + m[i][3] * rhs.m[3][j];
            out.m[i][j] = acc;
        }
    return out;
}
Vector3d Transform::transform_point(const Vector3d& p) const {
    Vector3d r;
    double* out[3] = {&r.x, &r.y, &r.z};
    for (int i = 0; i < 3; i++) *out[i] = ((p.x * m[i][0] + p.y * m[i][1]) + p.z * m[i][2]) + m[i][3];
    return r;
}
Vector3d Transform::transform_vector(const Vector3d& v) const {
    Vector3d r;
    double* out[3] = {&r.x, &r.y, &r.z};
    for (int i = 0; i < 3; i++) *out[i] = (v.x * m[i][0] + v.y * m[i][1]) + v.z * m[i][2];
    return r;
}
Vector3d Transform::transform_normal(const Vector3d& n) const {
    Vector3d r;
    double* out[3] = {&r.x, &r.y, &r.z};
    for (int j = 0; j < 3; j++) *out[j] = (n.x * m[0][j] + n.y * m[1][j]) + n.z * m[2][j];
    return r;
}

InversableTransform::InversableTransform(const Vector3d& t, const Vector3d& r, const Vector3d& s)
    : translate(t), rotate(r), scale(s) {
    direct = Transform::translate(t) * Transform::rotate(r) * Transform::scale(s);
    inverse = Transform::scale(Vector3d(1.0 / s.x, 1.0 / s.y, 1.0 / s.z)) *
              Transform::rotate_inverse(Vector3d(-r.x, -r.y, -r.z)) *
              Transform::translate(Vector3d(-t.x, -t.y, -t.z));
}

}  // namespace transform
}  // namespace algebra

// ------------------------------------------------------------------------------------------------
// camera
// ------------------------------------------------------------------------------------------------
namespace camera {

Camera::Camera(const Vector3d& position, const Vector3d& direction, const Vector3d& up_vector,
               double focal_length, double fov)
    : position_(position), fov_(fov), focal_length_(focal_length) {
    Vector3d right_vec = direction.cross(up_vector).normalize();
    direction_ = direction.normalize();
    up_ = right_vec.cross(direction).normalize();
    rigth_ = right_vec;
}

void Camera::set_direction(const Vector3d& d) {
    direction_ = d.normalize();
    rigth_ = direction_.cross(up_).normalize();
    up_ = rigth_.cross(direction_).normalize();
}

Camera Camera::from_pod(const rt_camera& c) {
    Camera cam;
    cam.position_ = Vector3d(c.position.x, c.position.y, c.position.z);
    cam.direction_ = Vector3d(c.direction.x, c.direction.y, c.direction.z);
    cam.up_ = Vector3d(c.up.x, c.up.y, c.up.z);
    cam.rigth_ = Vector3d(c.right.x, c.right.y, c.right.z);
    cam.fov_ = c.fov_rad;
    cam.focal_length_ = c.focal_length;
    return cam;
}

rt_camera Camera::to_pod() const {
    rt_camera c;
    c.position = rt_vec3{position_.x, position_.y, position_.z};
    c.direction = rt_vec3{direction_.x, direction_.y, direction_.z};
    c.up = rt_vec3{up_.x, up_.y, up_.z};
    c.right = rt_vec3{rigth_.x, rigth_.y, rigth_.z};
    c.fov_rad = fov_;
    c.focal_length = focal_length_;
    return c;
}

}  // namespace camera

// ------------------------------------------------------------------------------------------------
// world: JSON -> Scene -> FlatScene
// ------------------------------------------------------------------------------------------------
namespace world {

static ImageLoaderFn g_image_loader = nullptr;
void set_image_loader(ImageLoaderFn fn) { g_image_loader = fn; }

rt_scene_desc FlatScene::desc() const {
    rt_scene_desc d;
    d.n_shapes = (uint32_t)kind.size();
    d.kind = kind.data();
    d.flags = flags.data();
    d.inverse = inverse.data();
    d.direct = direct.data();
    d.params = params.data();
    d.material = material.data();
    d.n_materials = (uint32_t)materials.size();
    d.materials = materials.data();
    d.n_textures = (uint32_t)textures.size();
    d.textures = textures.data();
    d.n_images = (uint32_t)images.size();
    d.images = images.data();
    d.n_noise = (uint32_t)noise.size();
    d.noise = noise.data();
    return d;
}

namespace {

using rtjson::Value;

// Vector3d derives Deserialize: serde accepts both the map {"x","y","z"} and the sequence [x,y,z]
Vector3d parse_vec3(const Value& v) {
    if (v.kind == Value::Array) {
        if (v.arr.size() != 3) throw std::runtime_error("Vector3d: expected 3 elements");
        return Vector3d(v.arr[0]->as_number(), v.arr[1]->as_number(), v.arr[2]->as_number());
    }
    if (v.kind == Value::Object)
        return Vector3d(v.at("x").as_number(), v.at("y").as_number(), v.at("z").as_number());
    throw std::runtime_error("Vector3d: expected an array or an object");
}

InversableTransform parse_transform(const Value& v) {  // transform.rs:120-187
    return InversableTransform(parse_vec3(v.at("translate")), parse_vec3(v.at("rotate")),
                               parse_vec3(v.at("scale")));
}

bool load_ppm(const std::string& path, uint32_t* w, uint32_t* h, std::vector<uint8_t>* rgba) {
    std::ifstream f(path, std::ios::binary);
    if (!f) return false;
    std::string magic;
    f >> magic;
    if (magic != "P6") return false;
    auto next_int = [&]() -> long {
        for (;;) {
            int c = f.peek();
            if (c == '#') { std::string line; std::getline(f, line); }
            else if (isspace(c)) f.get();
            else break;
        }
        long x; f >> x; return x;
    };
    long W = next_int(), H = next_int(), maxv = next_int();
    f.get();
    if (!f || W <= 0 || H <= 0 || maxv != 255) return false;
    std::vector<uint8_t> rgb((size_t)W * H * 3);
    f.read((char*)rgb.data(), (std::streamsize)rgb.size());
    if (!f) return false;
    rgba->resize((size_t)W * H * 4);
    for (size_t i = 0; i < (size_t)W * H; i++) {
        (*rgba)[4 * i + 0] = rgb[3 * i + 0];
        (*rgba)[4 * i + 1] = rgb[3 * i + 1];
        (*rgba)[4 * i + 2] = rgb[3 * i + 2];
        (*rgba)[4 * i + 3] = 255;
    }
    *w = (uint32_t)W;
    *h = (uint32_t)H;
    return true;
}

// xoshiro256** seeded through splitmix64: the reproducible stand-in for rand::thread_rng()
struct HostRng {
    uint64_t s[4];
    explicit HostRng(uint64_t seed) {
        uint64_t x = seed;
        for (int i = 0; i < 4; i++) {
            uint64_t z = (x += 0x9E3779B97F4A7C15ull);
            z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
            z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
            s[i] = z ^ (z >> 31);
        }
    }
    static uint64_t rotl(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
    uint64_t next_u64() {
        uint64_t result = rotl(s[1] * 5, 7) * 9;
        uint64_t t = s[1] << 17;
        s[2] ^= s[0]; s[3] ^= s[1]; s[1] ^= s[2]; s[0] ^= s[3];
        s[2] ^= t;
        s[3] = rotl(s[3], 45);
        return result;
    }
    double gen() {  // rng.gen::<f64>(): 53 random bits scaled to [0,1)
        return (double)(next_u64() >> 11) * (1.0 / 9007199254740992.0);
    }
};

// Perlin::new, src/algebra/noise.rs:24-41.  The reference shuffles with thread_rng (unreproducible); the
// tables here come from the scene seed: Fisher-Yates like SliceRandom::shuffle (i from the top, j uniform
// in 0..=i), ranvec = Vector3d::random(-1.0, 1.0) = min + (max - min) * gen() per component.
rt_perlin make_perlin(uint64_t seed) {
    HostRng rng(seed ^ 0x5045524C494E0001ull);
    rt_perlin pn;
    uint32_t* perms[3] = {pn.perm_x, pn.perm_y, pn.perm_z};
    for (int a = 0; a < 3; a++) {
        for (uint32_t i = 0; i < 256; i++) perms[a][i] = i;
        for (uint32_t i = 255; i > 0; i--) {
            uint32_t j = (uint32_t)(rng.next_u64() % (uint64_t)(i + 1));
            std::swap(perms[a][i], perms[a][j]);
        }
    }
    for (int i = 0; i < 256; i++) (void)rng.gen();  // ranfloat (drawn, never used by noise / turb)
    for (int i = 0; i < 256; i++) {
        double x = -1.0 + (1.0 - -1.0) * rng.gen();
        double y = -1.0 + (1.0 - -1.0) * rng.gen();
        double z = -1.0 + (1.0 - -1.0) * rng.gen();
        pn.ranvec[i] = rt_vec3{x, y, z};
    }
    return pn;
}

struct Builder {
    FlatScene& fs;
    std::map<std::string, uint32_t> material_by_name;
    uint64_t seed = 1;
    explicit Builder(FlatScene& f) : fs(f) {}

    uint32_t add_solid(const Vector3d& c) {
        rt_texture t;
        memset(&t, 0, sizeof t);
        t.kind = RT_TEX_SOLID;
        t.color = rt_vec3{c.x, c.y, c.z};
        fs.textures.push_back(t);
        return (uint32_t)fs.textures.size() - 1;
    }

    uint32_t add_texture(const Value& v, int depth = 0) {  // typetag "type" dispatch, texture.rs:5
        if (depth > RT_TEX_MAX_DEPTH) throw std::runtime_error("texture nesting too deep");
        const std::string& type = v.at("type").as_string();
        rt_texture t;
        memset(&t, 0, sizeof t);
        if (type == "SolidColor") {
            return add_solid(parse_vec3(v.at("color")));
        } else if (type == "CheckerTexture") {
            t.kind = RT_TEX_CHECKER;
            Vector3d m = parse_vec3(v.at("multipliers"));
            t.color = rt_vec3{m.x, m.y, m.z};
            t.odd = add_texture(v.at("odd"), depth + 1);
            t.even = add_texture(v.at("even"), depth + 1);
        } else if (type == "UVChecker") {
            t.kind = RT_TEX_UV_CHECKER;
            const Value& m = v.at("multipliers");  // (f64, f64) tuple == 2-element sequence
            if (m.kind != Value::Array || m.arr.size() != 2)
                throw std::runtime_error("UVChecker.multipliers: expected [f64, f64]");
            t.color = rt_vec3{m.arr[0]->as_number(), m.arr[1]->as_number(), 0.0};
            t.odd = add_texture(v.at("odd"), depth + 1);
            t.even = add_texture(v.at("even"), depth + 1);
        } else if (type == "ImageTexture") {
            t.kind = RT_TEX_IMAGE;
            const std::string& fn = v.at("image_filename").as_string();
            uint32_t w = 0, h = 0;
            std::vector<uint8_t> rgba;
            bool ok = load_ppm(fn, &w, &h, &rgba);
            if (!ok && g_image_loader) {
                uint8_t* data = nullptr;
                if (g_image_loader(fn.c_str(), &w, &h, &data) && data) {
                    rgba.assign(data, data + (size_t)w * h * 4);
                    free(data);
                    ok = true;
                }
            }
            // the reference panics: "Could not open texture file: ..." (texture.rs:130-133)
            if (!ok) throw std::runtime_error("Could not open texture file: " + fn);
            fs.image_data.push_back(std::move(rgba));
            rt_image im;
            im.width = w;
            im.height = h;
            im.rgba = nullptr;  // fixed up after all images are stored (vector may reallocate)
            fs.images.push_back(im);
            t.image = (uint32_t)fs.images.size() - 1;
        } else if (type == "NoiseTexture") {  // texture.rs:54-68; `noise` is #[serde(skip)] -> Perlin::default()
            t.kind = RT_TEX_NOISE;
            t.color = rt_vec3{v.at("scale").as_number(), 0.0, 0.0};
            fs.noise.push_back(make_perlin(seed + 0x9E37ull * (uint64_t)fs.noise.size()));
            t.image = (uint32_t)fs.noise.size() - 1;
        } else {
            throw std::runtime_error("unknown variant `" + type + "` for Texture");
        }
        fs.textures.push_back(t);
        return (uint32_t)fs.textures.size() - 1;
    }

    uint32_t add_material(const std::string& name, const Value& v) {  // material.rs:22
        const std::string& type = v.at("type").as_string();
        rt_material m;
        memset(&m, 0, sizeof m);
        if (type == "Lambertian") {
            m.kind = RT_MAT_LAMBERTIAN;
            m.texture = add_texture(v.at("albedo"));
        } else if (type == "Metal") {
            m.kind = RT_MAT_METAL;
            m.texture = add_texture(v.at("albedo"));
            m.scalar = v.at("fuzz").as_number();
        } else if (type == "Dielectric") {
            m.kind = RT_MAT_DIELECTRIC;
            m.scalar = v.at("index_of_refraction").as_number();
        } else if (type == "DiffuseLight") {
            m.kind = RT_MAT_DIFFUSE_LIGHT;
            m.texture = add_texture(v.at("emit"));
        } else if (type == "EmptyMaterial") {
            m.kind = RT_MAT_EMPTY;
        } else {
            throw std::runtime_error("unknown variant `" + type + "` for Material");
        }
        fs.materials.push_back(m);
        fs.material_names.push_back(name);
        return (uint32_t)fs.materials.size() - 1;
    }

    void push_shape(int kind, uint8_t flags, const InversableTransform& tr, const double* params8,
                    uint32_t material, const std::string& name) {
        fs.kind.push_back((uint8_t)kind);
        fs.flags.push_back(flags);
        for (int r = 0; r < 3; r++)
            for (int c = 0; c < 4; c++) {
                fs.inverse.push_back(tr.inverse.m[r][c]);
                fs.direct.push_back(tr.direct.m[r][c]);
            }
        for (int k = 0; k < RT_SHAPE_PARAMS; k++) fs.params.push_back(params8 ? params8[k] : 0.0);
        fs.material.push_back(material);
        fs.shape_names.push_back(name);
    }

    uint32_t material_index(const Value& shape) {
        const std::string& name = shape.at("material").as_string();
        auto it = material_by_name.find(name);
        // the reference indexes the HashMap and panics on a missing key (shapes/mod.rs:760)
        if (it == material_by_name.end()) throw std::runtime_error("material `" + name + "` not found");
        return it->second;
    }

    void add_shape(const Value& v) {  // ShapeJson typetag dispatch, json_models.rs:15
        const std::string& type = v.at("type").as_string();
        const Value* nm = v.find("name");
        std::string name = (nm && nm->kind == Value::String) ? nm->str : type;
        double p[RT_SHAPE_PARAMS] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (type == "Sphere") {  // shapes/mod.rs:741-764
            (void)v.at("name");
            const Value* inv = v.find("inverse_normal");
            uint8_t flags = (inv && inv->as_bool()) ? RT_SHAPE_FLAG_INVERSE_NORMAL : 0;
            push_shape(RT_SHAPE_SPHERE, flags, parse_transform(v.at("transform")), p, material_index(v), name);
        } else if (type == "Cube") {  // :818-837
            (void)v.at("name");
            push_shape(RT_SHAPE_CUBE, 0, parse_transform(v.at("transform")), p, material_index(v), name);
        } else if (type == "Rectangle") {  // :791-816
            p[0] = v.at("x0").as_number();
            p[1] = v.at("y0").as_number();
            p[2] = v.at("x1").as_number();
            p[3] = v.at("y1").as_number();
            push_shape(RT_SHAPE_RECTANGLE, 0, parse_transform(v.at("transform")), p, material_index(v), name);
        } else if (type == "BruteForsableShape") {  // ray_marching.rs:532-556
            const Value& sh = v.at("shape");
            const std::string& st = sh.at("type").as_string();
            int surf;
            if (st == "Heart") surf = RT_SURF_HEART;                         // :563-571
            else if (st == "Sine") { surf = RT_SURF_SINE; p[3] = sh.at("a").as_number(); }
            else if (st == "Star") { surf = RT_SURF_STAR; p[3] = sh.at("a").as_number(); }
            else if (st == "DupinCyclide") {
                surf = RT_SURF_DUPIN;
                p[3] = sh.at("a").as_number();
                p[4] = sh.at("b").as_number();
                p[5] = sh.at("c").as_number();
                p[6] = sh.at("d").as_number();
            } else if (st == "HuntsSurface") surf = RT_SURF_HUNTS;
            else if (st == "Cushion") surf = RT_SURF_CUSHION;
            else throw std::runtime_error("unknown variant `" + st + "` for BruteForceShapeJson");
            if (surf != RT_SURF_HEART) p[7] = sh.at("sphere_radius").as_number();
            p[0] = (double)surf;
            p[1] = v.at("step").as_number();
            const Value* d = v.find("depth");
            double depth = d ? d->as_number() : 4.0;  // default_depth, :528-530
            if (depth < 0 || depth > 255 || depth != std::floor(depth))
                throw std::runtime_error("BruteForsableShape.depth: expected u8");
            p[2] = depth;
            push_shape(RT_SHAPE_MARCH, 0, parse_transform(v.at("transform")), p, material_index(v), name);
        } else if (type == "Torus") {  // shapes/mod.rs:766-789
            (void)v.at("name");
            p[0] = v.at("radius").as_number();
            p[1] = v.at("tube_radius").as_number();
            push_shape(RT_SHAPE_TORUS, 0, parse_transform(v.at("transform")), p, material_index(v), name);
        } else {
            throw std::runtime_error("unknown variant `" + type + "` for ShapeJson");
        }
    }
};

// json_models.rs:50-133
void add_random_spheres(Builder& b, uint64_t seed) {
    HostRng rng(seed);
    for (int a = -11; a < 11; a++) {
        for (int bb = -11; bb < 11; bb++) {  // cartesian_product: a outer, b inner
            double cx = (double)a + 0.9 * rng.gen();
            double cz = (double)bb + 0.9 * rng.gen();
            Vector3d center(cx, 0.2, cz);
            double rad = 0.2;
            Vector3d diff(center.x - 4.0, center.y - 0.2, center.z - 0.0);
            if (!(diff.length() > 0.9)) continue;
            double mat_choice = rng.gen();
            rt_material m;
            memset(&m, 0, sizeof m);
            if (mat_choice < 0.8) {
                Vector3d rc(rng.gen(), rng.gen(), rng.gen());  // Vector3d::random(0.0, 1.0)
                m.kind = RT_MAT_LAMBERTIAN;
                m.texture = b.add_solid(Vector3d(rc.x * rc.x, rc.y * rc.y, rc.z * rc.z));
            } else if (mat_choice < 0.95) {
                Vector3d rc(rng.gen(), rng.gen(), rng.gen());
                m.kind = RT_MAT_METAL;
                m.texture = b.add_solid(Vector3d(0.5 * (1.0 - rc.x), 0.5 * (1.0 - rc.y), 0.5 * (1.0 - rc.z)));
                m.scalar = 0.5 * rng.gen();
            } else {
                m.kind = RT_MAT_DIELECTRIC;
                m.scalar = 1.5;
            }
            char name[64];
            snprintf(name, sizeof name, "Sphere_%d_%d", a, bb);
            b.fs.materials.push_back(m);
            b.fs.material_names.push_back(std::string("#") + name);
            InversableTransform tr(center, Vector3d(0.0, 0.0, 0.0), Vector3d(rad, rad, rad));
            b.push_shape(RT_SHAPE_SPHERE, 0, tr, nullptr, (uint32_t)b.fs.materials.size() - 1, name);
        }
    }
}

thread_local std::string g_host_error;

}  // namespace

std::shared_ptr<Scene> Scene::from_json(const std::string& data, uint64_t seed, bool add_spheres) {
    rtjson::ValuePtr root = rtjson::parse(data);
    if (root->kind != Value::Object) throw std::runtime_error("scene: expected a JSON object");
    std::shared_ptr<Scene> sc(new Scene());

    // SceneJson, json_models.rs:23-29: all four fields are required
    const Value& cam = root->at("camera");  // CameraJson, camera/mod.rs:12-19,48-58 (fov in degrees)
    const double kPi = 3.14159265358979323846264338327950288;
    sc->camera_ = camera::Camera(parse_vec3(cam.at("position")), parse_vec3(cam.at("direction")),
                                 parse_vec3(cam.at("up")), cam.at("focal_length").as_number(),
                                 cam.at("fov").as_number() * (kPi / 180.0));
    sc->background_ = parse_vec3(root->at("background"));

    Builder b(sc->flat_);
    b.seed = seed;
    const Value& mats = root->at("materials");
    if (mats.kind != Value::Object) throw std::runtime_error("materials: expected a map");
    for (auto& kv : mats.obj) b.material_by_name[kv.first] = b.add_material(kv.first, *kv.second);
    const Value& shapes = root->at("shapes");
    if (shapes.kind != Value::Array) throw std::runtime_error("shapes: expected a sequence");
    for (auto& s : shapes.arr) b.add_shape(*s);
    if (add_spheres) add_random_spheres(b, seed);
    for (size_t i = 0; i < sc->flat_.images.size(); i++) sc->flat_.images[i].rgba = sc->flat_.image_data[i].data();
    return sc;
}

Scene::~Scene() {
    for (auto& kv : dev_) rt_scene_destroy(kv.second);
    for (auto& kv : multi_) rt_scene_destroy(kv.second);
}

void Scene::assign_material(uint32_t shape_index, const std::string& material_name) {
    if (!dev_.empty() || !multi_.empty()) throw std::runtime_error("assign_material: the scene is already on the device");
    if (shape_index >= flat_.material.size()) throw std::runtime_error("assign_material: bad shape index");
    for (size_t i = 0; i < flat_.material_names.size(); i++)
        if (flat_.material_names[i] == material_name) {
            flat_.material[shape_index] = (uint32_t)i;
            return;
        }
    throw std::runtime_error("material `" + material_name + "` not found");
}

void Scene::set_transforms(uint32_t n, const uint32_t* index, const double* direct16, const double* inverse16) {
    if (n == 0) return;
    if (!index || !direct16 || !inverse16) throw std::runtime_error("set_transforms: null array");
    std::vector<uint32_t> sorted(index, index + n);
    std::sort(sorted.begin(), sorted.end());
    if (sorted.back() >= shape_count()) throw std::runtime_error("set_transforms: bad shape index");
    if (std::adjacent_find(sorted.begin(), sorted.end()) != sorted.end())
        throw std::runtime_error("set_transforms: a shape index is listed twice");
    std::vector<double> inv((size_t)12 * n), dir((size_t)12 * n);   // rows 0..2, the rows the description holds
    for (uint32_t k = 0; k < n; k++)
        for (int j = 0; j < 12; j++) {
            inv[(size_t)12 * k + j] = inverse16[(size_t)16 * k + j];
            dir[(size_t)12 * k + j] = direct16[(size_t)16 * k + j];
        }
    std::vector<rt_scene*> handles;
    for (auto& kv : dev_) handles.push_back(kv.second);
    for (auto& kv : multi_) handles.push_back(kv.second);
    for (rt_scene* h : handles)
        if (rt_scene_update_transforms(h, n, index, inv.data(), dir.data()) != RT_OK)
            throw std::runtime_error(std::string("rt_scene_update_transforms: ") + rt_last_error());
    for (uint32_t k = 0; k < n; k++)
        for (int j = 0; j < 12; j++) {
            flat_.inverse[(size_t)12 * index[k] + j] = inv[(size_t)12 * k + j];
            flat_.direct[(size_t)12 * index[k] + j] = dir[(size_t)12 * k + j];
        }
}

// One rt_scene per device, created on first use and kept until the Scene dies: a handle given out for one device
// (GpuRenderer, DistributedRenderer, the Python helpers) stays valid when another device is asked for.
rt_scene* Scene::device_scene(int device) {
    auto it = dev_.find(device);
    if (it != dev_.end()) return it->second;
    rt_scene_desc d = flat_.desc();
    rt_scene* h = nullptr;
    int rc = rt_scene_create(&d, device, &h);
    if (rc != RT_OK) throw std::runtime_error(std::string("rt_scene_create: ") + rt_last_error());
    dev_[device] = h;
    return h;
}

rt_scene* Scene::device_scene(const std::vector<int>& devices) {
    if (devices.empty()) throw std::runtime_error("device_scene: empty device list");
    if (devices.size() == 1) return device_scene(devices[0]);
    auto it = multi_.find(devices);
    if (it != multi_.end()) return it->second;
    rt_scene_desc d = flat_.desc();
    rt_scene* h = nullptr;
    int rc = rt_scene_create_multi(&d, (int)devices.size(), devices.data(), &h);
    if (rc != RT_OK) throw std::runtime_error(std::string("rt_scene_create_multi: ") + rt_last_error());
    multi_[devices] = h;
    return h;
}

std::vector<RayHit> Scene::closest_hit(const std::vector<Ray>& rays, double min_t, double max_t, int mode,
                                       int device) {
    rt_scene* ds = device_scene(device);
    size_t n = rays.size();
    std::vector<int32_t> idx(n);
    std::vector<double> t(n), uv(2 * n);
    std::vector<rt_vec3> nrm(n), pt(n);
    std::vector<uint8_t> ff(n);
    static_assert(sizeof(Ray) == sizeof(rt_ray), "Ray must be layout-identical to rt_ray");
    int rc = rt_intersect_batch(ds, (const rt_ray*)rays.data(), n, min_t, max_t, mode, idx.data(), t.data(),
                                nrm.data(), pt.data(), uv.data(), ff.data());
    if (rc != RT_OK) throw std::runtime_error(std::string("rt_intersect_batch: ") + rt_last_error());
    std::vector<RayHit> out(n);
    for (size_t i = 0; i < n; i++) {
        out[i].shape_index = idx[i];
        out[i].distance = t[i];
        out[i].normal = Vector3d(nrm[i].x, nrm[i].y, nrm[i].z);
        out[i].point = Vector3d(pt[i].x, pt[i].y, pt[i].z);
        out[i].u = uv[2 * i];
        out[i].v = uv[2 * i + 1];
        out[i].is_front_face = ff[i] != 0;
    }
    return out;
}

}  // namespace world

// ------------------------------------------------------------------------------------------------
// renderer
// ------------------------------------------------------------------------------------------------
namespace renderer {

GpuRenderer::GpuRenderer(std::shared_ptr<world::Scene> scene, uint32_t /*thread_number*/, uint32_t depth,
                         int device, uint64_t seed)
    : scene_(scene), depth_(depth), device_(device), seed_(seed), started_(false), pixels_(0) {
    scene_->device_scene(device_);  // upload now, like ThreadPoolRenderer::new spawning its workers
}

GpuRenderer::GpuRenderer(std::shared_ptr<world::Scene> scene, uint32_t /*thread_number*/, uint32_t depth,
                         const std::vector<int>& devices, uint64_t seed)
    : scene_(scene), depth_(depth), device_(devices.empty() ? 0 : devices[0]), devices_(devices), seed_(seed),
      started_(false), pixels_(0) {
    if (devices_.size() == 1) devices_.clear();
    handle();
}

rt_scene* GpuRenderer::handle() const {
    return devices_.empty() ? scene_->device_scene(device_) : scene_->device_scene(devices_);
}

void GpuRenderer::start_rendering(std::shared_ptr<camera::Camera> camera, const camera::ImageParams& img,
                                  uint32_t samples_number) {
    rt_render_params p;
    memset(&p, 0, sizeof p);
    p.image = rt_image_params{img.width, img.height};
    p.samples_number = samples_number;
    p.max_depth = depth_;
    p.seed = seed_;
    p.shard_count = 1;
    rt_camera c = camera->to_pod();
    int rc = rt_render_start(handle(), &c, &p);
    if (rc != RT_OK) throw std::runtime_error(std::string("rt_render_start: ") + rt_last_error());
    started_ = true;
    pixels_ = (uint64_t)img.width * img.height;
}

bool GpuRenderer::render_step(std::vector<Vector3d>& buffer) { return render_step(buffer.data(), buffer.size()); }

bool GpuRenderer::render_step(Vector3d* buffer, size_t len) {
    if (!started_) return false;  // the reference's try_iter simply finds nothing
    static_assert(sizeof(Vector3d) == sizeof(rt_vec3), "Vector3d must be layout-identical to rt_vec3");
    // the reference indexes buffer[index] and panics when it is too short (step_by_step.rs:116)
    if (len < pixels_) throw std::runtime_error("render_step: buffer shorter than width*height");
    int done = 0;
    int rc = rt_render_poll(handle(), (rt_vec3*)buffer, &done);
    if (rc != RT_OK) throw std::runtime_error(std::string("rt_render_poll: ") + rt_last_error());
    if (done) started_ = false;
    return done != 0;
}

void GpuRenderer::stop_rendering() {
    if (started_) rt_render_stop(handle());
    started_ = false;
}

}  // namespace renderer
}  // namespace ray_tracing
