// raytracer.hpp -- host-side C++ mirror of the reference's scene / camera / material API,
// sitting on top of the C ABI (include/b200rt.h).
//
// A program written against DeltaPavonis/cpp_raytracer -- build a `Scene` out of `Sphere`,
// `Parallelogram` and `Box` objects holding `Lambertian` / `Metal` / `Dielectric` /
// `DiffuseLight` materials, configure a `Camera` with the fluent setters and call
// `.render(world).send_as_ppm(path)` (reference src/main.cpp:13-650) -- compiles against this
// header unchanged (the compatibility headers base/*.h, shapes/*.h, util/*.h, math/*.h next to
// this directory forward here).  Same names, same argument meaning, same defaults, same error
// convention (message on std::cout, then std::exit(-1); reference image.h:39-42, rgb.h:136-141).
//
// What is different by design: objects here only DESCRIBE the scene.  There is no CPU
// intersection or shading code in this header: `Camera::render` flattens the scene into the flat
// arrays of B200rtSceneDesc and calls b200rt_render_scene, i.e. the CUDA path.  Unknown
// `Hittable` / `Material` subclasses are an error (closed set), never silently skipped.
//
// Reference lines each piece follows are cited inline.
#pragma once

#include <algorithm>
#include <array>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <iostream>
#include <memory>
#include <mutex>
#include <numbers>
#include <optional>
#include <random>
#include <span>
#include <string>
#include <thread>
#include <type_traits>
#include <typeinfo>
#include <limits>
#include <unordered_map>
#include <utility>
#include <vector>

#include "../../../../include/b200rt.h"

// ===== util/rand_util.h ====================================================================
// Bit-exact restatement of the reference's generators (rand_util.h:11-127): scenes are built
// with these, so a scene function gives the same spheres here as in the reference.
class SeedSeqGenerator {
    using seed_type = uint32_t;
    std::optional<seed_type> custom_seed;
    std::mutex mtx;
    SeedSeqGenerator() = default;
public:
    static SeedSeqGenerator &get_instance() { static SeedSeqGenerator s; return s; }
    SeedSeqGenerator(const SeedSeqGenerator &) = delete;
    SeedSeqGenerator &operator=(const SeedSeqGenerator &) = delete;
    seed_type next_seed() {                                           // rand_util.h:51-69
        std::lock_guard<std::mutex> g(mtx);
        if (!custom_seed) {
            custom_seed = std::random_device{}();
            std::cout << "SeedSeqGenerator: No random seed provided, using " << *custom_seed
                      << " (Use SeedSeqGenerator::get_instance().set_seed([custom seed]) to set a custom seed)" << std::endl;
        }
        custom_seed = 2'483'477u * (*custom_seed) + 2'987'434'823u;
        return *custom_seed;
    }
    void set_seed(seed_type seed) {                                   // rand_util.h:75-79
        std::cout << "SeedSeqGenerator: Using user-provided random seed " << seed << '\n' << std::endl;
        custom_seed = seed;
    }
};

inline double rand_double(double min = 0, double max = 1) {          // rand_util.h:85-117
    thread_local uint32_t seed = SeedSeqGenerator::get_instance().next_seed();
    seed = 1'664'525u * seed + 1'013'904'223u;
    constexpr double SCALE = 1 / static_cast<double>(std::numeric_limits<uint32_t>::max() - 1);
    return min + (max - min) * static_cast<double>(seed) * SCALE;
}

inline int rand_int(int min = 0, int max = 1) {                      // rand_util.h:120-127
    thread_local std::mt19937 generator{SeedSeqGenerator::get_instance().next_seed()};
    thread_local std::uniform_int_distribution<> dist;
    dist.param(std::uniform_int_distribution<>::param_type{min, max});
    return dist(generator);
}

// ===== math/interval.h (the parts scene code can touch) ====================================
struct Interval {
    double min, max;
    Interval(double min_, double max_) : min{min_}, max{max_} {}
    bool contains_inclusive(double d) const { return min <= d && d <= max; }
    bool contains_exclusive(double d) const { return min < d && d < max; }
    double size() const { return max - min; }
    static Interval with_min(double m) { return Interval(m, std::numeric_limits<double>::infinity()); }
};

// ===== math/vec3d.h ==========================================================================
struct Vec3D {
    double x = 0, y = 0, z = 0;                                       // aggregate, as in the reference
    const double &operator[](size_t a) const { return a == 0 ? x : (a == 1 ? y : z); }
    double &operator[](size_t a) { return a == 0 ? x : (a == 1 ? y : z); }
    Vec3D operator-() const { return Vec3D{-x, -y, -z}; }
    Vec3D &operator+=(const Vec3D &r) { x += r.x; y += r.y; z += r.z; return *this; }
    Vec3D &operator-=(const Vec3D &r) { x -= r.x; y -= r.y; z -= r.z; return *this; }
    Vec3D &operator*=(double d) { x *= d; y *= d; z *= d; return *this; }
    Vec3D &operator/=(double d) { return *this *= (1 / d); }         // vec3d.h:31
    double mag() const { return std::sqrt(x * x + y * y + z * z); }
    double mag_squared() const { return x * x + y * y + z * z; }
    Vec3D unit_vector() const;
    bool near_zero(double eps = 1e-8) const { return std::fabs(x) < eps && std::fabs(y) < eps && std::fabs(z) < eps; }
    static Vec3D zero() { return Vec3D{0, 0, 0}; }
    static Vec3D random(double min = 0, double max = 1) {            // braced list: x, y, z in order (vec3d.h:60)
        return Vec3D{rand_double(min, max), rand_double(min, max), rand_double(min, max)};
    }
};
inline Vec3D operator+(const Vec3D &a, const Vec3D &b) { auto r = a; r += b; return r; }
inline Vec3D operator-(const Vec3D &a, const Vec3D &b) { auto r = a; r -= b; return r; }
inline Vec3D operator*(const Vec3D &a, double d) { auto r = a; r *= d; return r; }
inline Vec3D operator*(double d, const Vec3D &a) { return a * d; }
inline Vec3D operator/(const Vec3D &a, double d) { auto r = a; r /= d; return r; }
inline double dot(const Vec3D &a, const Vec3D &b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline Vec3D cross(const Vec3D &a, const Vec3D &b) {
    return Vec3D{a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x};
}
inline Vec3D Vec3D::unit_vector() const { return *this / this->mag(); }
inline std::ostream &operator<<(std::ostream &os, const Vec3D &v) { return os << "(" << v.x << ", " << v.y << ", " << v.z << ")"; }
using Point3D = Vec3D;

struct Ray3D {                                                        // math/ray3d.h
    Point3D origin{0, 0, 0};
    Vec3D dir{0, 0, 0};
    Point3D operator()(double t) const { return origin + t * dir; }
};

// ===== util/rgb.h =============================================================================
class RGB {
    RGB(double r_, double g_, double b_) : r{r_}, g{g_}, b{b_} {}
public:
    double r, g, b;
    double luminance() const { return 0.2126 * r + 0.7152 * g + 0.0722 * b; }                 // rgb.h:28-30
    static RGB from_mag(double red, double green, double blue) { return RGB(red, green, blue); }
    static RGB from_mag(double v) { return from_mag(v, v, v); }
    static RGB from_rgb(double red, double green, double blue, double max_magnitude = 255) {
        return RGB(red / max_magnitude, green / max_magnitude, blue / max_magnitude);
    }
    static RGB from_rgb(double v, double max_magnitude = 255) { return from_rgb(v, v, v, max_magnitude); }
    static RGB zero() { return from_mag(0); }
    // rgb.h:64-66 passes three rand_double() calls as function ARGUMENTS, whose evaluation order
    // is unspecified; g++ (the compiler the reference is built with) evaluates them last to first.
    // The order is made explicit here so that scenes come out identical with any compiler; the
    // scene-dump test pins it against reference-built scenes.
    static RGB random(double min = 0, double max = 1) {
        const double blue = rand_double(min, max);
        const double green = rand_double(min, max);
        const double red = rand_double(min, max);
        return from_mag(red, green, blue);
    }
    RGB &operator+=(const RGB &o) { r += o.r; g += o.g; b += o.b; return *this; }
    RGB &operator*=(double d) { r *= d; g *= d; b *= d; return *this; }
    RGB &operator/=(double d) { return *this *= (1 / d); }
    // rgb.h:90-113: Reinhard by luminance, gamma, int(scale * v); no clamp.
    std::string as_string(std::string delimiter = " ", std::string surrounding = "", double max_magnitude = 255,
                          double gamma = 2, bool use_tone_mapping = true) const {
        double r2 = r, g2 = g, b2 = b;
        if (use_tone_mapping) { const double L = luminance(); r2 /= 1 + L; g2 /= 1 + L; b2 /= 1 + L; }
        const double scale = max_magnitude + 0.999999;
        auto enc = [&](double v) { return std::to_string(static_cast<int>(scale * std::pow(v, 1 / gamma))); };
        return (surrounding.empty() ? "" : std::string{surrounding[0]}) + enc(r2) + delimiter + enc(g2) + delimiter + enc(b2) +
               (surrounding.empty() ? "" : std::string{surrounding[1]});
    }
};
inline RGB operator+(const RGB &a, const RGB &b) { return RGB::from_mag(a.r + b.r, a.g + b.g, a.b + b.b); }
inline RGB operator*(const RGB &a, double d) { auto r = a; r *= d; return r; }
inline RGB operator*(double d, const RGB &a) { return a * d; }
inline RGB operator*(const RGB &a, const RGB &b) { return RGB::from_mag(a.r * b.r, a.g * b.g, a.b * b.b); }
inline RGB lerp(const RGB &a, const RGB &b, double d) {                                         // rgb.h:133-148
    if (!Interval(0, 1).contains_inclusive(d)) {
        std::cout << "Error: In `lerp(...)`, lerp proportion " << d << " is not in the range [0, 1]." << std::endl;
        std::exit(-1);
    }
    return RGB::from_mag((1 - d) * a.r + d * b.r, (1 - d) * a.g + d * b.g, (1 - d) * a.b + d * b.b);
}

// ===== base/material.h ========================================================================
// Parameter holders.  kind()/colour()/param() are what the flattening step reads.
struct Material {
    virtual int kind() const = 0;                  // B200RT_MAT_*
    virtual RGB colour() const = 0;
    virtual double param() const = 0;
    virtual RGB emit() const { return RGB::zero(); }                                            // material.h:38-40
    virtual void print_to(std::ostream &os) const = 0;
    virtual ~Material() = default;
};
inline std::ostream &operator<<(std::ostream &os, const Material &m) { m.print_to(os); return os; }

class Lambertian : public Material {                                                            // material.h:58-95
    RGB intrinsic_color;
public:
    Lambertian(const RGB &c) : intrinsic_color{c} {}
    int kind() const override { return B200RT_MAT_LAMBERTIAN; }
    RGB colour() const override { return intrinsic_color; }
    double param() const override { return 0; }
    void print_to(std::ostream &os) const override { os << "Lambertian {color: " << intrinsic_color.as_string(", ", "()") << "} " << std::flush; }
};
class Metal : public Material {                                                                 // material.h:105-152
    RGB intrinsic_color;
    double fuzz_factor;
public:
    Metal(const RGB &c, double fuzz = 0) : intrinsic_color{c}, fuzz_factor{std::fmin(fuzz, 1.)} {}
    int kind() const override { return B200RT_MAT_METAL; }
    RGB colour() const override { return intrinsic_color; }
    double param() const override { return fuzz_factor; }
    void print_to(std::ostream &os) const override {
        os << "Metal {color: " << intrinsic_color.as_string(", ", "()") << ", fuzz factor: " << fuzz_factor << "} " << std::flush;
    }
};
class Dielectric : public Material {                                                            // material.h:164-227
    double refr_index;
public:
    Dielectric(double refractive_index) : refr_index{refractive_index} {}
    int kind() const override { return B200RT_MAT_DIELECTRIC; }
    RGB colour() const override { return RGB::from_mag(1, 1, 1); }
    double param() const override { return refr_index; }
    void print_to(std::ostream &os) const override { os << "Dielectric {refractive index: " << refr_index << "} " << std::flush; }
};
class DiffuseLight : public Material {                                                          // material.h:231-275
    RGB intrinsic_color;
    double intensity;
public:
    DiffuseLight(const RGB &c, double intensity_) : intrinsic_color{c}, intensity{intensity_} {}
    int kind() const override { return B200RT_MAT_LIGHT; }
    RGB colour() const override { return intrinsic_color; }
    double param() const override { return intensity; }
    RGB emit() const override { return intensity * intrinsic_color; }
    void print_to(std::ostream &os) const override {
        os << "DiffuseLight {color: " << intrinsic_color.as_string(", ", "()") << ", intensity: " << intensity << "} " << std::flush;
    }
};

// ===== base/hittable.h, shapes/*, base/scene.h ================================================
// base/hittable.h:20-71.  What a closest-hit query reports; the query itself runs on the GPU
// (BVH::hit_by below), the face orientation rule is the reference's.
struct hit_info {
    double hit_time;
    Point3D hit_point;
    Vec3D unit_surface_normal;
    bool hit_from_outside = false;
    const Material *material;
    hit_info(double hit_time_, const Point3D &hit_point_, const Vec3D &outward_unit_surface_normal, const Ray3D &ray,
             const std::shared_ptr<Material> &material_)
        : hit_time{hit_time_}, hit_point{hit_point_}, material{material_.get()} {
        hit_from_outside = !(dot(ray.dir, outward_unit_surface_normal) > 0);                    // hittable.h:56-70
        unit_surface_normal = hit_from_outside ? outward_unit_surface_normal : -outward_unit_surface_normal;
    }
};
inline std::ostream &operator<<(std::ostream &os, const hit_info &info) {                       // hittable.h:75-80
    os << "hit_info {\n\thit_time: " << info.hit_time << "\n\thit_point: " << info.hit_point << "\n\tsurface_normal: "
       << info.unit_surface_normal << "\n\thit_from_outside: " << info.hit_from_outside << "\n}\n";
    return os;
}

struct Hittable {
    // Compound objects return their parts; primitives return {} (hittable.h:112-117).
    virtual std::vector<std::shared_ptr<Hittable>> get_primitive_components() const { return {}; }
    // Extension used by the flattening step: the same canonical order as get_primitive_components(), as plain
    // pointers and without copying three million shared_ptrs.  Parts a compound creates on the fly are kept alive in `keep`.
    virtual void append_primitive_ptrs(std::vector<const Hittable *> &out, std::vector<std::shared_ptr<Hittable>> &keep) const {
        auto parts = get_primitive_components();
        if (parts.empty()) { out.push_back(this); return; }
        for (auto &p : parts) { keep.push_back(p); p->append_primitive_ptrs(out, keep); }
    }
    virtual void print_to(std::ostream &os) const = 0;
    virtual ~Hittable() = default;
};
inline std::ostream &operator<<(std::ostream &os, const Hittable &h) { h.print_to(os); return os; }

struct Sphere : public Hittable {                                                               // sphere.h:16-22,112
    Point3D center;
    double radius;
    std::shared_ptr<Material> material;
    Sphere(const Point3D &center_, double radius_, std::shared_ptr<Material> material_)
        : center{center_}, radius{radius_}, material{std::move(material_)} {}
    void print_to(std::ostream &os) const override {
        os << "Sphere {center: " << center << ", radius: " << radius << ", material: " << *material << "} " << std::flush;
    }
};

class Parallelogram : public Hittable {                                                         // parallelogram.h:14-48,269
    Point3D vertex;
    Vec3D side1, side2;
    std::shared_ptr<Material> material;
public:
    Parallelogram(const Point3D &vertex_, const Vec3D &side1_, const Vec3D &side2_, std::shared_ptr<Material> material_)
        : vertex{vertex_}, side1{side1_}, side2{side2_}, material{std::move(material_)} {}
    const Point3D &get_vertex() const { return vertex; }
    const Vec3D &get_side1() const { return side1; }
    const Vec3D &get_side2() const { return side2; }
    const std::shared_ptr<Material> &get_material() const { return material; }
    void print_to(std::ostream &os) const override {
        os << "Parallelogram {vertex: " << vertex << ", side 1 vector: " << side1 << ", side 2 vector: " << side2 << " } " << std::flush;
    }
};

class Scene : public Hittable {                                                                 // scene.h:12-125
    std::vector<std::shared_ptr<Hittable>> objects;
public:
    operator auto &() { return objects; }
    operator const auto &() const { return objects; }
    auto size() const { return objects.size(); }
    void clear() { objects.clear(); }
    auto &operator[](size_t i) { return objects[i]; }
    const auto &operator[](size_t i) const { return objects[i]; }
    auto begin() { return objects.begin(); }
    auto begin() const { return objects.cbegin(); }
    auto end() { return objects.end(); }
    auto end() const { return objects.cend(); }
    void add(std::shared_ptr<Hittable> object) { objects.push_back(std::move(object)); }
    void add(const Scene &scene) { for (const auto &o : scene) add(o); }
    // scene.h:85-105: compounds expanded in place, primitives kept, insertion order preserved.
    std::vector<std::shared_ptr<Hittable>> get_primitive_components() const override {
        std::vector<std::shared_ptr<Hittable>> ret;
        for (const auto &obj : objects) {
            if (auto parts = obj->get_primitive_components(); !parts.empty())
                ret.insert(ret.end(), std::make_move_iterator(parts.begin()), std::make_move_iterator(parts.end()));
            else
                ret.push_back(obj);
        }
        return ret;
    }
    void append_primitive_ptrs(std::vector<const Hittable *> &out, std::vector<std::shared_ptr<Hittable>> &keep) const override {
        for (const auto &obj : objects) obj->append_primitive_ptrs(out, keep);   // the objects live as long as the scene
    }
    void print_to(std::ostream &os) const override {
        os << "Scene with " << size() << " objects:\n";
        for (const auto &o : objects) { o->print_to(os); os << '\n'; }
        os << std::flush;
    }
    Scene() = default;
    Scene(std::span<const std::shared_ptr<Hittable>> objs) { for (const auto &o : objs) add(o); }
};

class Box : public Hittable {                                                                   // box.h:53-84
    Scene faces;
    std::shared_ptr<Material> material;
public:
    Box(const Point3D &vertex, const Point3D &opposite_vertex, std::shared_ptr<Material> material_) : material{std::move(material_)} {
        Point3D lo, hi;
        for (int i = 0; i < 3; ++i) { lo[i] = std::fmin(vertex[i], opposite_vertex[i]); hi[i] = std::fmax(vertex[i], opposite_vertex[i]); }
        const Vec3D sx{hi.x - lo.x, 0, 0}, sy{0, hi.y - lo.y, 0}, sz{0, 0, hi.z - lo.z};
        faces.add(std::make_shared<Parallelogram>(lo, sx, sy, material));
        faces.add(std::make_shared<Parallelogram>(lo, sx, sz, material));
        faces.add(std::make_shared<Parallelogram>(lo, sy, sz, material));
        faces.add(std::make_shared<Parallelogram>(hi, -sx, -sy, material));
        faces.add(std::make_shared<Parallelogram>(hi, -sx, -sz, material));
        faces.add(std::make_shared<Parallelogram>(hi, -sy, -sz, material));
    }
    std::vector<std::shared_ptr<Hittable>> get_primitive_components() const override { return faces.get_primitive_components(); }
    void append_primitive_ptrs(std::vector<const Hittable *> &out, std::vector<std::shared_ptr<Hittable>> &keep) const override {
        faces.append_primitive_ptrs(out, keep);
    }
    void print_to(std::ostream &os) const override { os << "Box {faces: " << faces << "} " << std::flush; }
};

// ===== util/image.h ===========================================================================
class Image {
    size_t w, h;
    std::vector<std::vector<RGB>> pixels;
    Image(size_t w_, size_t h_) : w{w_}, h{h_}, pixels(h_, std::vector<RGB>(w_, RGB::zero())) {}
    explicit Image(const std::vector<std::vector<RGB>> &rows) : w{rows.empty() ? 0 : rows[0].size()}, h{rows.size()}, pixels{rows} {}
    [[noreturn]] static void ppm_error(const std::string &file_name, const std::string &what) {
        std::cout << "Error: In Image::from_ppm_file(\"" << file_name << "\"), " << what << std::endl;
        std::exit(-1);
    }
public:
    auto width() const { return w; }
    auto height() const { return h; }
    auto &operator[](size_t row) { return pixels[row]; }
    const auto &operator[](size_t row) const { return pixels[row]; }
    double aspect_ratio() const { return static_cast<double>(w) / static_cast<double>(h); }
    static Image with_dimensions(size_t width, size_t height) { return Image(width, height); }
    // image.h:74-95: the missing dimension is round()ed from the aspect ratio, never below 1
    static Image with_width_and_aspect_ratio(size_t width, double aspect_ratio) {
        return Image(width, std::max(size_t{1}, static_cast<size_t>(std::round(static_cast<double>(width) / aspect_ratio))));
    }
    static Image with_height_and_aspect_ratio(size_t height, double aspect_ratio) {
        return Image(std::max(size_t{1}, static_cast<size_t>(std::round(static_cast<double>(height) * aspect_ratio))), height);
    }
    static Image from_data(const std::vector<std::vector<RGB>> &img) { return Image(img); }
    // image.h:57-66: a white one-pixel frame
    Image &outline_border() {
        if (w == 0 || h == 0) return *this;
        for (auto &row : pixels) row.front() = row.back() = RGB::from_mag(1);
        for (size_t c = 0; c < w; ++c) pixels.front()[c] = pixels.back()[c] = RGB::from_mag(1);
        return *this;
    }
    // image.h:100-164: ASCII P3 only; channel values are divided by the file's own maximum.
    static Image from_ppm_file(const std::string &file_name) {
        std::ifstream fin(file_name);
        if (!fin.is_open()) {
            std::cout << "Error: In Image::from_ppm_file(), could not find/open the file \"" << file_name << "\"" << std::endl;
            std::exit(-1);
        }
        std::string magic;
        std::getline(fin, magic);
        if (magic != "P3") ppm_error(file_name, "first line of file was not \"P3\", but instead was " + magic);
        size_t width = 0, height = 0;
        int max_magnitude = 0;
        if (!(fin >> width >> height)) ppm_error(file_name, "could not parse image width and height (two integers) on second line");
        if (!(fin >> max_magnitude)) ppm_error(file_name, "could not parse RGB max magnitude (one integer) after the image width and height");
        Image img(width, height);
        for (size_t i = 0; i < width * height; ++i) {
            int r, g, b;
            if (!(fin >> r >> g >> b)) ppm_error(file_name, "failed to parse color #" + std::to_string(i + 1) + " (three integers (r, g, b))");
            if (r < 0 || g < 0 || b < 0)
                ppm_error(file_name, "found negative RGB channel value; color #" + std::to_string(i + 1) + " was (" + std::to_string(r) +
                                         ", " + std::to_string(g) + ", " + std::to_string(b) + ")");
            img.pixels[i / width][i % width] = RGB::from_rgb(r, g, b, max_magnitude);
        }
        return img;
    }
    // image.h:38-56: ASCII P3, one "r g b" line per pixel through RGB::as_string() defaults.
    // The integers come from the tone-map kernel (b200rt_tonemap), formatting stays on the host.
    void send_as_ppm(const std::string &destination) const {
        std::ofstream fout(destination);
        if (!fout.is_open()) {
            std::cout << "Error: In Image::print_as_ppm(), could not open the file \"" << destination << "\"" << std::endl;
            std::exit(-1);
        }
        std::vector<float> hdr(w * h * 3);
        for (size_t r = 0; r < h; ++r)
            for (size_t c = 0; c < w; ++c) {
                hdr[(r * w + c) * 3 + 0] = (float)pixels[r][c].r;
                hdr[(r * w + c) * 3 + 1] = (float)pixels[r][c].g;
                hdr[(r * w + c) * 3 + 2] = (float)pixels[r][c].b;
            }
        std::vector<int32_t> ldr(w * h * 3);
        if (b200rt_tonemap(hdr.data(), (int64_t)(w * h), ldr.data(), 0) != B200RT_OK) {
            std::cout << "Error: In Image::send_as_ppm(), tone mapping failed: " << b200rt_last_error() << std::endl;
            std::exit(-1);
        }
        fout << "P3\n" << w << " " << h << "\n255\n";
        for (size_t i = 0; i < w * h; ++i) fout << ldr[3 * i] << ' ' << ldr[3 * i + 1] << ' ' << ldr[3 * i + 2] << '\n';
        std::cout << "Image successfully saved to \"" << destination << "\"" << std::endl;
    }
};

// image.h:168-262: a P3 writer that takes the pixels one at a time (top to bottom, left to right) and keeps
// none of them -- the sink for progressive / tiled output.  Each pixel goes through RGB::as_string().
class ImagePPMStream {
    std::string file;
    std::ofstream fout;
    size_t w, h, written = 0;
    ImagePPMStream(const std::string &file_, size_t w_, size_t h_) : file{file_}, fout{file_}, w{w_}, h{h_} {
        fout << "P3\n" << w << " " << h << "\n255\n";
    }
public:
    size_t width() const { return w; }
    size_t height() const { return h; }
    size_t size() const { return w * h; }
    double aspect_ratio() const { return static_cast<double>(w) / static_cast<double>(h); }
    // Redirect to another file and start the image over there (a partly written first file is reported).
    // The reference calls open() on the still-open stream (image.h:195), which only sets failbit and
    // silently drops every later pixel; this does what its comment describes: close, reopen, new header.
    void set_file(const std::string &file_name) {
        fout.close();
        fout.clear();
        fout.open(file_name);
        if (!fout.is_open()) {
            std::cout << "Error: In ImagePPMStream::set_file(), could not open the file \"" << file_name << "\"" << std::endl;
            std::exit(-1);
        }
        if (written > 0)
            std::cout << "Warning: In ImagePPMStream::set_file(\"" << file_name << "\"), original file \"" << file
                      << "\" is left incomplete; " << written << " out of " << size() << " pixels printed" << std::endl;
        file = file_name;
        written = 0;
        fout << "P3\n" << w << " " << h << "\n255\n";
    }
    void add(const RGB &rgb) {
        if (written == size()) {
            std::cout << "Error: Called ImagePPMStream::add() " << size() + 1 << " times for image of size " << size() << std::endl;
            std::exit(-1);
        }
        fout << rgb.as_string() << '\n';
        ++written;
    }
    static ImagePPMStream with_dimensions(size_t width, size_t height, const std::string &file_name) {
        return ImagePPMStream(file_name, width, height);
    }
    static ImagePPMStream with_width_and_aspect_ratio(size_t width, double aspect_ratio, const std::string &file_name) {
        return with_dimensions(width, std::max(size_t{1}, static_cast<size_t>(std::round(static_cast<double>(width) / aspect_ratio))), file_name);
    }
    static ImagePPMStream with_height_and_aspect_ratio(size_t height, double aspect_ratio, const std::string &file_name) {
        return with_dimensions(std::max(size_t{1}, static_cast<size_t>(std::round(static_cast<double>(height) * aspect_ratio))), height, file_name);
    }
    ~ImagePPMStream() {
        if (written == size()) std::cout << "Image successfully saved to \"" << file << "\"" << std::endl;
        else
            std::cout << "Warning: ImagePPMStream to \"" << file << "\" incomplete; " << written << " out of (" << w << " * " << h
                      << ") = " << size() << " RGB strings printed at time of destruction" << std::endl;
    }
};

// ===== scene flattening (the host half of the drop-in boundary) ==============================
namespace b200rt_host {

// Plain uninitialised storage for the flat arrays: a std::vector would zero 100+ MB on one thread (and take the page
// faults there) before the parallel fill overwrites every byte.
template <typename T>
class FlatArray {
    T *p = nullptr;
    size_t n = 0;
public:
    FlatArray() = default;
    FlatArray(const FlatArray &) = delete;
    FlatArray &operator=(const FlatArray &) = delete;
    FlatArray(FlatArray &&o) noexcept : p{o.p}, n{o.n} { o.p = nullptr; o.n = 0; }
    FlatArray &operator=(FlatArray &&o) noexcept { if (this != &o) { std::free(p); p = o.p; n = o.n; o.p = nullptr; o.n = 0; } return *this; }
    ~FlatArray() { std::free(p); }
    void resize_uninitialised(size_t count) {
        std::free(p);
        p = count ? static_cast<T *>(std::malloc(count * sizeof(T))) : nullptr;
        n = p ? count : 0;
        if (count && !p) { std::cout << "Error: out of memory while flattening the scene" << std::endl; std::exit(-1); }
    }
    size_t size() const { return n; }
    bool empty() const { return n == 0; }
    T *data() { return p; }
    const T *data() const { return p; }
    T &operator[](size_t i) { return p[i]; }
    const T &operator[](size_t i) const { return p[i]; }
    const T *begin() const { return p; }
    const T *end() const { return p + n; }
};

struct FlatScene {
    FlatArray<B200rtMaterial> materials;
    FlatArray<B200rtSphere> spheres;
    FlatArray<B200rtQuad> quads;
    B200rtSceneDesc desc() const {
        return B200rtSceneDesc{materials.size(), spheres.size(), quads.size(), materials.data(), spheres.data(), quads.data()};
    }
};

// Runs body(chunk, lo, hi) over [0, n) in `chunks` contiguous pieces on that many threads (inline when one).
template <typename F>
inline void for_chunks(size_t n, unsigned chunks, F body) {
    if (chunks <= 1) { body(0u, (size_t)0, n); return; }
    std::vector<std::thread> th;
    for (unsigned c = 0; c < chunks; ++c) th.emplace_back([=, &body] { body(c, n * c / chunks, n * (c + 1) / chunks); });
    for (auto &t : th) t.join();
}

// Canonical primitive order = get_primitive_components() order (scene.h:85-105); materials are shared by pointer, as
// the reference's shared_ptr<Material> members are, and numbered in order of first appearance.
//   The reference's big scenes hold 2-3 million primitives, each a heap object with its OWN material: walking that
// pointer graph is latency bound (about 2 s single-threaded with a hash map for the materials -- five times the 8-GPU
// render of the same scene).  So the walk runs on all host threads, in chunks of top-level objects: pass 1 expands and
// classifies a chunk and counts; a short serial step turns the counts into offsets and numbers the materials that
// somebody else also holds (a material with use_count() == 1 never enters the hash map); pass 2 fills the flat arrays,
// first-touching their pages in parallel.  The result is byte for byte what a serial walk produces
// (tests/test_host_api_cpu.py compares all ten scenes with dumps of the reference-built objects).
inline bool flatten(const Scene &world, FlatScene &out, std::string &err) {
    out = FlatScene{};
    const std::vector<std::shared_ptr<Hittable>> &objects = world;
    const size_t n_obj = objects.size();
    unsigned T = n_obj < (1u << 15) ? 1u : std::min(32u, std::max(1u, std::thread::hardware_concurrency()));
    if (const char *e = std::getenv("B200RT_FLATTEN_THREADS")) T = (unsigned)std::max(1, std::min(64, std::atoi(e)));
    // What pass 1 leaves per chunk: the chunk's flat records in order (material and primitive indices still to be
    // filled in), one tag per primitive, and the materials somebody else also holds (to be numbered globally).
    enum : uint8_t { kQuad = 1, kShared = 2, kFirst = 4 };
    struct Chunk {
        std::vector<B200rtSphere> sph;
        std::vector<B200rtQuad> quads;
        std::vector<B200rtMaterial> mats;                    // materials only this primitive holds, in order
        std::vector<uint8_t> tag;                            // per primitive
        std::vector<const Material *> shared;                // per primitive with kShared, in order
        std::vector<uint32_t> shared_u;                      // ... and how many unshared materials preceded it in the chunk
        std::vector<std::shared_ptr<Hittable>> keep;
        bool bad = false;
    };
    std::vector<Chunk> chunks(T);
    const bool trace = std::getenv("B200RT_TRACE") != nullptr;
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t0 = trace ? now() : 0;
    auto material_record = [](const Material *m) {
        B200rtMaterial fm{};
        fm.kind = (uint32_t)m->kind();
        const RGB col = m->colour();
        fm.rgb[0] = col.r; fm.rgb[1] = col.g; fm.rgb[2] = col.b;
        fm.param = m->param();
        return fm;
    };
    // pass 1: expand compounds, classify, read every object ONCE
    for_chunks(n_obj, T, [&](unsigned c, size_t lo, size_t hi) {
        Chunk &ch = chunks[c];
        std::vector<const Hittable *> prims;
        prims.reserve(hi - lo);
        for (size_t o = lo; o < hi; ++o) objects[o]->append_primitive_ptrs(prims, ch.keep);
        ch.tag.resize(prims.size());
        ch.mats.reserve(prims.size());
        for (size_t k = 0; k < prims.size(); ++k) {
            const Hittable *h = prims[k];
            const std::type_info &ti = typeid(*h);               // exact-type fast path; subclasses go through dynamic_cast
            const Sphere *s = ti == typeid(Sphere) ? static_cast<const Sphere *>(h) : nullptr;
            const Parallelogram *q = (!s && ti == typeid(Parallelogram)) ? static_cast<const Parallelogram *>(h) : nullptr;
            if (!s && !q) { s = dynamic_cast<const Sphere *>(h); if (!s) q = dynamic_cast<const Parallelogram *>(h); }
            const std::shared_ptr<Material> *mp;
            uint8_t tag = 0;
            if (s) {
                B200rtSphere f{};
                f.c[0] = s->center.x; f.c[1] = s->center.y; f.c[2] = s->center.z; f.r = s->radius;
                ch.sph.push_back(f);
                mp = &s->material;
            } else if (q) {
                B200rtQuad f{};
                const Point3D &v = q->get_vertex(); const Vec3D &a = q->get_side1(), &b = q->get_side2();
                f.v[0] = v.x; f.v[1] = v.y; f.v[2] = v.z;
                f.s1[0] = a.x; f.s1[1] = a.y; f.s1[2] = a.z;
                f.s2[0] = b.x; f.s2[1] = b.y; f.s2[2] = b.z;
                ch.quads.push_back(f);
                mp = &q->get_material();
                tag = kQuad;
            } else { ch.bad = true; return; }
            if (mp->use_count() == 1) ch.mats.push_back(material_record(mp->get()));
            else { tag |= kShared; ch.shared.push_back(mp->get()); ch.shared_u.push_back((uint32_t)ch.mats.size()); }
            ch.tag[k] = tag;
        }
    });
    for (const Chunk &ch : chunks)
        if (ch.bad) { err = "unsupported Hittable subclass (the device path knows Sphere, Parallelogram, Box and Scene)"; return false; }
    const double t1 = trace ? now() : 0;
    // serial step: offsets, and the first appearances of the shared materials in canonical order
    std::vector<size_t> prim_base(T + 1, 0), sph_base(T + 1, 0), quad_base(T + 1, 0), uniq_base(T + 1, 0), first_base(T + 1, 0);
    for (unsigned c = 0; c < T; ++c) {
        prim_base[c + 1] = prim_base[c] + chunks[c].tag.size();
        sph_base[c + 1] = sph_base[c] + chunks[c].sph.size();
        quad_base[c + 1] = quad_base[c] + chunks[c].quads.size();
        uniq_base[c + 1] = uniq_base[c] + chunks[c].mats.size();
    }
    if (prim_base[T] > 0x7FFFFFFFull) { err = "too many primitives"; return false; }
    std::unordered_map<const Material *, uint32_t> shared_id;
    std::vector<std::vector<uint8_t>> is_first(T);           // per chunk, per shared entry
    {
        size_t firsts = 0;
        for (unsigned c = 0; c < T; ++c) {
            first_base[c] = firsts;
            is_first[c].assign(chunks[c].shared.size(), 0);
            for (size_t j = 0; j < chunks[c].shared.size(); ++j) {
                const Material *m = chunks[c].shared[j];
                if (shared_id.count(m)) continue;
                is_first[c][j] = 1;
                // id = materials that appeared before this primitive: the unshared ones + the shared ones first seen before it
                shared_id[m] = (uint32_t)(uniq_base[c] + chunks[c].shared_u[j] + firsts);
                ++firsts;
            }
        }
        first_base[T] = firsts;
    }
    out.spheres.resize_uninitialised(sph_base[T]);
    out.quads.resize_uninitialised(quad_base[T]);
    out.materials.resize_uninitialised(uniq_base[T] + first_base[T]);
    const double t2 = trace ? now() : 0;
    // pass 2: stream the chunk records into the flat arrays with their final indices (every element written exactly once)
    for_chunks(T, T, [&](unsigned, size_t c_lo, size_t c_hi) {
      for (size_t c = c_lo; c < c_hi; ++c) {
        const Chunk &ch = chunks[c];
        size_t si = 0, qi = 0, ui = 0, shj = 0, firsts = first_base[c];
        for (size_t k = 0; k < ch.tag.size(); ++k) {
            const uint8_t tag = ch.tag[k];
            uint32_t mat;
            if (!(tag & kShared)) {
                mat = (uint32_t)(uniq_base[c] + ui + firsts);
                out.materials[mat] = ch.mats[ui++];
            } else {
                const Material *m = ch.shared[shj];
                mat = shared_id.find(m)->second;
                if (is_first[c][shj]) { out.materials[mat] = material_record(m); ++firsts; }
                ++shj;
            }
            const uint32_t prim = (uint32_t)(prim_base[c] + k);
            if (tag & kQuad) { B200rtQuad f = ch.quads[qi]; f.mat = mat; f.prim = prim; out.quads[quad_base[c] + qi++] = f; }
            else { B200rtSphere f = ch.sph[si]; f.mat = mat; f.prim = prim; out.spheres[sph_base[c] + si++] = f; }
        }
      }
    });
    if (trace) {
        const double t3 = now();
        chunks.clear();
        std::fprintf(stderr, "flatten: %u threads, pass 1 %.1f ms, offsets %.1f ms, pass 2 %.1f ms, release %.1f ms\n", T, t1 - t0, t2 - t1, t3 - t2, now() - t3);
    }
    return true;
}

}  // namespace b200rt_host

namespace b200rt_host {
// The GPUs a render uses when the program does not say (Camera::set_devices / the BVH constructor): the environment
// variable B200RT_DEVICES -- "all", a count ("8" = devices 0..7) or a comma-separated list of CUDA ordinals ("0,2,3");
// unset or unparsable = device 0.  This is how an UNMODIFIED reference program reaches config 5's sample split across
// 8 x B200: B200RT_DEVICES=all ./raytracer.
inline std::vector<int32_t> default_devices() {
    std::vector<int32_t> out;
    const char *env = std::getenv("B200RT_DEVICES");
    if (env && *env) {
        const std::string v = env;
        const int have = b200rt_device_count();
        if (v == "all") {
            for (int d = 0; d < have; ++d) out.push_back(d);
        } else if (v.find(',') == std::string::npos) {
            const int n = std::atoi(v.c_str());
            for (int d = 0; d < n; ++d) out.push_back(d);
        } else {
            size_t pos = 0;
            while (pos <= v.size()) {
                const size_t comma = std::min(v.find(',', pos), v.size());
                if (comma > pos) out.push_back(std::atoi(v.substr(pos, comma - pos).c_str()));
                pos = comma + 1;
            }
        }
    }
    if (out.empty()) out.push_back(0);
    return out;
}
}  // namespace b200rt_host

// ===== acceleration/bvh.h =====================================================================
// BVH(world) (bvh.h:754-776) = the scene made resident on the GPU: primitives flattened, the wide BVH built
// (host SAH or device LBVH by size) and uploaded, ONCE; every Camera::render(bvh) / hit_by afterwards reuses
// it.  Copies share the device scene (the reference's BVH is a value type over shared primitives).
class BVH : public Hittable {
    struct Resident {
        void *handle = nullptr;
        B200rtSceneInfo info{};
        ~Resident() { if (handle) b200rt_scene_destroy(handle); }
    };
    std::shared_ptr<Resident> dev;
    std::vector<std::shared_ptr<Hittable>> primitives;                                          // canonical order

public:
    // num_buckets / max_primitives_in_node keep their reference meaning (SAH bins per axis, leaf capacity;
    // the device leaf format holds at most 8) and their reference defaults select the library's own.
    template <typename T>
        requires std::is_base_of_v<Hittable, T>
    BVH(const T &world, size_t num_buckets = 32, size_t max_primitives_in_node = 12, std::vector<int32_t> devices = {})
        : primitives{world.get_primitive_components()} {
        if (devices.empty()) devices = b200rt_host::default_devices();
        b200rt_host::FlatScene flat;
        std::string err;
        bool ok;
        if constexpr (std::is_same_v<T, Scene>) {
            ok = b200rt_host::flatten(world, flat, err);        // same canonical order, without a second copy of every shared_ptr
        } else {
            Scene flat_world;
            if (primitives.empty()) primitives.push_back(std::shared_ptr<Hittable>(std::shared_ptr<Hittable>{}, const_cast<T *>(&world)));
            for (const auto &p : primitives) flat_world.add(p);
            ok = b200rt_host::flatten(flat_world, flat, err);
        }
        if (!ok) {
            std::cout << "Error: In BVH::BVH(), " << err << std::endl;
            std::exit(-1);
        }
        std::cout << "Building BVH over " << primitives.size() << " primitives..." << std::endl;
        B200rtBuildOpts opts{};
        opts.device = devices[0];
        if (num_buckets != 32) opts.sah_bins = (int32_t)num_buckets;
        if (max_primitives_in_node != 12) opts.max_leaf_prims = (int32_t)max_primitives_in_node;
        const B200rtSceneDesc desc = flat.desc();
        dev = std::make_shared<Resident>();
        // one device: a plain resident scene; several: built once on devices[0] and copied to the others, and every
        // Camera::render(bvh) splits the samples of each pixel across them inside the library
        if (b200rt_scene_create_multi(&desc, &opts, devices.data(), (int32_t)devices.size(), &dev->handle) != B200RT_OK ||
            b200rt_scene_info(dev->handle, &dev->info) != B200RT_OK) {
            std::cout << "Error: In BVH::BVH(), " << b200rt_last_error() << std::endl;
            std::exit(-1);
        }
        std::cout << "Constructed BVH in " << dev->info.build_ms << "ms (created " << dev->info.n_nodes << " BVHNodes total)\n" << std::endl;
    }

    void *handle() const { return dev->handle; }
    const B200rtSceneInfo &info() const { return dev->info; }
    auto size() const { return primitives.size(); }

    // bvh.h:585-715 for a batch of rays in one launch (b200rt_raycast): closest hit with
    // ray_times.min < t < ray_times.max per ray, exact ties to the lowest primitive index.
    std::vector<std::optional<hit_info>> hit_by(std::span<const Ray3D> rays, const Interval &ray_times) const {
        std::vector<double> packed(rays.size() * 6);
        for (size_t i = 0; i < rays.size(); ++i) {
            const Ray3D &r = rays[i];
            double *q = &packed[i * 6];
            q[0] = r.origin.x; q[1] = r.origin.y; q[2] = r.origin.z; q[3] = r.dir.x; q[4] = r.dir.y; q[5] = r.dir.z;
        }
        std::vector<int32_t> prim(rays.size());
        std::vector<double> t(rays.size());
        if (b200rt_raycast(dev->handle, packed.data(), (int64_t)rays.size(), ray_times.min, ray_times.max, prim.data(), t.data()) != B200RT_OK) {
            std::cout << "Error: In BVH::hit_by(), " << b200rt_last_error() << std::endl;
            std::exit(-1);
        }
        std::vector<std::optional<hit_info>> out(rays.size());
        for (size_t i = 0; i < rays.size(); ++i) {
            if (prim[i] < 0) continue;
            const Hittable *h = primitives[(size_t)prim[i]].get();
            const Point3D hit_point = rays[i](t[i]);
            if (auto s = dynamic_cast<const Sphere *>(h))
                out[i].emplace(t[i], hit_point, (hit_point - s->center) / s->radius, rays[i], s->material);          // sphere.h:94
            else if (auto q = dynamic_cast<const Parallelogram *>(h))
                out[i].emplace(t[i], hit_point, cross(q->get_side1(), q->get_side2()).unit_vector(), rays[i], q->get_material());  // parallelogram.h:225,273
        }
        return out;
    }
    std::optional<hit_info> hit_by(const Ray3D &ray, const Interval &ray_times) const {
        return hit_by(std::span<const Ray3D>(&ray, 1), ray_times)[0];
    }
    std::vector<std::shared_ptr<Hittable>> get_primitive_components() const override { return primitives; }
    void print_to(std::ostream &os) const override {
        os << "BVH {" << dev->info.n_nodes << " 4-wide nodes, depth " << dev->info.tree_depth << ", " << primitives.size()
           << " primitives, " << dev->info.device_bytes << " bytes on the device} " << std::flush;
    }
};

// ===== base/camera.h ==========================================================================
class Camera {
    size_t image_w = 1280, image_h = 720;                                                       // camera.h:16
    Ray3D camera{.origin = Point3D{0, 0, 0}, .dir = Vec3D{0, 0, -1}};                           // camera.h:29
    std::optional<Point3D> camera_lookat;
    Vec3D view_up_dir{0, 1, 0};
    std::optional<double> focus_dist;
    double defocus_angle = 0;
    size_t samples_per_pixel = 1, max_depth = 10;                                               // camera.h:67-69
    std::optional<double> vertical_fov{90}, horizontal_fov;                                     // camera.h:78 (sic: 90 radians)
    RGB background{RGB::from_mag(0.5)};
    uint64_t rng_seed = 0xB200;
    std::vector<int32_t> devices;                                                               // empty: B200RT_DEVICES, else device 0
    B200rtStats last_stats{};
    B200rtSceneInfo last_info{};

public:
    // Setter-level state -> the C ABI camera; Camera::init()'s derivation happens in b200rt_camera_init.
    B200rtCamera to_abi() const {
        B200rtCamera c{};
        c.image_w = image_w; c.image_h = image_h; c.spp = samples_per_pixel; c.max_depth = max_depth;
        const Vec3D dir = camera_lookat ? (*camera_lookat - camera.origin) : camera.dir;        // camera.h:95-97
        c.center[0] = camera.origin.x; c.center[1] = camera.origin.y; c.center[2] = camera.origin.z;
        c.dir[0] = dir.x; c.dir[1] = dir.y; c.dir[2] = dir.z;
        c.up[0] = view_up_dir.x; c.up[1] = view_up_dir.y; c.up[2] = view_up_dir.z;
        c.focus_dist = focus_dist.value_or(-1);
        c.defocus_angle = defocus_angle;
        c.vfov = vertical_fov.value_or(-1); c.hfov = horizontal_fov.value_or(-1);
        c.background[0] = background.r; c.background[1] = background.g; c.background[2] = background.b;
        if (b200rt_camera_init(&c) != B200RT_OK) {
            std::cout << "Error: In Camera::init(), " << b200rt_last_error() << std::endl;
            std::exit(-1);
        }
        return c;
    }

    template <typename V>
    static Image to_image(const std::vector<V> &hdr, size_t w, size_t h, double scale = 1.0) {
        Image img = Image::with_dimensions(w, h);
        const unsigned T = w * h < (1u << 20) ? 1u : std::min(16u, std::max(1u, std::thread::hardware_concurrency()));
        b200rt_host::for_chunks(h, T, [&](unsigned, size_t lo, size_t hi) {          // rows are independent
            for (size_t r = lo; r < hi; ++r)
                for (size_t c = 0; c < w; ++c) {
                    const V *p = &hdr[(r * w + c) * 3];
                    img[r][c] = RGB::from_mag(p[0] * scale, p[1] * scale, p[2] * scale);
                }
        });
        return img;
    }

    // camera.h:264-297 with T = BVH: renders from the scene already resident on the GPU (no build, no
    // upload) -- the call to use for several frames / cameras over one world.
    Image render(const BVH &bvh) {
        const B200rtCamera cam = to_abi();
        B200rtRenderOpts opts{};
        opts.seed = rng_seed;
        std::vector<float> hdr(image_w * image_h * 3);
        if (b200rt_render(bvh.handle(), &cam, &opts, hdr.data(), &last_stats) != B200RT_OK) {
            std::cout << "Error: In Camera::render(), " << b200rt_last_error() << std::endl;
            std::exit(-1);
        }
        last_info = bvh.info();
        return to_image(hdr, image_w, image_h);
    }

    // camera.h:264-297 for any other Hittable (a single Sphere, a Box, ...): its primitive components are
    // rendered exactly as a Scene holding it would be.
    template <typename T>
        requires(std::is_base_of_v<Hittable, T> && !std::is_same_v<T, Scene> && !std::is_same_v<T, BVH>)
    Image render(const T &world) {
        return render(BVH(world));
    }

    // Progressive output (extension; SURVEY 8(f)-4): the frame in passes of `samples_per_pass` samples over
    // the resident scene; after each pass `on_pass(image so far, samples done)` sees the running mean.  Pass k
    // renders samples [k*spp_pass, ...) of the same per-sample streams, so the final image is the one
    // render(bvh) returns up to FP32 summation order.
    template <typename F>
    Image render_progressive(const BVH &bvh, size_t samples_per_pass, F &&on_pass) {
        const B200rtCamera cam = to_abi();
        std::vector<float> sum(image_w * image_h * 3, 0.0f), pass(image_w * image_h * 3);
        B200rtStats total{};
        size_t done = 0;
        samples_per_pass = std::max<size_t>(1, samples_per_pass);
        while (done < samples_per_pixel) {
            B200rtRenderOpts opts{};
            opts.seed = rng_seed;
            opts.sample_offset = done;
            opts.sample_count = std::min(samples_per_pass, samples_per_pixel - done);
            opts.flags = B200RT_FLAG_SUM;
            B200rtStats st{};
            if (b200rt_render(bvh.handle(), &cam, &opts, pass.data(), &st) != B200RT_OK) {
                std::cout << "Error: In Camera::render_progressive(), " << b200rt_last_error() << std::endl;
                std::exit(-1);
            }
            for (size_t i = 0; i < sum.size(); ++i) sum[i] += pass[i];
            done += opts.sample_count;
            total.kernel_ms += st.kernel_ms; total.total_ms += st.total_ms; total.paths += st.paths; total.rays += st.rays;
            total.kernel_launches += st.kernel_launches; total.d2h_bytes += st.d2h_bytes;
            on_pass(to_image(sum, image_w, image_h, 1.0 / (double)done), done);
        }
        last_stats = total;
        last_info = bvh.info();
        return to_image(sum, image_w, image_h, 1.0 / (double)std::max<size_t>(1, done));
    }

    // Sample variance of one pixel channel from the mean of x and the mean of x^2 over n samples: n/(n-1) (m2 - mean^2),
    // in double; +inf when n < 2.  Both planes come from FP32 frames (and x^2 is summed in 2^-24 units), so a difference
    // within their resolution -- 2^-20 of m2, plus 2^-24 -- is no evidence of noise and counts as 0: a pixel whose
    // samples are all equal (one that sees only the background) reports exactly 0.
    static double sample_variance(double mean, double m2, size_t n) {
        if (n < 2) return std::numeric_limits<double>::infinity();
        const double d = m2 - mean * mean;
        if (d <= std::ldexp(m2, -20) + std::ldexp(1.0, -24)) return 0.0;
        return (double)n / (double)(n - 1) * d;
    }

    // Extension: render(bvh) and, per pixel and channel, the standard error of that mean, sqrt(s^2 / n) with s^2 the
    // sample variance of the pixel's n = samples_per_pixel samples (b200rt_render_moments).  The first image is the one
    // render(bvh) returns, bit for bit, up to 2^16 samples per pixel.
    std::pair<Image, Image> render_with_noise(const BVH &bvh) {
        const B200rtCamera cam = to_abi();
        B200rtRenderOpts opts{};
        opts.seed = rng_seed;
        std::vector<float> hdr(image_w * image_h * 3), m2(image_w * image_h * 3);
        if (b200rt_render_moments(bvh.handle(), &cam, &opts, hdr.data(), m2.data(), &last_stats) != B200RT_OK) {
            std::cout << "Error: In Camera::render_with_noise(), " << b200rt_last_error() << std::endl;
            std::exit(-1);
        }
        last_info = bvh.info();
        std::vector<double> se(hdr.size());
        for (size_t i = 0; i < hdr.size(); ++i) se[i] = std::sqrt(sample_variance(hdr[i], m2[i], samples_per_pixel) / (double)samples_per_pixel);
        return {to_image(hdr, image_w, image_h), to_image(se, image_w, image_h)};
    }

    // Extension: renders until the frame is as clean as asked.  Passes of `samples_per_pass` samples over the resident
    // scene, as render_progressive, each through b200rt_render_moments as SUM planes that are added on the host in
    // double; stops after the first pass whose frame relative noise is <= rel_noise, or when samples_per_pixel samples
    // are done.  Returns the mean image; stats().paths / (width * height) is the number of samples it used.
    //   Frame relative noise = sqrt(mean over all pixels and channels of se^2) / (mean over all pixels and channels of
    // the image), where se^2 = s^2 / n is the squared standard error of a pixel channel's mean (s^2: sample_variance).
    // Channels, not luminance, because the moments are per channel.  +inf while fewer than 2 samples are done; 0 for a
    // black, noise-free frame.
    Image render_to_noise(const BVH &bvh, double rel_noise, size_t samples_per_pass) {
        const B200rtCamera cam = to_abi();
        const size_t n_fl = image_w * image_h * 3;
        std::vector<double> sum(n_fl, 0.0), sum2(n_fl, 0.0);
        std::vector<float> pass(n_fl), pass2(n_fl);
        B200rtStats total{};
        size_t done = 0;
        samples_per_pass = std::max<size_t>(1, samples_per_pass);
        while (done < samples_per_pixel) {
            B200rtRenderOpts opts{};
            opts.seed = rng_seed;
            opts.sample_offset = done;
            opts.sample_count = std::min(samples_per_pass, samples_per_pixel - done);
            opts.flags = B200RT_FLAG_SUM;
            B200rtStats st{};
            if (b200rt_render_moments(bvh.handle(), &cam, &opts, pass.data(), pass2.data(), &st) != B200RT_OK) {
                std::cout << "Error: In Camera::render_to_noise(), " << b200rt_last_error() << std::endl;
                std::exit(-1);
            }
            for (size_t i = 0; i < n_fl; ++i) { sum[i] += pass[i]; sum2[i] += pass2[i]; }
            done += opts.sample_count;
            total.kernel_ms += st.kernel_ms; total.total_ms += st.total_ms; total.paths += st.paths; total.rays += st.rays;
            total.kernel_launches += st.kernel_launches; total.d2h_bytes += st.d2h_bytes;
            if (frame_relative_noise(sum, sum2, done) <= rel_noise) break;
        }
        last_stats = total;
        last_info = bvh.info();
        return to_image(sum, image_w, image_h, 1.0 / (double)std::max<size_t>(1, done));
    }

    // Extension: adaptive sampling.  Each pixel gets samples until ITS noise reaches the target (b200rt_render_adaptive):
    // min_spp in the first pass, then samples_per_pass per pass while the pixel or a neighbour is still noisy, up to
    // samples_per_pixel.  A pixel is converged when the standard error of its mean, sqrt(mean of the channel variances /
    // n), is <= rel_noise x its mean radiance.  Returns the mean image and each pixel's sample count (row-major); every
    // pixel is the one render(bvh) gives at that pixel's count.  stats().paths is the sum of the counts.
    std::pair<Image, std::vector<uint32_t>> render_adaptive(const BVH &bvh, double rel_noise, size_t min_spp, size_t samples_per_pass) {
        const B200rtCamera cam = to_abi();
        B200rtRenderOpts opts{};
        opts.seed = rng_seed;
        B200rtAdaptiveOpts aopts{};
        aopts.min_spp = (uint32_t)std::min<size_t>(min_spp, 0xFFFFFFFFu);
        aopts.step_spp = (uint32_t)std::min<size_t>(samples_per_pass, 0xFFFFFFFFu);
        aopts.rel_noise = rel_noise;
        std::vector<float> hdr(image_w * image_h * 3);
        std::vector<uint32_t> spp(image_w * image_h);
        if (b200rt_render_adaptive(bvh.handle(), &cam, &opts, &aopts, hdr.data(), nullptr, spp.data(), &last_stats) != B200RT_OK) {
            std::cout << "Error: In Camera::render_adaptive(), " << b200rt_last_error() << std::endl;
            std::exit(-1);
        }
        last_info = bvh.info();
        return {to_image(hdr, image_w, image_h), std::move(spp)};
    }

    // The frame relative noise (see render_to_noise) of SUM planes over n samples.
    static double frame_relative_noise(const std::vector<double> &sum, const std::vector<double> &sum2, size_t n) {
        if (n < 2 || sum.empty()) return std::numeric_limits<double>::infinity();
        double se2 = 0, img = 0;
        for (size_t i = 0; i < sum.size(); ++i) {
            const double mean = sum[i] / (double)n;
            se2 += sample_variance(mean, sum2[i] / (double)n, n) / (double)n;
            img += mean;
        }
        se2 /= (double)sum.size();
        img /= (double)sum.size();
        if (!(img > 0)) return se2 > 0 ? std::numeric_limits<double>::infinity() : 0.0;
        return std::sqrt(se2) / img;
    }

    // camera.h:301-303.  Builds the acceleration structure, uploads, renders on the GPU and
    // returns the linear HDR image, all inside this call.
    Image render(const Scene &world) {
        const auto t_flat = std::chrono::steady_clock::now();
        b200rt_host::FlatScene flat;
        std::string err;
        if (!b200rt_host::flatten(world, flat, err)) {
            std::cout << "Error: In Camera::render(), " << err << std::endl;
            std::exit(-1);
        }
        const B200rtCamera cam = to_abi();
        const B200rtSceneDesc desc = flat.desc();
        B200rtRenderOpts opts{};
        opts.seed = rng_seed;
        std::vector<float> hdr(image_w * image_h * 3);
        std::cout << "Rendering " << image_w << " x " << image_h << " image (" << flat.spheres.size() + flat.quads.size()
                  << " primitives, " << samples_per_pixel << " spp) on the GPU..." << std::endl;
        const std::vector<int32_t> devs = devices.empty() ? b200rt_host::default_devices() : devices;
        const auto t_call = std::chrono::steady_clock::now();
        if (b200rt_render_scene_multi(&desc, &cam, &opts, nullptr, devs.data(), (int32_t)devs.size(), hdr.data(), &last_stats, &last_info) != B200RT_OK) {
            std::cout << "Error: In Camera::render(), " << b200rt_last_error() << std::endl;
            std::exit(-1);
        }
        if (std::getenv("B200RT_TRACE"))
            std::fprintf(stderr, "Camera::render: flatten %.1f ms, b200rt_render_scene_multi %.1f ms\n",
                         std::chrono::duration<double, std::milli>(t_call - t_flat).count(),
                         std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_call).count());
        std::cout << "Constructed BVH in " << last_info.build_ms << "ms (created " << last_info.n_nodes << " BVHNodes total); rendered in "
                  << last_stats.kernel_ms << "ms (" << (double)last_stats.paths / last_stats.kernel_ms / 1e3 << " Mpaths/s)\n" << std::endl;
        return to_image(hdr, image_w, image_h);
    }
    const B200rtStats &stats() const { return last_stats; }
    const B200rtSceneInfo &scene_info() const { return last_info; }
    Camera &set_rng_seed(uint64_t s) { rng_seed = s; return *this; }   // extension: the GPU RNG key
    // extension: the GPUs render(const Scene&) splits the samples of every pixel across (CUDA ordinals; the
    // acceleration structure is built once on the first and copied to the others).  Not called: B200RT_DEVICES.
    Camera &set_devices(std::vector<int32_t> d) { devices = std::move(d); return *this; }
    Camera &set_device_count(int n) { devices.clear(); for (int d = 0; d < n; ++d) devices.push_back(d); return *this; }

    // camera.h:308-406
    Camera &set_camera_center(const Point3D &p) { camera.origin = p; return *this; }
    Camera &set_camera_direction(const Vec3D &dir) { camera.dir = dir; return *this; }
    Camera &set_camera_direction_towards(const Point3D &p) { camera.dir = p - camera.origin; camera_lookat.reset(); return *this; }
    Camera &set_camera_lookat(const Point3D &p) { camera_lookat = p; return *this; }
    Camera &set_focus_distance(double d) { focus_dist = d; return *this; }
    Camera &set_defocus_angle(double degrees) { defocus_angle = degrees * std::numbers::pi / 180; return *this; }
    Camera &turn_blur_off() { defocus_angle = 0; return *this; }
    Camera &set_camera_up_direction(const Vec3D &dir) { view_up_dir = dir; return *this; }
    Camera &set_image_width(size_t w) { image_w = w; return *this; }
    Camera &set_image_height(size_t h) { image_h = h; return *this; }
    Camera &set_image_dimensions(size_t w, size_t h) { image_w = w; image_h = h; return *this; }
    Camera &set_image_by_width_and_aspect_ratio(size_t width, double aspect_ratio) {
        auto height = static_cast<size_t>(std::round(static_cast<double>(width) / aspect_ratio));
        return set_image_dimensions(width, std::max(size_t{1}, height));
    }
    Camera &set_image_by_height_and_aspect_ratio(size_t height, double aspect_ratio) {
        auto width = static_cast<size_t>(std::round(static_cast<double>(height) * aspect_ratio));
        return set_image_dimensions(std::max(size_t{1}, width), height);
    }
    Camera &set_samples_per_pixel(size_t s) { samples_per_pixel = s; return *this; }
    Camera &set_max_depth(size_t d) { max_depth = d; return *this; }
    Camera &set_vertical_fov(double degrees) { vertical_fov = degrees * std::numbers::pi / 180; horizontal_fov.reset(); return *this; }
    Camera &set_horizontal_fov(double degrees) { horizontal_fov = degrees * std::numbers::pi / 180; vertical_fov.reset(); return *this; }
    Camera &set_background(const RGB &c) { background = c; return *this; }
};
