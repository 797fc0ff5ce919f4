"""The API-compatible C++ host layer (cpp_raytracer_b200/host): programs written against the
reference's Scene / Sphere / Parallelogram / Box / material / Camera API compile against it, and
the scene functions restated with it (host/scenes.hpp) produce, after flattening to the C ABI
structs, EXACTLY the bytes a dump of the reference-built scene holds (tests/golden/*.scene.gz were
dumped from the reference's own objects).  That pins: the bit-exact LCG (rand_util.h:85-117),
SeedSeqGenerator, rand_int, RGB::random's draw order, Box -> 6 faces in constructor order,
material sharing by pointer, canonical primitive order, and Camera::init through
b200rt_camera_init."""
import gzip
import hashlib
import json
import os
import subprocess

import pytest

from conftest import GOLDEN, ROOT, SMALL_SCENES


@pytest.fixture(scope="module")
def scenes_bin():
    from cpp_raytracer_b200 import build
    build.build()
    return build.build_host()


@pytest.mark.parametrize("name", SMALL_SCENES)
def test_host_scene_builders_match_reference_dumps(scenes_bin, name, tmp_path):
    out = str(tmp_path / f"{name}.scene")
    subprocess.run([scenes_bin, name, "dump", out], check=True, capture_output=True)
    want = gzip.open(os.path.join(GOLDEN, f"{name}.scene.gz"), "rb").read()
    got = open(out, "rb").read()
    assert got == want, f"{name}: host-built scene differs from the reference-built scene"


@pytest.mark.parametrize("threads", ["1", "3", "16"])
def test_parallel_flatten_is_byte_identical_whatever_the_chunking(scenes_bin, threads, tmp_path):
    """Flattening walks the object graph on several host threads in chunks of top-level objects (two passes with
    prefix sums; materials held by one primitive only never enter the hash map).  Primitive order, material numbering
    by first appearance -- shared materials included (Boxes: six faces one material; the Cornell walls) -- must not depend
    on how the objects fall into chunks: forced to 1, 3 and 16 threads, all seven fixture scenes give the reference's bytes."""
    for name in SMALL_SCENES:
        out = str(tmp_path / f"{name}.scene")
        subprocess.run([scenes_bin, name, "dump", out], check=True, capture_output=True,
                       env=dict(os.environ, B200RT_FLATTEN_THREADS=threads))
        want = gzip.open(os.path.join(GOLDEN, f"{name}.scene.gz"), "rb").read()
        assert open(out, "rb").read() == want, (name, threads)


@pytest.mark.parametrize("name", ["raining", "millions_lights"])
def test_host_big_scene_builders_match_reference_live(scenes_bin, ref_bridge, name, tmp_path):
    """2.2 M quads / 3.1 M spheres: too big to commit, so compare against the reference binary
    live (oracle/_ref travels with the repo)."""
    if ref_bridge is None:
        pytest.skip("oracle/_ref/ref_bridge not built")
    mine, ref = str(tmp_path / "mine.scene"), str(tmp_path / "ref.scene")
    subprocess.run([scenes_bin, name, "dump", mine], check=True, capture_output=True)
    subprocess.run([ref_bridge, name, "dump", ref], check=True, capture_output=True)
    assert subprocess.run(["cmp", "-s", mine, ref]).returncode == 0


@pytest.mark.parametrize("name", ["raining", "millions_lights"])
def test_host_big_scene_builders_match_recorded_digest(scenes_bin, name, tmp_path):
    """The same two scenes against the byte length and SHA-256 of their dumps recorded in
    tests/golden/big_scenes.json (tests/golden/make_big_golden.py), so a change to the scene code or
    the flattening shows up without the reference binary."""
    want = json.load(open(os.path.join(GOLDEN, "big_scenes.json")))[name]
    out = str(tmp_path / f"{name}.scene")
    subprocess.run([scenes_bin, name, "dump", out], check=True, capture_output=True)
    data = open(out, "rb").read()
    assert len(data) == want["bytes"] and hashlib.sha256(data).hexdigest() == want["sha256"], name


def test_reference_style_program_compiles_unchanged(tmp_path):
    """A src/main.cpp-style translation unit (same includes, same fluent calls) builds against
    host/include and libb200rt.so without modification."""
    src = tmp_path / "prog.cpp"
    src.write_text('''
#include "util/rand_util.h"
#include "base/scene.h"
#include "base/material.h"
#include "base/camera.h"
#include "shapes/shapes.h"
int main() {
    SeedSeqGenerator::get_instance().set_seed(42);
    Scene world;
    auto ground = std::make_shared<Lambertian>(RGB::from_mag(0.5, 0.5, 0.5));
    world.add(std::make_shared<Sphere>(Point3D(0, -1000, 0), 1000, ground));
    world.add(std::make_shared<Sphere>(Point3D(0, 1, 0), 1.0, std::make_shared<Dielectric>(1.5)));
    world.add(std::make_shared<Parallelogram>(Point3D(-2, 0, -2), Vec3D(4, 0, 0), Vec3D(0, 4, 0),
                                              std::make_shared<Metal>(RGB::random(0.5, 1), rand_double(0, 0.5))));
    world.add(std::make_shared<Box>(Point3D(2, 0, 2), Point3D(3, 1, 3), std::make_shared<DiffuseLight>(RGB::from_mag(1), 4)));
    if (world.size() != 4 || world.get_primitive_components().size() != 9) return 3;
    // Scene container API (scene.h:19-56): add(const Scene&) copies the objects in, not the scene
    Scene outer;
    outer.add(world);
    outer.add(std::make_shared<Sphere>(Point3D{9, 9, 9}, 0.5, ground));
    if (outer.size() != 5 || outer[4] == nullptr || outer.begin() == outer.end()) return 5;
    size_t spheres = 0;
    for (const auto &obj : outer) if (std::dynamic_pointer_cast<Sphere>(obj)) ++spheres;
    if (spheres != 3) return 6;
    outer.clear();
    if (outer.size() != 0) return 7;
    // value-level helpers the scene functions rely on
    if (RGB::from_rgb(255, 0, 51).r != 1.0 || RGB::from_mag(0.5).g != 0.5 || RGB::zero().b != 0.0) return 8;
    if ((Vec3D{1, 2, 3} - Vec3D{1, 2, 3}).mag() != 0.0 || dot(Vec3D{1, 0, 0}, cross(Vec3D{0, 1, 0}, Vec3D{0, 0, 1})) != 1.0) return 9;
    if (RGB::from_mag(10, 0.2, 0.01).as_string() != "447 63 14") return 10;          // rgb.h:90-113, the reference's own answer (kat.json)
    if (Metal(RGB::from_mag(1), 7.0).param() != 1.0) return 11;                     // fuzz clamped to 1 (material.h:150-151)
    Camera cam;
    cam.set_image_by_width_and_aspect_ratio(64, 16. / 9.).set_vertical_fov(20).set_camera_center(Point3D{13, 2, 3})
       .set_camera_lookat(Point3D{0, 0, 0}).set_camera_up_direction(Vec3D{0, 1, 0}).set_defocus_angle(0.6)
       .set_focus_distance(10).set_samples_per_pixel(4).set_max_depth(5).set_background(RGB::from_mag(0.7, 0.8, 1));
    if (cam.to_abi().image_h != 36) return 4;            // round(64 / (16/9)) = 36 (camera.h:366-370)
    if (std::getenv("RUN_RENDER")) cam.render(world).send_as_ppm(std::getenv("RUN_RENDER"));
    return 0;
}
''')
    exe = str(tmp_path / "prog")
    env = dict(os.environ)
    env.pop("CXX", None); env.pop("CC", None)
    inc = os.path.join(ROOT, "cpp_raytracer_b200", "host", "include")
    lib = os.path.join(ROOT, "cpp_raytracer_b200")
    subprocess.run(["g++", "-std=c++20", "-O1", f"-I{inc}", "-o", exe, str(src), f"-L{lib}", "-lb200rt", f"-Wl,-rpath,{lib}"],
                   check=True, env=env)
    assert subprocess.run([exe], capture_output=True).returncode == 0


def test_host_rand_double_matches_reference_stream(golden, tmp_path):
    """rand_double / SeedSeqGenerator of the host layer vs the reference's own stream
    (tests/golden/kat.json: set_seed(12345), then the first 16 draws of the main thread)."""
    kat = golden.kat()
    src = tmp_path / "lcg.cpp"
    src.write_text('''
#include <cstdio>
#include "util/rand_util.h"
int main() {
    SeedSeqGenerator::get_instance().set_seed(%d);
    for (int i = 0; i < 16; ++i) std::printf("%%.17g\\n", rand_double());
    return 0;
}
''' % kat["rand_double_seed"])
    exe = str(tmp_path / "lcg")
    env = dict(os.environ)
    env.pop("CXX", None); env.pop("CC", None)
    inc = os.path.join(ROOT, "cpp_raytracer_b200", "host", "include")
    lib = os.path.join(ROOT, "cpp_raytracer_b200")
    subprocess.run(["g++", "-std=c++20", "-O1", f"-I{inc}", "-o", exe, str(src), f"-L{lib}", "-lb200rt", f"-Wl,-rpath,{lib}"],
                   check=True, env=env)
    out = subprocess.run([exe], capture_output=True, text=True, check=True).stdout
    got = [float(x) for x in out.splitlines() if x and x[0].isdigit()]
    assert got == kat["rand_double_next16"]


def _compile(tmp_path, name, text):
    src = tmp_path / f"{name}.cpp"
    src.write_text(text)
    exe = str(tmp_path / name)
    env = dict(os.environ)
    env.pop("CXX", None); env.pop("CC", None)
    inc = os.path.join(ROOT, "cpp_raytracer_b200", "host", "include")
    lib = os.path.join(ROOT, "cpp_raytracer_b200")
    subprocess.run(["g++", "-std=c++20", "-O1", f"-I{inc}", "-o", exe, str(src), f"-L{lib}", "-lb200rt", f"-Wl,-rpath,{lib}"],
                   check=True, env=env)
    return exe


def test_image_io_surface(tmp_path):
    """image.h: named constructors, outline_border, the streaming P3 writer (ImagePPMStream) and the P3
    reader (Image::from_ppm_file).  Host-only I/O: no device involved."""
    out1, out2, inp = tmp_path / "a.ppm", tmp_path / "b.ppm", tmp_path / "in.ppm"
    inp.write_text("P3\n2 2\n100\n50 0 100\n0 25 0\n1 2 3\n100 100 100\n")
    exe = _compile(tmp_path, "imgio", r'''
#include <cstdio>
#include "util/image.h"
int main(int argc, char **argv) {
    if (Image::with_width_and_aspect_ratio(64, 16. / 9.).height() != 36) return 1;
    if (Image::with_height_and_aspect_ratio(36, 16. / 9.).width() != 64) return 2;
    if (Image::with_width_and_aspect_ratio(1, 100.).height() != 1) return 3;
    auto img = Image::with_dimensions(4, 3);
    img.outline_border();
    if (img[0][2].r != 1 || img[1][0].g != 1 || img[1][3].b != 1 || img[2][1].r != 1 || img[1][1].r != 0 || img[1][2].r != 0) return 4;
    auto data = Image::from_data({{RGB::from_mag(1), RGB::from_mag(0.25)}});
    if (data.width() != 2 || data.height() != 1 || data[0][1].g != 0.25) return 5;
    {
        auto s = ImagePPMStream::with_dimensions(3, 2, argv[1]);
        if (s.size() != 6 || s.aspect_ratio() != 1.5) return 6;
        s.add(RGB::from_mag(10, 0.2, 0.01));                 // "447 63 14": the reference's own answer (kat.json)
        s.add(RGB::zero());
        s.set_file(argv[2]);                                 // restart in a second file
        for (int i = 0; i < 6; ++i) s.add(RGB::from_mag(i == 5 ? 10 : 0, i == 5 ? 0.2 : 0, i == 5 ? 0.01 : 0));
    }
    auto in = Image::from_ppm_file(argv[3]);
    if (in.width() != 2 || in.height() != 2) return 7;
    if (in[0][0].r != 0.5 || in[0][0].g != 0 || in[0][0].b != 1 || in[0][1].g != 0.25 || in[1][0].b != 0.03 || in[1][1].r != 1) return 8;
    return 0;
}
''')
    r = subprocess.run([exe, str(out1), str(out2), str(inp)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout
    assert out1.read_text() == "P3\n3 2\n255\n447 63 14\n0 0 0\n"
    assert out2.read_text() == "P3\n3 2\n255\n" + "0 0 0\n" * 5 + "447 63 14\n"      # set_file starts the image over
    assert "left incomplete; 2 out of 6" in r.stdout and "Image successfully saved" in r.stdout
    bad = tmp_path / "bad.ppm"
    bad.write_text("P6\n1 1\n255\n")
    exe2 = _compile(tmp_path, "imgbad", '#include "util/image.h"\nint main(int, char **argv) { Image::from_ppm_file(argv[1]); return 0; }\n')
    r = subprocess.run([exe2, str(bad)], capture_output=True, text=True)
    assert r.returncode != 0 and 'was not "P3"' in r.stdout


def test_bvh_reuse_program_compiles(tmp_path):
    """The program of tests/test_gpu_host_api.py (BVH reuse, hit_by, progressive render, render<T>) builds
    here without a GPU; it runs in the -m gpu suite."""
    from test_gpu_host_api import PROGRAM
    assert os.path.exists(_compile(tmp_path, "bvhprog", PROGRAM))
