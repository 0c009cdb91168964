// render_test.cpp -- headless C++ mirror of the reference driver RenderTest/Sample/RayTracing4.fs
// (DoRayTrace4: InitSceneState -> new Scene -> Window.Run calling Scene.Render every frame), with
// the Silk.NET/ImGui window (EngineCore/Core/Film.fs:38-92) replaced by PFM + PPM files.  It is the
// host side a maintainer would write in F# (INTEGRATION.md) expressed in the toolchain this image
// has; it talks to the GPU only through the C ABI of include/mafrix_cuda.h.
//
//   render_test [--obj file.obj] [--frames N] [--spp S] [--size WxH] [--depth D] [--exact] [--gpus N] [--out prefix]
//
// --gpus N: the same single-threaded loop over mfx_multi_* -- the library replicates the scene on N devices and
// every device keeps the Film (Film.fs:13-34) of its own stripes (mfx_multi_film_*); only the last frame's texture and
// the screen cross PCIe.
//
// Without --obj it renders the reference's default scene: the Cornell box of Scene.xml
// (RayTracing4.fs:9-72: camera (0,1,3) looking -z, fov 120, 300x300, three Lambert materials,
// area light 10,10,10, maxDepth 3 as hard-coded at Scene/Scene.fs:304, 1 spp per frame, :332).
#include "../include/mafrix_cuda.h"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

static void die(const char *what)
{
    fprintf(stderr, "render_test: %s: %s\n", what, mfx_last_error());
    exit(1);
}
#define CHECK(call) do { if ((call) != MFX_OK) die(#call); } while (0)

struct P3 { double x, y, z; };
static P3 sub(P3 a, P3 b) { return { a.x - b.x, a.y - b.y, a.z - b.z }; }
static P3 cross(P3 a, P3 b) { return { a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x }; }
static double dot(P3 a, P3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }

static MfxPrim make_rect(P3 p0, P3 p1, P3 p2, P3 p3, P3 facing, int material)
{
    // the reference never flips normals towards the ray (quirk Q4): orient (v1-v0)x(v2-v0) along `facing`
    if (dot(cross(sub(p1, p0), sub(p2, p0)), facing) < 0) std::swap(p1, p3);
    MfxPrim r; memset(&r, 0, sizeof(r));
    r.kind = MFX_RECT; r.material = material;
    const P3 v[4] = { p0, p1, p2, p3 };
    for (int i = 0; i < 4; i++) { r.v[3 * i] = v[i].x; r.v[3 * i + 1] = v[i].y; r.v[3 * i + 2] = v[i].z; }
    return r;
}

static void add_box(std::vector<MfxPrim> &out, const P3 top[4], int material)
{
    P3 c = { 0, 0, 0 };
    for (int i = 0; i < 4; i++) { c.x += top[i].x / 4; c.y += top[i].y / 4; c.z += top[i].z / 4; }
    out.push_back(make_rect(top[0], top[1], top[2], top[3], { 0, 1, 0 }, material));
    for (int k = 0; k < 4; k++) {
        P3 a = top[k], b = top[(k + 1) % 4], a0 = a, b0 = b;
        a0.y = 0; b0.y = 0;
        P3 outw = { (a.x + b.x) / 2 - c.x, 0, (a.z + b.z) / 2 - c.z };
        out.push_back(make_rect(a0, a, b, b0, outw, material));
    }
}

// Scene.xml re-authored (CornellBox-Original.obj is absent from the reference repo, Scene.xml:10)
static std::vector<MfxPrim> cornell_box()
{
    std::vector<MfxPrim> p;
    p.push_back(make_rect({ -1.01, 0, 0.99 }, { 1, 0, 0.99 }, { 1, 0, -1.04 }, { -0.99, 0, -1.04 }, { 0, 1, 0 }, 0));          // floor
    p.push_back(make_rect({ -1.02, 1.99, 0.99 }, { -1.02, 1.99, -1.04 }, { 1, 1.99, -1.04 }, { 1, 1.99, 0.99 }, { 0, -1, 0 }, 0)); // ceiling
    p.push_back(make_rect({ -0.99, 0, -1.04 }, { 1, 0, -1.04 }, { 1, 1.99, -1.04 }, { -1.02, 1.99, -1.04 }, { 0, 0, 1 }, 0));     // backWall
    p.push_back(make_rect({ 1, 0, -1.04 }, { 1, 0, 0.99 }, { 1, 1.99, 0.99 }, { 1, 1.99, -1.04 }, { -1, 0, 0 }, 1));              // rightWall
    p.push_back(make_rect({ -1.01, 0, 0.99 }, { -0.99, 0, -1.04 }, { -1.02, 1.99, -1.04 }, { -1.02, 1.99, 0.99 }, { 1, 0, 0 }, 2)); // leftWall
    const P3 shortTop[4] = { { 0.53, 0.6, 0.75 }, { 0.70, 0.6, 0.17 }, { 0.13, 0.6, 0.0 }, { -0.05, 0.6, 0.57 } };
    const P3 tallTop[4] = { { -0.53, 1.2, 0.09 }, { 0.04, 1.2, -0.09 }, { -0.14, 1.2, -0.67 }, { -0.71, 1.2, -0.49 } };
    add_box(p, shortTop, 0);
    add_box(p, tallTop, 0);
    return p;
}

// OBJ faces the way ObjModelLoader.Face.ToHitable reads them (Models/ObjModelLoader.fs:63-92):
// 3 vertices -> Triangle, 4 -> Rect, only the geometric index of a/b/c, negative indices from the end.
static std::vector<MfxPrim> load_obj(const std::string &path, int material)
{
    std::ifstream in(path);
    if (!in) { fprintf(stderr, "render_test: cannot open %s\n", path.c_str()); exit(1); }
    std::vector<P3> v;
    std::vector<MfxPrim> out;
    std::string line;
    while (std::getline(in, line)) {
        std::istringstream ls(line);
        std::string tag;
        ls >> tag;
        if (tag == "v") { P3 p; ls >> p.x >> p.y >> p.z; v.push_back(p); }
        else if (tag == "f") {
            std::vector<int> idx;
            std::string ref;
            while (ls >> ref) {
                int i = atoi(ref.substr(0, ref.find('/')).c_str());
                idx.push_back(i > 0 ? i - 1 : (int)v.size() + i);
            }
            if (idx.size() != 3 && idx.size() != 4) { fprintf(stderr, "render_test: face with %zu vertices\n", idx.size()); exit(1); }
            MfxPrim p; memset(&p, 0, sizeof(p));
            p.kind = idx.size() == 4 ? MFX_RECT : MFX_TRIANGLE; p.material = material;
            for (size_t k = 0; k < idx.size(); k++) { p.v[3 * k] = v[idx[k]].x; p.v[3 * k + 1] = v[idx[k]].y; p.v[3 * k + 2] = v[idx[k]].z; }
            out.push_back(p);
        }
    }
    return out;
}

static void write_pfm(const std::string &path, const std::vector<double> &tex, int w, int h)
{
    FILE *f = fopen(path.c_str(), "wb");
    fprintf(f, "PF\n%d %d\n-1.0\n", w, h);
    for (int y = h - 1; y >= 0; y--)
        for (int x = 0; x < w; x++) {
            const double *c = &tex[((size_t)x * h + y) * 4];     // Color[w,h] is x-major
            float rgb[3] = { (float)c[0], (float)c[1], (float)c[2] };
            fwrite(rgb, 4, 3, f);
        }
    fclose(f);
}

static void write_ppm(const std::string &path, const std::vector<uint8_t> &rgba, int w, int h)
{
    FILE *f = fopen(path.c_str(), "wb");
    fprintf(f, "P6\n%d %d\n255\n", w, h);
    for (size_t p = 0; p < (size_t)w * h; p++) fwrite(&rgba[4 * p], 1, 3, f);
    fclose(f);
}

int main(int argc, char **argv)
{
    std::string obj, out = "render_test";
    int frames = 16, spp = 1, w = 300, h = 300, depth = 3, precision = MFX_FAST_F32, gpus = 0;
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i];
        if (a == "--obj" && i + 1 < argc) obj = argv[++i];
        else if (a == "--frames" && i + 1 < argc) frames = atoi(argv[++i]);
        else if (a == "--spp" && i + 1 < argc) spp = atoi(argv[++i]);
        else if (a == "--depth" && i + 1 < argc) depth = atoi(argv[++i]);
        else if (a == "--size" && i + 1 < argc) sscanf(argv[++i], "%dx%d", &w, &h);
        else if (a == "--out" && i + 1 < argc) out = argv[++i];
        else if (a == "--exact") precision = MFX_EXACT_F64;
        else if (a == "--gpus" && i + 1 < argc) gpus = atoi(argv[++i]);
        else { fprintf(stderr, "usage: render_test [--obj f.obj] [--frames N] [--spp S] [--size WxH] [--depth D] [--exact] [--gpus N] [--out prefix]\n"); return 2; }
    }
    CHECK(mfx_init(0));                                     // no GPU -> MFX_ERR_NO_DEVICE, no CPU fallback

    std::vector<MfxPrim> prims;
    MfxAreaLight light; memset(&light, 0, sizeof(light));
    double pos[3], dir[3];
    if (obj.empty()) {
        prims = cornell_box();
        const double lp[12] = { -0.24, 1.98, 0.16, -0.24, 1.98, -0.22, 0.23, 1.98, -0.22, 0.23, 1.98, 0.16 };   // Scene.fs:194
        memcpy(light.p, lp, sizeof(lp));
        pos[0] = 0; pos[1] = 1; pos[2] = 3; dir[0] = 0; dir[1] = 0; dir[2] = -1;                                // Scene.xml:3-4
    } else {
        prims = load_obj(obj, 0);
        double lo[3] = { 1e300, 1e300, 1e300 }, hi[3] = { -1e300, -1e300, -1e300 };
        for (const MfxPrim &p : prims)
            for (int k = 0; k < (p.kind == MFX_RECT ? 4 : 3); k++)
                for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], p.v[3 * k + a]); hi[a] = std::max(hi[a], p.v[3 * k + a]); }
        const double ext = std::max(hi[0] - lo[0], std::max(hi[1] - lo[1], hi[2] - lo[2]));
        const double cx = (lo[0] + hi[0]) / 2, cz = (lo[2] + hi[2]) / 2, top = hi[1] + ext;
        prims.push_back(make_rect({ cx - 4 * ext, lo[1], cz - 4 * ext }, { cx - 4 * ext, lo[1], cz + 4 * ext },
                                  { cx + 4 * ext, lo[1], cz + 4 * ext }, { cx + 4 * ext, lo[1], cz - 4 * ext }, { 0, 1, 0 }, 0));
        const double s = ext / 3;
        const double lp[12] = { cx - s, top, cz + s, cx - s, top, cz - s, cx + s, top, cz - s, cx + s, top, cz + s };
        memcpy(light.p, lp, sizeof(lp));
        pos[0] = cx; pos[1] = (lo[1] + hi[1]) / 2; pos[2] = lo[2] - 1.6 * ext; dir[0] = 0; dir[1] = 0; dir[2] = 1;
    }
    light.normal[1] = -1;
    light.color[0] = light.color[1] = light.color[2] = 10.0;                                                    // Scene.xml:55
    MfxMaterial mats[3]; memset(mats, 0, sizeof(mats));
    const double albedo[3][3] = { { 0.725, 0.71, 0.68 }, { 0.14, 0.45, 0.091 }, { 0.63, 0.065, 0.05 } };        // Scene.xml:15,18,21
    for (int m = 0; m < 3; m++) { mats[m].kind = MFX_LAMBERT; memcpy(mats[m].albedo, albedo[m], 24); }

    MfxSceneDesc desc; memset(&desc, 0, sizeof(desc));
    desc.prims = prims.data(); desc.n_prims = (int)prims.size();
    desc.materials = mats; desc.n_materials = 3;
    desc.nodes = nullptr; desc.indices = nullptr;                  // Bvh.Build reproduced on the host by the library
    desc.light = light;
    CHECK(mfx_camera_pinhole(pos, dir, 120.0, (double)w / h, &desc.camera));   // PinholeCamera(pos, dir, 120, aspect)
    desc.width = w; desc.height = h; desc.max_depth = depth; desc.integrator = MFX_PATH_INTEGRATOR;

    if (gpus > 0) {
        // N GPUs behind the same single-threaded host loop: the library shards, this thread sees IPixelIntegrator.Sample
        if (mfx_device_count() < gpus) { fprintf(stderr, "render_test: --gpus %d but %d device(s) visible\n", gpus, mfx_device_count()); return 1; }
        MfxMulti *multi = nullptr; MfxMultiFilm *film = nullptr;
        CHECK(mfx_multi_create(&desc, nullptr, gpus, &multi));
        CHECK(mfx_multi_film_create(multi, &film));                 // every device keeps the Film of its own stripes
        std::vector<double> target((size_t)w * h * 4);
        std::vector<uint8_t> screen((size_t)w * h * 4);
        double ms = 0; uint64_t rays = 0;
        for (int f = 0; f < frames; f++) {
            MfxSampleParams sp; memset(&sp, 0, sizeof(sp));
            sp.precision = precision; sp.spp = spp; sp.seed = 1; sp.first_sample = f * spp; sp.world = 1;
            CHECK(mfx_multi_film_get_frame(film, &sp, f + 1 == frames ? target.data() : nullptr));   // Film.GetFrame(integrator, spp)
            MfxStats st; CHECK(mfx_multi_get_stats(multi, &st, nullptr));
            ms += st.ms_total; rays += st.closest_rays + st.shadow_rays;
        }
        CHECK(mfx_multi_film_post_process(film, screen.data()));     // PostProcessAndToScreenBuffer
        write_pfm(out + ".pfm", target, w, h);
        write_ppm(out + ".ppm", screen, w, h);
        printf("%s: %zu primitives, %dx%d, %d frames x %d spp, depth %d, %s, %d GPUs: %.2f ms on the slowest device, %.1f Mrays/s -> %s.pfm / .ppm\n",
               obj.empty() ? "cornell" : obj.c_str(), prims.size(), w, h, frames, spp, depth,
               precision == MFX_FAST_F32 ? "f32" : "f64", gpus, ms, rays / (ms * 1e3), out.c_str());
        mfx_multi_film_destroy(film);
        mfx_multi_destroy(multi);
        return 0;
    }

    MfxScene *scene = nullptr; MfxFilm *film = nullptr;
    CHECK(mfx_scene_create(&desc, &scene));                       // new Scene(state)
    CHECK(mfx_film_create(scene, &film));
    std::vector<double> target((size_t)w * h * 4);
    std::vector<uint8_t> screen((size_t)w * h * 4);
    double ms = 0; uint64_t rays = 0;
    for (int f = 0; f < frames; f++) {                            // window.Run(): scene.Render per frame
        MfxSampleParams sp; memset(&sp, 0, sizeof(sp));
        sp.precision = precision; sp.spp = spp; sp.seed = 1; sp.first_sample = f * spp; sp.world = 1;
        CHECK(mfx_film_get_frame(film, &sp, f + 1 == frames ? target.data() : nullptr));   // Film.GetFrame(integrator, spp)
        MfxStats st; CHECK(mfx_get_stats(scene, &st));
        ms += st.ms_total; rays += st.closest_rays + st.shadow_rays;
    }
    CHECK(mfx_film_post_process(film, screen.data()));           // PostProcessAndToScreenBuffer
    write_pfm(out + ".pfm", target, w, h);
    write_ppm(out + ".ppm", screen, w, h);
    printf("%s: %zu primitives, %dx%d, %d frames x %d spp, depth %d, %s: %.2f ms on the device, %.1f Mrays/s -> %s.pfm / .ppm\n",
           obj.empty() ? "cornell" : obj.c_str(), prims.size(), w, h, frames, spp, depth,
           precision == MFX_FAST_F32 ? "f32" : "f64", ms, rays / (ms * 1e3), out.c_str());
    mfx_film_destroy(film);
    mfx_scene_destroy(scene);
    return 0;
}
