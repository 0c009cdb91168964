// CPU model of the shipped traversal (k_f_trace6, csrc/mfx_fast.cu) over the library's own tree (csrc/mfx_build.cpp):
// counts 128-byte records fetched and triangle tests per ray for a C2-like path population (primary rays, uniform
// hemisphere bounces to depth 5, one shadow ray per vertex towards the quad light), with the kernel's rules -- sorted
// 4-wide node step, nearest child first (shadow queries: farthest first), deferred hits culled by their entry distance
// at pop time, leaves of the chosen child tested at once, first hit ends a shadow ray, a ray never re-hits the triangle
// it starts on.  One thread, f32.
// It also reports the traversal stack's height per query kind: the peak, and how many rays push deeper than the
// entries the kernels keep in shared memory (MFX_STACK_SMEM, default 12) and so use the spill columns in global memory,
// against 3*depth, the bound those columns are sized for (csrc/mfx_host.cpp flatten_fast).
// The GPU's own counters (MFX_SAMPLE_COUNT_OWN_TREE, bench.py `own_tree`) are what validates this model: C2 measures
// 3.35 records + 2.07 triangle tests per closest-hit ray and, with shadow queries still nearest-first
// (SIM_ANY_NEAREST=1 here), 4.19 + 1.65 per shadow ray.
//
// build:  g++ -O2 -std=c++17 -pthread -I /usr/local/cuda/include -I mafrixraytracing_b200/csrc -o /tmp/own_tree_sim \
//             tools/own_tree_sim.cpp mafrixraytracing_b200/csrc/mfx_build.cpp
// usage:  own_tree_sim tris.bin n [width height [camera and light, see main]]      tris.bin = n x 9 doubles (tools/own_tree_sim.py)
// env:    MFX_COLLAPSE_DP / MFX_SAH_MAX_LEAF / MFX_SAH_TRAV_COST_PCT   the builder's knobs
//         SIM_ANY_NEAREST=1         shadow queries visit the nearest child first (the kernel up to the last GPU run of round 1)
//         MFX_STACK_SMEM=k          the stack entries kept in shared memory, for the count of rays above it (default 12)
//         SIM_SHADOW_FROM_LIGHT=1   trace every shadow ray from the light sample towards the surface point instead (same
//                                   segment, same answer); the run always prints both directions split by outcome
#include "mfx_build.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <vector>

int mfx_fail(int code, const char *fmt, ...) { va_list ap; va_start(ap, fmt); vfprintf(stderr, fmt, ap); va_end(ap); return code; }
long mfx_env_long(const char *name, long dflt) { const char *v = getenv(name); return (v && *v) ? atol(v) : dflt; }

struct V { float x, y, z; };
static inline V operator-(V a, V b) { return { a.x - b.x, a.y - b.y, a.z - b.z }; }
static inline V operator+(V a, V b) { return { a.x + b.x, a.y + b.y, a.z + b.z }; }
static inline V operator*(V a, float s) { return { a.x * s, a.y * s, a.z * s }; }
static inline float dot(V a, V b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static inline V cross(V a, V b) { return { a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x }; }
static inline V norm(V a) { const float l = std::sqrt(dot(a, a)); return a * (1.f / l); }
static int as_int(float f) { int i; memcpy(&i, &f, 4); return i; }
static unsigned as_uint(float f) { unsigned i; memcpy(&i, &f, 4); return i; }
static float as_float(unsigned u) { float f; memcpy(&f, &u, 4); return f; }

static bool g_any_nearest = false;
static int g_smem = 12;         // MFX_STACK_SMEM
static int g_quant = 0;          // SIM_QUANT: 1 = boxes replaced by their 8-bit grid planes (QuadC), 2 = plus the kernel's one-fma plane arithmetic
struct Tri { V v0, e1, e2, n; };
struct Counts { double rays = 0, records = 0, tris = 0, leaf_visits = 0, deep = 0; int peak = 0; };   // deep: rays whose stack rose above g_smem

struct Sim {
    const MfxOwnTree *t;
    const std::vector<QuadC> *cq = nullptr;
    std::vector<Tri> tri;        // leaf order
    bool test_leaf(int leaf, V o, V d, float tmin, int src, float &best, int &best_slot, Counts &c) const
    {
        c.leaf_visits++;
        const int first = leaf >> 3, cnt = leaf & 7;
        bool found = false;
        for (int k = 0; k < cnt; k++) {         // Moller-Trumbore with the acceptance rules of leaf_f3 (Trangle.fs:130-148)
            const Tri &T = tri[first + k];
            c.tris++;
            const V s1 = cross(d, T.e2);
            const float div = dot(s1, T.e1);
            const float inv = 1.f / div;
            const V dd = o - T.v0;
            const float b1 = dot(dd, s1) * inv;
            const V s2 = cross(dd, T.e1);
            const float b2 = dot(d, s2) * inv;
            const float tt = dot(T.e2, s2) * inv;
            if (std::fabs(div) >= 1e-6f && b1 >= 0.f && b1 <= 1.f && b2 >= 0.f && (b1 + b2) < 1.f && tt > tmin && tt < best && (first + k) != src) {
                best = tt; best_slot = first + k; found = true;
            }
        }
        return found;
    }
    // returns the slot hit (or -1); any = shadow query
    int trace(V o, V d, float tmin, float tmax, int src, bool any, float &t_out, Counts &c) const
    {
        const V id = { 1.f / d.x, 1.f / d.y, 1.f / d.z };
        const V ood = { o.x * id.x, o.y * id.y, o.z * id.z };
        float best = tmax; int best_slot = -1;
        struct E { unsigned key; int rec; };
        E stack[256]; int sp = 0, peak = 0;
        int node = 0, leaf = -1; bool need_pop = false;
        c.rays++;
        for (;;) {
            if (leaf < 0 && !need_pop) {                            // node step
                const QuadF &q = t->quads[node];
                c.records++;
                const float *lo[3] = { &q.lox.x, &q.loy.x, &q.loz.x }, *hi[3] = { &q.hix.x, &q.hiy.x, &q.hiz.x };
                unsigned key[4];
                for (int s = 0; s < 4; s++) {
                    float x0 = lo[0][s] * id.x - ood.x, x1 = hi[0][s] * id.x - ood.x;
                    float y0 = lo[1][s] * id.y - ood.y, y1 = hi[1][s] * id.y - ood.y;
                    float z0 = lo[2][s] * id.z - ood.z, z1 = hi[2][s] * id.z - ood.z;
                    if (g_quant == 2) {         // k_f_trace6<CMP>: t = (2^23 + q) * S + (C - 2^23 * S)
                        const QuadC &c = (*cq)[node];
                        const float S[3] = { c.sx * id.x, c.sy * id.y, c.sz * id.z };
                        const float Cc[3] = { std::fmaf(-8388608.f, S[0], std::fmaf(c.ox, id.x, -ood.x)), std::fmaf(-8388608.f, S[1], std::fmaf(c.oy, id.y, -ood.y)),
                                              std::fmaf(-8388608.f, S[2], std::fmaf(c.oz, id.z, -ood.z)) };
                        const unsigned wl[3] = { c.lox, c.loy, c.loz }, wh[3] = { c.hix, c.hiy, c.hiz };
                        float *out[3][2] = { { &x0, &x1 }, { &y0, &y1 }, { &z0, &z1 } };
                        for (int a = 0; a < 3; a++) {
                            *out[a][0] = std::fmaf(as_float(0x4B000000u | ((wl[a] >> (8 * s)) & 255u)), S[a], Cc[a]);
                            *out[a][1] = std::fmaf(as_float(0x4B000000u | ((wh[a] >> (8 * s)) & 255u)), S[a], Cc[a]);
                        }
                    }
                    const float tn = std::max(std::max(std::min(x0, x1), std::min(y0, y1)), std::max(std::min(z0, z1), tmin));
                    const float tf = std::min(std::min(std::max(x0, x1), std::max(y0, y1)), std::min(std::max(z0, z1), best));
                    const int mt = as_int((&q.meta.x)[s]);
                    // closest hit: nearest child first; shadow query: farthest first (as shipped; SIM_ANY_NEAREST=1: the old order)
                    const unsigned ord = (any && !g_any_nearest) ? (0x7f7ffff8u - (as_uint(tn) & ~7u)) : (as_uint(tn) & ~7u);
                    key[s] = (tn <= tf && mt != MFX_QUAD_EMPTY) ? (ord | (mt >= 0 ? 4u : 0u) | (unsigned)s) : 0x7f800000u;
                }
                std::sort(key, key + 4);
                for (int k = 3; k >= 1; k--) if (key[k] != 0x7f800000u) stack[sp++] = { key[k], node };      // nearest on top
                peak = std::max(peak, sp);
                need_pop = true;
                if (key[0] != 0x7f800000u) {
                    const int link = as_int((&q.meta.x)[key[0] & 3u]);
                    if (key[0] & 4u) leaf = link; else { node = ~link; need_pop = false; }
                }
            }
            if (leaf >= 0) {
                const bool found = test_leaf(leaf, o, d, tmin, src, best, best_slot, c);
                leaf = -1;
                if (any && found) break;
            }
            if (need_pop) {
                bool got = false;
                while (sp > 0) {
                    const E e = stack[--sp];
                    if (any || as_float(e.key & ~7u) <= best) {
                        const int link = as_int((&t->quads[e.rec].meta.x)[e.key & 3u]);
                        if (e.key & 4u) leaf = link; else { node = ~link; need_pop = false; }
                        got = true;
                        break;
                    }
                }
                if (!got) break;
            }
        }
        c.peak = std::max(c.peak, peak);
        if (peak > g_smem) c.deep++;
        t_out = best;
        return best_slot;
    }
};

static double g_st[2][2][2], g_cnt[2], g_mism;
int main(int argc, char **argv)
{
    if (argc < 3) { fprintf(stderr, "usage: own_tree_sim tris.bin n [width height]\n"); return 2; }
    const int n = atoi(argv[2]);
    g_any_nearest = getenv("SIM_ANY_NEAREST") != nullptr;
    g_smem = (int)std::max(1L, mfx_env_long("MFX_STACK_SMEM", 12));
    const int W = argc > 3 ? atoi(argv[3]) : 480, H = argc > 4 ? atoi(argv[4]) : 270;
    FILE *f = fopen(argv[1], "rb");
    if (!f) { fprintf(stderr, "cannot open %s\n", argv[1]); return 2; }
    std::vector<double> raw(9 * (size_t)n);
    if (fread(raw.data(), 72, n, f) != (size_t)n) { fprintf(stderr, "short read\n"); return 2; }
    fclose(f);
    std::vector<float> lo(3 * (size_t)n), hi(3 * (size_t)n);
    for (int i = 0; i < n; i++) for (int a = 0; a < 3; a++) {
        const double v0 = raw[9 * (size_t)i + a], v1 = raw[9 * (size_t)i + 3 + a], v2 = raw[9 * (size_t)i + 6 + a];
        lo[3 * (size_t)i + a] = std::nextafterf((float)std::min(v0, std::min(v1, v2)), -INFINITY);
        hi[3 * (size_t)i + a] = std::nextafterf((float)std::max(v0, std::max(v1, v2)), INFINITY);
    }
    MfxOwnTree tree;
    const auto tb0 = std::chrono::steady_clock::now();
    mfx_build_own_tree(lo.data(), hi.data(), n, (int)mfx_env_long("MFX_SAH_MAX_LEAF", 4), (float)mfx_env_long("MFX_SAH_TRAV_COST_PCT", 100) * 0.01f, 3, tree);
    g_quant = (int)mfx_env_long("SIM_QUANT", 0);
    std::vector<QuadC> cq;
    if (g_quant) {
        mfx_compress_quads(tree.quads, cq);
        double infl[2] = { 0, 0 }, cnt[2] = { 0, 0 };
        for (size_t i = 0; i < cq.size(); i++) {
            QuadF &q = tree.quads[i]; const QuadC &c = cq[i];
            float *lo[3] = { &q.lox.x, &q.loy.x, &q.loz.x }, *hi[3] = { &q.hix.x, &q.hiy.x, &q.hiz.x };
            const float org[3] = { c.ox, c.oy, c.oz }, st[3] = { c.sx, c.sy, c.sz };
            const unsigned wl[3] = { c.lox, c.loy, c.loz }, wh[3] = { c.hix, c.hiy, c.hiz };
            for (int s = 0; s < 4; s++) {
                const int m = as_int((&q.meta.x)[s]);
                if (m == MFX_QUAD_EMPTY) continue;
                double e0[3], e1[3];
                for (int a = 0; a < 3; a++) {
                    e0[a] = (double)hi[a][s] - lo[a][s];
                    const float nl = org[a] + (float)((wl[a] >> (8 * s)) & 255u) * st[a], nh = org[a] + (float)((wh[a] >> (8 * s)) & 255u) * st[a];
                    if (nl > lo[a][s] || nh < hi[a][s]) { fprintf(stderr, "record %zu child %d axis %d: grid planes inside the box\n", i, s, a); return 1; }
                    lo[a][s] = nl; hi[a][s] = nh;
                    e1[a] = (double)nh - nl;
                }
                const double a0 = e0[0] * e0[1] + e0[1] * e0[2] + e0[2] * e0[0], a1 = e1[0] * e1[1] + e1[1] * e1[2] + e1[2] * e1[0];
                if (a0 > 0.) { infl[m >= 0] += a1 / a0; cnt[m >= 0] += 1; }
            }
        }
        printf("8-bit grids: mean surface-area ratio of a child box, interior %.4f, leaf %.4f\n", infl[0] / cnt[0], infl[1] / cnt[1]);
    }
    printf("own tree built in %.2f ms\n", std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - tb0).count());
    Sim sim; sim.t = &tree; sim.cq = &cq; sim.tri.resize(n);
    for (int k = 0; k < n; k++) {
        const double *p = &raw[9 * (size_t)tree.order[k]];
        const V v0 = { (float)p[0], (float)p[1], (float)p[2] };
        const V e1 = { (float)(p[3] - p[0]), (float)(p[4] - p[1]), (float)(p[5] - p[2]) }, e2 = { (float)(p[6] - p[0]), (float)(p[7] - p[1]), (float)(p[8] - p[2]) };
        sim.tri[k] = { v0, e1, e2, norm(cross(e1, e2)) };
    }
    // record statistics
    long kids_hist[5] = { 0, 0, 0, 0, 0 }, leaf_hist[8] = { 0 };
    for (const QuadF &q : tree.quads) {
        int kids = 0;
        for (int s = 0; s < 4; s++) { const int m = as_int((&q.meta.x)[s]); if (m != MFX_QUAD_EMPTY) { kids++; if (m >= 0) leaf_hist[m & 7]++; } }
        kids_hist[kids]++;
    }
    printf("tree: %zu records, depth %d; children per record 1..4: %ld %ld %ld %ld; leaf sizes 1..4: %ld %ld %ld %ld\n", tree.quads.size(), tree.depth,
           kids_hist[1], kids_hist[2], kids_hist[3], kids_hist[4], leaf_hist[1], leaf_hist[2], leaf_hist[3], leaf_hist[4]);

    // camera and light: C2's by default -- PinholeCamera((0, 0.1, -2.6), (0, 0, 1), fov 120 -> effective 60 deg, aspect 16/9),
    // light quad 1x1 at y = 2.5 -- or 19 numbers after width/height: pos(3) dir(3) fov aspect, light p0(3) p1(3) p3(3), max_depth
    float cv[19] = { 0.f, 0.1f, -2.6f, 0.f, 0.f, 1.f, 120.f, 16.f / 9.f, -0.5f, 2.5f, 0.5f, -0.5f, 2.5f, -0.5f, 0.5f, 2.5f, 0.5f, 5.f, 0.f };
    for (int k = 0; k < 18 && 5 + k < argc; k++) cv[k] = (float)atof(argv[5 + k]);
    const int D = (int)cv[17];
    const V pos = { cv[0], cv[1], cv[2] };
    const float hs = std::tan(0.5f * cv[6] * 3.14159265f / 360.f), vs = hs / cv[7];
    const V fwd = norm(V{ cv[3], cv[4], cv[5] }), hori = cross(fwd, V{ 0, 1, 0 }), vert = cross(hori, fwd);
    const V right = hori * hs, up = vert * vs, down = up * -1.f;
    const V tl = pos + fwd * 0.5f - right * 0.5f + up * 0.5f;
    const V l0 = { cv[8], cv[9], cv[10] }, le1 = V{ cv[11], cv[12], cv[13] } - l0, le3 = V{ cv[14], cv[15], cv[16] } - l0;
    std::mt19937 rng(12345);
    std::uniform_real_distribution<float> U(0.f, 1.f);
    Counts cl[6], sh[6];
    for (int j = 0; j < H; j++) for (int i = 0; i < W; i++) {
        const float u = (i + U(rng)) / W, v = (j + U(rng)) / H;
        V o = pos, d = norm(tl + right * u + down * v - pos);
        int src = -1;
        for (int b = 0; b <= D && b <= 5; b++) {
            float t;
            const int slot = sim.trace(o, d, 1e-6f, 99999999.f, src, false, t, cl[b]);
            if (slot < 0) break;
            const V p = o + d * t, nm = sim.tri[slot].n;
            // light sample (uniform on the quad is close enough for a count), shadow ray unless the contribution is zero
            const V lp = l0 + le1 * U(rng) + le3 * U(rng);
            const V toL = lp - p;
            const float dist = std::sqrt(dot(toL, toL));
            if (dot(toL, V{ 0, -1, 0 }) < 0.f && dot(toL, nm) != 0.f) {
                float ts, t2;
                Counts a, r;
                const int hf = sim.trace(p, toL * (1.f / dist), 1e-6f, dist - 1e-6f, slot, true, ts, a);
                const int hr = sim.trace(lp, toL * (-1.f / dist), 1e-6f, dist - 1e-6f, slot, true, t2, r);
                const int occ = hf >= 0;
                g_cnt[occ]++; if ((hf >= 0) != (hr >= 0)) g_mism++;
                g_st[occ][0][0] += a.records; g_st[occ][0][1] += a.tris; g_st[occ][1][0] += r.records; g_st[occ][1][1] += r.tris;
                const Counts &use = getenv("SIM_SHADOW_FROM_LIGHT") ? r : a;
                sh[b].rays += 1; sh[b].records += use.records; sh[b].tris += use.tris;
                sh[b].deep += use.deep; sh[b].peak = std::max(sh[b].peak, use.peak);
            }
            // uniform hemisphere about the (unflipped) geometric normal
            const float z = 1.f - 2.f * U(rng), r = std::sqrt(std::max(0.f, 1.f - z * z)), ph = 6.2831853f * U(rng);
            V w = { r * std::cos(ph), r * std::sin(ph), z };
            if (dot(w, nm) < 0.f) w = w * -1.f;
            o = p; d = w; src = slot;
        }
    }
    for (int o2 = 0; o2 < 2; o2++)
        printf("shadow rays, %s: %.0f rays; from the surface %.3f records %.3f tris | from the light %.3f records %.3f tris  (answers that differ: %.0f)\n",
               o2 ? "occluded" : "clear", g_cnt[o2], g_st[o2][0][0] / g_cnt[o2], g_st[o2][0][1] / g_cnt[o2], g_st[o2][1][0] / g_cnt[o2], g_st[o2][1][1] / g_cnt[o2], g_mism);
    Counts C, S;
    for (int b = 0; b <= 5; b++) {
        printf("bounce %d: closest %9.0f rays %.3f records %.3f tris | shadow %9.0f rays %.3f records %.3f tris\n", b, cl[b].rays,
               cl[b].records / std::max(cl[b].rays, 1.0), cl[b].tris / std::max(cl[b].rays, 1.0), sh[b].rays, sh[b].records / std::max(sh[b].rays, 1.0), sh[b].tris / std::max(sh[b].rays, 1.0));
        C.rays += cl[b].rays; C.records += cl[b].records; C.tris += cl[b].tris; S.rays += sh[b].rays; S.records += sh[b].records; S.tris += sh[b].tris;
        C.deep += cl[b].deep; S.deep += sh[b].deep; C.peak = std::max(C.peak, cl[b].peak); S.peak = std::max(S.peak, sh[b].peak);
    }
    printf("all: closest %.3f records + %.3f tris per ray (GPU counters on C2: 3.35 + 2.07); shadow %.3f + %.3f (GPU, nearest-first shadow queries: 4.19 + 1.65)\n",
           C.records / C.rays, C.tris / C.rays, S.records / S.rays, S.tris / S.rays);
    for (int k = 0; k < 2; k++) {
        const Counts &q = k ? S : C;
        printf("stack, %s: peak %d entries, 3*depth %d; %.0f of %.0f rays above %d entries (%.4f)\n", k ? "shadow" : "closest", q.peak, 3 * tree.depth,
               q.deep, q.rays, g_smem, q.deep / std::max(q.rays, 1.0));
    }
    return 0;
}
