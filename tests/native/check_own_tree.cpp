// CPU-only check of the fast path's own tree builder (csrc/mfx_build.cpp); built and run by tests/test_host_abi.py.
// usage: check_own_tree <n> <mode>   mode 0: random small boxes, 1: all boxes identical, 2: a few huge + many small
//        check_own_tree <n> 3 <tris.bin>   boxes of n triangles (9 doubles each) read from a file; prints histograms
#include "mfx_build.h"

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <random>

int mfx_fail(int code, const char *fmt, ...) { va_list ap; va_start(ap, fmt); vfprintf(stderr, fmt, ap); va_end(ap); return code; }
long mfx_env_long(const char *name, long dflt) { const char *v = getenv(name); return (v && *v) ? atol(v) : dflt; }

static int as_int(float f) { int i; memcpy(&i, &f, 4); return i; }
#define REQUIRE(c) do { if (!(c)) { fprintf(stderr, "FAILED %s (line %d)\n", #c, __LINE__); return 1; } } while (0)

int main(int argc, char **argv)
{
    const int n = argc > 1 ? atoi(argv[1]) : 1000, mode = argc > 2 ? atoi(argv[2]) : 0, max_leaf = 4;
    std::mt19937 rng(n * 7 + mode);
    std::uniform_real_distribution<float> U(-10.f, 10.f), S(0.01f, 0.3f);
    std::vector<float> lo(3 * (size_t)n), hi(3 * (size_t)n);
    for (int i = 0; i < n; i++)
        for (int a = 0; a < 3; a++) {
            float c = mode == 1 ? 1.f : U(rng), e = mode == 1 ? 0.5f : S(rng);
            if (mode == 2 && i < 4) { c = 0.f; e = 12.f; }
            lo[3 * (size_t)i + a] = c - e; hi[3 * (size_t)i + a] = c + e;
        }
    if (mode == 3 && argc > 3) {
        FILE *f = fopen(argv[3], "rb");
        if (!f) { fprintf(stderr, "cannot open %s\n", argv[3]); return 2; }
        std::vector<double> tri(9 * (size_t)n);
        if (fread(tri.data(), 72, n, f) != (size_t)n) { fprintf(stderr, "short read\n"); return 2; }
        fclose(f);
        for (int i = 0; i < n; i++) for (int a = 0; a < 3; a++) {
            const double v0 = tri[9 * (size_t)i + a], v1 = tri[9 * (size_t)i + 3 + a], v2 = tri[9 * (size_t)i + 6 + a];
            lo[3 * (size_t)i + a] = (float)std::min(v0, std::min(v1, v2)) - 1e-6f; hi[3 * (size_t)i + a] = (float)std::max(v0, std::max(v1, v2)) + 1e-6f;
        }
    }
    MfxOwnTree t;
    mfx_build_own_tree(lo.data(), hi.data(), n, max_leaf, 1.0f, (int)mfx_env_long("MFX_BVH_BUILD_PAR_DEPTH", 3), t);
    REQUIRE((int)t.order.size() == n);
    std::vector<int> seen(n, 0);
    for (int v : t.order) { REQUIRE(v >= 0 && v < n); seen[v]++; }
    for (int i = 0; i < n; i++) REQUIRE(seen[i] == 1);
    REQUIRE(!t.quads.empty());
    size_t visited = 0; int depth = 0; long leaf_slots = 0;
    // returns the true bounds of the subtree of record r and checks every stored child box against them
    std::function<bool(int, int, float *, float *)> walk = [&](int r, int level, float *blo, float *bhi) -> bool {
        if (r < 0 || r >= (int)t.quads.size()) return false;
        visited++; depth = std::max(depth, level + 1);
        const QuadF &q = t.quads[r];
        const float *L[3] = { &q.lox.x, &q.loy.x, &q.loz.x }, *H[3] = { &q.hix.x, &q.hiy.x, &q.hiz.x };
        int kids = 0;
        for (int s = 0; s < 4; s++) {
            const int link = as_int((&q.meta.x)[s]);
            if (link == MFX_QUAD_EMPTY) continue;
            kids++;
            float clo[3] = { 3e38f, 3e38f, 3e38f }, chi[3] = { -3e38f, -3e38f, -3e38f };
            if (link >= 0) {
                const int first = link >> 3, cnt = link & 7;
                if (cnt < 1 || cnt > max_leaf || first < 0 || first + cnt > n) return false;
                leaf_slots += cnt;
                for (int k = 0; k < cnt; k++) for (int a = 0; a < 3; a++) {
                    clo[a] = std::min(clo[a], lo[3 * (size_t)t.order[first + k] + a]); chi[a] = std::max(chi[a], hi[3 * (size_t)t.order[first + k] + a]);
                }
            } else if (!walk(~link, level + 1, clo, chi)) return false;
            for (int a = 0; a < 3; a++) {
                if (L[a][s] > clo[a] || H[a][s] < chi[a]) return false;            // stored box must contain its subtree
                blo[a] = std::min(blo[a], clo[a]); bhi[a] = std::max(bhi[a], chi[a]);
            }
        }
        return kids >= 1;
    };
    float blo[3] = { 3e38f, 3e38f, 3e38f }, bhi[3] = { -3e38f, -3e38f, -3e38f };
    REQUIRE(walk(0, 0, blo, bhi));
    REQUIRE(visited == t.quads.size());
    REQUIRE(leaf_slots == n);
    REQUIRE(depth == t.depth);
    // SAH cost of the records: every record costs one step per unit of its area, every leaf child one test per slot
    double cost = 0.;
    for (const QuadF &q : t.quads) {
        const float *L[3] = { &q.lox.x, &q.loy.x, &q.loz.x }, *H[3] = { &q.hix.x, &q.hiy.x, &q.hiz.x };
        double rlo[3] = { 3e38, 3e38, 3e38 }, rhi[3] = { -3e38, -3e38, -3e38 };
        for (int s = 0; s < 4; s++) {
            const int link = as_int((&q.meta.x)[s]);
            if (link == MFX_QUAD_EMPTY) continue;
            const double x = (double)H[0][s] - L[0][s], y = (double)H[1][s] - L[1][s], z = (double)H[2][s] - L[2][s];
            if (link >= 0) cost += (x * y + y * z + z * x) * (link & 7);
            for (int a = 0; a < 3; a++) { rlo[a] = std::min(rlo[a], (double)L[a][s]); rhi[a] = std::max(rhi[a], (double)H[a][s]); }
        }
        const double x = rhi[0] - rlo[0], y = rhi[1] - rlo[1], z = rhi[2] - rlo[2];
        cost += x * y + y * z + z * x;
    }
    // FNV-1a over the records and the slot order: equal trees print equal hashes
    unsigned long long hash = 1469598103934665603ull;
    auto mix = [&](const void *p, size_t bytes) { for (size_t k = 0; k < bytes; k++) hash = (hash ^ ((const unsigned char *)p)[k]) * 1099511628211ull; };
    mix(t.quads.data(), t.quads.size() * sizeof(QuadF));
    mix(t.order.data(), t.order.size() * sizeof(int));
    printf("ok n=%d mode=%d records=%zu depth=%d cost=%.6g tree=%016llx\n", n, mode, t.quads.size(), t.depth, cost, hash);
    if (mode == 3) {
        long kids[5] = { 0, 0, 0, 0, 0 }, leafsz[8] = { 0, 0, 0, 0, 0, 0, 0, 0 }, leaves = 0, inner = 0;
        for (const QuadF &q : t.quads) {
            int k = 0;
            for (int s = 0; s < 4; s++) {
                const int link = as_int((&q.meta.x)[s]);
                if (link == MFX_QUAD_EMPTY) continue;
                k++;
                if (link >= 0) { leaves++; leafsz[link & 7]++; } else inner++;
            }
            kids[k]++;
        }
        printf("children per record: 1:%ld 2:%ld 3:%ld 4:%ld   leaf children %ld, interior children %ld\n", kids[1], kids[2], kids[3], kids[4], leaves, inner);
        printf("slots per leaf: 1:%ld 2:%ld 3:%ld 4:%ld 5+:%ld\n", leafsz[1], leafsz[2], leafsz[3], leafsz[4], leafsz[5] + leafsz[6] + leafsz[7]);
    }
    return 0;
}
