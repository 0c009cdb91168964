// mfx_build.cpp -- host tree builders.
//   * mfx_bvh_build: the reference's Bvh.Build (BvhNode.fs:24-61) reproduced bit for bit (the exact path and the
//     instrumented counters traverse this tree);
//   * mfx_build_own_tree: the fast path's own tree (binned SAH, four children per record).
// Compiled with -ffp-contract=off like the rest of the host code.
#include "mfx_build.h"
#include <functional>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstring>
#include <deque>
#include <future>

#define fail mfx_fail
#define env_long mfx_env_long

static float int_bits(int v) { float f; memcpy(&f, &v, 4); return f; }

// ------------------------------------------------------------------ Bvh.Build reproduction
struct HBound { double lo[3], hi[3]; };

// F# min/max on floats are System.Math.Min/Max: NaN propagates, -0.0 < +0.0.
static inline double net_min(double a, double b)
{
    if (a < b) return a;
    if (b < a) return b;
    if (a != a) return a;
    return std::signbit(a) ? a : b;
}
static inline double net_max(double a, double b)
{
    if (a > b) return a;
    if (b > a) return b;
    if (a != a) return a;
    return std::signbit(a) ? b : a;
}

static HBound prim_bound(const MfxPrim &p)
{
    HBound b;
    if (p.kind == MFX_SPHERE) {                                 // Sphere.fs:17-20: Bound(c - v, c + v)
        for (int a = 0; a < 3; a++) {
            double m0 = p.v[a] - p.v[3], m1 = p.v[a] + p.v[3];
            b.lo[a] = net_min(m0, m1); b.hi[a] = net_max(m0, m1);
        }
        return b;
    }
    const int nv = (p.kind == MFX_RECT) ? 4 : 3;                // Trangle.fs:113, Rect.fs:23
    for (int a = 0; a < 3; a++) {
        double lo = p.v[a], hi = p.v[a];
        for (int k = 1; k < nv; k++) { lo = net_min(lo, p.v[3 * k + a]); hi = net_max(hi, p.v[3 * k + a]); }
        b.lo[a] = lo; b.hi[a] = hi;
    }
    return b;
}

struct BuildCtx {
    const std::vector<HBound> *pb;
    MfxBvhNode *nodes;
    int32_t *indices;
    int32_t n_slots;
};

static MfxBvhNode init_node(const BuildCtx &c, int start, int count)    // BvhNode.fs:32-37
{
    MfxBvhNode n;
    const HBound &b0 = (*c.pb)[c.indices[start]];
    for (int a = 0; a < 3; a++) { n.pmin[a] = b0.lo[a]; n.pmax[a] = b0.hi[a]; }
    for (int i = 1; i < count; i++) {
        const HBound &b = (*c.pb)[c.indices[start + i]];
        for (int a = 0; a < 3; a++) { n.pmin[a] = net_min(n.pmin[a], b.lo[a]); n.pmax[a] = net_max(n.pmax[a], b.hi[a]); }
    }
    n.first = start; n.count = count;
    return n;
}

// Bvh.Subdivide (BvhNode.fs:42-61) for the subtree rooted at heap slot `root`.  Subtrees are independent (disjoint
// index ranges and heap slots), so the top `par_depth` levels hand their left child to another thread: the result
// is identical to the serial recursion, a 10 M-primitive build just finishes ~4x sooner.
static int subdivide(const BuildCtx &c, int root, int par_depth)
{
    std::vector<std::pair<double, int32_t>> scratch;
    std::vector<int> todo{ root };
    std::vector<std::future<int>> spawned;
    int rc = MFX_OK;
    while (!todo.empty()) {
        const int i = todo.back(); todo.pop_back();
        const MfxBvhNode node = c.nodes[i];
        if (node.count <= MFX_LEAF_NODE_COUNT) continue;
        // Bound.MaximumExtent, Aggregate.fs:29-36
        const double dx = node.pmax[0] - node.pmin[0], dy = node.pmax[1] - node.pmin[1], dz = node.pmax[2] - node.pmin[2];
        const int axis = (dx > dy && dx > dz) ? 0 : (dy > dz ? 1 : 2);
        scratch.resize(node.count);
        for (int k = 0; k < node.count; k++) {
            const int32_t id = c.indices[node.first + k];
            const HBound &b = (*c.pb)[id];
            const double dig = (b.hi[axis] - b.lo[axis]) * 0.5;           // b.Diagnal() * 0.5
            scratch[k] = { b.lo[axis] + dig, id };                        // b.pMin + dig
        }
        // Array.sortInPlaceBy is an unstable introsort in .NET (quirk Q9); ties are fixed to "stable"
        std::stable_sort(scratch.begin(), scratch.end(),
                         [](const std::pair<double, int32_t> &a, const std::pair<double, int32_t> &b) { return a.first < b.first; });
        for (int k = 0; k < node.count; k++) c.indices[node.first + k] = scratch[k].second;
        const int leftcount = node.count / 2;
        const int li = i * 2 + 1, ri = i * 2 + 2;
        if (ri >= c.n_slots) { rc = fail(MFX_ERR_INVALID_ARGUMENT, "mfx_bvh_build: heap index %d exceeds %d slots", ri, c.n_slots); break; }
        c.nodes[li] = init_node(c, node.first, leftcount);
        c.nodes[ri] = init_node(c, node.first + leftcount, node.count - leftcount);
        if (par_depth > 0 && i == root && node.count > (1 << 16)) {
            spawned.push_back(std::async(std::launch::async, [&c, li, par_depth]() { return subdivide(c, li, par_depth - 1); }));
            root = ri; par_depth--;                                       // keep splitting the right child on this thread
            todo.push_back(ri);
        } else {
            todo.push_back(ri);
            todo.push_back(li);
        }
    }
    for (auto &f : spawned) { const int r = f.get(); if (r != MFX_OK) rc = r; }
    return rc;
}

extern "C" int mfx_bvh_build(const MfxPrim *prims, int32_t n, MfxBvhNode *nodes_out, int32_t n_slots, int32_t *indices_out)
{
    if (!prims || !nodes_out || !indices_out || n <= 0) return fail(MFX_ERR_INVALID_ARGUMENT, "mfx_bvh_build: null/empty input");
    if (n_slots != 2 * n - 1) return fail(MFX_ERR_INVALID_ARGUMENT, "mfx_bvh_build: n_slots must be 2n-1 = %d, got %d", 2 * n - 1, n_slots);
    std::vector<HBound> pb(n);
    for (int i = 0; i < n; i++) {
        if (prims[i].kind < 0 || prims[i].kind > 2) return fail(MFX_ERR_INVALID_ARGUMENT, "primitive %d: unknown kind %d", i, prims[i].kind);
        pb[i] = prim_bound(prims[i]);
    }
    for (int i = 0; i < n; i++) indices_out[i] = i;
    memset(nodes_out, 0, sizeof(MfxBvhNode) * (size_t)n_slots);
    BuildCtx c{ &pb, nodes_out, indices_out, n_slots };
    nodes_out[0] = init_node(c, 0, n);
    return subdivide(c, 0, (int)env_long("MFX_BVH_BUILD_PAR_DEPTH", 5));
}

// ---- flatten: fast layout over the library's own tree (binned SAH, collapsed to four children per record)
struct SahNode { float lo[3], hi[3]; int left, right, first, count; };   // count > 0: leaf over order[first .. first+count)
struct SahCtx {
    const float (*lo)[3]; const float (*hi)[3];
    int *idx;
    SahNode *nodes;
    std::atomic<int> next{ 0 };
    int max_leaf;
    float c_trav;       // cost of one node step relative to one primitive test
    int sweep_below;    // nodes with at most this many primitives get the exact sweep, larger ones 32 bins
};
static inline float half_area(const float *lo, const float *hi)
{
    const float x = hi[0] - lo[0], y = hi[1] - lo[1], z = hi[2] - lo[2];
    return x * y + y * z + z * x;
}
static inline void grow(float *lo, float *hi, const float *blo, const float *bhi)
{
    for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], blo[a]); hi[a] = std::max(hi[a], bhi[a]); }
}
static const float SAH_INF = 3.0e38f;

// Splits idx[first .. first+count) by the surface-area heuristic; returns the size of the left part (0 = keep as leaf).
static int sah_split(SahCtx &c, const SahNode &nd)
{
    const int first = nd.first, count = nd.count;
    const float area = half_area(nd.lo, nd.hi);
    const float leaf_cost = (float)count;                    // in units of (node area x primitive test)
    float best = SAH_INF; int best_axis = -1, best_pos = -1, best_bal = 0x7fffffff;
    float clo[3] = { SAH_INF, SAH_INF, SAH_INF }, chi[3] = { -SAH_INF, -SAH_INF, -SAH_INF };
    for (int k = 0; k < count; k++) {
        const int id = c.idx[first + k];
        for (int a = 0; a < 3; a++) { const float ce = 0.5f * (c.lo[id][a] + c.hi[id][a]); clo[a] = std::min(clo[a], ce); chi[a] = std::max(chi[a], ce); }
    }
    const float inv_area = area > 0.f ? 1.0f / area : 0.f;
    if (count <= c.sweep_below) {
        // exact sweep: sort by centroid on each axis (stable), try every split position
        static thread_local std::vector<std::pair<float, int>> key;
        static thread_local std::vector<float> right;
        static thread_local std::vector<int> best_order;
        key.resize(count); right.resize(count); best_order.resize(count);
        for (int ax = 0; ax < 3; ax++) {
            if (count <= 24) {
                for (int k = 0; k < count; k++) {
                    const int id = c.idx[first + k];
                    const std::pair<float, int> e{ c.lo[id][ax] + c.hi[id][ax], id };
                    int j = k;
                    while (j > 0 && key[j - 1].first > e.first) { key[j] = key[j - 1]; j--; }
                    key[j] = e;
                }
            } else {
                for (int k = 0; k < count; k++) { const int id = c.idx[first + k]; key[k] = { c.lo[id][ax] + c.hi[id][ax], id }; }
                std::stable_sort(key.begin(), key.end(), [](const std::pair<float, int> &x, const std::pair<float, int> &y) { return x.first < y.first; });
            }
            float lo[3] = { SAH_INF, SAH_INF, SAH_INF }, hi[3] = { -SAH_INF, -SAH_INF, -SAH_INF };
            for (int k = count - 1; k > 0; k--) { grow(lo, hi, c.lo[key[k].second], c.hi[key[k].second]); right[k] = half_area(lo, hi); }
            for (int a = 0; a < 3; a++) { lo[a] = SAH_INF; hi[a] = -SAH_INF; }
            bool improved = false;
            for (int k = 1; k < count; k++) {
                grow(lo, hi, c.lo[key[k - 1].second], c.hi[key[k - 1].second]);
                const float cost = c.c_trav + (half_area(lo, hi) * k + right[k] * (count - k)) * inv_area;
                // equal costs (coincident boxes): take the most balanced split, or the tree degenerates into a chain
                const int bal = std::abs(2 * k - count);
                if (cost < best || (cost == best && bal < best_bal)) { best = cost; best_bal = bal; best_axis = ax; best_pos = k; improved = true; }
            }
            if (improved) for (int k = 0; k < count; k++) best_order[k] = key[k].second;
        }
        if (best_axis < 0 || (count <= c.max_leaf && leaf_cost <= best)) return count <= c.max_leaf ? 0 : count / 2;
        for (int k = 0; k < count; k++) c.idx[first + k] = best_order[k];
        return best_pos;
    }
    // binned: up to 1024 centroid bins per axis.  Few bins are not enough here: one outlier (the floor quad under a
    // 6 k-triangle model) stretches the centroid range until the model falls into three or four of 32 bins, and the
    // tree built that way needs a third more node steps per ray than the exact sweep's (C2: 4.4 vs 3.3 records/ray).
    const int NBMAX = 1024;
    const int NB = std::min(NBMAX, std::max(32, count / 2));
    int best_bin = -1;
    static thread_local std::vector<float> bin_box;     // [NB][6] lo.xyz hi.xyz
    static thread_local std::vector<int> bin_n;
    static thread_local std::vector<float> right_area;
    static thread_local std::vector<int> right_n;
    bin_box.resize((size_t)NB * 6); bin_n.resize(NB); right_area.resize(NB); right_n.resize(NB);
    for (int ax = 0; ax < 3; ax++) {
        const float ext = chi[ax] - clo[ax];
        if (!(ext > 0.f)) continue;
        const float scale = (float)NB * (1.0f - 1e-6f) / ext;
        float *bb = bin_box.data(); int *bn = bin_n.data(); float *right = right_area.data(); int *rn = right_n.data();
        for (int b = 0; b < NB; b++) { bn[b] = 0; for (int a = 0; a < 3; a++) { bb[6 * b + a] = SAH_INF; bb[6 * b + 3 + a] = -SAH_INF; } }
        for (int k = 0; k < count; k++) {
            const int id = c.idx[first + k];
            int b = (int)((0.5f * (c.lo[id][ax] + c.hi[id][ax]) - clo[ax]) * scale);
            b = b < 0 ? 0 : (b >= NB ? NB - 1 : b);
            bn[b]++; grow(bb + 6 * b, bb + 6 * b + 3, c.lo[id], c.hi[id]);
        }
        float lo[3] = { SAH_INF, SAH_INF, SAH_INF }, hi[3] = { -SAH_INF, -SAH_INF, -SAH_INF };
        int cnt = 0;
        for (int b = NB - 1; b > 0; b--) { if (bn[b]) grow(lo, hi, bb + 6 * b, bb + 6 * b + 3); cnt += bn[b]; right[b] = cnt ? half_area(lo, hi) : 0.f; rn[b] = cnt; }
        for (int a = 0; a < 3; a++) { lo[a] = SAH_INF; hi[a] = -SAH_INF; }
        cnt = 0;
        for (int b = 1; b < NB; b++) {
            if (bn[b - 1]) grow(lo, hi, bb + 6 * (b - 1), bb + 6 * (b - 1) + 3);
            cnt += bn[b - 1];
            if (cnt == 0 || rn[b] == 0) continue;
            const float cost = c.c_trav + (half_area(lo, hi) * cnt + right[b] * rn[b]) * inv_area;
            if (cost < best) { best = cost; best_axis = ax; best_bin = b; }
        }
    }
    if (best_axis < 0) {
        // all centroids coincide: nothing to choose between, cut the list in half
        return count / 2;
    }
    const float scale = (float)NB * (1.0f - 1e-6f) / (chi[best_axis] - clo[best_axis]);
    int *mid = std::partition(c.idx + first, c.idx + first + count, [&](int id) {
        int b = (int)((0.5f * (c.lo[id][best_axis] + c.hi[id][best_axis]) - clo[best_axis]) * scale);
        b = b < 0 ? 0 : (b >= NB ? NB - 1 : b);
        return b < best_bin;
    });
    const int left = (int)(mid - (c.idx + first));
    return (left == 0 || left == count) ? count / 2 : left;
}

static void sah_bound(const SahCtx &c, SahNode &nd)
{
    for (int a = 0; a < 3; a++) { nd.lo[a] = SAH_INF; nd.hi[a] = -SAH_INF; }
    for (int k = 0; k < nd.count; k++) grow(nd.lo, nd.hi, c.lo[c.idx[nd.first + k]], c.hi[c.idx[nd.first + k]]);
}

// Builds the subtree of node `root` (its first/count/bounds are set).  Disjoint ranges => the top levels fork.
static void sah_build(SahCtx &c, int root, int par_depth)
{
    std::vector<int> todo{ root };
    std::vector<std::future<void>> spawned;
    while (!todo.empty()) {
        const int i = todo.back(); todo.pop_back();
        SahNode nd = c.nodes[i];
        if (nd.count <= 1) continue;
        const int left = sah_split(c, nd);
        if (left == 0) continue;                                 // stays a leaf
        const int li = c.next.fetch_add(2), ri = li + 1;
        SahNode &L = c.nodes[li], &R = c.nodes[ri];
        L.first = nd.first; L.count = left; L.left = L.right = -1;
        R.first = nd.first + left; R.count = nd.count - left; R.left = R.right = -1;
        sah_bound(c, L); sah_bound(c, R);
        c.nodes[i].left = li; c.nodes[i].right = ri; c.nodes[i].count = 0;
        if (par_depth > 0 && i == root && nd.count > 1024) {
            spawned.push_back(std::async(std::launch::async, [&c, li, par_depth]() { sah_build(c, li, par_depth - 1); }));
            root = ri; par_depth--;
            todo.push_back(ri);
        } else {
            todo.push_back(ri); todo.push_back(li);
        }
    }
    for (auto &f : spawned) f.get();
}

// The forked levels of sah_build take their node indices from one counter in whatever order the threads reach it; the
// splits themselves do not depend on the schedule.  The reinsertion pass breaks ties by node index, so before it runs
// the nodes are renumbered in the order a serial build allocates them: the same tree for any fork depth and schedule.
static void sah_renumber_serial(std::vector<SahNode> &nodes)
{
    std::vector<SahNode> out(nodes.size());
    std::vector<std::pair<int, int>> todo{ { 0, 0 } };         // (index in `nodes`, index in `out`)
    int next = 1;
    while (!todo.empty()) {
        const auto [from, to] = todo.back(); todo.pop_back();
        SahNode nd = nodes[from];
        if (nd.count == 0) {
            todo.push_back({ nd.right, next + 1 }); todo.push_back({ nd.left, next });
            nd.left = next; nd.right = next + 1;
            next += 2;
        }
        out[to] = nd;
    }
    nodes.swap(out);
}

// Insertion-based optimisation of the binary tree (after Bittner, Hapala, Havran 2013): take a subtree out, let its sibling
// move up, and put it back where the sum of the interior nodes' areas grows least -- found by branch and bound from the
// root (induced cost = what the ancestors of a candidate grow by; a subtree can never cost less than its own area).
// The best position includes the old one, so the SAH cost never rises; primitives and leaves are untouched.  Sequential
// (every move changes the boxes the next search reads); `passes` sweeps over the `max_cand` largest nodes, largest first.
static void sah_reinsert(SahNode *nodes, int nn, int passes, size_t max_cand)
{
    std::vector<int> parent(nn, -1), cand;
    {
        std::vector<int> st{ 0 };
        while (!st.empty()) {
            const int i = st.back(); st.pop_back();
            if (nodes[i].count == 0) { parent[nodes[i].left] = i; parent[nodes[i].right] = i; st.push_back(nodes[i].left); st.push_back(nodes[i].right); }
            if (i != 0) cand.push_back(i);
        }
    }
    auto refit = [&](int i) {           // from node i up to the root
        for (; i >= 0; i = parent[i]) {
            SahNode &n = nodes[i];
            if (n.count > 0) continue;
            const SahNode &l = nodes[n.left], &r = nodes[n.right];
            float lo[3], hi[3];
            for (int a = 0; a < 3; a++) { lo[a] = std::min(l.lo[a], r.lo[a]); hi[a] = std::max(l.hi[a], r.hi[a]); }
            bool same = true;
            for (int a = 0; a < 3; a++) same = same && lo[a] == n.lo[a] && hi[a] == n.hi[a];
            if (same) break;
            for (int a = 0; a < 3; a++) { n.lo[a] = lo[a]; n.hi[a] = hi[a]; }
        }
    };
    auto union_area = [&](const SahNode &x, const SahNode &y) {
        float lo[3], hi[3];
        for (int a = 0; a < 3; a++) { lo[a] = std::min(x.lo[a], y.lo[a]); hi[a] = std::max(x.hi[a], y.hi[a]); }
        return half_area(lo, hi);
    };
    struct Item { float ind; int node; bool operator<(const Item &o) const { return ind > o.ind; } };
    std::vector<Item> heap;
    for (int pass = 0; pass < passes; pass++) {
        std::sort(cand.begin(), cand.end(), [&](int x, int y) {
            const float ax = half_area(nodes[x].lo, nodes[x].hi), ay = half_area(nodes[y].lo, nodes[y].hi);
            return ax > ay || (ax == ay && x < y);
        });
        // the largest subtrees matter most (every ray meets them) and the cost of a pass is bounded by their number
        for (size_t ci = 0; ci < cand.size() && ci < max_cand; ci++) {
            const int N = cand[ci];
            const int P = parent[N];
            if (P <= 0) continue;                                   // children of the root stay (the root keeps index 0)
            const int G = parent[P];
            const int S = nodes[P].left == N ? nodes[P].right : nodes[P].left;
            // take N (and its parent P) out: S moves up
            (nodes[G].left == P ? nodes[G].left : nodes[G].right) = S;
            parent[S] = G;
            refit(G);
            // branch and bound for the cheapest new sibling X
            const float aN = half_area(nodes[N].lo, nodes[N].hi);
            // the position it came from is the one to beat, STRICTLY: among equal costs (coincident boxes) nothing moves,
            // or every subtree would end up beside the root and the tree would degenerate into a chain
            float best, ind0 = 0.f; int bestX = S;
            for (int A = G; A >= 0; A = parent[A]) ind0 += union_area(nodes[A], nodes[N]) - half_area(nodes[A].lo, nodes[A].hi);
            best = ind0 + union_area(nodes[S], nodes[N]);
            heap.clear(); heap.push_back({ 0.f, 0 });
            while (!heap.empty()) {
                std::pop_heap(heap.begin(), heap.end()); const Item it = heap.back(); heap.pop_back();
                if (it.ind + aN >= best) break;
                const SahNode &X = nodes[it.node];
                const float direct = union_area(X, nodes[N]);
                const float total = it.ind + direct;
                if (total < best * 0.99999f) { best = total; bestX = it.node; }
                const float child_ind = total - half_area(X.lo, X.hi);
                if (X.count == 0 && child_ind + aN < best) {
                    heap.push_back({ child_ind, X.left }); std::push_heap(heap.begin(), heap.end());
                    heap.push_back({ child_ind, X.right }); std::push_heap(heap.begin(), heap.end());
                }
            }
            // put P (with children bestX and N) where bestX was
            const int X = bestX, XP = parent[X];
            if (XP < 0) {                                            // new sibling is the root: the root record must stay node 0
                // swap roles: node 0 keeps being the root, P takes over the old root's content
                nodes[P] = nodes[0];
                if (nodes[P].count == 0) { parent[nodes[P].left] = P; parent[nodes[P].right] = P; }
                nodes[0].count = 0; nodes[0].left = P; nodes[0].right = N; nodes[0].first = 0;
                parent[P] = 0; parent[N] = 0;
                refit(0);
                // force a full refit of the new root
                for (int a = 0; a < 3; a++) { nodes[0].lo[a] = std::min(nodes[P].lo[a], nodes[N].lo[a]); nodes[0].hi[a] = std::max(nodes[P].hi[a], nodes[N].hi[a]); }
                continue;
            }
            (nodes[XP].left == X ? nodes[XP].left : nodes[XP].right) = P;
            parent[P] = XP;
            nodes[P].left = X; nodes[P].right = N; nodes[P].count = 0;
            parent[X] = P; parent[N] = P;
            for (int a = 0; a < 3; a++) { nodes[P].lo[a] = std::min(nodes[X].lo[a], nodes[N].lo[a]); nodes[P].hi[a] = std::max(nodes[X].hi[a], nodes[N].hi[a]); }
            refit(XP);
        }
    }
}

void mfx_build_own_tree(const float *lo, const float *hi, int ns, int max_leaf, float trav_cost, int par_depth, MfxOwnTree &out)
{
    std::vector<int> idx(ns);
    for (int k = 0; k < ns; k++) idx[k] = k;
    std::vector<SahNode> nodes((size_t)2 * ns + 2);
    SahCtx c;
    c.lo = reinterpret_cast<const float (*)[3]>(lo); c.hi = reinterpret_cast<const float (*)[3]>(hi);
    c.idx = idx.data(); c.nodes = nodes.data(); c.next = 1;
    c.max_leaf = max_leaf;
    c.c_trav = trav_cost;
    c.sweep_below = (int)std::max(24L, env_long("MFX_SAH_SWEEP_BELOW", 64));
    nodes[0].first = 0; nodes[0].count = ns; nodes[0].left = nodes[0].right = -1;
    sah_bound(c, nodes[0]);
    sah_build(c, 0, par_depth);
    sah_renumber_serial(nodes);
    c.nodes = nodes.data();
    // MFX_TREE_OPT = reinsertion passes over the binary tree before it is collapsed (0: off), each over the
    // MFX_TREE_OPT_NODES largest subtrees; scenes above MFX_TREE_OPT_MAX primitives skip it (the pass is sequential)
    {
        const int passes = (int)env_long("MFX_TREE_OPT", 2);
        if (passes > 0 && nodes[0].count == 0 && ns <= env_long("MFX_TREE_OPT_MAX", 500000))
            sah_reinsert(nodes.data(), c.next.load(), passes, (size_t)std::max(1L, env_long("MFX_TREE_OPT_NODES", 32768)));
    }

    // MFX_COLLAPSE_DP = cost of one record step in percent of one primitive test (default 100; 0 = the greedy
    // largest-area-first collapse of round 1; measured on B200: +1.0 % C2, +1.0 % C3, +0.5 % C4, same build time):
    // choose the <= 4 slots of every record by dynamic programming over the binary tree instead of greedily --
    //   slot(n)   = min( area(n) * prims(n)                          if prims(n) <= max_leaf: n becomes ONE leaf,
    //                    area(n) * c_rec + min_k F(left, k) + F(right, 4 - k)          : n becomes a record )
    //   F(n, j)   = min( F(n, j - 1), min_k F(left, k) + F(right, j - k) ),  F(n, 1) = slot(n)
    // (the wide-BVH construction of Ylitie, Karras, Laine 2017, four wide).  Evaluated with tools/own_tree_sim.cpp.
    const float dp_rec = (float)env_long("MFX_COLLAPSE_DP", 100) * 0.01f;
    const bool dp = dp_rec > 0.f && nodes[0].count == 0;
    const int nn = c.next.load();
    std::vector<int> np;                    // prims below a binary node
    std::vector<float> fcost;               // F(n, j), j = 1..4 at [4n + j - 1]
    std::vector<unsigned char> as_leaf, fsplit;     // slot(n) is a leaf; fsplit[4n + j - 1] = k (0: take F(n, j - 1))
    if (dp) {
        np.assign(nn, 0); fcost.assign((size_t)4 * nn, 0.f); as_leaf.assign(nn, 0); fsplit.assign((size_t)4 * nn, 0);
        // children are allocated after their parent (fetch_add), so a descending index order is a post-order
        std::vector<int> orderv; orderv.reserve(nn);
        { std::vector<int> st{ 0 }; while (!st.empty()) { const int i = st.back(); st.pop_back(); orderv.push_back(i); if (nodes[i].count == 0) { st.push_back(nodes[i].left); st.push_back(nodes[i].right); } } }
        for (size_t r = orderv.size(); r-- > 0;) {
            const int i = orderv[r];
            const SahNode &nd = nodes[i];
            const float ar = half_area(nd.lo, nd.hi);
            float *F = &fcost[(size_t)4 * i];
            if (nd.count > 0) {
                np[i] = nd.count; as_leaf[i] = 1;
                for (int j = 0; j < 4; j++) F[j] = ar * (float)nd.count;
                continue;
            }
            const int L = nd.left, R = nd.right;
            np[i] = np[L] + np[R];
            const float *FL = &fcost[(size_t)4 * L], *FR = &fcost[(size_t)4 * R];
            // as a record: the best way to spend four slots on the two subtrees
            float rec = SAH_INF;
            for (int k = 1; k <= 3; k++) rec = std::min(rec, FL[k - 1] + FR[3 - k]);
            rec += ar * dp_rec;
            const float leaf = np[i] <= max_leaf ? ar * (float)np[i] : SAH_INF;
            as_leaf[i] = leaf <= rec;
            F[0] = std::min(leaf, rec);
            for (int j = 2; j <= 4; j++) {
                float best = F[j - 2]; int bk = 0;
                for (int k = 1; k < j; k++) { const float v = FL[k - 1] + FR[j - k - 1]; if (v < best) { best = v; bk = k; } }
                F[j - 1] = best; fsplit[(size_t)4 * i + j - 1] = (unsigned char)bk;
            }
        }
    }
    // the slots the DP gives subtree n when it may use up to j of them
    std::function<void(int, int, int *, int &)> dp_expand = [&](int n, int j, int *kids, int &nk) {
        while (j > 1 && fsplit[(size_t)4 * n + j - 1] == 0) j--;
        if (j == 1 || nodes[n].count > 0) { kids[nk++] = n; return; }
        const int k = fsplit[(size_t)4 * n + j - 1];
        dp_expand(nodes[n].left, k, kids, nk); dp_expand(nodes[n].right, j - k, kids, nk);
    };
    auto slot_prims = [&](int b) { return dp ? (as_leaf[b] ? np[b] : 0) : nodes[b].count; };   // > 0: the slot is a leaf

    // collapse to four children per record, depth-first; leaves of a record get consecutive slots
    std::vector<QuadF> &quads = out.quads;
    quads.clear();
    std::vector<int> &order = out.order;
    order.clear(); order.reserve(ns);
    int own_depth = 0;
    struct Item { int bnode; int level; int parent; int pslot; };
    std::vector<Item> todo{ { 0, 0, -1, 0 } };
    quads.reserve((size_t)ns / 2 + 4);
    const float FAR = 1e30f;
    while (!todo.empty()) {
        const Item it = todo.back(); todo.pop_back();
        const int qi = (int)quads.size();
        if (it.parent >= 0) reinterpret_cast<int *>(&quads[it.parent].meta)[it.pslot] = ~qi;
        own_depth = std::max(own_depth, it.level + 1);
        int kids[4], nk = 0;
        if (nodes[it.bnode].count > 0) kids[nk++] = it.bnode;           // a one-leaf tree: the root record holds it
        else if (dp) {
            const float *FL = &fcost[(size_t)4 * nodes[it.bnode].left], *FR = &fcost[(size_t)4 * nodes[it.bnode].right];
            int bk = 1; float best = SAH_INF;
            for (int k = 1; k <= 3; k++) { const float v = FL[k - 1] + FR[3 - k]; if (v < best) { best = v; bk = k; } }
            dp_expand(nodes[it.bnode].left, bk, kids, nk); dp_expand(nodes[it.bnode].right, 4 - bk, kids, nk);
        }
        else { kids[nk++] = nodes[it.bnode].left; kids[nk++] = nodes[it.bnode].right; }
        while (!dp && nk < 4) {
            int pick = -1; float pa = -1.f;
            for (int k = 0; k < nk; k++) if (nodes[kids[k]].count == 0) { const float ar = half_area(nodes[kids[k]].lo, nodes[kids[k]].hi); if (ar > pa) { pa = ar; pick = k; } }
            if (pick < 0) break;
            const int b = kids[pick];
            kids[pick] = nodes[b].left; kids[nk++] = nodes[b].right;
        }
        QuadF q; memset(&q, 0, sizeof(q));
        float lo[3][4], hi[3][4]; int meta[4];
        for (int sl = 0; sl < 4; sl++) { for (int a = 0; a < 3; a++) { lo[a][sl] = FAR; hi[a][sl] = FAR; } meta[sl] = MFX_QUAD_EMPTY; }
        for (int k = 0; k < nk; k++) {
            const SahNode &nd = nodes[kids[k]];
            for (int a = 0; a < 3; a++) { lo[a][k] = nd.lo[a]; hi[a][k] = nd.hi[a]; }
            const int cnt = slot_prims(kids[k]);
            if (cnt > 0) {
                meta[k] = ((int)order.size() << 3) | cnt;
                // (a binary subtree merged into one leaf: its primitives are gathered leaf by leaf -- after the reinsertion
                //  pass they are no longer one range of idx)
                int st[16], sp = 0; st[sp++] = kids[k];
                while (sp > 0) {
                    const SahNode &g = nodes[st[--sp]];
                    if (g.count > 0) { for (int j = 0; j < g.count; j++) order.push_back(idx[g.first + j]); }
                    else { st[sp++] = g.right; st[sp++] = g.left; }
                }
            }
        }
        q.lox = make_float4(lo[0][0], lo[0][1], lo[0][2], lo[0][3]); q.hix = make_float4(hi[0][0], hi[0][1], hi[0][2], hi[0][3]);
        q.loy = make_float4(lo[1][0], lo[1][1], lo[1][2], lo[1][3]); q.hiy = make_float4(hi[1][0], hi[1][1], hi[1][2], hi[1][3]);
        q.loz = make_float4(lo[2][0], lo[2][1], lo[2][2], lo[2][3]); q.hiz = make_float4(hi[2][0], hi[2][1], hi[2][2], hi[2][3]);
        q.meta = make_float4(int_bits(meta[0]), int_bits(meta[1]), int_bits(meta[2]), int_bits(meta[3]));
        quads.push_back(q);
        for (int k = nk - 1; k >= 0; k--) if (slot_prims(kids[k]) == 0) todo.push_back({ kids[k], it.level + 1, qi, k });
    }
    out.depth = own_depth;
}
