// mfx_build.h -- the two host tree builders (mfx_build.cpp) and the error / environment plumbing shared by the
// host translation units.  Nothing here crosses the C ABI except mfx_bvh_build (declared in include/mafrix_cuda.h).
#pragma once
#include "../../include/mafrix_cuda.h"
#include "mfx_internal.h"
#include <vector>

int mfx_fail(int code, const char *fmt, ...);           // sets mfx_last_error(), returns `code` (mfx_host.cpp)
long mfx_env_long(const char *name, long dflt);

// The fast path's own tree: binned-SAH binary BVH over n primitive slots (bounds lo/hi, [n][3] floats), collapsed to
// four children per 128 B record, records depth-first, the leaves of a record owning consecutive output slots.
struct MfxOwnTree {
    std::vector<QuadF> quads;   // links: leaf first<<3|count (indices into `order`), interior ~record, MFX_QUAD_EMPTY
    std::vector<int>   order;   // output slot -> input slot
    int depth = 0;              // number of record levels (the traversal stack holds <= 3 entries per level)
};
void mfx_build_own_tree(const float *lo, const float *hi, int n, int max_leaf, float trav_cost, int par_depth, MfxOwnTree &out);
