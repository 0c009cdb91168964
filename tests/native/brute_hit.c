/* brute_hit.c -- brute-force f64 classifier of closest-hit and any-hit queries, for the f32 traversal tests
 * (tests/test_gpu_f32_traversal.py, and tests/test_gpu_f32_from_surface.py for rays that start on a primitive).  Test
 * infrastructure only: no tree, every ray against every primitive.
 *
 * Semantics are those of the fast path (DESIGN.md 4.3, leaf_f3 in mfx_fast.cu), not the reference's quirks:
 *   - a triangle is Moller-Trumbore with leaf_f3's acceptance predicate: |div| >= 1e-6 absolute, b1 in [0,1],
 *     b2 >= 0, b1 + b2 < 1, tMin < t < tMax (triangles honour tMax: quirk Q2 is not reproduced);
 *   - a Rect is two independent triangles, (v0,v1,v2) as sub 0 and (v0,v2,v3) as sub 1, the nearer wins (no Q3);
 *   - a sphere solves Sphere.Hit's quadratic (a = 1: the direction is taken as a unit vector, so spheres are only
 *     queried with unit directions) and takes the near root if it lies in the window, otherwise the far root; big
 *     spheres (r >= 32, the kernel's f64 branch) get the same treatment;
 *   - a ray may start on a source primitive (brute_classify_from, SOURCE RULES below); brute_classify has none.
 *
 * Every (ray, primitive) pair is a CLEAR HIT, a CLEAR MISS or AMBIGUOUS, with margins taken from the f32 kernel's error.
 * The kernel sees o, d, v0 (a sphere's centre) and the edges e1 = v1 - v0, e2 = v2 - v0 rounded to f32, 2^-24 relative
 * each; it forms dd = o - v0 and cross and dot products of dd, d and the edges (a few roundings of 2^-24 of the
 * magnitudes involved each) and divides with rcp.approx (2^-23).  Carried to the plane of the primitive as a
 * displacement of the hit point relative to the ray:
 *   - rounding o and v0 moves it by at most sqrt(3) 2^-24 (|o|_inf + max_abs), max_abs the largest coordinate
 *     magnitude of the scene (sphere centre +- radius included);
 *   - rounding the edges and d, the products and rcp.approx move it by at most about 12 2^-24 (|dd| + t|d| + |e1| +
 *     |e2|), and the hit distance t|d| is at most |dd| + |e1| + |e2| (a sphere: |o - c| + r for |dd|, r for the edges);
 * so, with a factor of two to spare on each term,
 *     eps = 2^-24 (K_IN (max_abs + |o|_inf) + K_AR (|dd| + |e1| + |e2|)),  K_IN = 4,  K_AR = 48.
 * eps is per pair: a small mesh far from the origin is limited by where it is (the first term), not by how far the
 * ray travels to it.  A displacement eps perpendicular to the ray moves the hit point in the plane by eps/|cos| (cos:
 * between the ray and the plane's normal) and t by eps/(|d||cos|); the margins below carry that factor.  The f32 slab
 * tests of the tree need no margin of their own: their roundings are of the same kind and size (o * rcp(d) and the
 * fma with a box bound: 2^-24 of |o| and of the bound, 2^-23 of |bound - o|), and a box misses a point of its
 * primitive only if that point lies within that rounding of two of its faces at once; the only such points of a
 * triangle lie within eps of one of its edges or vertices (DESIGN.md 4.3).
 *
 * A pair is AMBIGUOUS when it is not a clear miss and any of these holds:
 *   - the hit point lies within eps/|cos| of a triangle edge line, or the ray passes within eps of the sphere's
 *     silhouette (|h - r| < eps, h the distance from the centre to the ray);
 *   - t lies within u + 1e-5 t of tMin or tMax, u = eps / (|d| |cos|) the t uncertainty (a sphere's cos is the
 *     one at the chosen root, sqrt(disc) / r);
 *   - |div| lies within 1e-3 relative of the 1e-6 threshold;
 *   - the ray meets the triangle's plane at |cos| < 1e-3.
 * A pair is a clear miss when |div| < 1e-6 (1 - 1e-3), when the hit point lies beyond eps/|cos| outside an edge line,
 * when h >= r + eps, or when the chosen t lies beyond its margin outside the window.
 *
 * A ray's answer is ROBUST when every way of resolving its ambiguous pairs gives the same answer:
 *   - closest hit: no candidate (clear or ambiguous) at all -- a robust miss -- or a nearest clear hit t_w that lies
 *     before every other candidate (its least possible t) by at least 1e-4 t_w + u_w + u_j (coincident copies and
 *     shared Rect diagonals are therefore not robust);
 *   - any hit: occluded if a clear hit lies in the window, clear if there is no candidate at all.
 *
 * SOURCE RULES (leaf_f3: the rays of bounces >= 1 and the shadow rays start on the primitive they left, src = its index):
 *   - a source triangle or Rect is a clear miss, both halves of a Rect (the kernel compares the id without the half
 *     bit), a non-planar Rect included;
 *   - a source sphere is decided by the sign of hb = (o - c).d (d a unit vector): the kernel skips it when its f32 hb
 *     is >= 0 (leaving) and otherwise takes the far root, or the chord -2 hb when its f32 discriminant comes out <= 0.
 *     The kernel's hb differs from the f64 one by the rounding of o and c (sqrt(3) 2^-24 (|o|_inf + |c|_inf)), of d
 *     (sqrt(3) 2^-24 |o - c|, d unit), of the subtraction o - c (sqrt(3) 2^-24 |o - c|) and of the three products and
 *     two sums of the dot product (3 2^-24 |o - c|): at most about 2^-24 (2 (|c|_inf + |o|_inf) + 7 |o - c|).  With a
 *     factor of two to spare, in the constants of eps,
 *         eps_h = 2^-24 (K_IN (|c|_inf + |o|_inf) + K_AR |o - c|),
 *     and a big sphere (r >= 32, solved in f64 from its f64 centre) drops |c|_inf: only o and d are rounded there.
 *       hb >= eps_h: clear miss (leaving);
 *       hb <= -eps_h: the far root, when the f64 discriminant hb^2 - (|o - c|^2 - r^2) is within its rounding of 0
 *         the chord -2 hb (on a point exactly on the surface the two are the same).  The kernel's t lies in
 *           [max(t - u, |hb| - eps_h),  min(t + u, 2 (|hb| + eps_h) + sqrt(4 r eps_h))],
 *         u = eps / (|d| cos) the t margin above (cos = sqrt(disc) / r at the far root, |hb| / r at the chord), and
 *         the pair is classified by that interval (its centre and half-width stand for t and u).  The second bound
 *         of each end holds whichever of the root or the chord fires: the far root -hb + sqrt(disc) is at least
 *         |hb_f32| and the chord is 2 |hb_f32|, |hb_f32| >= |hb| - eps_h; the f32 discriminant is hb_f32^2 plus an
 *         error delta -- the origin's distance from the surface (at most eps_h / 2, times 2 r), the error of the
 *         perpendicular part of o - c (at most eps_h, times 2 r) and the roundings of r^2 and |perp|^2 (4 2^-24 r^2)
 *         -- so |delta| <= 4 r eps_h and the root is at most 2 |hb_f32| + sqrt(4 r eps_h).  Near the tangent plane,
 *         where u exceeds t and the kernel's chord fires (|hb| up to ~1e-3 r), an entering ray is therefore a clear
 *         hit of its source once |hb| - eps_h clears tMin: the chord rule is held ray by ray;
 *       |hb| < eps_h: ambiguous (skipped, or re-entered at a t anywhere from 0 to the f32 root's error), at tMin.
 *   - every other pair is classified as without a source.
 */
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define K_IN 4.0
#define K_AR 48.0
#define MISS 0
#define HIT 1
#define AMB 2

typedef struct {
    int prim, sub, sphere;
    double v0[3], e1[3], e2[3];     /* triangle */
    double ha, hb, hc, nl;          /* |n|/|e2|, |n|/|e1|, |n|/|e2 - e1|, |n| = |e1 x e2| */
    double size;                    /* |e1| + |e2|; a sphere: r */
    double c[3], r;                 /* sphere */
} BPrim;

typedef struct {
    const BPrim *p; int np;
    const double *o, *d; int n;
    double tmin, tmax, max_abs;
    int any_hit, normalize;
    const int32_t *src;             /* caller's index of the primitive ray i starts on, -1 none; NULL: none at all */
    int8_t *robust; int32_t *prim, *sub, *n_amb; double *t, *terr, *eps;
    int next; pthread_mutex_t mu;
} Job;

typedef struct { double t, u; } Cand;

static inline double dot3(const double *a, const double *b) { return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]; }
static inline void cross3(const double *a, const double *b, double *o)
{
    o[0] = a[1] * b[2] - a[2] * b[1]; o[1] = a[2] * b[0] - a[0] * b[2]; o[2] = a[0] * b[1] - a[1] * b[0];
}

/* where x lies in the window (tmin, tmax) with margin m: -1 below, 0 inside, 1 ambiguous, 2 above */
static inline int window(double x, double m, double tmin, double tmax)
{
    if (x <= tmin - m) return -1;
    if (x >= tmax + m) return 2;
    if (x < tmin + m || x > tmax - m) return 1;
    return 0;
}

static int classify_tri(const BPrim *p, const double *o, const double *d, double dl, double eps_in, double tmin, double tmax,
                        double *t_out, double *u_out, double *eps_out)
{
    double s1[3], s2[3], dd[3];
    cross3(d, p->e2, s1);
    const double div = dot3(s1, p->e1), adiv = fabs(div);
    if (adiv < 1e-6 * (1.0 - 1e-3) || p->nl == 0.0) return MISS;
    int amb = adiv < 1e-6 * (1.0 + 1e-3);
    const double cosv = adiv / (dl * p->nl);
    const double inv = 1.0 / div;
    for (int k = 0; k < 3; k++) dd[k] = o[k] - p->v0[k];
    const double eps = eps_in + K_AR * ldexp(1.0, -24) * (sqrt(dot3(dd, dd)) + p->size);
    *eps_out = eps;
    const double b1 = dot3(dd, s1) * inv;
    cross3(dd, p->e1, s2);
    const double b2 = dot3(d, s2) * inv;
    const double t = dot3(p->e2, s2) * inv;
    const double m = eps / cosv;
    const double sa = b1 * p->ha, sb = b2 * p->hb, sc = (1.0 - b1 - b2) * p->hc;
    if (sa < -m || sb < -m || sc < -m) return MISS;
    if (sa <= m || sb <= m || sc <= m || cosv < 1e-3) amb = 1;
    const double u = eps / (dl * cosv);
    const int w = window(t, u + 1e-5 * fabs(t), tmin, tmax);
    if (w == -1 || w == 2) return MISS;
    if (w == 1) amb = 1;
    *t_out = t; *u_out = u;
    return amb ? AMB : HIT;
}

static int classify_sphere(const BPrim *p, const double *o, const double *d, double dl, double eps_in, double tmin, double tmax,
                           double *t_out, double *u_out, double *eps_out)
{
    double oc[3], perp[3];
    for (int k = 0; k < 3; k++) oc[k] = o[k] - p->c[k];
    const double eps = eps_in + K_AR * ldexp(1.0, -24) * (sqrt(dot3(oc, oc)) + 2.0 * p->size);
    *eps_out = eps;
    const double hb = dot3(oc, d), cc = dot3(oc, oc) - p->r * p->r;
    const double dl2 = dl * dl;
    for (int k = 0; k < 3; k++) perp[k] = oc[k] - d[k] * (hb / dl2);
    const double h = sqrt(dot3(perp, perp));
    if (h >= p->r + eps) return MISS;
    const double disc = hb * hb - cc;
    const double root = sqrt(fmax(disc, 0.0));
    const double q = (hb < 0.0) ? -(hb - root) : -(hb + root);
    const double t1 = (q != 0.0) ? cc / q : q;
    const double lo = fmin(q, t1), hi = fmax(q, t1);
    const double cosv = root / (p->r * dl);
    const double u = eps / (dl * fmax(cosv, 1e-300));
    if (h > p->r - eps) {                                   /* grazes the silhouette */
        if (hi + u + 1e-5 * fabs(hi) <= tmin || lo - u - 1e-5 * fabs(lo) >= tmax) return MISS;
        *t_out = fmax(lo, tmin); *u_out = u;
        return AMB;
    }
    const int wl = window(lo, u + 1e-5 * fabs(lo), tmin, tmax);
    *u_out = u;
    if (wl == 0) { *t_out = lo; return HIT; }
    if (wl == 1) { *t_out = lo; return AMB; }
    if (wl == 2) return MISS;
    const int wh = window(hi, u + 1e-5 * fabs(hi), tmin, tmax);
    if (wh == 0) { *t_out = hi; return HIT; }
    if (wh == 1) { *t_out = hi; return AMB; }
    return MISS;
}

/* a sphere the ray starts on (SOURCE RULES in the header); eps_o = K_IN 2^-24 |o|_inf, the rounding of o alone */
static int classify_src_sphere(const BPrim *p, const double *o, const double *d, double dl, double eps_in, double eps_o,
                               double tmin, double tmax, double *t_out, double *u_out, double *eps_out)
{
    double oc[3];
    for (int k = 0; k < 3; k++) oc[k] = o[k] - p->c[k];
    const double oc2 = dot3(oc, oc), ocl = sqrt(oc2);
    const double eps = eps_in + K_AR * ldexp(1.0, -24) * (ocl + 2.0 * p->size);
    *eps_out = eps;
    const double cmax = fmax(fabs(p->c[0]), fmax(fabs(p->c[1]), fabs(p->c[2])));
    const double eps_h = eps_o + K_AR * ldexp(1.0, -24) * ocl + (p->r >= 32.0 ? 0.0 : K_IN * ldexp(1.0, -24) * cmax);
    const double hb = dot3(oc, d);
    if (hb >= eps_h) return MISS;                                           /* leaving */
    if (hb > -eps_h) { *t_out = tmin; *u_out = 0.0; return AMB; }           /* along the tangent plane */
    const double cc = oc2 - p->r * p->r, disc = hb * hb - cc;
    double t, cosv;
    if (disc <= 4.0 * ldexp(1.0, -52) * (hb * hb + oc2 + p->r * p->r)) { t = -2.0 * hb; cosv = -hb / (p->r * dl); }
    else {
        const double root = sqrt(disc), q = root - hb;                      /* hb < 0: q is the far root */
        t = fmax(q, cc / q);
        cosv = root / (p->r * dl);
    }
    const double u = eps / (dl * cosv);
    const double lo = fmax(t - u, -hb - eps_h), hi = fmin(t + u, 2.0 * (eps_h - hb) + sqrt(4.0 * p->r * eps_h));
    const double tc = 0.5 * (lo + hi), uc = 0.5 * (hi - lo);
    *t_out = tc; *u_out = uc;
    const int w = window(tc, uc + 1e-5 * tc, tmin, tmax);
    if (w == -1 || w == 2) return MISS;
    return w == 1 ? AMB : HIT;
}

static void classify_ray(Job *J, int i, Cand **buf, int *cap)
{
    double d[3] = { J->d[3 * i], J->d[3 * i + 1], J->d[3 * i + 2] };
    const double *o = J->o + 3 * i;
    double dl = sqrt(dot3(d, d));
    if (J->normalize) { for (int k = 0; k < 3; k++) d[k] /= dl; dl = sqrt(dot3(d, d)); }
    const double omax = fmax(fabs(o[0]), fmax(fabs(o[1]), fabs(o[2])));
    const double eps_in = K_IN * ldexp(1.0, -24) * (J->max_abs + omax), eps_o = K_IN * ldexp(1.0, -24) * omax;
    const int src = J->src ? J->src[i] : -1;
    int nc = 0, namb = 0, any_clear = 0;
    int wp = -1, ws = 0; double wt = INFINITY, wu = 0.0, weps = eps_in;
    for (int j = 0; j < J->np; j++) {
        const BPrim *p = J->p + j;
        double t = 0.0, u = 0.0, eps = 0.0;
        int c;
        if (p->prim == src) c = p->sphere ? classify_src_sphere(p, o, d, dl, eps_in, eps_o, J->tmin, J->tmax, &t, &u, &eps) : MISS;
        else c = p->sphere ? classify_sphere(p, o, d, dl, eps_in, J->tmin, J->tmax, &t, &u, &eps)
                           : classify_tri(p, o, d, dl, eps_in, J->tmin, J->tmax, &t, &u, &eps);
        if (c == MISS) continue;
        if (c == AMB) namb++;
        else {
            any_clear = 1;
            if (t < wt) { wt = t; wu = u; wp = p->prim; ws = p->sub; weps = eps; }
        }
        if (nc == *cap) { *cap = *cap ? 2 * *cap : 64; *buf = (Cand *)realloc(*buf, (size_t)*cap * sizeof(Cand)); }
        (*buf)[nc].t = t; (*buf)[nc].u = u; nc++;
    }
    J->n_amb[i] = namb;
    J->eps[i] = weps;
    J->prim[i] = -1; J->sub[i] = 0; J->t[i] = 0.0; J->terr[i] = 0.0;
    if (J->any_hit) {
        J->robust[i] = (any_clear || nc == 0) ? 1 : 0;
        J->prim[i] = any_clear ? 0 : -1;
        return;
    }
    if (nc == 0) { J->robust[i] = 1; return; }
    if (wp < 0) { J->robust[i] = 0; return; }
    int robust = 1, seen_w = 0;
    for (int k = 0; k < nc && robust; k++) {
        const Cand *c = *buf + k;
        if (!seen_w && c->t == wt && c->u == wu) { seen_w = 1; continue; }          /* the winner itself */
        if (c->t < wt + 1e-4 * wt + wu + c->u) robust = 0;
    }
    J->robust[i] = (int8_t)robust;
    J->prim[i] = wp; J->sub[i] = ws; J->t[i] = wt;
    J->terr[i] = 1e-5 * wt + 4.0 * wu;
}

static void *worker(void *arg)
{
    Job *J = (Job *)arg;
    Cand *buf = NULL; int cap = 0;
    for (;;) {
        pthread_mutex_lock(&J->mu);
        const int i0 = J->next; J->next += 256;
        pthread_mutex_unlock(&J->mu);
        if (i0 >= J->n) break;
        const int i1 = i0 + 256 < J->n ? i0 + 256 : J->n;
        for (int i = i0; i < i1; i++) classify_ray(J, i, &buf, &cap);
    }
    free(buf);
    return NULL;
}

static void set_tri(BPrim *b, const double *a, const double *p1, const double *p2)
{
    double n[3], e21[3];
    for (int k = 0; k < 3; k++) { b->v0[k] = a[k]; b->e1[k] = p1[k] - a[k]; b->e2[k] = p2[k] - a[k]; }
    cross3(b->e1, b->e2, n);
    for (int k = 0; k < 3; k++) e21[k] = b->e2[k] - b->e1[k];
    b->nl = sqrt(dot3(n, n));
    b->size = sqrt(dot3(b->e1, b->e1)) + sqrt(dot3(b->e2, b->e2));
    b->ha = b->nl / sqrt(dot3(b->e2, b->e2));
    b->hb = b->nl / sqrt(dot3(b->e1, b->e1));
    b->hc = b->nl / sqrt(dot3(e21, e21));
}

/* kind[i]: 0 triangle, 1 Rect, 2 sphere; v: 12 doubles per primitive (the MfxPrim layout).  tmin / tmax: the query's
 * window; any_hit selects the query; normalize: divide each direction by its length first (the sphere sample's Ray).
 * Out per ray: robust flag, expected (prim, sub, t) -- prim >= 0 means occluded for an any-hit query -- the allowed
 * |t_f32 - t| of a robust closest hit, eps of the nearest clear hit (of a ray without one: its first term) and the
 * number of ambiguous pairs.  src: per ray, the caller's index of the primitive it starts on or -1 (NULL: -1 for every
 * ray); indices outside [0, n_prims) match no primitive.  Returns max_abs. */
double brute_classify_from(int n_prims, const int32_t *kind, const double *v, int n, const double *o, const double *d,
                           const int32_t *src, double tmin, double tmax, int any_hit, int normalize, int threads,
                           int8_t *robust, int32_t *prim, int32_t *sub, double *t, double *terr, double *eps, int32_t *n_amb)
{
    BPrim *P = (BPrim *)calloc((size_t)2 * n_prims + 1, sizeof(BPrim));
    int np = 0;
    double max_abs = 0.0;
    for (int i = 0; i < n_prims; i++) {
        const double *q = v + 12 * i;
        if (kind[i] == 2) {
            BPrim *b = P + np++;
            b->prim = i; b->sub = 0; b->sphere = 1;
            memcpy(b->c, q, 3 * sizeof(double)); b->r = b->size = fabs(q[3]);
            for (int k = 0; k < 3; k++) max_abs = fmax(max_abs, fabs(q[k]) + b->r);
            continue;
        }
        const int nt = kind[i] == 1 ? 2 : 1;
        for (int s = 0; s < nt; s++) {
            BPrim *b = P + np++;
            b->prim = i; b->sub = s; b->sphere = 0;
            set_tri(b, q, q + 3 * (1 + s), q + 3 * (2 + s));
        }
        for (int k = 0; k < 3 * (nt + 2); k++) max_abs = fmax(max_abs, fabs(q[k]));
    }
    Job J;
    memset(&J, 0, sizeof(J));
    J.p = P; J.np = np; J.o = o; J.d = d; J.n = n; J.tmin = tmin; J.tmax = tmax; J.max_abs = max_abs;
    J.any_hit = any_hit; J.normalize = normalize; J.src = src;
    J.robust = robust; J.prim = prim; J.sub = sub; J.t = t; J.terr = terr; J.eps = eps; J.n_amb = n_amb;
    pthread_mutex_init(&J.mu, NULL);
    if (threads < 1) threads = 1;
    pthread_t *th = (pthread_t *)malloc((size_t)threads * sizeof(pthread_t));
    for (int k = 0; k < threads; k++) pthread_create(th + k, NULL, worker, &J);
    for (int k = 0; k < threads; k++) pthread_join(th[k], NULL);
    free(th);
    pthread_mutex_destroy(&J.mu);
    free(P);
    return max_abs;
}

/* the rays of brute_classify_from without a source primitive */
double brute_classify(int n_prims, const int32_t *kind, const double *v, int n, const double *o, const double *d,
                      double tmin, double tmax, int any_hit, int normalize, int threads,
                      int8_t *robust, int32_t *prim, int32_t *sub, double *t, double *terr, double *eps, int32_t *n_amb)
{
    return brute_classify_from(n_prims, kind, v, n, o, d, NULL, tmin, tmax, any_hit, normalize, threads,
                               robust, prim, sub, t, terr, eps, n_amb);
}
