// Eval geometry metrics (the igl half of the reference's _scripts/eval/measure.py:141-201) on the device:
// area-weighted surface sampling, an LBVH over the faces and exact point-to-mesh distances, all in float64.
// The contract is written out in oracle/metrics3d_oracle.py; every operation below is rounded separately
// (__d*_rn, no FMA contraction) so the oracle's numpy float64 gives the same bits.
//
//   sample: k_pm_area     |cross(b-a, c-a)| per face
//           cub::DeviceReduce::Max -> k_pm_weights  floor(area / max * 2^32) as uint64
//           cub::DeviceScan::InclusiveSum (exact: integers) -> k_pm_sample  face by upper_bound, point by bary2cart order
//   build:  k_pm_bounds   centroid bounding box (order-preserving uint64 atomics: exact, so run-to-run identical)
//           k_pm_morton   key = morton30(centroid) << 32 | face   (all keys distinct)
//           cub::DeviceRadixSort::SortKeys
//           k_pm_topology Karras (2012), one thread per internal node
//           k_pm_refit    one thread per leaf, the second arrival at a node unions its children (min / max: exact)
//   query:  k_pm_query    one thread per point, nearest child first, explicit 64-entry stack of far children
// No kernel needs a host synchronisation; failures that only the device can see are OR-ed into a status word.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_reduce.cuh>
#include <cub/device/device_scan.cuh>

#include "p3d_common.cuh"
#include "../../include/p3d_geom.h"

namespace p3d {
namespace {

constexpr int NT = 256;
constexpr int STACK = 64;                 // distinct 64-bit keys: at most 64 internal levels, only far children pushed
constexpr double PRUNE_MARGIN = 1.0 + 0x1p-40;

// ---------------------------------------------------------------- fp64 vector ops, each rounded separately
struct D3 {
    double x, y, z;
};
__device__ __forceinline__ D3 ld3(const double* __restrict__ p, long long i) {
    return D3{__ldg(p + 3 * i), __ldg(p + 3 * i + 1), __ldg(p + 3 * i + 2)};
}
__device__ __forceinline__ D3 sub(D3 a, D3 b) { return D3{__dsub_rn(a.x, b.x), __dsub_rn(a.y, b.y), __dsub_rn(a.z, b.z)}; }
__device__ __forceinline__ double dot(D3 a, D3 b) {
    return __dadd_rn(__dadd_rn(__dmul_rn(a.x, b.x), __dmul_rn(a.y, b.y)), __dmul_rn(a.z, b.z));
}
__device__ __forceinline__ D3 axpy(D3 a, double t, D3 u) {          // a + t*u
    return D3{__dadd_rn(a.x, __dmul_rn(t, u.x)), __dadd_rn(a.y, __dmul_rn(t, u.y)), __dadd_rn(a.z, __dmul_rn(t, u.z))};
}

// closest point on segment a-b (a when the projection is <= 0, b when it is >= |ab|^2)
__device__ __forceinline__ D3 closest_on_segment(D3 p, D3 a, D3 b) {
    const D3 ab = sub(b, a);
    const double t = dot(sub(p, a), ab), den = dot(ab, ab);
    if (!(t > 0.0)) return a;
    if (t >= den) return b;
    return axpy(a, __ddiv_rn(t, den), ab);
}

// Ericson, Real-Time Collision Detection 5.1.5.  Returns false on a zero denominator (degenerate face).
__device__ __forceinline__ bool closest_ericson(D3 p, D3 a, D3 b, D3 c, D3& q) {
    const D3 ab = sub(b, a), ac = sub(c, a), ap = sub(p, a);
    const double d1 = dot(ab, ap), d2 = dot(ac, ap);
    if (d1 <= 0.0 && d2 <= 0.0) { q = a; return true; }
    const D3 bp = sub(p, b);
    const double d3 = dot(ab, bp), d4 = dot(ac, bp);
    if (d3 >= 0.0 && d4 <= d3) { q = b; return true; }
    const double vc = __dsub_rn(__dmul_rn(d1, d4), __dmul_rn(d3, d2));
    if (vc <= 0.0 && d1 >= 0.0 && d3 <= 0.0) {
        const double den = __dsub_rn(d1, d3);
        if (den == 0.0) return false;
        q = axpy(a, __ddiv_rn(d1, den), ab);
        return true;
    }
    const D3 cp = sub(p, c);
    const double d5 = dot(ab, cp), d6 = dot(ac, cp);
    if (d6 >= 0.0 && d5 <= d6) { q = c; return true; }
    const double vb = __dsub_rn(__dmul_rn(d5, d2), __dmul_rn(d1, d6));
    if (vb <= 0.0 && d2 >= 0.0 && d6 <= 0.0) {
        const double den = __dsub_rn(d2, d6);
        if (den == 0.0) return false;
        q = axpy(a, __ddiv_rn(d2, den), ac);
        return true;
    }
    const double va = __dsub_rn(__dmul_rn(d3, d6), __dmul_rn(d5, d4));
    const double e43 = __dsub_rn(d4, d3), e56 = __dsub_rn(d5, d6);
    if (va <= 0.0 && e43 >= 0.0 && e56 >= 0.0) {
        const double den = __dadd_rn(e43, e56);
        if (den == 0.0) return false;
        q = axpy(b, __ddiv_rn(e43, den), sub(c, b));
        return true;
    }
    const double sum = __dadd_rn(__dadd_rn(va, vb), vc);
    if (sum == 0.0) return false;
    const double inv = __ddiv_rn(1.0, sum), v = __dmul_rn(vb, inv), w = __dmul_rn(vc, inv);
    q = axpy(axpy(a, v, ab), w, ac);
    return true;
}

__device__ __forceinline__ double dist2(D3 p, D3 q) {
    const D3 d = sub(p, q);
    return dot(d, d);
}

// The closest point of face (a, b, c) to p, clamped into the face's bounding box (so it lies inside every box that
// holds the face: the BVH's lower bounds stay valid for the computed point), and its squared distance.
__device__ __forceinline__ double closest_on_triangle(D3 p, D3 a, D3 b, D3 c, D3& q) {
    if (!closest_ericson(p, a, b, c, q)) {          // degenerate: nearest of the edges ab, bc, ca (first on ties)
        q = closest_on_segment(p, a, b);
        double best = dist2(p, q);
        const D3 q1 = closest_on_segment(p, b, c);
        const double e1 = dist2(p, q1);
        if (e1 < best) { best = e1; q = q1; }
        const D3 q2 = closest_on_segment(p, c, a);
        if (dist2(p, q2) < best) q = q2;
    }
    q.x = fmin(fmax(q.x, fmin(fmin(a.x, b.x), c.x)), fmax(fmax(a.x, b.x), c.x));
    q.y = fmin(fmax(q.y, fmin(fmin(a.y, b.y), c.y)), fmax(fmax(a.y, b.y), c.y));
    q.z = fmin(fmax(q.z, fmin(fmin(a.z, b.z), c.z)), fmax(fmax(a.z, b.z), c.z));
    return dist2(p, q);
}

__device__ __forceinline__ void load_face(const double* __restrict__ v, const int32_t* __restrict__ f, long long i, D3& a, D3& b, D3& c) {
    a = ld3(v, __ldg(f + 3 * i));
    b = ld3(v, __ldg(f + 3 * i + 1));
    c = ld3(v, __ldg(f + 3 * i + 2));
}

// ---------------------------------------------------------------- sampler
__global__ void __launch_bounds__(NT) k_pm_area(const double* __restrict__ v, const int32_t* __restrict__ f, long long nf,
                                                double* __restrict__ area) {
    const long long i = (long long)blockIdx.x * NT + threadIdx.x;
    if (i >= nf) return;
    D3 a, b, c;
    load_face(v, f, i, a, b, c);
    const D3 u = sub(b, a), w = sub(c, a);
    const D3 x{__dsub_rn(__dmul_rn(u.y, w.z), __dmul_rn(u.z, w.y)), __dsub_rn(__dmul_rn(u.z, w.x), __dmul_rn(u.x, w.z)),
               __dsub_rn(__dmul_rn(u.x, w.y), __dmul_rn(u.y, w.x))};
    area[i] = __dsqrt_rn(dot(x, x));
}

__global__ void __launch_bounds__(NT) k_pm_weights(const double* __restrict__ area, const double* __restrict__ amax, long long nf,
                                                   unsigned long long* __restrict__ w) {
    const long long i = (long long)blockIdx.x * NT + threadIdx.x;
    if (i >= nf) return;
    const double m = *amax;
    // area <= max, so the quotient is in [0, 1] and the weight in [0, 2^32]; the scale by 2^32 is exact
    w[i] = m > 0.0 ? __double2ull_rz(__dmul_rn(__ddiv_rn(area[i], m), 4294967296.0)) : 0ull;
}

__global__ void __launch_bounds__(NT) k_pm_sample(const double* __restrict__ v, const int32_t* __restrict__ f, long long nf,
                                                  const unsigned long long* __restrict__ cdf, long long n, uint64_t seed, unsigned sid,
                                                  const unsigned long long* __restrict__ face_bits, const double* __restrict__ bary_u,
                                                  double* __restrict__ bary, int64_t* __restrict__ face, double* __restrict__ pts,
                                                  int* __restrict__ status) {
    const long long i = (long long)blockIdx.x * NT + threadIdx.x;
    if (i >= n) return;
    const unsigned long long total = cdf[nf - 1];
    if (total == 0) {                               // every face has zero area
        if (i == 0) atomicOr(status, P3D_GEOM_ZERO_AREA);
        face[i] = -1;
        for (int k = 0; k < 3; ++k) {
            bary[3 * i + k] = __longlong_as_double(0x7ff8000000000000ll);
            if (pts) pts[3 * i + k] = __longlong_as_double(0x7ff8000000000000ll);
        }
        return;
    }
    unsigned long long k;
    double a, b;
    if (face_bits) {
        k = face_bits[i];
        a = bary_u[2 * i];
        b = bary_u[2 * i + 1];
    } else {
        const Philox4 r = philox4x32_10(seed, (uint64_t)i, sid);
        k = ((unsigned long long)r.x << 32) | r.y;
        a = (double)r.z * 0x1p-32;
        b = (double)r.w * 0x1p-32;
    }
    const unsigned long long t = __umul64hi(k, total);            // in [0, total)
    long long lo = 0, hi = nf;                                       // first face with cdf > t
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (__ldg(cdf + mid) > t) hi = mid; else lo = mid + 1;
    }
    if (__dadd_rn(a, b) > 1.0) { a = __dsub_rn(1.0, a); b = __dsub_rn(1.0, b); }
    const double b0 = __dsub_rn(__dsub_rn(1.0, a), b);
    face[i] = lo;
    bary[3 * i] = b0; bary[3 * i + 1] = a; bary[3 * i + 2] = b;
    if (pts) {
        D3 p0, p1, p2;
        load_face(v, f, lo, p0, p1, p2);
        pts[3 * i] = __dadd_rn(__dadd_rn(__dmul_rn(p0.x, b0), __dmul_rn(p1.x, a)), __dmul_rn(p2.x, b));
        pts[3 * i + 1] = __dadd_rn(__dadd_rn(__dmul_rn(p0.y, b0), __dmul_rn(p1.y, a)), __dmul_rn(p2.y, b));
        pts[3 * i + 2] = __dadd_rn(__dadd_rn(__dmul_rn(p0.z, b0), __dmul_rn(p1.z, a)), __dmul_rn(p2.z, b));
    }
}

// ---------------------------------------------------------------- BVH
// Internal node: both children's boxes (fp32, rounded outward from the fp64 geometry) and ids: an internal child is its
// index >= 0, a leaf child is ~face.  64 bytes, read as four 16-byte loads.
struct __align__(16) Node {
    float box[2][6];          // lo xyz, hi xyz per child
    int child[2];
    int pad[2];
};
static_assert(sizeof(Node) == 64, "Node layout");

__device__ __forceinline__ unsigned long long dbl_to_ordered(double d) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(d);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
__device__ __forceinline__ double ordered_to_dbl(unsigned long long u) {
    return __longlong_as_double((long long)((u >> 63) ? (u & 0x7fffffffffffffffull) : ~u));
}

__device__ __forceinline__ D3 centroid(D3 a, D3 b, D3 c) {
    return D3{__ddiv_rn(__dadd_rn(__dadd_rn(a.x, b.x), c.x), 3.0), __ddiv_rn(__dadd_rn(__dadd_rn(a.y, b.y), c.y), 3.0),
              __ddiv_rn(__dadd_rn(__dadd_rn(a.z, b.z), c.z), 3.0)};
}

// bounds[0..2] = ordered min, [3..5] = ordered max of the centroids (initialised to ~0 / 0)
__global__ void __launch_bounds__(NT) k_pm_bounds(const double* __restrict__ v, const int32_t* __restrict__ f, long long nf,
                                                  unsigned long long* __restrict__ bounds) {
    const long long i = (long long)blockIdx.x * NT + threadIdx.x;
    unsigned long long m[6] = {~0ull, ~0ull, ~0ull, 0ull, 0ull, 0ull};
    if (i < nf) {
        D3 a, b, c;
        load_face(v, f, i, a, b, c);
        const D3 g = centroid(a, b, c);
        m[0] = m[3] = dbl_to_ordered(g.x);
        m[1] = m[4] = dbl_to_ordered(g.y);
        m[2] = m[5] = dbl_to_ordered(g.z);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            m[k] = min(m[k], __shfl_xor_sync(0xffffffffu, m[k], o));
            m[k + 3] = max(m[k + 3], __shfl_xor_sync(0xffffffffu, m[k + 3], o));
        }
    }
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            if (m[k] != ~0ull) atomicMin(bounds + k, m[k]);
            if (m[k + 3] != 0ull) atomicMax(bounds + k + 3, m[k + 3]);
        }
    }
}

__device__ __forceinline__ unsigned expand10(unsigned x) {          // 10 bits -> every third bit of 30
    x &= 0x3ffu;
    x = (x | (x << 16)) & 0x030000ffu;
    x = (x | (x << 8)) & 0x0300f00fu;
    x = (x | (x << 4)) & 0x030c30c3u;
    x = (x | (x << 2)) & 0x09249249u;
    return x;
}
__device__ __forceinline__ unsigned quant10(double c, double lo, double hi) {
    if (!(hi > lo)) return 0;
    const double t = (c - lo) / (hi - lo) * 1024.0;
    return t <= 0.0 ? 0u : t >= 1023.0 ? 1023u : (unsigned)t;
}

__global__ void __launch_bounds__(NT) k_pm_morton(const double* __restrict__ v, const int32_t* __restrict__ f, long long nf,
                                                  const unsigned long long* __restrict__ bounds, unsigned long long* __restrict__ keys) {
    const long long i = (long long)blockIdx.x * NT + threadIdx.x;
    if (i >= nf) return;
    D3 a, b, c;
    load_face(v, f, i, a, b, c);
    const D3 g = centroid(a, b, c);
    const unsigned m = (expand10(quant10(g.x, ordered_to_dbl(bounds[0]), ordered_to_dbl(bounds[3]))) << 2) |
                       (expand10(quant10(g.y, ordered_to_dbl(bounds[1]), ordered_to_dbl(bounds[4]))) << 1) |
                       expand10(quant10(g.z, ordered_to_dbl(bounds[2]), ordered_to_dbl(bounds[5])));
    keys[i] = ((unsigned long long)m << 32) | (unsigned long long)i;
}

__device__ __forceinline__ int common_prefix(const unsigned long long* __restrict__ k, long long n, long long i, long long j) {
    if (j < 0 || j >= n) return -1;
    return __clzll(k[i] ^ k[j]);                                       // keys are distinct: never 64
}

// Karras, "Maximizing parallelism in the construction of BVHs, octrees, and k-d trees" (HPG 2012), one thread per
// internal node i in [0, n-1): the range it covers, its split, and its two children.
__global__ void __launch_bounds__(NT) k_pm_topology(const unsigned long long* __restrict__ keys, long long n, Node* __restrict__ nodes,
                                                    int* __restrict__ parent_int, int* __restrict__ parent_leaf) {
    const long long i = (long long)blockIdx.x * NT + threadIdx.x;
    if (i >= n - 1) return;
    const int d = common_prefix(keys, n, i, i + 1) - common_prefix(keys, n, i, i - 1) >= 0 ? 1 : -1;
    const int dmin = common_prefix(keys, n, i, i - d);
    long long lmax = 2;
    while (common_prefix(keys, n, i, i + lmax * d) > dmin) lmax <<= 1;
    long long l = 0;
    for (long long t = lmax >> 1; t >= 1; t >>= 1)
        if (common_prefix(keys, n, i, i + (l + t) * d) > dmin) l += t;
    const long long j = i + l * d;
    const int dnode = common_prefix(keys, n, i, j);
    long long s = 0, t = l;
    do {
        t = (t + 1) >> 1;
        if (common_prefix(keys, n, i, i + (s + t) * d) > dnode) s += t;
    } while (t > 1);
    const long long gamma = i + s * d + min(d, 0);
    const long long lo = min(i, j), hi = max(i, j);
    int c0, c1;
    if (lo == gamma) { c0 = ~(int)(unsigned)keys[gamma]; parent_leaf[gamma] = (int)i; }
    else { c0 = (int)gamma; parent_int[gamma] = (int)i; }
    if (hi == gamma + 1) { c1 = ~(int)(unsigned)keys[gamma + 1]; parent_leaf[gamma + 1] = (int)i; }
    else { c1 = (int)(gamma + 1); parent_int[gamma + 1] = (int)i; }
    nodes[i].child[0] = c0;
    nodes[i].child[1] = c1;
}

__device__ __forceinline__ void put_box(Node* nd, int slot, const float b[6]) {
#pragma unroll
    for (int k = 0; k < 6; ++k) __stcg(&nd->box[slot][k], b[k]);
}

// One thread per leaf (sorted position k): write the face's box into its parent's slot, then climb.  The first thread to
// arrive at a node stops; the second (whose sibling's box is then complete: written and fenced before its atomic) unions
// both slots and carries on.  All node reads bypass L1 (__ldcg) so a sibling's box is never read stale.
__global__ void __launch_bounds__(NT) k_pm_refit(const double* __restrict__ v, const int32_t* __restrict__ f, long long n,
                                                 const unsigned long long* __restrict__ keys, Node* __restrict__ nodes,
                                                 const int* __restrict__ parent_int, const int* __restrict__ parent_leaf,
                                                 int* __restrict__ arrivals) {
    const long long k = (long long)blockIdx.x * NT + threadIdx.x;
    if (k >= n) return;
    const int face = (int)(unsigned)keys[k];
    D3 a, b, c;
    load_face(v, f, face, a, b, c);
    float box[6] = {__double2float_rd(fmin(fmin(a.x, b.x), c.x)), __double2float_rd(fmin(fmin(a.y, b.y), c.y)),
                    __double2float_rd(fmin(fmin(a.z, b.z), c.z)), __double2float_ru(fmax(fmax(a.x, b.x), c.x)),
                    __double2float_ru(fmax(fmax(a.y, b.y), c.y)), __double2float_ru(fmax(fmax(a.z, b.z), c.z))};
    int me = ~face;
    int p = parent_leaf[k];
    while (true) {
        Node* nd = nodes + p;
        const int slot = __ldcg(&nd->child[0]) == me ? 0 : 1;
        put_box(nd, slot, box);
        __threadfence();
        if (atomicAdd(arrivals + p, 1) == 0) return;
        __threadfence();
#pragma unroll
        for (int q = 0; q < 3; ++q) {
            box[q] = fminf(__ldcg(&nd->box[0][q]), __ldcg(&nd->box[1][q]));
            box[q + 3] = fmaxf(__ldcg(&nd->box[0][q + 3]), __ldcg(&nd->box[1][q + 3]));
        }
        if (p == 0) return;
        me = p;
        p = parent_int[p];
    }
}

// squared distance from p to the box (lo, hi), every step rounded down: a lower bound of the true squared distance
__device__ __forceinline__ double box_lower_bound(D3 p, float lx, float ly, float lz, float hx, float hy, float hz) {
    const double lo[3] = {lx, ly, lz}, hi[3] = {hx, hy, hz}, q[3] = {p.x, p.y, p.z};
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double g = q[k] < lo[k] ? __dsub_rd(lo[k], q[k]) : q[k] > hi[k] ? __dsub_rd(q[k], hi[k]) : 0.0;
        s = __dadd_rd(s, __dmul_rd(g, g));
    }
    return s;
}

struct Best {
    double d2;
    int face;
    D3 q;
};

__device__ __forceinline__ void test_face(D3 p, const double* __restrict__ v, const int32_t* __restrict__ f, int face, Best& best) {
    D3 a, b, c, q;
    load_face(v, f, face, a, b, c);
    const double d2 = closest_on_triangle(p, a, b, c, q);
    if (d2 < best.d2 || (d2 == best.d2 && face < best.face)) { best.d2 = d2; best.face = face; best.q = q; }
}

// A node is pruned only when its lower bound exceeds best * (1 + 2^-40) (rounded up): the closest point of every face
// lies in the face's box, so its computed squared distance is at least (1 - 2^-53)^5 times the box's lower bound, i.e.
// strictly more than the best so far - no face that exhaustive search would pick (ties included) is ever skipped.
__global__ void __launch_bounds__(NT) k_pm_query(const double* __restrict__ pts, long long np, const double* __restrict__ v,
                                                 const int32_t* __restrict__ f, long long nf, const Node* __restrict__ nodes,
                                                 double* __restrict__ out_d2, int64_t* __restrict__ out_face,
                                                 double* __restrict__ out_q, int* __restrict__ status) {
    const long long i = (long long)blockIdx.x * NT + threadIdx.x;
    if (i >= np) return;
    const D3 p = ld3(pts, i);
    Best best{__longlong_as_double(0x7ff0000000000000ll), 0x7fffffff, D3{0.0, 0.0, 0.0}};
    bool overflow = false;
    if (nf == 1) {
        test_face(p, v, f, 0, best);
    } else {
        unsigned long long stack[STACK];          // (float lower bound, rounded down) << 32 | node
        int sp = 0, node = 0;
        while (true) {
            const float4* nd = reinterpret_cast<const float4*>(nodes + node);
            const float4 r0 = __ldg(nd), r1 = __ldg(nd + 1), r2 = __ldg(nd + 2), r3 = __ldg(nd + 3);
            const int c0 = __float_as_int(r3.x), c1 = __float_as_int(r3.y);
            const double l0 = box_lower_bound(p, r0.x, r0.y, r0.z, r0.w, r1.x, r1.y);
            const double l1 = box_lower_bound(p, r1.z, r1.w, r2.x, r2.y, r2.z, r2.w);
            const double thr = __dmul_ru(best.d2, PRUNE_MARGIN);
            bool go0 = l0 <= thr, go1 = l1 <= thr;
            if (go0 && c0 < 0) { test_face(p, v, f, ~c0, best); go0 = false; }
            if (go1 && c1 < 0) { test_face(p, v, f, ~c1, best); go1 = false; }
            if (go0 && go1) {
                const bool first0 = l0 <= l1;
                if (sp == STACK) { overflow = true; break; }
                const double lf = first0 ? l1 : l0;
                stack[sp++] = ((unsigned long long)__float_as_uint(__double2float_rd(lf)) << 32) | (unsigned)(first0 ? c1 : c0);
                node = first0 ? c0 : c1;
                continue;
            }
            if (go0) { node = c0; continue; }
            if (go1) { node = c1; continue; }
            const double t = __dmul_ru(best.d2, PRUNE_MARGIN);
            node = -1;
            while (sp > 0) {
                const unsigned long long e = stack[--sp];
                if ((double)__uint_as_float((unsigned)(e >> 32)) <= t) { node = (int)(unsigned)e; break; }
            }
            if (node < 0) break;
        }
    }
    if (overflow) atomicOr(status, P3D_GEOM_STACK_OVERFLOW);
    out_d2[i] = best.d2;
    out_face[i] = best.face == 0x7fffffff ? -1 : best.face;
    if (out_q) { out_q[3 * i] = best.q.x; out_q[3 * i + 1] = best.q.y; out_q[3 * i + 2] = best.q.z; }
}

// ---------------------------------------------------------------- host
size_t take(size_t& o, size_t bytes) {
    const size_t at = o;
    o = (o + bytes + 255) & ~(size_t)255;
    return at;
}

struct SampleLayout {
    size_t area, amax, w, cdf, temp, temp_bytes, total;
};
int sample_layout(long long nf, SampleLayout* L) {
    P3D_REQUIRE(nf >= 1 && nf < (1ll << 31), "p3d_surface_sample: n_faces must be in [1, 2^31) (got %lld)", nf);
    size_t o = 0, tr = 0, ts = 0;
    L->area = take(o, 8ull * nf);
    L->amax = take(o, 8);
    L->w = take(o, 8ull * nf);
    L->cdf = take(o, 8ull * nf);
    P3D_CUDA_TRY(cub::DeviceReduce::Max(nullptr, tr, (const double*)nullptr, (double*)nullptr, (int)nf));
    P3D_CUDA_TRY(cub::DeviceScan::InclusiveSum(nullptr, ts, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, (int)nf));
    L->temp_bytes = tr > ts ? tr : ts;
    L->temp = take(o, L->temp_bytes);
    L->total = o;
    return P3D_OK;
}

struct BvhLayout {
    size_t keys_in, keys, nodes, parent_int, parent_leaf, arrivals, bounds, temp, temp_bytes, total;
};
int bvh_layout(long long nf, BvhLayout* L) {
    P3D_REQUIRE(nf >= 1 && nf < (1ll << 31), "p3d_bvh: n_faces must be in [1, 2^31) (got %lld)", nf);
    size_t o = 0;
    const long long ni = nf > 1 ? nf - 1 : 1;
    L->keys_in = take(o, 8ull * nf);
    L->keys = take(o, 8ull * nf);
    L->nodes = take(o, sizeof(Node) * ni);
    L->parent_int = take(o, 4ull * ni);
    L->parent_leaf = take(o, 4ull * nf);
    L->arrivals = take(o, 4ull * ni);
    L->bounds = take(o, 6 * 8);
    L->temp_bytes = 0;
    P3D_CUDA_TRY(cub::DeviceRadixSort::SortKeys(nullptr, L->temp_bytes, (const unsigned long long*)nullptr, (unsigned long long*)nullptr, (int)nf));
    L->temp = take(o, L->temp_bytes);
    L->total = o;
    return P3D_OK;
}

int check_ws(const void* ws, size_t have, size_t need, const char* who) {
    P3D_REQUIRE(ws != nullptr && ((uintptr_t)ws & 255) == 0, "%s: workspace must be a 256-byte aligned device pointer", who);
    P3D_REQUIRE(have >= need, "%s: workspace of %zu bytes, %zu needed", who, have, need);
    return P3D_OK;
}

unsigned blocks(long long n) { return (unsigned)((n + NT - 1) / NT); }

}  // namespace
}  // namespace p3d

using namespace p3d;

extern "C" size_t p3d_surface_sample_workspace_bytes(int64_t n_faces) {
    SampleLayout L;
    return sample_layout(n_faces, &L) ? 0 : L.total;
}

extern "C" int p3d_surface_sample(const double* verts, const int32_t* faces, int64_t n_faces, int64_t n_samples, uint64_t seed,
                                  uint32_t stream_id, const uint64_t* face_bits, const double* bary_u, void* workspace,
                                  size_t workspace_bytes, double* bary, int64_t* face, double* points, int32_t* status, void* stream) {
    SampleLayout L;
    if (int rc = sample_layout(n_faces, &L)) return rc;
    P3D_REQUIRE(n_samples >= 0, "p3d_surface_sample: n_samples < 0");
    P3D_REQUIRE(verts && faces && bary && face && status, "p3d_surface_sample: NULL pointer");
    P3D_REQUIRE(!face_bits == !bary_u, "p3d_surface_sample: face_bits and bary_u are injected together");
    if (int rc = check_ws(workspace, workspace_bytes, L.total, "p3d_surface_sample")) return rc;
    if (n_samples == 0) return P3D_OK;
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    double *area = (double*)(ws + L.area), *amax = (double*)(ws + L.amax);
    unsigned long long *w = (unsigned long long*)(ws + L.w), *cdf = (unsigned long long*)(ws + L.cdf);
    k_pm_area<<<blocks(n_faces), NT, 0, st>>>(verts, faces, n_faces, area);
    P3D_LAUNCH_CHECK();
    size_t tb = L.temp_bytes;
    P3D_CUDA_TRY(cub::DeviceReduce::Max(ws + L.temp, tb, area, amax, (int)n_faces, st));
    count_launch();
    k_pm_weights<<<blocks(n_faces), NT, 0, st>>>(area, amax, n_faces, w);
    P3D_LAUNCH_CHECK();
    tb = L.temp_bytes;
    P3D_CUDA_TRY(cub::DeviceScan::InclusiveSum(ws + L.temp, tb, w, cdf, (int)n_faces, st));
    count_launch();
    k_pm_sample<<<blocks(n_samples), NT, 0, st>>>(verts, faces, n_faces, cdf, n_samples, seed, stream_id,
                                                  (const unsigned long long*)face_bits, bary_u, bary, face, points, status);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

extern "C" size_t p3d_bvh_workspace_bytes(int64_t n_faces) {
    BvhLayout L;
    return bvh_layout(n_faces, &L) ? 0 : L.total;
}

extern "C" int p3d_bvh_build(const double* verts, const int32_t* faces, int64_t n_faces, void* workspace, size_t workspace_bytes,
                             void* stream) {
    BvhLayout L;
    if (int rc = bvh_layout(n_faces, &L)) return rc;
    P3D_REQUIRE(verts && faces, "p3d_bvh_build: NULL pointer");
    if (int rc = check_ws(workspace, workspace_bytes, L.total, "p3d_bvh_build")) return rc;
    if (n_faces == 1) return P3D_OK;                                  // the root is the leaf: nothing to build
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    unsigned long long *keys_in = (unsigned long long*)(ws + L.keys_in), *keys = (unsigned long long*)(ws + L.keys);
    unsigned long long* bounds = (unsigned long long*)(ws + L.bounds);
    Node* nodes = (Node*)(ws + L.nodes);
    int *parent_int = (int*)(ws + L.parent_int), *parent_leaf = (int*)(ws + L.parent_leaf), *arrivals = (int*)(ws + L.arrivals);
    P3D_CUDA_TRY(cudaMemsetAsync(bounds, 0xff, 3 * 8, st));
    P3D_CUDA_TRY(cudaMemsetAsync(bounds + 3, 0, 3 * 8, st));
    P3D_CUDA_TRY(cudaMemsetAsync(arrivals, 0, 4ull * (n_faces - 1), st));
    k_pm_bounds<<<blocks(n_faces), NT, 0, st>>>(verts, faces, n_faces, bounds);
    P3D_LAUNCH_CHECK();
    k_pm_morton<<<blocks(n_faces), NT, 0, st>>>(verts, faces, n_faces, bounds, keys_in);
    P3D_LAUNCH_CHECK();
    size_t tb = L.temp_bytes;
    P3D_CUDA_TRY(cub::DeviceRadixSort::SortKeys(ws + L.temp, tb, keys_in, keys, (int)n_faces, 0, 64, st));
    count_launch();
    k_pm_topology<<<blocks(n_faces - 1), NT, 0, st>>>(keys, n_faces, nodes, parent_int, parent_leaf);
    P3D_LAUNCH_CHECK();
    k_pm_refit<<<blocks(n_faces), NT, 0, st>>>(verts, faces, n_faces, keys, nodes, parent_int, parent_leaf, arrivals);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

extern "C" int p3d_point_mesh_distance(const double* points, int64_t n_points, const double* verts, const int32_t* faces,
                                       int64_t n_faces, const void* bvh_workspace, size_t workspace_bytes, double* dist2,
                                       int64_t* face, double* closest, int32_t* status, void* stream) {
    BvhLayout L;
    if (int rc = bvh_layout(n_faces, &L)) return rc;
    P3D_REQUIRE(n_points >= 0, "p3d_point_mesh_distance: n_points < 0");
    P3D_REQUIRE(points && verts && faces && dist2 && face && status, "p3d_point_mesh_distance: NULL pointer");
    if (int rc = check_ws(bvh_workspace, workspace_bytes, L.total, "p3d_point_mesh_distance")) return rc;
    if (n_points == 0) return P3D_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const Node* nodes = (const Node*)((const char*)bvh_workspace + L.nodes);
    k_pm_query<<<blocks(n_points), NT, 0, st>>>(points, n_points, verts, faces, n_faces, nodes, dist2, face, closest, status);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}
