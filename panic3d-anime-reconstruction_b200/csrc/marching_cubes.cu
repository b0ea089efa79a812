// Marching cubes (SURVEY 8f-2, after the volume query): the configuration the reference hard-codes in
// _util/eg3d_metrics3d.py:186-210 (skimage 'lewiner', spacing 1, 'descent', allow_degenerate=False) on the device.
// The contract - vertex order, fp32 positions, the in-cell loop walk with the asymptotic decider, fan order,
// degenerate merging - is written out in oracle/mesh_oracle.py; the kernels below implement exactly that.
//
// Every pass is one thread per lattice corner; corner (i,j,k) owns the 3 edges leaving it towards +axis (edge key
// 3*lin + a, which is also the vertex order) and, when it is not on a far border, the cell whose lowest corner it is.
//   count:  k_mc_classify  min/max, crossing count, rep[corner] = lowest edge key whose vertex sits exactly on it
//           k_mc_cells     loop walk per cell; faces left after merging vertices onto rep; marks referenced vertices
//           k_mc_pack      (referenced vertices << 32 | kept faces) per corner -> one cub::DeviceScan -> totals
//   emit:   k_mc_verts     position / normal / value / colour of every referenced vertex at its scanned id
//           k_mc_faces     the loop walk again, faces written at their scanned offset
// No atomics decide any output position (only the min/max/count reductions use them), so the mesh is bit-identical
// run to run.  All of it is integer / compare work over a 67 MB volume that sits in L2: no tensor cores.
#include <cub/device/device_scan.cuh>

#include "p3d_common.cuh"
#include "../../include/p3d_mesh.h"

namespace p3d {
namespace {

constexpr int NT = 256;
constexpr unsigned NO_REP = 0xffffffffu;

// ---------------------------------------------------------------- cube geometry (folds to constants when unrolled)
// cell corner c = 4*d0 + 2*d1 + d2 (its offsets along axis 0, 1, 2): ascending c is ascending linear index
__host__ __device__ constexpr int off(int c, int a) { return (c >> (2 - a)) & 1; }
// local id of the edge leaving corner c along axis a (off(c, a) == 0): the 12 cell edges in ascending key order
__host__ __device__ constexpr int edge_id(int c, int a) {
    int n = 0;
    for (int c2 = 0; c2 < c; ++c2) n += 3 - off(c2, 0) - off(c2, 1) - off(c2, 2);
    for (int a2 = 0; a2 < a; ++a2) n += 1 - off(c, a2);
    return n;
}
// face f = 2*n + s (normal axis n, side s): corner q of the ring counter-clockwise about the outward normal
__host__ __device__ constexpr int ring_corner(int f, int q) {
    const int n = f >> 1, s = f & 1, up = (n + 1) % 3, wp = (n + 2) % 3;       // e_up x e_wp = e_n
    // s = 1: (u',w') = (1,0) (1,1) (0,1) (0,0); s = 0: the reverse turn, (0,0) (0,1) (1,1) (1,0)
    const int pu = s ? (q < 2) : (q >= 2), pw = (q == 1 || q == 2);
    return (s << (2 - n)) | (pu << (2 - up)) | (pw << (2 - wp));
}
// the edge from ring corner q to ring corner q+1
__host__ __device__ constexpr int ring_edge(int f, int q) {
    const int c0 = ring_corner(f, q), c1 = ring_corner(f, (q + 1) & 3), x = c0 ^ c1;
    return edge_id(c0 & c1, x == 4 ? 0 : x == 2 ? 1 : 2);
}
// corner q of the face in lattice order (a, b, c, d) = (u,w) offsets (0,0), (0,1), (1,0), (1,1), u < w
__host__ __device__ constexpr int lat_corner(int f, int q) {
    const int n = f >> 1, s = f & 1, u = n == 0 ? 1 : 0, w = n == 2 ? 1 : 2;
    return (s << (2 - n)) | ((q >> 1) << (2 - u)) | ((q & 1) << (2 - w));
}

struct Vol {
    const float* v;
    int d[3];
    unsigned s[3];       // element strides of the three axes
    unsigned n;          // d0*d1*d2 (3n < 2^31: checked on the host)
    float level;
};

__device__ __forceinline__ float edge_t(float lo, float hi, float level) {
    return __fdiv_rn(__fsub_rn(level, lo), __fsub_rn(hi, lo));
}
__device__ __forceinline__ void decompose(const Vol& g, unsigned idx, int p[3]) {
    p[2] = (int)(idx % (unsigned)g.d[2]);
    unsigned r = idx / (unsigned)g.d[2];
    p[1] = (int)(r % (unsigned)g.d[1]);
    p[0] = (int)(r / (unsigned)g.d[1]);
}

// Loop walk of one cell: directed face segments -> closed loops -> fans.  Returns the triangle count; tri[] holds
// (local edge) triples packed 4 bits each.  ins: inside bits by corner; f: values minus level by corner.
__device__ __forceinline__ int cell_triangles(unsigned ins, const float f[8], unsigned tri[10]) {
    unsigned long long nxt = ~0ull;                   // 4 bits per local edge: the edge its segment leads to (15: none)
#pragma unroll
    for (int fc = 0; fc < 6; ++fc) {
        int ib[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) ib[q] = (ins >> ring_corner(fc, q)) & 1;
        unsigned cm = 0;                                  // ring edges q (corner q -> q+1) that cross
#pragma unroll
        for (int q = 0; q < 4; ++q) cm |= (unsigned)(ib[q] != ib[(q + 1) & 3]) << q;
        if (cm == 0) continue;
        bool joined = false;
        if (cm == 0xf) {   // asymptotic decider, in the face's lattice order so both cells of the face agree bit for bit
            const float a = f[lat_corner(fc, 0)], b = f[lat_corner(fc, 1)], c = f[lat_corner(fc, 2)], d = f[lat_corner(fc, 3)];
            const float det = __fsub_rn(__fmul_rn(a, d), __fmul_rn(b, c));
            joined = ((ins >> lat_corner(fc, 0)) & 1) ? det > 0.f : det < 0.f;
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (!((cm >> q) & 1) || ib[q]) continue;        // only outside -> inside crossings start a segment
            // the segment ends at the next crossing along the ring (separated), or the previous one (joined)
            int e_to = 0;
#pragma unroll
            for (int r = 3; r >= 1; --r) {
                const int qq = joined ? (q + 4 - r) & 3 : (q + r) & 3;
                if ((cm >> qq) & 1) e_to = ring_edge(fc, qq);
            }
            const int e_from = ring_edge(fc, q);
            nxt = (nxt & ~(0xfull << (4 * e_from))) | ((unsigned long long)e_to << (4 * e_from));
        }
    }
    int nt = 0;
    unsigned seen = 0;
    for (int e = 0; e < 12; ++e) {                     // ascending local id = ascending vertex id: loops start at their minimum
        const unsigned n1 = (unsigned)(nxt >> (4 * e)) & 0xf;
        if (n1 == 0xf || ((seen >> e) & 1)) continue;
        seen |= (1u << e) | (1u << n1);
        unsigned prev = n1, cur = (unsigned)(nxt >> (4 * n1)) & 0xf;
        while (cur != (unsigned)e) {
            tri[nt++] = (unsigned)e | (prev << 4) | (cur << 8);
            seen |= 1u << cur;
            prev = cur;
            cur = (unsigned)(nxt >> (4 * cur)) & 0xf;
        }
    }
    return nt;
}

// One cell (lowest corner idx, coordinates p): triangles and, per local edge, the key of the vertex it finally uses
// (its own, or rep[] of the lattice corner its vertex sits exactly on).  Returns 0 for cells without a crossing.
__device__ __forceinline__ int cell_setup(const Vol& g, unsigned idx, const int p[3], const unsigned* __restrict__ rep,
                                          unsigned tri[10], unsigned mk[12]) {
    float v[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) v[c] = __ldg(g.v + idx + off(c, 0) * g.s[0] + off(c, 1) * g.s[1] + off(c, 2));
    unsigned ins = 0;
#pragma unroll
    for (int c = 0; c < 8; ++c) ins |= (v[c] > g.level ? 1u : 0u) << c;
    if (ins == 0 || ins == 0xff) return 0;
    float f[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) f[c] = __fsub_rn(v[c], g.level);
    const int nt = cell_triangles(ins, f, tri);
#pragma unroll
    for (int c = 0; c < 8; ++c) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (off(c, a)) continue;
            const int c1 = c | (1 << (2 - a));
            if (!(((ins >> c) ^ (ins >> c1)) & 1)) continue;
            const unsigned lin = idx + off(c, 0) * g.s[0] + off(c, 1) * g.s[1] + off(c, 2);
            const float base = (float)p[a], pos = __fadd_rn(base, edge_t(v[c], v[c1], g.level));
            mk[edge_id(c, a)] = pos == base ? __ldg(rep + lin) : pos == base + 1.f ? __ldg(rep + lin + g.s[a]) : 3u * lin + a;
        }
    }
    return nt;
}

__device__ __forceinline__ bool is_cell(const Vol& g, const int p[3]) {
    return p[0] < g.d[0] - 1 && p[1] < g.d[1] - 1 && p[2] < g.d[2] - 1;
}

// ---------------------------------------------------------------- count
struct Stats {                 // device-side reductions + totals, copied to the host by p3d_mc_count
    unsigned vmin, vmax;       // order-preserving uint images of the min / max
    unsigned long long crossings;
    unsigned long long totals; // (vertices << 32) | faces
};

__global__ void __launch_bounds__(NT) k_mc_classify(Vol g, unsigned* __restrict__ rep, Stats* __restrict__ st) {
    __shared__ float s_min[NT / 32], s_max[NT / 32];
    __shared__ unsigned s_cnt[NT / 32];
    const unsigned idx = blockIdx.x * NT + threadIdx.x;
    float lo = INFINITY, hi = -INFINITY;
    unsigned cnt = 0;
    if (idx < g.n) {
        int p[3];
        decompose(g, idx, p);
        const float v = __ldg(g.v + idx);
        lo = hi = v;
        const bool in = v > g.level;
        unsigned best = NO_REP;
        // edges ending here (owned by the lower neighbours) have the smaller keys, ascending in a
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (p[a] == 0) continue;
            const float vl = __ldg(g.v + idx - g.s[a]);
            if ((vl > g.level) != in && __fadd_rn((float)(p[a] - 1), edge_t(vl, v, g.level)) == (float)p[a])
                best = min(best, 3u * (idx - g.s[a]) + a);
        }
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (p[a] + 1 >= g.d[a]) continue;
            const float vh = __ldg(g.v + idx + g.s[a]);
            if ((vh > g.level) == in) continue;
            ++cnt;
            if (__fadd_rn((float)p[a], edge_t(v, vh, g.level)) == (float)p[a]) best = min(best, 3u * idx + a);
        }
        rep[idx] = best;
    }
    lo = warp_min(lo); hi = warp_max(hi);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) { s_min[w] = lo; s_max[w] = hi; s_cnt[w] = cnt; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < NT / 32; ++k) { lo = fminf(lo, s_min[k]); hi = fmaxf(hi, s_max[k]); cnt += s_cnt[k]; }
        atomicMin(&st->vmin, float_to_ordered(lo));
        atomicMax(&st->vmax, float_to_ordered(hi));
        if (cnt) atomicAdd(&st->crossings, (unsigned long long)cnt);
    }
}

__global__ void __launch_bounds__(NT) k_mc_cells(Vol g, const unsigned* __restrict__ rep, uint8_t* __restrict__ ref,
                                                 uint8_t* __restrict__ fcount) {
    const unsigned idx = blockIdx.x * NT + threadIdx.x;
    if (idx >= g.n) return;
    int p[3];
    decompose(g, idx, p);
    int kept = 0;
    if (is_cell(g, p)) {
        unsigned tri[10], mk[12];
        const int nt = cell_setup(g, idx, p, rep, tri, mk);
        for (int t = 0; t < nt; ++t) {
            const unsigned a = mk[tri[t] & 0xf], b = mk[(tri[t] >> 4) & 0xf], c = mk[tri[t] >> 8];
            if (a == b || b == c || a == c) continue;              // collapsed onto a lattice corner
            ++kept;
            ref[a] = 1; ref[b] = 1; ref[c] = 1;                    // same value from every writer
        }
    }
    fcount[idx] = (uint8_t)kept;
}

__global__ void __launch_bounds__(NT) k_mc_pack(unsigned n, const uint8_t* __restrict__ ref, const uint8_t* __restrict__ fcount,
                                                unsigned long long* __restrict__ cnt) {
    const unsigned idx = blockIdx.x * NT + threadIdx.x;
    if (idx >= n) return;
    const unsigned nv = ref[3 * idx] + ref[3 * idx + 1] + ref[3 * idx + 2];
    cnt[idx] = ((unsigned long long)nv << 32) | fcount[idx];
}

__global__ void k_mc_total(unsigned n, const unsigned long long* __restrict__ cnt, const unsigned long long* __restrict__ base,
                           Stats* __restrict__ st) {
    st->totals = base[n - 1] + cnt[n - 1];
}

// ---------------------------------------------------------------- emit
// -dV/dx_b at corner (lin, coordinate q) by numpy.gradient rules: central inside, one-sided on the border
__device__ __forceinline__ float neg_grad(const float* __restrict__ v, unsigned lin, int q, int d, unsigned s) {
    float gr;
    if (q == 0) gr = __fsub_rn(__ldg(v + lin + s), __ldg(v + lin));
    else if (q == d - 1) gr = __fsub_rn(__ldg(v + lin), __ldg(v + lin - s));
    else gr = __fmul_rn(__fsub_rn(__ldg(v + lin + s), __ldg(v + lin - s)), 0.5f);
    return -gr;
}

struct EmitArgs {
    const uint8_t* ref;
    const unsigned long long* base;
    const float* rgb;
    long long rs[4];
    float *verts, *normals, *values, *colors;
    int* faces;
};

__global__ void __launch_bounds__(NT) k_mc_verts(Vol g, EmitArgs e) {
    const unsigned idx = blockIdx.x * NT + threadIdx.x;
    if (idx >= g.n) return;
    const uint8_t r0 = e.ref[3 * idx], r1 = e.ref[3 * idx + 1], r2 = e.ref[3 * idx + 2];
    if (!(r0 | r1 | r2)) return;
    int p[3];
    decompose(g, idx, p);
    unsigned id = (unsigned)(e.base[idx] >> 32);
    const float v = __ldg(g.v + idx);
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        if (!(a == 0 ? r0 : a == 1 ? r1 : r2)) continue;
        const unsigned hi = idx + g.s[a];
        const float t = edge_t(v, __ldg(g.v + hi), g.level);
        float pos[3] = {(float)p[0], (float)p[1], (float)p[2]};
        pos[a] = __fadd_rn(pos[a], t);
        float nrm[3];
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            const float glo = neg_grad(g.v, idx, p[b], g.d[b], g.s[b]);
            const float ghi = neg_grad(g.v, hi, p[b] + (b == a), g.d[b], g.s[b]);
            nrm[b] = __fadd_rn(glo, __fmul_rn(t, __fsub_rn(ghi, glo)));
        }
        const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(nrm[0], nrm[0]), __fmul_rn(nrm[1], nrm[1])), __fmul_rn(nrm[2], nrm[2])));
        // value: max over the lowest-index cell containing the edge
        unsigned cell = idx;
#pragma unroll
        for (int b = 0; b < 3; ++b)
            if (b != a && p[b] > 0) cell -= g.s[b];
        float vmax = -INFINITY;
#pragma unroll
        for (int c = 0; c < 8; ++c) vmax = fmaxf(vmax, __ldg(g.v + cell + off(c, 0) * g.s[0] + off(c, 1) * g.s[1] + off(c, 2)));
#pragma unroll
        for (int b = 0; b < 3; ++b) {
            e.verts[3 * (size_t)id + b] = pos[b];
            e.normals[3 * (size_t)id + b] = len > 0.f ? __fdiv_rn(nrm[b], len) : 0.f;
        }
        e.values[id] = vmax;
        if (e.rgb) {       // rgbs[:3, a, b, c] at verts.astype(int): the truncated fp32 position, not the edge's corner
            const long long o = (long long)(int)pos[0] * e.rs[1] + (long long)(int)pos[1] * e.rs[2] + (long long)(int)pos[2] * e.rs[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) e.colors[3 * (size_t)id + c] = __ldg(e.rgb + o + c * e.rs[0]);
        }
        ++id;
    }
}

// final id of the vertex with key m: its corner's scanned base + the referenced edges of that corner below its axis
__device__ __forceinline__ int final_id(const EmitArgs& e, unsigned m) {
    const unsigned c = m / 3, a = m - 3 * c;
    unsigned id = (unsigned)(e.base[c] >> 32);
    if (a > 0) id += e.ref[3 * c];
    if (a > 1) id += e.ref[3 * c + 1];
    return (int)id;
}

__global__ void __launch_bounds__(NT) k_mc_faces(Vol g, const unsigned* __restrict__ rep, EmitArgs e) {
    const unsigned idx = blockIdx.x * NT + threadIdx.x;
    if (idx >= g.n) return;
    int p[3];
    decompose(g, idx, p);
    if (!is_cell(g, p)) return;
    unsigned tri[10], mk[12];
    const int nt = cell_setup(g, idx, p, rep, tri, mk);
    if (nt == 0) return;
    size_t out = (size_t)(unsigned)e.base[idx];
    for (int t = 0; t < nt; ++t) {
        const unsigned a = mk[tri[t] & 0xf], b = mk[(tri[t] >> 4) & 0xf], c = mk[tri[t] >> 8];
        if (a == b || b == c || a == c) continue;
        e.faces[3 * out] = final_id(e, a);
        e.faces[3 * out + 1] = final_id(e, b);
        e.faces[3 * out + 2] = final_id(e, c);
        ++out;
    }
}

// ---------------------------------------------------------------- host
struct Layout {
    size_t rep, ref, fcount, cnt, base, stats, temp, temp_bytes, total;
};

int make_vol(const float* vol, int32_t d0, int32_t d1, int32_t d2, double level, Vol* g) {
    P3D_REQUIRE(d0 >= 2 && d1 >= 2 && d2 >= 2, "p3d_mc: every volume dimension must be >= 2 (got %d x %d x %d)", d0, d1, d2);
    P3D_REQUIRE(3ll * d0 * d1 * d2 < (1ll << 31), "p3d_mc: volume %d x %d x %d too large for int32 vertex ids", d0, d1, d2);
    g->v = vol;
    g->d[0] = d0; g->d[1] = d1; g->d[2] = d2;
    g->s[0] = (unsigned)d1 * (unsigned)d2; g->s[1] = (unsigned)d2; g->s[2] = 1;
    g->n = (unsigned)d0 * g->s[0];
    g->level = (float)level;
    return P3D_OK;
}

int make_layout(unsigned n, Layout* L) {
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t at = o; o = (o + bytes + 255) & ~(size_t)255; return at; };
    L->rep = take(4ull * n);
    L->ref = take(3ull * n);
    L->fcount = take(n);
    L->cnt = take(8ull * n);
    L->base = take(8ull * n);
    L->stats = take(sizeof(Stats));
    L->temp_bytes = 0;
    P3D_CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, L->temp_bytes, (unsigned long long*)nullptr, (unsigned long long*)nullptr, (int)n));
    L->temp = take(L->temp_bytes);
    L->total = o;
    return P3D_OK;
}

int check_workspace(const Vol& g, void* ws, size_t ws_bytes, Layout* L) {
    if (int rc = make_layout(g.n, L)) return rc;
    P3D_REQUIRE(ws != nullptr && ((uintptr_t)ws & 255) == 0, "p3d_mc: workspace must be a 256-byte aligned device pointer");
    P3D_REQUIRE(ws_bytes >= L->total, "p3d_mc: workspace of %zu bytes, %zu needed (p3d_mc_workspace_bytes)", ws_bytes, L->total);
    return P3D_OK;
}

}  // namespace
}  // namespace p3d

using namespace p3d;

extern "C" size_t p3d_mc_workspace_bytes(int32_t d0, int32_t d1, int32_t d2) {
    Vol g;
    Layout L;
    if (make_vol(nullptr, d0, d1, d2, 0.0, &g) || make_layout(g.n, &L)) return 0;
    return L.total;
}

extern "C" int p3d_mc_count(const float* vol, int32_t d0, int32_t d1, int32_t d2, double level, void* workspace, size_t workspace_bytes,
                            int64_t* out_counts, float* out_range, void* stream) {
    Vol g;
    Layout L;
    if (int rc = make_vol(vol, d0, d1, d2, level, &g)) return rc;
    P3D_REQUIRE(vol && out_counts && out_range, "p3d_mc_count: NULL pointer");
    if (int rc = check_workspace(g, workspace, workspace_bytes, &L)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    unsigned* rep = (unsigned*)(ws + L.rep);
    uint8_t *ref = (uint8_t*)(ws + L.ref), *fcount = (uint8_t*)(ws + L.fcount);
    unsigned long long *cnt = (unsigned long long*)(ws + L.cnt), *base = (unsigned long long*)(ws + L.base);
    Stats* stats = (Stats*)(ws + L.stats);
    const Stats init{0xffffffffu, 0u, 0ull, 0ull};
    P3D_CUDA_TRY(cudaMemcpyAsync(stats, &init, sizeof(Stats), cudaMemcpyHostToDevice, st));
    P3D_CUDA_TRY(cudaMemsetAsync(ref, 0, 3ull * g.n, st));
    const unsigned grid = (g.n + NT - 1) / NT;
    k_mc_classify<<<grid, NT, 0, st>>>(g, rep, stats);
    P3D_LAUNCH_CHECK();
    k_mc_cells<<<grid, NT, 0, st>>>(g, rep, ref, fcount);
    P3D_LAUNCH_CHECK();
    k_mc_pack<<<grid, NT, 0, st>>>(g.n, ref, fcount, cnt);
    P3D_LAUNCH_CHECK();
    size_t tb = L.temp_bytes;
    P3D_CUDA_TRY(cub::DeviceScan::ExclusiveSum(ws + L.temp, tb, cnt, base, (int)g.n, st));
    count_launch();
    k_mc_total<<<1, 1, 0, st>>>(g.n, cnt, base, stats);
    P3D_LAUNCH_CHECK();
    Stats h;
    P3D_CUDA_TRY(cudaMemcpyAsync(&h, stats, sizeof(Stats), cudaMemcpyDeviceToHost, st));
    P3D_CUDA_TRY(cudaStreamSynchronize(st));
    out_counts[0] = (int64_t)(h.totals >> 32);
    out_counts[1] = (int64_t)(h.totals & 0xffffffffull);
    out_counts[2] = (int64_t)h.crossings;
    out_range[0] = ordered_to_float(h.vmin);
    out_range[1] = ordered_to_float(h.vmax);
    return P3D_OK;
}

extern "C" int p3d_mc_emit(const float* vol, int32_t d0, int32_t d1, int32_t d2, double level, void* workspace, size_t workspace_bytes,
                           const float* rgb, int64_t rgb_stride_c, int64_t rgb_stride_0, int64_t rgb_stride_1, int64_t rgb_stride_2,
                           float* verts, float* normals, float* values, float* colors, int32_t* faces, void* stream) {
    Vol g;
    Layout L;
    if (int rc = make_vol(vol, d0, d1, d2, level, &g)) return rc;
    P3D_REQUIRE(vol && verts && normals && values && faces, "p3d_mc_emit: NULL pointer");
    P3D_REQUIRE(!rgb || colors, "p3d_mc_emit: rgb given without a colors output");
    if (int rc = check_workspace(g, workspace, workspace_bytes, &L)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    char* ws = (char*)workspace;
    EmitArgs e;
    e.ref = (const uint8_t*)(ws + L.ref);
    e.base = (const unsigned long long*)(ws + L.base);
    e.rgb = rgb;
    e.rs[0] = rgb_stride_c; e.rs[1] = rgb_stride_0; e.rs[2] = rgb_stride_1; e.rs[3] = rgb_stride_2;
    e.verts = verts; e.normals = normals; e.values = values; e.colors = colors; e.faces = faces;
    const unsigned grid = (g.n + NT - 1) / NT;
    k_mc_verts<<<grid, NT, 0, st>>>(g, e);
    P3D_LAUNCH_CHECK();
    k_mc_faces<<<grid, NT, 0, st>>>(g, (const unsigned*)(ws + L.rep), e);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}
