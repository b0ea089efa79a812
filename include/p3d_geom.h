/*
 * p3d_geom.h - C ABI of the eval geometry metrics: surface sampling, a BVH over a triangle mesh and exact
 * point-to-mesh distances (the igl calls of the reference's _scripts/eval/measure.py:141-201, whose Chamfer distance
 * and F1 scores panic3d_b200.metrics3d computes on the device).
 *
 * All geometry is float64: verts (V,3), points (n,3), contiguous, device pointers; faces (F,3) int32 indices into
 * verts.  Every arithmetic operation is rounded separately (no FMA contraction), so oracle/metrics3d_oracle.py's numpy
 * float64 restatement gives the same bits.  Return codes / p3d_last_error() as in p3d_render.h.
 *
 * status: a caller-zeroed device int32 into which the kernels OR the P3D_GEOM_* bits below; reading it is the caller's
 * only host synchronisation, so several calls can share one status word and be checked once.
 */
#ifndef P3D_GEOM_H_
#define P3D_GEOM_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define P3D_GEOM_ZERO_AREA      1   /* p3d_surface_sample: every face has zero area; outputs are NaN / face -1 */
#define P3D_GEOM_STACK_OVERFLOW 2   /* p3d_point_mesh_distance: traversal stack bound exceeded; results invalid */

/* ---------------------------------------------------------------- area-weighted surface sampling
 * Face f has integer weight floor(|cross(b-a, c-a)| / max_f |cross| * 2^32); the exact uint64 inclusive scan of the
 * weights is the CDF.  Sample i takes a 64-bit word k and two uniforms a, b in [0,1): its face is the first f with
 * cdf[f] > mulhi64(k, total) (zero-weight faces are never drawn); if a + b > 1 then (a, b) = (1-a, 1-b); barycentrics
 * (1-a-b, a, b); point = (v0*b0 + v1*b1) + v2*b2.  Random bits: one Philox4x32-10 call per sample (key seed,
 * counter i, stream_id): k = x << 32 | y, a = z * 2^-32, b = w * 2^-32 - unless face_bits (n) / bary_u (n,2) are given,
 * which replace k / (a, b). */
size_t p3d_surface_sample_workspace_bytes(int64_t n_faces);
/* bary (n,3) fp64, face (n) int64, points (n,3) fp64 or NULL.  No host synchronisation. */
int p3d_surface_sample(const double* verts, const int32_t* faces, int64_t n_faces, int64_t n_samples, uint64_t seed,
                       uint32_t stream_id, const uint64_t* face_bits, const double* bary_u, void* workspace,
                       size_t workspace_bytes, double* bary, int64_t* face, double* points, int32_t* status, void* stream);

/* ---------------------------------------------------------------- LBVH over the faces
 * 30-bit Morton codes of the face centroids in the centroids' bounding box, keys (morton << 32 | face), one radix sort,
 * Karras (2012) topology, bottom-up refit; child boxes stored in their parent as fp32 rounded outward.  The workspace
 * IS the tree: pass the same buffer (unchanged verts / faces) to p3d_point_mesh_distance.  No host synchronisation. */
size_t p3d_bvh_workspace_bytes(int64_t n_faces);
int p3d_bvh_build(const double* verts, const int32_t* faces, int64_t n_faces, void* workspace, size_t workspace_bytes,
                  void* stream);

/* Closest point on the mesh to each point (Ericson, Real-Time Collision Detection 5.1.5, clamped to the face's box; a
 * zero denominator falls back to the nearest of the three edges): dist2 (n) fp64, face (n) int64, closest (n,3) fp64
 * (closest may be NULL).  Equal to exhaustive search over all faces bit for bit, ties to the smallest face id.
 * No host synchronisation. */
int p3d_point_mesh_distance(const double* points, int64_t n_points, const double* verts, const int32_t* faces,
                            int64_t n_faces, const void* bvh_workspace, size_t workspace_bytes, double* dist2,
                            int64_t* face, double* closest, int32_t* status, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* P3D_GEOM_H_ */
