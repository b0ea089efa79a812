/*
 * p3d_mesh.h - C ABI of the marching-cubes mesh extraction (SURVEY.md 8f-2, the step after the volume query).
 *
 * The reference extracts the eval mesh with skimage.measure.marching_cubes(vol, level, spacing=(1,1,1),
 * gradient_direction='descent', step_size=1, allow_degenerate=False, method='lewiner', mask=None)
 * (_util/eg3d_metrics3d.py:186-210, called by _scripts/eval/generate.py:98-103).  This is that configuration on the
 * device; the exact contract (vertex order, positions, in-cell triangulation, degenerate removal) is written out in
 * oracle/mesh_oracle.py, which the tests compare against array for array.
 *
 * Two calls per volume, sharing one caller-allocated workspace:
 *   p3d_mc_count   classify cells, resolve degenerates, scan the counts; returns the mesh size to the host
 *                  (the only host synchronisation: the caller needs it to size the outputs);
 *   p3d_mc_emit    writes the mesh into outputs of exactly that size.
 * The volume, level and workspace passed to p3d_mc_emit must be those of the preceding p3d_mc_count.
 *
 * Volume: fp32, contiguous, shape (d0, d1, d2), device pointer; every dimension >= 2 and 3*d0*d1*d2 < 2^31 (int32
 * vertex ids).  Return codes / p3d_last_error() as in p3d_render.h.
 */
#ifndef P3D_MESH_H_
#define P3D_MESH_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Workspace bytes for a (d0, d1, d2) volume (about 24 bytes per voxel); 0 for a shape p3d_mc_count rejects. */
size_t p3d_mc_workspace_bytes(int32_t d0, int32_t d1, int32_t d2);

/* out_counts[0] = vertices, [1] = faces of the final mesh (after degenerate removal), [2] = crossing edges before it;
   out_range[0], [1] = min and max of the volume (the caller's level check).  Synchronises `stream`. */
int p3d_mc_count(const float* vol, int32_t d0, int32_t d1, int32_t d2, double level, void* workspace, size_t workspace_bytes,
                 int64_t* out_counts, float* out_range, void* stream);

/* verts (V,3) index-space positions (axis0, axis1, axis2); normals (V,3); values (V); faces (F,3) int32.
   rgb: (3, d0, d1, d2) fp32 with element strides rgb_strides[0..3] (any layout), or NULL; colors (V,3) receives
   rgb[:, floor(verts)] when rgb is given (colors may be NULL otherwise). */
int p3d_mc_emit(const float* vol, int32_t d0, int32_t d1, int32_t d2, double level, void* workspace, size_t workspace_bytes,
                const float* rgb, int64_t rgb_stride_c, int64_t rgb_stride_0, int64_t rgb_stride_1, int64_t rgb_stride_2,
                float* verts, float* normals, float* values, float* colors, int32_t* faces, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* P3D_MESH_H_ */
