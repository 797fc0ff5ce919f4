// scene_layout.cu -- the scene's primitive and material arrays, laid out on the device for either BVH builder.
//
// A builder (bvh_builder.cpp on the host, lbvh.cu on the device) decides only the tree and the leaf order:
// sphere_order[i] / quad_order[i] is the caller's index of the sphere / quad at leaf position i.  This step turns the
// caller's records, already on the device as they are, into what the kernels read (traverse.cuh DeviceScene):
// spheres and quads gathered into leaf order with the quad constants computed, materials converted, and every
// per-primitive index and material kind of the description checked.  One implementation for both builders is what
// keeps the records, and so hit times and images, the same bits whichever builder ran (tests/test_gpu_lbvh.py).
#include "../../include/b200rt.h"
#include "devmem.h"
#include "kernels.h"

namespace b200rt {

namespace {

// bad[0]: a material or canonical primitive index out of range; bad[1]: an unknown material kind

__global__ void gather_spheres(const B200rtSphere *__restrict__ raw, const uint32_t *__restrict__ order, uint32_t n,
                               uint32_t n_prims, uint32_t n_materials, double2 *__restrict__ out, uint2 *__restrict__ meta, int *bad) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const B200rtSphere s = raw[order[i]];
    if (s.mat >= n_materials || s.prim >= n_prims) bad[0] = 1;
    out[2 * (size_t)i] = make_double2(s.c[0], s.c[1]);
    out[2 * (size_t)i + 1] = make_double2(s.c[2], s.r);
    meta[i] = make_uint2(s.prim, s.mat);
}

__global__ void gather_quads(const B200rtQuad *__restrict__ raw, const uint32_t *__restrict__ order, uint32_t n,
                             uint32_t n_prims, uint32_t n_materials, double2 *__restrict__ out, uint2 *__restrict__ meta, int *bad) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const B200rtQuad q = raw[order[i]];
    if (q.mat >= n_materials || q.prim >= n_prims) bad[0] = 1;
    // parallelogram.h:275-279: n = cross(s1, s2); unit = n * (1 / |n|); w = n * (1 / |n|^2), in the reference's
    // operation order (no FMA contraction: -fmad=false)
    const double nx = q.s1[1] * q.s2[2] - q.s1[2] * q.s2[1], ny = q.s1[2] * q.s2[0] - q.s1[0] * q.s2[2],
                 nz = q.s1[0] * q.s2[1] - q.s1[1] * q.s2[0];
    const double m2 = nx * nx + ny * ny + nz * nz;
    const double im = 1 / sqrt(m2), im2 = 1 / m2;
    const double f[16] = {nx * im, ny * im, nz * im, q.v[0], q.v[1], q.v[2], nx * im2, ny * im2, nz * im2,
                          q.s1[0], q.s1[1], q.s1[2], q.s2[0], q.s2[1], q.s2[2], 0.0};
    for (int k = 0; k < 8; ++k) out[8 * (size_t)i + k] = make_double2(f[2 * k], f[2 * k + 1]);
    meta[i] = make_uint2(q.prim, q.mat);
}

// B200rtMaterial (the caller's 40-byte records) -> DeviceMaterial: lights pre-multiplied by their intensity
// (material.h:261-263), metal fuzz clamped to 1 (material.h:150-151).  The reference's big scenes carry one material
// PER PRIMITIVE (millions), which is why this runs on the device.
__global__ void convert_materials(const B200rtMaterial *__restrict__ raw, uint32_t n, DeviceMaterial *__restrict__ out, int *bad) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const B200rtMaterial m = raw[i];
    if (m.kind > B200RT_MAT_LIGHT) bad[1] = 1;
    DeviceMaterial dm;
    const double k = m.kind == B200RT_MAT_LIGHT ? m.param : 1.0;
    dm.r = (float)(k * m.rgb[0]); dm.g = (float)(k * m.rgb[1]); dm.b = (float)(k * m.rgb[2]);
    dm.kind = m.kind;
    dm.param = m.kind == B200RT_MAT_METAL ? fmin(m.param, 1.0) : m.param;
    dm.pad = 0.0;
    out[i] = dm;
}

}  // namespace

// Fills the scene's leaf-ordered sphere / quad / meta arrays and its materials from the caller's records (all pointers
// device memory, enqueued on the legacy default stream) and returns once they are written, with bad_out[0] set if a
// material or primitive index is out of range and bad_out[1] if a material kind is unknown.
cudaError_t assemble_scene_device(const B200rtSphere *sph, const uint32_t *sphere_order, uint32_t n_sph, const B200rtQuad *quads,
                                  const uint32_t *quad_order, uint32_t n_quad, const B200rtMaterial *mats, uint32_t n_mat,
                                  double2 *out_sph, uint2 *out_sph_meta, double2 *out_quads, uint2 *out_quad_meta,
                                  DeviceMaterial *out_mats, int bad_out[2]) {
    bad_out[0] = bad_out[1] = 0;
    int *bad = nullptr;
    cudaError_t e = dev_alloc_async(&bad, 2 * sizeof(int), 0);
    if (e != cudaSuccess) return e;
    e = cudaMemsetAsync(bad, 0, 2 * sizeof(int), 0);
    const uint32_t n_prims = n_sph + n_quad, B = 256;
    if (e == cudaSuccess && n_sph)
        gather_spheres<<<(n_sph + B - 1) / B, B>>>(sph, sphere_order, n_sph, n_prims, n_mat, out_sph, out_sph_meta, bad);
    if (e == cudaSuccess && n_quad)
        gather_quads<<<(n_quad + B - 1) / B, B>>>(quads, quad_order, n_quad, n_prims, n_mat, out_quads, out_quad_meta, bad);
    if (e == cudaSuccess && n_mat) convert_materials<<<(n_mat + B - 1) / B, B>>>(mats, n_mat, out_mats, bad);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(bad_out, bad, 2 * sizeof(int), cudaMemcpyDeviceToHost, 0);
    if (e == cudaSuccess) e = cudaStreamSynchronize(0);
    dev_free(bad);
    return e;
}

}  // namespace b200rt
