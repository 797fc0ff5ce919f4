// shade.cuh -- camera ray generation, surface interaction and scattering for the path kernels.
//
// Stands in for Camera::random_ray_through_pixel (reference include/base/camera.h:184-200),
// the hit_info constructor (hittable.h:46-71), Lambertian/Metal/Dielectric/DiffuseLight
// scatter+emit (material.h:64-263) and reflected/refracted (math/vec3d.h:144-200).
// Geometry (origins, directions, normals) stays in FP64 like the reference; colours and
// random numbers are FP32.  Random directions are drawn by direct sampling from one Philox
// block per ray segment instead of the reference's rejection loops (vec3d.h:64-85): the
// distributions are identical (uniform on the unit sphere / in the unit disk), the streams
// necessarily are not.
#pragma once
#include "../../include/b200rt.h"
#include "rng.cuh"
#include "traverse.cuh"

namespace b200rt {

struct CameraParams {
    double center[3], pixel00[3], delta_x[3], delta_y[3], disk_x[3], disk_y[3];
    float background[3];
    uint32_t defocus;   // defocus_angle > 0 (camera.h:186)
    uint32_t w, h, max_depth;
};

struct PathState {
    float tr, tg, tb;   // throughput (product of attenuations so far)
};

// Uniform direction on the unit sphere from two uniforms (what random_unit_vector() produces
// after normalisation, vec3d.h:64-75).
__device__ __forceinline__ void sample_unit_sphere(float u1, float u2, double &x, double &y, double &z) {
    const float cz = 1.0f - 2.0f * u1;
    const float r = sqrtf(fmaxf(0.0f, 1.0f - cz * cz));
    float s, c;
    sincospif(2.0f * u2, &s, &c);
    x = (double)(r * c);
    y = (double)(r * s);
    z = (double)cz;
}

// Uniform point in the unit disk from two uniforms (what random_vector_in_unit_disk() produces, vec3d.h:79-85).
__device__ __forceinline__ void sample_unit_disk(float u1, float u2, double &x, double &y) {
    const float rad = sqrtf(u1);
    float s, c;
    sincospif(2.0f * u2, &s, &c);
    x = (double)(rad * c);
    y = (double)(rad * s);
}

// camera.h:184-200 (+ :160-168 for the defocus disk)
__device__ __forceinline__ void camera_ray(const CameraParams &C, uint32_t px, uint32_t py, const Philox4 &rnd,
                                           Ray &r, PathState &p) {
    double ox = C.center[0], oy = C.center[1], oz = C.center[2];
    if (C.defocus) {
        double ax, ay;
        sample_unit_disk(u01(rnd.z), u01(rnd.w), ax, ay);
        ox = (C.center[0] + ax * C.disk_x[0]) + ay * C.disk_y[0];
        oy = (C.center[1] + ax * C.disk_x[1]) + ay * C.disk_y[1];
        oz = (C.center[2] + ax * C.disk_x[2]) + ay * C.disk_y[2];
    }
    const double row = (double)py, col = (double)px;
    const double jx = (double)u01(rnd.x) - 0.5, jy = (double)u01(rnd.y) - 0.5;
    const double sx = ((C.pixel00[0] + row * C.delta_y[0]) + col * C.delta_x[0]) + jx * C.delta_x[0] + jy * C.delta_y[0];
    const double sy = ((C.pixel00[1] + row * C.delta_y[1]) + col * C.delta_x[1]) + jx * C.delta_x[1] + jy * C.delta_y[1];
    const double sz = ((C.pixel00[2] + row * C.delta_y[2]) + col * C.delta_x[2]) + jx * C.delta_x[2] + jy * C.delta_y[2];
    r.ox = ox; r.oy = oy; r.oz = oz;
    r.dx = sx - ox; r.dy = sy - oy; r.dz = sz - oz;   // NOT normalised (camera.h:199)
    p.tr = p.tg = p.tb = 1.0f;
}

// Applies one surface interaction.  Returns true if the path continues with the new ray in `r`.
// Emitted light is added to (acc_r, acc_g, acc_b) weighted by the path throughput: the sum over a
// path of throughput x emission is what ray_color's recursion returns (camera.h:233-234).
__device__ __forceinline__ bool shade_hit(const DeviceScene &S, const Hit &h, const Philox4 &rnd, Ray &r, PathState &p,
                                          float &acc_r, float &acc_g, float &acc_b) {
    // hit point: ray(t) = origin + t * dir (ray3d.h:16)
    const double hx = r.ox + h.t * r.dx, hy = r.oy + h.t * r.dy, hz = r.oz + h.t * r.dz;
    double nx, ny, nz;
    uint32_t mat_id;
    if (h.ref & kQuadFlagD) {
        const uint32_t qi = h.ref & ~kQuadFlagD;
        const double2 q0 = __ldg(S.quads + (size_t)qi * 8), q1 = __ldg(S.quads + (size_t)qi * 8 + 1);
        nx = q0.x; ny = q0.y; nz = q1.x;                      // unit_plane_normal (parallelogram.h:234)
        mat_id = __ldg(&S.quad_meta[qi]).y;
    } else {
        const double2 s0 = __ldg(S.spheres + (size_t)h.ref * 2), s1 = __ldg(S.spheres + (size_t)h.ref * 2 + 1);
        const double inv_r = 1.0 / s1.y;                      // (hit_point - center) / radius, via *= 1/d (vec3d.h:31, sphere.h:94)
        nx = (hx - s0.x) * inv_r; ny = (hy - s0.y) * inv_r; nz = (hz - s1.x) * inv_r;
        mat_id = __ldg(&S.sphere_meta[h.ref]).y;
    }
    // front/back face (hittable.h:56-70)
    const bool inside = (r.dx * nx + r.dy * ny + r.dz * nz) > 0;
    if (inside) { nx = -nx; ny = -ny; nz = -nz; }

#ifdef B200RT_DEBUG_BOUNDS
    if (!B200RT_CHECK(S, mat_id < S.dbg.n_materials, 2)) return false;
#endif
    const float4 m0 = __ldg((const float4 *)(S.materials + mat_id));
    const uint32_t kind = __float_as_uint(m0.w);
    if (kind == B200RT_MAT_LIGHT) {   // DiffuseLight: emits on both faces, never scatters (material.h:248-263)
        acc_r += p.tr * m0.x; acc_g += p.tg * m0.y; acc_b += p.tb * m0.z;
        return false;
    }
    double sx, sy, sz;
    if (kind == B200RT_MAT_LAMBERTIAN) {   // Lambertian (material.h:64-86)
        double ux, uy, uz;
        sample_unit_sphere(u01(rnd.x), u01(rnd.y), ux, uy, uz);
        sx = nx + ux; sy = ny + uy; sz = nz + uz;
        if (fabs(sx) < 1e-8 && fabs(sy) < 1e-8 && fabs(sz) < 1e-8) { sx = nx; sy = ny; sz = nz; }
        p.tr *= m0.x; p.tg *= m0.y; p.tb *= m0.z;
    } else {
        // unit_vector(): *this / mag(), and operator/= multiplies by 1/d (vec3d.h:31,127-130)
        const double inv_len = 1.0 / sqrt(r.dx * r.dx + r.dy * r.dy + r.dz * r.dz);
        const double vx = r.dx * inv_len, vy = r.dy * inv_len, vz = r.dz * inv_len;
        const double vdotn = vx * nx + vy * ny + vz * nz;
        // reflected(v, n) = v - 2*dot(v,n)*n (vec3d.h:144-155)
        const double rx = vx - (2 * vdotn) * nx, ry = vy - (2 * vdotn) * ny, rz = vz - (2 * vdotn) * nz;
        if (kind == B200RT_MAT_METAL) {   // Metal (material.h:116-139)
            const double fuzz = __ldg(&S.materials[mat_id].param);
            double ux, uy, uz;
            sample_unit_sphere(u01(rnd.x), u01(rnd.y), ux, uy, uz);
            sx = rx + fuzz * ux; sy = ry + fuzz * uy; sz = rz + fuzz * uz;
            if (nx * sx + ny * sy + nz * sz < 0) return false;   // absorbed
            p.tr *= m0.x; p.tg *= m0.y; p.tb *= m0.z;
        } else {            // Dielectric (material.h:185-218, vec3d.h:168-200)
            const double ior = __ldg(&S.materials[mat_id].param);
            const double eta = inside ? ior : 1.0 / ior;
            const double cos_theta = fmin(-vdotn, 1.0);
            const double sin_theta = sqrt(1 - cos_theta * cos_theta);
            bool reflect = eta * sin_theta > 1;                  // total internal reflection: no random drawn
            if (!reflect) {
                double r0 = (1 - eta) / (1 + eta);
                r0 *= r0;
                const double m = 1 - cos_theta;
                const double schlick = r0 + (1 - r0) * (m * m * m * m * m);
                reflect = (double)u01(rnd.z) < schlick;
            }
            if (reflect) { sx = rx; sy = ry; sz = rz; }
            else {
                const double ex = eta * (vx + cos_theta * nx), ey = eta * (vy + cos_theta * ny), ez = eta * (vz + cos_theta * nz);
                const double k = -sqrt(fabs(1 - (ex * ex + ey * ey + ez * ez)));
                sx = ex + k * nx; sy = ey + k * ny; sz = ez + k * nz;
            }
            // attenuation is (1,1,1) (material.h:217)
        }
    }
    r.ox = hx; r.oy = hy; r.oz = hz;   // scattered ray starts AT the hit point (no offset; tmin = 1e-5 guards acne)
    r.dx = sx; r.dy = sy; r.dz = sz;   // NOT normalised
    return true;
}

}  // namespace b200rt
