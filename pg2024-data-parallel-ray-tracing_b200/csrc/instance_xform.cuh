// instance_xform.cuh -- the instance arithmetic of the real-scene front end, one source for the host flatten
// (scene_flatten.cpp, g++ -ffp-contract=off) and the device flatten (instance_flatten.cu, --fmad=false): both give the same
// bits. The oracle restates it independently.
//   corner   p_w = M p          per row  fma(m2, z, fma(m1, y, fma(m0, x, m3)))                      (binary32)
//   normal   n_w = A^-T n       A = upper 3x3 of M; A^-T = cofactors / det evaluated in binary64 in the order written
//                               below, each entry rounded once to binary32; per row fma(g2, nz, fma(g1, ny, g0 * nx))
// M is the row-major 3x4 objectToWorld of dprt_instance_desc.
#pragma once
#include <cfloat>
#include <cmath>

#ifdef __CUDACC__
#define DPRT_XF_HD __host__ __device__ __forceinline__
#else
#define DPRT_XF_HD inline
#endif

namespace dprt {

// g = A^-T, row-major 3x3. false (g untouched) when det(A) is zero or not finite: such a transform is rejected.
DPRT_XF_HD bool instance_normal_matrix(const float* M, float* g) {
    const double a00 = M[0], a01 = M[1], a02 = M[2], a10 = M[4], a11 = M[5], a12 = M[6], a20 = M[8], a21 = M[9], a22 = M[10];
    const double c00 = a11 * a22 - a12 * a21, c01 = -(a10 * a22 - a12 * a20), c02 = a10 * a21 - a11 * a20;
    const double c10 = -(a01 * a22 - a02 * a21), c11 = a00 * a22 - a02 * a20, c12 = -(a00 * a21 - a01 * a20);
    const double c20 = a01 * a12 - a02 * a11, c21 = -(a00 * a12 - a02 * a10), c22 = a00 * a11 - a01 * a10;
    const double det = a00 * c00 + a01 * c01 + a02 * c02;
    if (!(det != 0.0) || !(fabs(det) <= DBL_MAX)) return false;
    const double inv = 1.0 / det;
    g[0] = (float)(c00 * inv); g[1] = (float)(c01 * inv); g[2] = (float)(c02 * inv);
    g[3] = (float)(c10 * inv); g[4] = (float)(c11 * inv); g[5] = (float)(c12 * inv);
    g[6] = (float)(c20 * inv); g[7] = (float)(c21 * inv); g[8] = (float)(c22 * inv);
    return true;
}

// o = M p (world-space corner)
DPRT_XF_HD void instance_corner(const float* M, const float* p, float* o) {
    o[0] = fmaf(M[2], p[2], fmaf(M[1], p[1], fmaf(M[0], p[0], M[3])));
    o[1] = fmaf(M[6], p[2], fmaf(M[5], p[1], fmaf(M[4], p[0], M[7])));
    o[2] = fmaf(M[10], p[2], fmaf(M[9], p[1], fmaf(M[8], p[0], M[11])));
}

// q = g n (world-space normal, not renormalised)
DPRT_XF_HD void instance_normal(const float* g, const float* n, float* q) {
    q[0] = fmaf(g[2], n[2], fmaf(g[1], n[1], g[0] * n[0]));
    q[1] = fmaf(g[5], n[2], fmaf(g[4], n[1], g[3] * n[0]));
    q[2] = fmaf(g[8], n[2], fmaf(g[7], n[1], g[6] * n[0]));
}

}  // namespace dprt
