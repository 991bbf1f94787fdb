// Axis-angle -> rotation matrix through the unit quaternion (pytorch3d.axis_angle_to_matrix, the route of
// core/utils/skeleton_utils.py:411-418), and its derivative.  Shared by the graph net (graphnet.cu: its inputs are the
// first two columns of these matrices) and the pose layer (pose.cu: its kinematic chain).
#pragma once
#include <math.h>

namespace danbo {

// R (row-major 3x3) of axis-angle aa, in the op order of pose_opt.axisang_to_rot / networks.axis_angle_to_matrix,
// including the |angle| < 1e-6 branch of the quaternion's vector scale.
__device__ __forceinline__ void axisang_to_rot(const float aa[3], float R[9]) {
    const float ax = aa[0], ay = aa[1], az = aa[2];
    const float ang = sqrtf(ax * ax + ay * ay + az * az), half = 0.5f * ang;
    const float k = fabsf(ang) < 1e-6f ? 0.5f - ang * ang / 48.f : sinf(half) / ang;
    const float qr = cosf(half), qi = ax * k, qj = ay * k, qk = az * k;
    const float two_s = 2.f / (qr * qr + qi * qi + qj * qj + qk * qk);
    R[0] = 1.f - two_s * (qj * qj + qk * qk); R[1] = two_s * (qi * qj - qk * qr); R[2] = two_s * (qi * qk + qj * qr);
    R[3] = two_s * (qi * qj + qk * qr); R[4] = 1.f - two_s * (qi * qi + qk * qk); R[5] = two_s * (qj * qk - qi * qr);
    R[6] = two_s * (qi * qk - qj * qr); R[7] = two_s * (qj * qk + qi * qr); R[8] = 1.f - two_s * (qi * qi + qj * qj);
}

// d aa = (d R / d aa)^T g for g = d loss / d R (row-major 3x3): back through q -> R (with s = 2 / |q|^2), then
// q = (cos(ang/2), aa k(ang)), then ang = |aa|.  As torch autograd of the forward: the branch of k that the forward
// did not take receives nothing, and ang = 0 gives the norm no gradient.
__device__ __forceinline__ void axisang_to_rot_bwd(const float aa[3], const float g[9], float d_aa[3]) {
    const float ax = aa[0], ay = aa[1], az = aa[2];
    const float ang = sqrtf(ax * ax + ay * ay + az * az), half = 0.5f * ang;
    const bool small = fabsf(ang) < 1e-6f;
    const float sh = sinf(half), ch = cosf(half);
    const float k = small ? 0.5f - ang * ang / 48.f : sh / ang;
    const float r = ch, i = ax * k, j = ay * k, kk = az * k;
    const float s = 2.f / (r * r + i * i + j * j + kk * kk);
    const float ds = -(j * j + kk * kk) * g[0] + (i * j - kk * r) * g[1] + (i * kk + j * r) * g[2]
                   + (i * j + kk * r) * g[3] - (i * i + kk * kk) * g[4] + (j * kk - i * r) * g[5]
                   + (i * kk - j * r) * g[6] + (j * kk + i * r) * g[7] - (i * i + j * j) * g[8];
    const float dn = -0.5f * s * s * ds;                                  // s = 2 / n, n = |q|^2
    const float dr = s * (-kk * g[1] + j * g[2] + kk * g[3] - i * g[5] - j * g[6] + i * g[7]) + 2.f * r * dn;
    const float di = s * (j * g[1] + kk * g[2] + j * g[3] - 2.f * i * g[4] - r * g[5] + kk * g[6] + r * g[7]
                          - 2.f * i * g[8]) + 2.f * i * dn;
    const float dj = s * (-2.f * j * g[0] + i * g[1] + r * g[2] + i * g[3] + kk * g[5] - r * g[6] + kk * g[7]
                          - 2.f * j * g[8]) + 2.f * j * dn;
    const float dk = s * (-2.f * kk * g[0] - r * g[1] + i * g[2] + r * g[3] - 2.f * kk * g[4] + j * g[5] + i * g[6]
                          + j * g[7]) + 2.f * kk * dn;
    const float dkk = di * ax + dj * ay + dk * az;                       // d k
    const float dkdang = small ? -ang / 24.f : (0.5f * ch * ang - sh) / (ang * ang);
    const float dang = -0.5f * sh * dr + dkdang * dkk;
    const float u = ang > 0.f ? dang / ang : 0.f;
    d_aa[0] = di * k + u * ax;
    d_aa[1] = dj * k + u * ay;
    d_aa[2] = dk * k + u * az;
}

}  // namespace danbo
