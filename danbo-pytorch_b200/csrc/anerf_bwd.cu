// AN1 backward to the poses: d loss / d skts of the A-NeRF encodings (pose refinement, --opt_pose).
//
// Reference being differentiated (autograd of, per sample):
//   core/encoders.py:288-303 transform_batch_pts, :442-444 bone align, :639-651 RelDistEncoder, :774-795 VecNormEncoder
//   core/cutoff_embedder.py:151-214 CutoffEmbedder._embed (pe_fn on the distances, dirs_pe_fn on the ray directions)
//   core/encoders.py:305-317 transform_batch_rays (rotation only), core/networks/nerf.py:222-279 encode_pts / encode_views
//
// The field reads the pose only through skts.  Per sample (embed_kernel, anerf.cu):
//   q_j = A_j (R_j p + t_j) + a_j,  v_j = |q_j|,  r_j = q_j / max(v_j, 1e-12),  w_j = 1 - sigmoid(tau (v_j - c))
//   xd[row f * 24 + j] = PE_f(c - v_j) w_j (15 rows),  xd[360 + 3j + a] = r_j[a],  xv[m * 72 + 3j + a] = enc_m(d_j)[a] w_j
// Per ray (ray_kernel): d_j = normalize(R_j d_ray), enc = [d, sin(2^f d), cos(2^f d)]_{f<4}.
// Given d xd (rows,432) and d xv (rows,648) (the A-NeRF MLP's input gradient), this kernel forms
//   dv_j = w'_j (sum_f dxd_f PE_f + sum_{m,a} dxv enc) + w_j sum_f dxd_f PE'_f,   dr_j = dxd[360 + 3j + a],
//   dq_j = dv_j r_j + (dr_j - (r_j . dr_j) r_j) / v_j,   d skts_j[0:3, :] += (A_j^T dq_j) (x) [p, 1]
// and, per ray, d d_j = sum_samples w_j dxv . d enc / d d_j,   d skts_j[0:3, 0:3] += (d d_j - (d_j . d d_j) d_j) / |R_j d_ray|
// (x) d_ray.  Row 3 of every d skts gets nothing.  Near/far (cylinders) and the sample depths come from the batch and
// are constants here, as on the DANBO pose path.
//
// Work layout: a warp per ray, lane j < 24 owns joint j and walks the ray's S samples.  A warp's loads of one row are
// then 24 consecutive floats per PE row, 72 for the unit vectors and 72 per direction-encoding row: every byte of the
// 4 320-byte fp32 gradient row is read by one coalesced access, with no shared-memory staging.  The 12 d skts entries
// of a joint stay in the lane's registers over the whole ray (all samples of a ray share its pose); the 4 warps of a
// block then reduce through shared memory and issue one set of 24 x 12 atomics per block when every ray of the block
// has the same pose (rays are image-major, so almost always), and per-warp atomics otherwise.
// 162 registers, no spills (-Xptxas -v): 4-warp blocks, 3 resident per SM.  With 8-warp blocks bounded to 2 per SM
// (128 registers) ptxas spills 176 bytes.
#include "field_common.cuh"

namespace danbo {
namespace anerf_bwd {

constexpr int kXD = 432, kXV = 648;
constexpr float kCutoff = 0.5f;          // cutoff_mm * ext_scale, as embed_kernel
constexpr int kWarps = 4;

__global__ void __launch_bounds__(kWarps * 32, 3)
embed_bwd_kernel(const float* __restrict__ rays, int ray_stride, int n_rays, int S, const float* __restrict__ z,
                 const float* __restrict__ pose_skts, int rays_per_pose, int n_poses, const float* __restrict__ align,
                 const float* __restrict__ ray_enc, float tau, const float* __restrict__ d_xd,
                 const float* __restrict__ d_xv, float* __restrict__ d_skts) {
    __shared__ float red[kWarps][DANBO_J][12];
    __shared__ int pose_of[kWarps];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int n = blockIdx.x * kWarps + wib;
    const bool live = n < n_rays;
    int pose = 0;
    if (live) { pose = n / rays_per_pose; if (pose >= n_poses) pose = n_poses - 1; }
    float acc[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) acc[i] = 0.f;
    if (live && lane < DANBO_J) {
        const int j = lane;
        const float* r = rays + (size_t)n * ray_stride;
        const float ox = r[0], oy = r[1], oz = r[2], dx = r[3], dy = r[4], dz = r[5];
        const float4* skt4 = reinterpret_cast<const float4*>(pose_skts + ((size_t)pose * DANBO_J + j) * 16);
        const float4* A4 = reinterpret_cast<const float4*>(align + j * 16);
        const float4 r0 = __ldg(skt4), r1 = __ldg(skt4 + 1), r2 = __ldg(skt4 + 2);
        const float4 a0 = __ldg(A4), a1 = __ldg(A4 + 1), a2 = __ldg(A4 + 2);
        // the ray's direction encoding of joint j (ray_kernel's fp32 values): enc[m][a]
        const float* e = ray_enc + (size_t)n * kXV + 3 * j;
        float enc[9][3];
#pragma unroll
        for (int m = 0; m < 9; ++m)
#pragma unroll
            for (int a = 0; a < 3; ++a) enc[m][a] = __ldg(e + m * 72 + a);
        float dd[3] = {0.f, 0.f, 0.f};            // d loss / d d_j, summed over the ray's samples
        for (int s = 0; s < S; ++s) {
            const size_t row = (size_t)n * S + s;
            const float* gx = d_xd + row * kXD;
            const float* gw = d_xv + row * kXV + 3 * j;
            float gpe[15], gr[3], gv[9][3];
#pragma unroll
            for (int f = 0; f < 15; ++f) gpe[f] = __ldg(gx + f * 24 + j);
#pragma unroll
            for (int a = 0; a < 3; ++a) gr[a] = __ldg(gx + 360 + 3 * j + a);
#pragma unroll
            for (int m = 0; m < 9; ++m)
#pragma unroll
                for (int a = 0; a < 3; ++a) gv[m][a] = __ldg(gw + m * 72 + a);
            // ---- forward recompute, embed_kernel's op order
            const float zz = __ldg(z + row);
            const float px = __fadd_rn(ox, __fmul_rn(dx, zz));
            const float py = __fadd_rn(oy, __fmul_rn(dy, zz));
            const float pz = __fadd_rn(oz, __fmul_rn(dz, zz));
            const float l0 = fmaf(r0.z, pz, fmaf(r0.y, py, fmaf(r0.x, px, r0.w)));
            const float l1 = fmaf(r1.z, pz, fmaf(r1.y, py, fmaf(r1.x, px, r1.w)));
            const float l2 = fmaf(r2.z, pz, fmaf(r2.y, py, fmaf(r2.x, px, r2.w)));
            const float q0 = __fadd_rn(fmaf(a0.z, l2, fmaf(a0.y, l1, __fmul_rn(a0.x, l0))), a0.w);
            const float q1 = __fadd_rn(fmaf(a1.z, l2, fmaf(a1.y, l1, __fmul_rn(a1.x, l0))), a1.w);
            const float q2 = __fadd_rn(fmaf(a2.z, l2, fmaf(a2.y, l1, __fmul_rn(a2.x, l0))), a2.w);
            const float v = sqrtf(q0 * q0 + q1 * q1 + q2 * q2);
            const float den = fmaxf(v, 1e-12f);
            const float rq[3] = {__fdiv_rn(q0, den), __fdiv_rn(q1, den), __fdiv_rn(q2, den)};
            const float w = 1.f - 1.f / (1.f + expf(-tau * (v - kCutoff)));
            const float wp = -tau * w * (1.f - w);                        // d w / d v
            const float inp = kCutoff - v;
            float sn, cs;
            sincosf(inp * (2.f / kCutoff) - 1.f, &sn, &cs);
            // ---- d v: T multiplies w' (the encodings' values), B multiplies w (their derivatives)
            float T = gpe[0] * inp, B = -gpe[0];
            float oct = 1.f;
#pragma unroll
            for (int f = 0; f < 7; ++f) {
                T = fmaf(gpe[1 + 2 * f], sn, fmaf(gpe[2 + 2 * f], cs, T));
                B = fmaf(oct * (-2.f / kCutoff), fmaf(gpe[1 + 2 * f], cs, -gpe[2 + 2 * f] * sn), B);
                if (f < 6) {
                    const float s2 = 2.f * sn * cs;
                    cs = 1.f - 2.f * sn * sn;
                    sn = s2;
                }
                oct *= 2.f;
            }
            // view input: value enc * w (-> T) and d enc / d d_j times w (-> dd)
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                float g = gv[0][a];                                          // d enc_0 / d d = 1
                T = fmaf(gv[0][a], enc[0][a], T);
#pragma unroll
                for (int f = 0; f < 4; ++f) {
                    const float fr = (float)(1 << f);
                    T = fmaf(gv[1 + 2 * f][a], enc[1 + 2 * f][a], fmaf(gv[2 + 2 * f][a], enc[2 + 2 * f][a], T));
                    g = fmaf(gv[1 + 2 * f][a], fr * enc[2 + 2 * f][a], g);   // d sin(2^f d) = 2^f cos(2^f d)
                    g = fmaf(gv[2 + 2 * f][a], -fr * enc[1 + 2 * f][a], g);  // d cos(2^f d) = -2^f sin(2^f d)
                }
                dd[a] = fmaf(w, g, dd[a]);
            }
            const float dv = fmaf(wp, T, w * B);
            // ---- d q = dv r + (dr - (r . dr) r) / v ; d l = A^T d q ; d [R | t] += d l (x) [p, 1]
            const float rdr = rq[0] * gr[0] + rq[1] * gr[1] + rq[2] * gr[2];
            float dq[3];
#pragma unroll
            for (int a = 0; a < 3; ++a) dq[a] = fmaf(dv, rq[a], (gr[a] - rdr * rq[a]) / den);
            const float dl[3] = {fmaf(a2.x, dq[2], fmaf(a1.x, dq[1], a0.x * dq[0])),
                                 fmaf(a2.y, dq[2], fmaf(a1.y, dq[1], a0.y * dq[0])),
                                 fmaf(a2.z, dq[2], fmaf(a1.z, dq[1], a0.z * dq[0]))};
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                acc[i * 4 + 0] = fmaf(dl[i], px, acc[i * 4 + 0]);
                acc[i * 4 + 1] = fmaf(dl[i], py, acc[i * 4 + 1]);
                acc[i * 4 + 2] = fmaf(dl[i], pz, acc[i * 4 + 2]);
                acc[i * 4 + 3] += dl[i];
            }
        }
        // ---- per ray: d_j = l / max(|l|, 1e-12), l = R_j d_ray (ray_kernel's op order)
        const float m0 = fmaf(r0.z, dz, fmaf(r0.y, dy, r0.x * dx));
        const float m1 = fmaf(r1.z, dz, fmaf(r1.y, dy, r1.x * dx));
        const float m2 = fmaf(r2.z, dz, fmaf(r2.y, dy, r2.x * dx));
        const float mden = fmaxf(sqrtf(m0 * m0 + m1 * m1 + m2 * m2), 1e-12f);
        const float ddd = enc[0][0] * dd[0] + enc[0][1] * dd[1] + enc[0][2] * dd[2];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float dm = (dd[i] - ddd * enc[0][i]) / mden;
            acc[i * 4 + 0] = fmaf(dm, dx, acc[i * 4 + 0]);
            acc[i * 4 + 1] = fmaf(dm, dy, acc[i * 4 + 1]);
            acc[i * 4 + 2] = fmaf(dm, dz, acc[i * 4 + 2]);
        }
    }
    // ---- reduction: one set of atomics per block when its rays share a pose
    if (lane < DANBO_J) {
#pragma unroll
        for (int i = 0; i < 12; ++i) red[wib][lane][i] = acc[i];
    }
    if (lane == 0) pose_of[wib] = live ? pose : -1;
    __syncthreads();
    const int p0 = pose_of[0];                 // warp 0 always holds a live ray
    bool uniform = true;
#pragma unroll
    for (int w = 1; w < kWarps; ++w) uniform = uniform && (pose_of[w] == p0 || pose_of[w] < 0);
    if (uniform) {
        for (int t = threadIdx.x; t < DANBO_J * 12; t += blockDim.x) {
            const int jj = t / 12, i = t % 12;
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < kWarps; ++w) s += red[w][jj][i];
            atomicAdd(d_skts + ((size_t)p0 * DANBO_J + jj) * 16 + (i >> 2) * 4 + (i & 3), s);
        }
    } else if (live && lane < DANBO_J) {
        float* dst = d_skts + ((size_t)pose * DANBO_J + lane) * 16;
#pragma unroll
        for (int i = 0; i < 12; ++i) atomicAdd(dst + (i >> 2) * 4 + (i & 3), acc[i]);
    }
}

}  // namespace anerf_bwd
}  // namespace danbo

using namespace danbo;

extern "C" int danbo_anerf_embed_bwd(const float* rays, int ray_stride, int n_rays, int S, const float* z,
                                     const float* pose_skts, int rays_per_pose, int n_poses, const float* align,
                                     const float* ray_enc, float tau, const float* d_xd, const float* d_xv,
                                     float* d_skts, void* stream) {
    if (n_rays <= 0) return 0;
    if (S <= 0 || ray_stride < 6 || rays_per_pose <= 0 || n_poses <= 0 || !d_skts || !d_xd || !d_xv) return -1;
    const int blocks = (n_rays + anerf_bwd::kWarps - 1) / anerf_bwd::kWarps;
    anerf_bwd::embed_bwd_kernel<<<blocks, anerf_bwd::kWarps * 32, 0, (cudaStream_t)stream>>>(
        rays, ray_stride, n_rays, S, z, pose_skts, rays_per_pose, n_poses, align, ray_enc, tau, d_xd, d_xv, d_skts);
    DANBO_CHECK_LAUNCH();
    return 0;
}
