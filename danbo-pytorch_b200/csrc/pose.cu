// The pose layer under --opt_pose: per-frame axis-angle parameters -> kinematic chain -> (kps, bones, skts) of the
// batch's poses, the trainer's pose regulariser, and the backward pass of both into the layer's gradient arena.
//
// Reference: PoseOptLayer core/pose_opt.py:132-339 (idx_to_params :210-224, the chain :264-339 with the pelvis shift,
// skts = inverse(l2ws)), axis_angle_to_matrix core/utils/skeleton_utils.py:411-418, Trainer._compute_kp_loss
// core/trainer.py:446-505 (without the temporal term).  The torch restatement is pose_opt.PoseOptLayer.calculate_kinematic
// and pose_opt.kp_loss; the kernels follow its op order:
//     R_j = R_parent(j) Rl_j,   t_j = R_parent(j) (rest_j - rest_parent(j)) + t_parent(j),   t_root = rest_root
//     kps_j = t_j + pelvis,     skts_j = [R_j^T | -R_j^T kps_j]
//     kp_loss = coef * mean_{pose, j >= 1} sum_c max((anchor - aa)^2 - tol, 0)      MPJPC = mean |anchor kps - kps| / ext
//
// Layout: one warp per pose, lane = joint (24 of 32 lanes).  A batch holds at most a few dozen poses of 24 joints, so
// the work is a few thousand flops: what matters is that it is one launch each way with no dependent global round
// trips.  The chain runs level by level (8 levels below the SMPL root): each level every lane reads its parent's
// (R, t) with 12 shuffles and the lanes of that depth update.  The backward pass recomputes the chain from the
// parameters (cheaper than saving it) and runs it leaf -> root through 1.1 KB of shared memory per warp: the lanes of
// a level write their contribution to the parent, the parents sum their children in a fixed order.  One block holds
// every pose (warp w takes poses w, w + warps, ...), so the regulariser and MPJPC are reduced in the block and written
// without atomics; the parameter gradients are added with atomics, since two poses of a batch may share a frame or a
// kp_map row.
#include "common.cuh"
#include "rotation.cuh"

namespace danbo {
namespace pose {

constexpr int kMaxWarps = 16;
constexpr int kLevels = 8;
__constant__ int c_parent[DANBO_J] = {0, 0, 0, 0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 9, 9, 12, 13, 14, 16, 17, 18, 19, 20, 21};
__constant__ int c_depth[DANBO_J] = {0, 1, 1, 1, 2, 2, 2, 3, 3, 3, 4, 4, 4, 4, 4, 5, 5, 5, 6, 6, 7, 7, 8, 8};

struct Layer {
    const float* pelvis;            // (F,3)
    const float* bones;             // (F,24,3), or (U,23,3) with kp_map
    const float* root_bones;        // (F,3) or NULL
    const long long* kp_map;        // (F) or NULL
    const float* rest;              // (R,24,3)
    int n_rest;
    const long long* rest_idx;      // (F) when n_rest > 1
    const long long* idx;           // frame of pose g: idx[g * idx_stride]
    int idx_stride;
    int n_poses;
};

// One lane's view of pose g: frame, axis-angle, rest position and offset to the parent.  Lanes >= 24 get joint 0's
// data so that they can take part in the shuffles; they store nothing.
struct Joint {
    long long f;
    int j, p, depth;
    float aa[3], rest[3], off[3];
};

__device__ __forceinline__ Joint load_joint(const Layer& L, int g, int lane) {
    Joint q;
    q.f = L.idx[(size_t)g * L.idx_stride];
    q.j = lane < DANBO_J ? lane : 0;
    q.p = c_parent[q.j];
    q.depth = lane < DANBO_J ? c_depth[q.j] : -1;
    const float* a;
    if (L.root_bones == nullptr) a = L.bones + ((size_t)q.f * DANBO_J + q.j) * 3;
    else if (q.j == 0) a = L.root_bones + (size_t)q.f * 3;
    else a = L.bones + ((size_t)L.kp_map[q.f] * (DANBO_J - 1) + q.j - 1) * 3;
    const long long row = L.n_rest == 1 ? 0 : L.rest_idx[q.f];
    const float* r = L.rest + (size_t)row * DANBO_J * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        q.aa[c] = a[c];
        q.rest[c] = r[q.j * 3 + c];
        q.off[c] = r[q.j * 3 + c] - r[q.p * 3 + c];
    }
    return q;
}

// World rotation and translation (before the pelvis shift) of every lane's joint; Rl = the joint's local rotation.
__device__ __forceinline__ void chain(const Joint& q, const float Rl[9], float R[9], float t[3]) {
#pragma unroll
    for (int m = 0; m < 9; ++m) R[m] = Rl[m];
#pragma unroll
    for (int c = 0; c < 3; ++c) t[c] = q.rest[c];
#pragma unroll 1
    for (int it = 1; it <= kLevels; ++it) {
        float pR[9], pt[3];
#pragma unroll
        for (int m = 0; m < 9; ++m) pR[m] = __shfl_sync(0xffffffffu, R[m], q.p);
#pragma unroll
        for (int c = 0; c < 3; ++c) pt[c] = __shfl_sync(0xffffffffu, t[c], q.p);
        if (q.depth == it) {
#pragma unroll
            for (int r = 0; r < 3; ++r) {
#pragma unroll
                for (int c = 0; c < 3; ++c)
                    R[r * 3 + c] = pR[r * 3] * Rl[c] + pR[r * 3 + 1] * Rl[3 + c] + pR[r * 3 + 2] * Rl[6 + c];
                t[r] = (pR[r * 3] * q.off[0] + pR[r * 3 + 1] * q.off[1] + pR[r * 3 + 2] * q.off[2]) + pt[r];
            }
        }
    }
}

__global__ void fwd_kernel(Layer L, const float* __restrict__ anchor_kps, const float* __restrict__ anchor_bones,
                           float tol, float coef, float ext_scale, float* __restrict__ kps, float* __restrict__ bones,
                           float* __restrict__ skts, float* __restrict__ stats) {
    __shared__ float red[2][kMaxWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    float reg = 0.f, pj = 0.f;
    for (int g = warp; g < L.n_poses; g += nw) {
        const Joint q = load_joint(L, g, lane);
        float Rl[9], R[9], t[3];
        axisang_to_rot(q.aa, Rl);
        chain(q, Rl, R, t);
#pragma unroll
        for (int c = 0; c < 3; ++c) t[c] += L.pelvis[(size_t)q.f * 3 + c];
        if (lane < DANBO_J) {
            const size_t at = (size_t)g * DANBO_J + q.j;
            float* s = skts + at * 16;
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                kps[at * 3 + r] = t[r];
                bones[at * 3 + r] = q.aa[r];
                s[r * 4 + 0] = R[0 * 3 + r];
                s[r * 4 + 1] = R[1 * 3 + r];
                s[r * 4 + 2] = R[2 * 3 + r];
                s[r * 4 + 3] = -(R[0 * 3 + r] * t[0] + R[1 * 3 + r] * t[1] + R[2 * 3 + r] * t[2]);
            }
            s[12] = 0.f; s[13] = 0.f; s[14] = 0.f; s[15] = 1.f;
            if (stats) {
                const float* ab = anchor_bones + ((size_t)q.f * DANBO_J + q.j) * 3;
                const float* ak = anchor_kps + ((size_t)q.f * DANBO_J + q.j) * 3;
                float e = 0.f;
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float d = (ab[c] - q.aa[c]) * (ab[c] - q.aa[c]);
                    if (q.j > 0 && d > tol) reg += d - tol;
                    e += (ak[c] - t[c]) * (ak[c] - t[c]);
                }
                pj += sqrtf(e);
            }
        }
    }
    if (!stats) return;
    reg = warp_sum(reg);
    pj = warp_sum(pj);
    if (lane == 0) { red[0][warp] = reg; red[1][warp] = pj; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = 0.f, b = 0.f;
        for (int w = 0; w < nw; ++w) { a += red[0][w]; b += red[1][w]; }
        stats[0] = a / (float)(L.n_poses * (DANBO_J - 1)) * coef;
        stats[1] = b / (float)(L.n_poses * DANBO_J) / ext_scale;
    }
}

__global__ void bwd_kernel(Layer L, const float* __restrict__ d_skts, const float* __restrict__ d_bones,
                           const float* __restrict__ d_kps, const float* __restrict__ anchor_bones,
                           const float* __restrict__ d_reg, float tol, float coef, float* __restrict__ g_pelvis,
                           float* __restrict__ g_bones, float* __restrict__ g_root_bones) {
    __shared__ float contrib[kMaxWarps][DANBO_J][12];          // a joint's (d R, d t) share for its parent
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const float reg_scale = d_reg ? *d_reg * coef * 2.f / (float)(L.n_poses * (DANBO_J - 1)) : 0.f;
    for (int g = warp; g < L.n_poses; g += nw) {
        const Joint q = load_joint(L, g, lane);
        float Rl[9], R[9], t[3];
        axisang_to_rot(q.aa, Rl);
        chain(q, Rl, R, t);
#pragma unroll
        for (int c = 0; c < 3; ++c) t[c] += L.pelvis[(size_t)q.f * 3 + c];
        float pR[9];
#pragma unroll
        for (int m = 0; m < 9; ++m) pR[m] = __shfl_sync(0xffffffffu, R[m], q.p);
        // direct gradients of this joint's outputs: skts = [R^T | -R^T t], kps = t
        float dR[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f}, dt[3] = {0.f, 0.f, 0.f};
        const size_t at = (size_t)g * DANBO_J + q.j;
        if (lane < DANBO_J) {
            const float* S = d_skts + at * 16;
            const float db[3] = {S[3], S[7], S[11]};
#pragma unroll
            for (int k = 0; k < 3; ++k) {
#pragma unroll
                for (int i = 0; i < 3; ++i) dR[k * 3 + i] = S[i * 4 + k] - t[k] * db[i];
                dt[k] = -(R[k * 3] * db[0] + R[k * 3 + 1] * db[1] + R[k * 3 + 2] * db[2]);
                if (d_kps) dt[k] += d_kps[at * 3 + k];
            }
        }
        // leaf -> root: a joint of depth `it` hands d R_p += dR Rl^T + dt off^T and d t_p += dt to its parent
#pragma unroll 1
        for (int it = kLevels; it >= 1; --it) {
            if (q.depth == it) {
                float* o = contrib[warp][q.j];
#pragma unroll
                for (int r = 0; r < 3; ++r) {
#pragma unroll
                    for (int c = 0; c < 3; ++c)
                        o[r * 3 + c] = dR[r * 3] * Rl[c * 3] + dR[r * 3 + 1] * Rl[c * 3 + 1] + dR[r * 3 + 2] * Rl[c * 3 + 2]
                                     + dt[r] * q.off[c];
                    o[9 + r] = dt[r];
                }
            }
            __syncwarp();
            if (q.depth == it - 1) {
                for (int k = 1; k < DANBO_J; ++k) {
                    if (c_parent[k] != q.j || c_depth[k] != it) continue;
                    const float* o = contrib[warp][k];
#pragma unroll
                    for (int m = 0; m < 9; ++m) dR[m] += o[m];
#pragma unroll
                    for (int c = 0; c < 3; ++c) dt[c] += o[9 + c];
                }
            }
            __syncwarp();
        }
        if (lane >= DANBO_J) continue;
        // d Rl = R_p^T d R (the root: Rl = R)
        float dRl[9];
#pragma unroll
        for (int r = 0; r < 3; ++r) {
#pragma unroll
            for (int c = 0; c < 3; ++c)
                dRl[r * 3 + c] = q.j == 0 ? dR[r * 3 + c]
                                          : pR[r] * dR[c] + pR[3 + r] * dR[3 + c] + pR[6 + r] * dR[6 + c];
        }
        float da[3];
        axisang_to_rot_bwd(q.aa, dRl, da);
        const float* ab = anchor_bones + ((size_t)q.f * DANBO_J + q.j) * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            if (d_bones) da[c] += d_bones[at * 3 + c];
            if (d_reg && q.j > 0) {
                const float e = q.aa[c] - ab[c];
                if (e * e > tol) da[c] += reg_scale * e;
            }
        }
        float* gb;
        if (L.root_bones == nullptr) gb = g_bones + ((size_t)q.f * DANBO_J + q.j) * 3;
        else if (q.j == 0) gb = g_root_bones + (size_t)q.f * 3;
        else gb = g_bones + ((size_t)L.kp_map[q.f] * (DANBO_J - 1) + q.j - 1) * 3;
#pragma unroll
        for (int c = 0; c < 3; ++c) atomicAdd(gb + c, da[c]);
        if (q.j == 0) {                              // the root's d t holds every joint's: t_j = ... + pelvis
#pragma unroll
            for (int c = 0; c < 3; ++c) atomicAdd(g_pelvis + (size_t)q.f * 3 + c, dt[c]);
        }
    }
}

// 2D keypoint reprojection term: joint j of pose g projects through P_g (3x4) to (u, v) = (P0 X, P1 X) / P2 X with
// X = [kps_j, 1]; the residual against the detection (u^, v^, c) is penalised per coordinate with Geman-McClure,
// rho(r) = s^2 r^2 / (s^2 + r^2), weighted by c.  loss = coef / (G * 24) * sum c (rho(r_u) + rho(r_v)); d kps is
// written in the same pass (d rho / d r = 2 s^4 r / (s^2 + r^2)^2, d u / d X = (P0 - u P2) / w).  A joint at or behind
// the camera (w <= 1e-6) adds nothing to the loss, the pixel error or the gradient.  Same layout as fwd_kernel: one
// block, warp w takes poses w, w + warps, ..., lane = joint; the loss and the pixel error are reduced in the block.
__global__ void kp2d_kernel(const float* __restrict__ kps, const float* __restrict__ kp2d, const float* __restrict__ proj,
                            int n_poses, float sigma, float coef, float* __restrict__ d_kps, float* __restrict__ stats) {
    __shared__ float red[3][kMaxWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const float s2 = sigma * sigma, scale = coef / (float)(n_poses * DANBO_J);
    float loss = 0.f, px = 0.f, seen = 0.f;
    for (int g = warp; g < n_poses; g += nw) {
        if (lane >= DANBO_J) continue;
        const size_t at = (size_t)g * DANBO_J + lane;
        const float* P = proj + (size_t)g * 12;
        const float X[3] = {kps[at * 3], kps[at * 3 + 1], kps[at * 3 + 2]};
        float h[3];
#pragma unroll
        for (int r = 0; r < 3; ++r) h[r] = P[r * 4] * X[0] + P[r * 4 + 1] * X[1] + P[r * 4 + 2] * X[2] + P[r * 4 + 3];
        const float c = kp2d[at * 3 + 2];
        float d[3] = {0.f, 0.f, 0.f};
        if (h[2] > 1e-6f) {
            const float u = h[0] / h[2], v = h[1] / h[2];
            const float ru = u - kp2d[at * 3], rv = v - kp2d[at * 3 + 1];
            const float qu = s2 + ru * ru, qv = s2 + rv * rv;
            loss += c * (s2 * ru * ru / qu + s2 * rv * rv / qv);
            if (c > 0.f) { px += sqrtf(ru * ru + rv * rv); seen += 1.f; }
            const float gu = scale * c * 2.f * s2 * s2 * ru / (qu * qu) / h[2];
            const float gv = scale * c * 2.f * s2 * s2 * rv / (qv * qv) / h[2];
#pragma unroll
            for (int k = 0; k < 3; ++k) d[k] = gu * (P[k] - u * P[8 + k]) + gv * (P[4 + k] - v * P[8 + k]);
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) d_kps[at * 3 + k] = d[k];
    }
    loss = warp_sum(loss);
    px = warp_sum(px);
    seen = warp_sum(seen);
    if (lane == 0) { red[0][warp] = loss; red[1][warp] = px; red[2][warp] = seen; }
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = 0.f, b = 0.f, n = 0.f;
        for (int w = 0; w < nw; ++w) { a += red[0][w]; b += red[1][w]; n += red[2][w]; }
        stats[0] = a * scale;
        stats[1] = n > 0.f ? b / n : 0.f;
    }
}

static int threads_for(int n_poses) { return 32 * (n_poses < kMaxWarps ? n_poses : kMaxWarps); }

static bool layer_ok(const Layer& L) {
    if (!L.pelvis || !L.bones || !L.rest || !L.idx || L.idx_stride <= 0 || L.n_rest <= 0) return false;
    if ((L.root_bones == nullptr) != (L.kp_map == nullptr)) return false;
    if (L.n_rest > 1 && !L.rest_idx) return false;
    return true;
}

}  // namespace pose
}  // namespace danbo

using namespace danbo;

extern "C" int danbo_pose_fwd(const float* pelvis, const float* bones, const float* root_bones, const long long* kp_map,
                              const float* rest_pose, int n_rest, const long long* rest_idx, const long long* idx,
                              int idx_stride, int n_poses, const float* anchor_kps, const float* anchor_bones, float tol,
                              float coef, float ext_scale, float* kps, float* bones_out, float* skts, float* stats,
                              void* stream) {
    if (n_poses <= 0) return 0;
    const pose::Layer L{pelvis, bones, root_bones, kp_map, rest_pose, n_rest, rest_idx, idx, idx_stride, n_poses};
    if (!pose::layer_ok(L) || !kps || !bones_out || !skts) return -1;
    if (stats && (!anchor_kps || !anchor_bones || !(ext_scale > 0.f))) return -1;
    pose::fwd_kernel<<<1, pose::threads_for(n_poses), 0, (cudaStream_t)stream>>>(
        L, anchor_kps, anchor_bones, tol, coef, ext_scale, kps, bones_out, skts, stats);
    DANBO_CHECK_LAUNCH();
    return 0;
}

extern "C" int danbo_pose_bwd(const float* pelvis, const float* bones, const float* root_bones, const long long* kp_map,
                              const float* rest_pose, int n_rest, const long long* rest_idx, const long long* idx,
                              int idx_stride, int n_poses, const float* d_skts, const float* d_bones, const float* d_kps,
                              const float* anchor_bones, const float* d_reg, float tol, float coef, float* g_pelvis,
                              float* g_bones, float* g_root_bones, void* stream) {
    if (n_poses <= 0) return 0;
    const pose::Layer L{pelvis, bones, root_bones, kp_map, rest_pose, n_rest, rest_idx, idx, idx_stride, n_poses};
    if (!pose::layer_ok(L) || !d_skts || !g_pelvis || !g_bones) return -1;
    if ((root_bones != nullptr) != (g_root_bones != nullptr)) return -1;
    if (d_reg && !anchor_bones) return -1;
    pose::bwd_kernel<<<1, pose::threads_for(n_poses), 0, (cudaStream_t)stream>>>(
        L, d_skts, d_bones, d_kps, anchor_bones, d_reg, tol, coef, g_pelvis, g_bones, g_root_bones);
    DANBO_CHECK_LAUNCH();
    return 0;
}

extern "C" int danbo_pose_kp2d(const float* kps, const float* kp2d, const float* proj, int n_poses, float sigma,
                               float coef, float* d_kps, float* stats, void* stream) {
    if (n_poses <= 0) return 0;
    if (!kps || !kp2d || !proj || !d_kps || !stats || !(sigma > 0.f)) return -1;
    pose::kp2d_kernel<<<1, pose::threads_for(n_poses), 0, (cudaStream_t)stream>>>(kps, kp2d, proj, n_poses, sigma, coef,
                                                                                  d_kps, stats);
    DANBO_CHECK_LAUNCH();
    return 0;
}
