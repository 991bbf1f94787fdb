// GN1 + GN2: the per-pose skeleton graph net (pose -> 24 x 240 bone feature lines), forward and backward.
//
// Reference: encode_graph_inputs core/encoders.py:460-473, AxisAngtoRot6DEncoder :859-877 (axis-angle -> quaternion ->
// matrix, first two columns), Embedder core/cutoff_embedder.py:62-73 (5 octaves), BodyGNN.forward
// core/networks/gnn_backbone.py:683-704 on FactorizeGNN: DensePNGCN :225-274 (per-joint linear, then the learned
// 24x24 mix adj_w * adj, shared bias), ParallelLinear core/networks/misc.py:174-183.
//     n0 = mask_root * w            lin0[j] = n0[j] W0[j]     pre0 = A0 lin0 + b0      n1 = relu(2 pre0)   (the x2: SURVEY F3)
//     lin1[j] = n1[j] W1[j]         pre1 = A1 lin1 + b1       n2 = relu(pre1)
//     n3 = relu(n2[j] W2[j] + b2[j])                          out[j] = n3[j] W3[j] + b3[j]
// The work is tiny (<= 16 poses x 24 nodes, 28 MFLOP forward) and latency bound: as PyTorch ops it was ~50 launches
// forward and ~100 backward of a 1.6 ms training iteration, and a first version with one block per node (24 blocks, a
// 128-long dependent chain of weight loads per thread) still took 0.35 ms.  Now every layer is one launch over
// (node, 32-column tile | 16-row slice, 16-pose group) blocks: forward blocks rebuild the node's input vector (the
// adjacency mix of the previous launch's output), split K over their 8 warps and reduce through shared memory;
// backward blocks own a 16-row slice of the node's weight matrix, for both its gradient (one owner thread per entry:
// plain += unless there are several pose groups) and the transposed product.  4 launches forward, 4 backward, fp32.
#include "common.cuh"
#include "rotation.cuh"
#include <math.h>

namespace danbo {
namespace gn {

constexpr int kG = 16;             // poses per block
constexpr int kW = 128;            // node width
constexpr int kIn = 66;            // 6 * (1 + 2 * 5)
constexpr int kOut = DANBO_VOL;    // 240
constexpr int kThreads = 256;
constexpr int kTile = 32;          // output columns per forward block
constexpr int kSlice = 16;         // weight rows per backward block
constexpr int kP = kW + 1;         // shared-memory pitch of a 128-wide row

struct Params {
    const float* w0; const float* adjw0; const float* adj0; const float* b0;     // (24,66,128) (24,24) (24,24) (128)
    const float* w1; const float* adjw1; const float* adj1; const float* b1;     // (24,128,128) ... (128)
    const float* w2; const float* b2;                                            // (24,128,128) (24,128)
    const float* w3; const float* b3;                                            // (24,128,240) (24,240)
};
struct Saved {                     // activations kept for the backward pass, all (G,24,*)
    float* w_in; float* lin0; float* n1; float* lin1; float* n2; float* n3;
};
struct Grads {                     // accumulated into (+=)
    float* w0; float* adjw0; float* b0; float* w1; float* adjw1; float* b1; float* w2; float* b2; float* w3; float* b3;
};

// Graph inputs of (pose g, joint j): rot6d of the axis-angle (quaternion route, skeleton_utils.py:411-418) and its
// 5-octave encoding [x, sin 2^0 x, cos 2^0 x, sin 2^1 x, ...] in blocks of 6, zeroed for the root (mask_root).
// One thread per (pose, rot6d component i): it writes the 11 entries that derive from component i.  It computes only
// the entry it needs rather than calling axisang_to_rot (rotation.cuh), which compiles one sum differently (an FADD
// becomes an FFMA) and would change the graph net's outputs in the last bit.
__device__ __forceinline__ void graph_inputs(const float* __restrict__ aa, int j, int i, float* row, float* keep) {
    const float ax = aa[0], ay = aa[1], az = aa[2];
    const float ang = sqrtf(ax * ax + ay * ay + az * az), half = 0.5f * ang;
    const float k = fabsf(ang) < 1e-6f ? 0.5f - ang * ang / 48.f : sinf(half) / ang;
    const float qr = cosf(half), qi = ax * k, qj = ay * k, qk = az * k;
    const float two_s = 2.f / (qr * qr + qi * qi + qj * qj + qk * qk);
    float r;
    switch (i) {                                                                   // R00 R01 R10 R11 R20 R21
        case 0: r = 1.f - two_s * (qj * qj + qk * qk); break;
        case 1: r = two_s * (qi * qj - qk * qr); break;
        case 2: r = two_s * (qi * qj + qk * qr); break;
        case 3: r = 1.f - two_s * (qi * qi + qk * qk); break;
        case 4: r = two_s * (qi * qk - qj * qr); break;
        default: r = two_s * (qj * qk + qi * qr); break;
    }
    const float root = j == 0 ? 0.f : 1.f;
    float v = r * root;
    row[i] = v;
    if (keep) keep[i] = v;
#pragma unroll
    for (int f = 0; f < 5; ++f) {
        const float x = r * (float)(1 << f);
        v = sinf(x) * root; row[6 + 12 * f + i] = v; if (keep) keep[6 + 12 * f + i] = v;
        v = cosf(x) * root; row[12 + 12 * f + i] = v; if (keep) keep[12 + 12 * f + i] = v;
    }
}

// dst[g][c] (c < 128) = sum_k A[j][k] src[g][k][c], A = adj_w * adj with zero entries skipped.  Thread = (column, half of
// the poses).  With kT the transposed mix (node k collects from the nodes j it feeds) for the backward pass.
template <bool kT>
__device__ __forceinline__ void mix(const float* __restrict__ adjw, const float* __restrict__ adj, int node,
                                    const float* __restrict__ src, int g0, int ng, float (&acc)[kG / 2]) {
    const int c = threadIdx.x & (kW - 1), half = threadIdx.x >> 7;
#pragma unroll
    for (int u = 0; u < kG / 2; ++u) acc[u] = 0.f;
    for (int o = 0; o < DANBO_J; ++o) {
        const int e = kT ? o * DANBO_J + node : node * DANBO_J + o;
        const float m = __ldg(adj + e);
        if (m == 0.f) continue;
        const float a = __ldg(adjw + e) * m;
#pragma unroll
        for (int u = 0; u < kG / 2; ++u) {
            const int g = half * (kG / 2) + u;
            if (g < ng) acc[u] = fmaf(a, src[((size_t)(g0 + g) * DANBO_J + o) * kW + c], acc[u]);
        }
    }
}

// ---- forward ----------------------------------------------------------------------------------------------------
// MODE 0: graph inputs -> lin0.   MODE 1: n1 = relu(2 (A0 lin0 + b0)) -> lin1.   MODE 2: n2 = relu(A1 lin1 + b1) ->
// n3 = relu(n2 W2 + b2).   MODE 3: n3 -> out = n3 W3 + b3.   Block = (node, 32-column tile, pose group).
template <int MODE>
__global__ void __launch_bounds__(kThreads)
fwd_kernel(const float* __restrict__ bones, int G, Params P, Saved S, float* __restrict__ out) {
    constexpr int n_in = MODE == 0 ? kIn : kW;
    constexpr int n_out = MODE == 3 ? kOut : kW;
    __shared__ float in_s[kG * kP];
    __shared__ float red_s[(kThreads / 32) * kG * kTile];
    const int j = blockIdx.x, c0 = blockIdx.y * kTile, g0 = blockIdx.z * kG, ng = min(kG, G - g0);
    const int tid = threadIdx.x;
    // ---- the node's input vector for every pose of the group
    if (MODE == 0) {
        for (int e = tid; e < kG * kP; e += kThreads) in_s[e] = 0.f;
        __syncthreads();
        if (tid < ng * 6) {
            const int g = tid / 6, i = tid - g * 6;
            graph_inputs(bones + ((size_t)(g0 + g) * DANBO_J + j) * 3, j, i, in_s + g * kP,
                         blockIdx.y == 0 ? S.w_in + ((size_t)(g0 + g) * DANBO_J + j) * kIn : nullptr);
        }
    } else if (MODE == 3) {
        for (int e = tid; e < kG * kW; e += kThreads) {
            const int g = e >> 7, c = e & (kW - 1);
            in_s[g * kP + c] = g < ng ? S.n3[((size_t)(g0 + g) * DANBO_J + j) * kW + c] : 0.f;
        }
    } else {
        float acc[kG / 2];
        mix<false>(MODE == 1 ? P.adjw0 : P.adjw1, MODE == 1 ? P.adj0 : P.adj1, j, MODE == 1 ? S.lin0 : S.lin1, g0, ng, acc);
        const int c = tid & (kW - 1), half = tid >> 7;
        const float b = __ldg((MODE == 1 ? P.b0 : P.b1) + c);
        float* keep = MODE == 1 ? S.n1 : S.n2;
#pragma unroll
        for (int u = 0; u < kG / 2; ++u) {
            const int g = half * (kG / 2) + u;
            const float pre = acc[u] + b;
            const float v = g < ng ? fmaxf(MODE == 1 ? pre + pre : pre, 0.f) : 0.f;
            in_s[g * kP + c] = v;
            if (g < ng && blockIdx.y == 0) keep[((size_t)(g0 + g) * DANBO_J + j) * kW + c] = v;
        }
    }
    __syncthreads();
    // ---- out[g][c0 + lane] = sum_i in[g][i] W[i][c0 + lane]: K split over the 8 warps (rows i = warp, warp + 8, ...)
    const float* W = MODE == 0 ? P.w0 + (size_t)j * kIn * kW : MODE == 1 ? P.w1 + (size_t)j * kW * kW
                   : MODE == 2 ? P.w2 + (size_t)j * kW * kW : P.w3 + (size_t)j * kW * kOut;
    const int lane = tid & 31, ks = tid >> 5, c = c0 + lane;
    float acc[kG];
#pragma unroll
    for (int g = 0; g < kG; ++g) acc[g] = 0.f;
    if (c < n_out) {
#pragma unroll 8
        for (int i = ks; i < n_in; i += kThreads / 32) {
            const float w = __ldg(W + (size_t)i * n_out + c);
#pragma unroll
            for (int g = 0; g < kG; ++g) acc[g] = fmaf(in_s[g * kP + i], w, acc[g]);
        }
    }
#pragma unroll
    for (int g = 0; g < kG; ++g) red_s[(ks * kG + g) * kTile + lane] = acc[g];
    __syncthreads();
    for (int o = tid; o < kG * kTile; o += kThreads) {
        const int g = o >> 5, l = o & 31, cc = c0 + l;
        float v = 0.f;
#pragma unroll
        for (int k = 0; k < kThreads / 32; ++k) v += red_s[(k * kG + g) * kTile + l];
        if (g >= ng || cc >= n_out) continue;
        const size_t at = (size_t)(g0 + g) * DANBO_J + j;
        if (MODE == 0) S.lin0[at * kW + cc] = v;
        else if (MODE == 1) S.lin1[at * kW + cc] = v;
        else if (MODE == 2) S.n3[at * kW + cc] = fmaxf(v + __ldg(P.b2 + j * kW + cc), 0.f);
        else out[at * kOut + cc] = v + __ldg(P.b3 + j * kOut + cc);
    }
}

// ---- backward ---------------------------------------------------------------------------------------------------
// MODE 3: d out -> dW3, db3, d pre2.   MODE 2: d pre2 -> dW2, db2, d pre1, db1.   MODE 1: d pre1 -> (un-mix) d lin1 ->
// dA1, dW1, d pre0, db0.   MODE 0: d pre0 -> d lin0 -> dA0, dW0.   Block = (node, 16-row slice of its weight matrix,
// pose group).  kGrads = false (pose-only backward, the graph net is frozen): the transposed products only, i.e. MODE
// 3..1 leave d pre2, d pre1 and d pre0 (what bwd_pose_kernel reads) and no weight, bias or adjacency gradient; MODE 0
// then has nothing to do and is not launched.
template <int MODE, bool kGrads>
__global__ void __launch_bounds__(kThreads)
bwd_kernel(int G, Params P, Saved S, const float* __restrict__ d_in, Grads Gr, float* __restrict__ d_next) {
    constexpr int n_in = MODE == 0 ? kIn : kW;              // rows of the weight matrix
    constexpr int n_out = MODE == 3 ? kOut : kW;            // its columns = width of d
    constexpr int pd = n_out + 1;
    __shared__ float d_s[kG * pd];                          // d (lin | pre | out) of this node, every pose
    __shared__ float w_s[MODE == 0 ? 1 : kSlice * pd];      // the slice's weight rows
    __shared__ float a_s[kG * kSlice];                      // the slice of the node's input activations
    __shared__ float red[kThreads / 32];
    const int node = blockIdx.x, i0 = blockIdx.y * kSlice, g0 = blockIdx.z * kG, ng = min(kG, G - g0);
    const int tid = threadIdx.x;
    const bool excl = gridDim.z == 1, first = blockIdx.y == 0;
    const int nr = min(kSlice, n_in - i0);
    // ---- d of this node
    if (MODE >= 2) {
        for (int e = tid; e < kG * n_out; e += kThreads) {
            const int g = e / n_out, c = e - g * n_out;
            d_s[g * pd + c] = g < ng ? d_in[((size_t)(g0 + g) * DANBO_J + node) * n_out + c] : 0.f;
        }
    } else {
        const float* adjw = MODE == 1 ? P.adjw1 : P.adjw0;
        const float* adj = MODE == 1 ? P.adj1 : P.adj0;
        float dl[kG / 2];
        mix<true>(adjw, adj, node, d_in, g0, ng, dl);
        const int c = tid & (kW - 1), half = tid >> 7;
#pragma unroll
        for (int u = 0; u < kG / 2; ++u) d_s[(half * (kG / 2) + u) * pd + c] = dl[u];
        if (kGrads && first) {
            // d A[j][node] = sum_{g,c} d pre[g][j][c] lin[g][node][c];  d adj_w = d A * adj
            const float* lin = MODE == 1 ? S.lin1 : S.lin0;
            float* d_adjw = MODE == 1 ? Gr.adjw1 : Gr.adjw0;
            float lk[kG / 2];
#pragma unroll
            for (int u = 0; u < kG / 2; ++u) {
                const int g = half * (kG / 2) + u;
                lk[u] = g < ng ? lin[((size_t)(g0 + g) * DANBO_J + node) * kW + c] : 0.f;
            }
            for (int j = 0; j < DANBO_J; ++j) {
                const float m = __ldg(adj + j * DANBO_J + node);             // block-uniform
                if (m == 0.f) continue;
                float dot = 0.f;
#pragma unroll
                for (int u = 0; u < kG / 2; ++u) {
                    const int g = half * (kG / 2) + u;
                    if (g < ng) dot = fmaf(d_in[((size_t)(g0 + g) * DANBO_J + j) * kW + c], lk[u], dot);
                }
                dot = warp_sum(dot);
                if ((tid & 31) == 0) red[tid >> 5] = dot;
                __syncthreads();
                if (tid == 0) {
                    float s = 0.f;
#pragma unroll
                    for (int w = 0; w < kThreads / 32; ++w) s += red[w];
                    if (excl) d_adjw[j * DANBO_J + node] += s * m; else atomicAdd(d_adjw + j * DANBO_J + node, s * m);
                }
                __syncthreads();
            }
        }
    }
    // ---- the slice's activations and weight rows
    const float* act = MODE == 3 ? S.n3 : MODE == 2 ? S.n2 : MODE == 1 ? S.n1 : S.w_in;
    {
        const int g = tid & (kG - 1), il = tid >> 4;
        a_s[g * kSlice + il] = (g < ng && il < nr) ? act[((size_t)(g0 + g) * DANBO_J + node) * n_in + i0 + il] : 0.f;
    }
    const float* W = MODE == 3 ? P.w3 + (size_t)node * kW * kOut : MODE == 2 ? P.w2 + (size_t)node * kW * kW
                   : P.w1 + (size_t)node * kW * kW;
    if (MODE >= 1) {
        for (int e = tid; e < kSlice * n_out; e += kThreads) {
            const int il = e / n_out, c = e - il * n_out;
            w_s[il * pd + c] = il < nr ? __ldg(W + (size_t)(i0 + il) * n_out + c) : 0.f;
        }
    }
    __syncthreads();
    // ---- dW[i][c] += sum_g act[g][i] d[g][c] for the slice's rows: one owner thread per entry
    float* dW = MODE == 3 ? Gr.w3 + (size_t)node * kW * kOut : MODE == 2 ? Gr.w2 + (size_t)node * kW * kW
              : MODE == 1 ? Gr.w1 + (size_t)node * kW * kW : Gr.w0 + (size_t)node * kIn * kW;
    for (int e = tid; kGrads && e < nr * n_out; e += kThreads) {
        const int il = e / n_out, c = e - il * n_out;
        float s = 0.f;
#pragma unroll
        for (int g = 0; g < kG; ++g) s = fmaf(a_s[g * kSlice + il], d_s[g * pd + c], s);
        float* dst = dW + (size_t)(i0 + il) * n_out + c;
        if (excl) *dst += s; else atomicAdd(dst, s);
    }
    // ---- per-joint bias of layers 2 and 3
    if (kGrads && MODE >= 2 && first) {
        float* db = MODE == 3 ? Gr.b3 + node * kOut : Gr.b2 + node * kW;
        for (int c = tid; c < n_out; c += kThreads) {
            float s = 0.f;
#pragma unroll
            for (int g = 0; g < kG; ++g) s += d_s[g * pd + c];
            if (excl) db[c] += s; else atomicAdd(db + c, s);
        }
    }
    // ---- d act[g][i] = sum_c d[g][c] W[i][c] for the slice's rows, through the ReLU, to the previous layer
    if (MODE >= 1) {
        const int g = tid & (kG - 1), il = tid >> 4;
        float s = 0.f;
#pragma unroll 8
        for (int c = 0; c < n_out; ++c) s = fmaf(d_s[g * pd + c], w_s[il * pd + c], s);
        float v = a_s[g * kSlice + il] > 0.f ? (MODE == 1 ? s + s : s) : 0.f;      // n1 = relu(2 pre0)
        if (g >= ng || il >= nr) v = 0.f;
        if (g < ng && il < nr) d_next[((size_t)(g0 + g) * DANBO_J + node) * kW + i0 + il] = v;
        if (kGrads && MODE <= 2) {                           // shared biases b1 / b0: summed over poses and nodes
            float sb = v;
#pragma unroll
            for (int o = kG / 2; o > 0; o >>= 1) sb += __shfl_xor_sync(0xffffffffu, sb, o);
            if (g == 0 && il < nr) atomicAdd((MODE == 2 ? Gr.b1 : Gr.b0) + i0 + il, sb);
        }
    }
}

// ---- d pose: layer 0's d pre-activation -> d axis-angle --------------------------------------------------------
// d lin0 = A0^T d pre0 (the transposed mix), d w_in = mask_root (W0[j] d lin0), then back through the 5-octave PE with
// the sin / cos values the forward kept in saved[0] (d sin(2^f x) / dx = 2^f cos(2^f x)), rot6d = (R00 R01 R10 R11
// R20 R21) and the quaternion route.  Block = (node, pose), 128 threads: thread = column of d lin0, then warp = rows of
// W0[j]; the root's row is zero (mask_root).
__global__ void __launch_bounds__(kW)
bwd_pose_kernel(const float* __restrict__ bones, Params P, Saved S, const float* __restrict__ d_pre0,
                float* __restrict__ d_bones) {
    __shared__ float dl[kW];
    __shared__ float dw[kIn];
    const int node = blockIdx.x, g = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    const size_t at = (size_t)g * DANBO_J + node;
    if (node == 0) {
        if (tid < 3) d_bones[at * 3 + tid] = 0.f;
        return;
    }
    float acc = 0.f;
    for (int o = 0; o < DANBO_J; ++o) {
        const int e = o * DANBO_J + node;
        const float m = __ldg(P.adj0 + e);
        if (m == 0.f) continue;
        acc = fmaf(__ldg(P.adjw0 + e) * m, d_pre0[((size_t)g * DANBO_J + o) * kW + tid], acc);
    }
    dl[tid] = acc;
    __syncthreads();
    for (int i = tid >> 5; i < kIn; i += kW / 32) {
        const float* w = P.w0 + ((size_t)node * kIn + i) * kW;
        float s = 0.f;
#pragma unroll
        for (int c = lane; c < kW; c += 32) s = fmaf(__ldg(w + c), dl[c], s);
        s = warp_sum(s);
        if (lane == 0) dw[i] = s;
    }
    __syncthreads();
    if (tid >= 32) return;
    float dx = 0.f;
    if (lane < 6) {
        const float* keep = S.w_in + at * kIn;
        dx = dw[lane];
#pragma unroll
        for (int f = 0; f < 5; ++f)
            dx += (float)(1 << f) * (keep[12 + 12 * f + lane] * dw[6 + 12 * f + lane]
                                     - keep[6 + 12 * f + lane] * dw[12 + 12 * f + lane]);
    }
    float gR[9] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    gR[0] = __shfl_sync(0xffffffffu, dx, 0); gR[1] = __shfl_sync(0xffffffffu, dx, 1);
    gR[3] = __shfl_sync(0xffffffffu, dx, 2); gR[4] = __shfl_sync(0xffffffffu, dx, 3);
    gR[6] = __shfl_sync(0xffffffffu, dx, 4); gR[7] = __shfl_sync(0xffffffffu, dx, 5);
    if (lane == 0) {
        const float a[3] = {bones[at * 3], bones[at * 3 + 1], bones[at * 3 + 2]};
        float da[3];
        axisang_to_rot_bwd(a, gR, da);
        d_bones[at * 3] = da[0]; d_bones[at * 3 + 1] = da[1]; d_bones[at * 3 + 2] = da[2];
    }
}

}  // namespace gn
}  // namespace danbo

using namespace danbo;

static gn::Params gn_params(const float* const* p) {
    gn::Params P;
    P.w0 = p[0]; P.adjw0 = p[1]; P.adj0 = p[2]; P.b0 = p[3]; P.w1 = p[4]; P.adjw1 = p[5]; P.adj1 = p[6]; P.b1 = p[7];
    P.w2 = p[8]; P.b2 = p[9]; P.w3 = p[10]; P.b3 = p[11];
    return P;
}
static gn::Saved gn_saved(float* const* s) { return gn::Saved{s[0], s[1], s[2], s[3], s[4], s[5]}; }

extern "C" int danbo_graph_net_fwd(const float* pose_bones, int n_poses, const float* const* params, float* const* saved,
                                   float* vol_out, void* stream) {
    if (n_poses <= 0) return 0;
    if (!pose_bones || !params || !saved || !vol_out) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    const gn::Params P = gn_params(params);
    const gn::Saved S = gn_saved(saved);
    const int groups = (n_poses + gn::kG - 1) / gn::kG;
    const dim3 g128(DANBO_J, gn::kW / gn::kTile, groups), g240(DANBO_J, (gn::kOut + gn::kTile - 1) / gn::kTile, groups);
    gn::fwd_kernel<0><<<g128, gn::kThreads, 0, st>>>(pose_bones, n_poses, P, S, nullptr);
    DANBO_CHECK_LAUNCH();
    gn::fwd_kernel<1><<<g128, gn::kThreads, 0, st>>>(pose_bones, n_poses, P, S, nullptr);
    DANBO_CHECK_LAUNCH();
    gn::fwd_kernel<2><<<g128, gn::kThreads, 0, st>>>(pose_bones, n_poses, P, S, nullptr);
    DANBO_CHECK_LAUNCH();
    gn::fwd_kernel<3><<<g240, gn::kThreads, 0, st>>>(pose_bones, n_poses, P, S, vol_out);
    DANBO_CHECK_LAUNCH();
    return 0;
}

// grads = NULL: the pose-only variant (three launches, no weight gradients); work then still holds d pre0 for
// danbo_graph_net_bwd_pose.
extern "C" int danbo_graph_net_bwd(int n_poses, const float* const* params, float* const* saved, const float* d_vol,
                                   float* const* grads, float* work /* 2 * n_poses*24*128 floats */, void* stream) {
    if (n_poses <= 0) return 0;
    if (!params || !saved || !d_vol || !work) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    const gn::Params P = gn_params(params);
    const gn::Saved S = gn_saved(saved);
    float* d_pre1 = work;
    float* d_pre0 = work + (size_t)n_poses * DANBO_J * gn::kW;
    const int groups = (n_poses + gn::kG - 1) / gn::kG;
    const dim3 g128(DANBO_J, gn::kW / gn::kSlice, groups), g66(DANBO_J, (gn::kIn + gn::kSlice - 1) / gn::kSlice, groups);
    if (grads == nullptr) {
        const gn::Grads none{};
        gn::bwd_kernel<3, false><<<g128, gn::kThreads, 0, st>>>(n_poses, P, S, d_vol, none, d_pre0);
        DANBO_CHECK_LAUNCH();
        gn::bwd_kernel<2, false><<<g128, gn::kThreads, 0, st>>>(n_poses, P, S, d_pre0, none, d_pre1);
        DANBO_CHECK_LAUNCH();
        gn::bwd_kernel<1, false><<<g128, gn::kThreads, 0, st>>>(n_poses, P, S, d_pre1, none, d_pre0);
        DANBO_CHECK_LAUNCH();
        return 0;
    }
    const gn::Grads Gr{grads[0], grads[1], grads[2], grads[3], grads[4], grads[5], grads[6], grads[7], grads[8], grads[9]};
    // d_pre2 lives in d_pre0's buffer: it is consumed (by <2>) before <1> writes d_pre0
    gn::bwd_kernel<3, true><<<g128, gn::kThreads, 0, st>>>(n_poses, P, S, d_vol, Gr, d_pre0);
    DANBO_CHECK_LAUNCH();
    gn::bwd_kernel<2, true><<<g128, gn::kThreads, 0, st>>>(n_poses, P, S, d_pre0, Gr, d_pre1);
    DANBO_CHECK_LAUNCH();
    gn::bwd_kernel<1, true><<<g128, gn::kThreads, 0, st>>>(n_poses, P, S, d_pre1, Gr, d_pre0);
    DANBO_CHECK_LAUNCH();
    gn::bwd_kernel<0, true><<<g66, gn::kThreads, 0, st>>>(n_poses, P, S, d_pre0, Gr, nullptr);
    DANBO_CHECK_LAUNCH();
    return 0;
}

extern "C" int danbo_graph_net_bwd_pose(const float* pose_bones, int n_poses, const float* const* params,
                                        float* const* saved, const float* work, float* d_pose_bones, void* stream) {
    if (n_poses <= 0) return 0;
    if (!pose_bones || !params || !saved || !work || !d_pose_bones) return -1;
    const gn::Params P = gn_params(params);
    const gn::Saved S = gn_saved(saved);
    const float* d_pre0 = work + (size_t)n_poses * DANBO_J * gn::kW;     // where danbo_graph_net_bwd leaves it
    gn::bwd_pose_kernel<<<dim3(DANBO_J, n_poses), gn::kW, 0, (cudaStream_t)stream>>>(pose_bones, P, S, d_pre0,
                                                                                      d_pose_bones);
    DANBO_CHECK_LAUNCH();
    return 0;
}
