// B*: backward of the field stages G1/G2, A1-A3 and the positional encoding (hand-written, fp32).
//
// Autograd of core/networks/danbo.py:261-302 + gnn_backbone.py:787-828 + misc.py:331-351 as reached from trainer.py:573:
//   d X (rows,208) -> d hbar -> d p_j, d h_j -> d logits (+ the soft-softmax gradient on confd) -> aggregation-net
//   parameters (V0, adjacency weights, biases, V1, V2), the bone feature lines (scatter-add into (G,24,240), the input
//   of the graph net's own autograd) and axis_scale (through the sampling coordinates x = t/|s|; the window is
//   detached, gnn_backbone.py:804).
// Same work layout as the forward: `field_rows_bwd` lane = row, `pair_logits_bwd` lane = (row, bone) pair with a warp
// holding 32 pairs of one bone; per-warp shared-memory tiles turn the per-pair outer products into per-weight sums.
#include "field_common.cuh"

namespace danbo {

__global__ void __launch_bounds__(128)
field_rows_bwd_kernel(const float* __restrict__ rays, int ray_stride, int n_rays, int S, const float* __restrict__ z,
                      const uint32_t* __restrict__ mask, const int* __restrict__ active_ids,
                      const int* __restrict__ active_count, int capacity, const float* __restrict__ pose_skts,
                      const float* __restrict__ pose_vol, int rays_per_pose, int n_poses, FieldConsts fc,
                      const float* __restrict__ logits, const float* __restrict__ hbar /* (rows,16) */,
                      const float* __restrict__ dX /* (rows,208) */, const float* __restrict__ g_logit_ext /* (n*S,24) or null */,
                      float* __restrict__ d_hbar /* (rows,16) */, float* __restrict__ d_logit /* (n*S,24) */,
                      int agg_mode /* 0 sigmoid, 1 masked softmax */) {
    int count = *active_count; if (count > capacity) count = capacity;
    const int total = n_rays * S;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < count; e += gridDim.x * blockDim.x) {
        const int id = active_ids[e];
        if (id >= total) continue;                      // empty entry: h = 0 is a constant
        const float* dx = dX + (size_t)e * 208;
        float dh[DANBO_FEAT];
#pragma unroll
        for (int i = 0; i < DANBO_FEAT; ++i) {
            const float h = hbar[(size_t)e * 16 + i];
            float sn, cs;
            sincosf(h, &sn, &cs);
            float g = dx[i], f = 1.f;
#pragma unroll
            for (int q = 0; q < 6; ++q) {
                g += f * (cs * dx[DANBO_FEAT + 30 * q + i] - sn * dx[DANBO_FEAT + 30 * q + DANBO_FEAT + i]);
                const float s2 = 2.f * sn * cs, c2 = 1.f - 2.f * sn * sn;
                sn = s2; cs = c2; f *= 2.f;
            }
            dh[i] = g;
            d_hbar[(size_t)e * 16 + i] = g;
        }
        const int n = id / S;
        const float* r = rays + (size_t)n * ray_stride;
        const float zz = z[id];
        const float px = __fadd_rn(r[0], __fmul_rn(r[3], zz));
        const float py = __fadd_rn(r[1], __fmul_rn(r[4], zz));
        const float pz = __fadd_rn(r[2], __fmul_rn(r[5], zz));
        int pose = n / rays_per_pose; if (pose >= n_poses) pose = n_poses - 1;
        const float* skt = pose_skts + (size_t)pose * DANBO_J * 16;
        const float* vol = pose_vol + (size_t)pose * DANBO_J * DANBO_VOL;
        const uint32_t vis = mask[id];
        const float* a_row = logits + (size_t)id * DANBO_J;
        float* da_row = d_logit + (size_t)id * DANBO_J;
        float amax = 0.f, inv_den = 0.f, dot = 0.f;      // softmax: dot = sum_j dL/dp_j p_j
        int amax_at = 0;
        if (agg_mode == 1) softmax_terms(a_row, vis, amax, inv_den, &amax_at);
        for (uint32_t m = vis; m;) {
            const int j = __ffs(m) - 1; m &= m - 1;
            float x0, x1, x2, h[DANBO_FEAT];
            bone_coords(skt + j * 16, fc.align + j * 16, fc.axis_scale + j * 3, px, py, pz, x0, x1, x2);
            bone_features(vol + j * DANBO_VOL, x0, x1, x2, h);
            float dp = 0.f;
#pragma unroll
            for (int i = 0; i < DANBO_FEAT; ++i) dp = fmaf(dh[i], h[i], dp);
            if (agg_mode == 1) {
                dot = fmaf(dp, expf(a_row[j] - amax) * inv_den, dot);
                da_row[j] = dp;                          // parked; turned into d a_j below
                continue;
            }
            const float sg = 1.f / (1.f + expf(-a_row[j]));
            float da = dp * 1.002f * sg * (1.f - sg);
            if (g_logit_ext) da += g_logit_ext[(size_t)id * DANBO_J + j];
            da_row[j] = da;
        }
        if (agg_mode == 1) {
            // p_j = e_j / D, e_j = v_j exp(a_j - M), D = sum_k e_k + 24 eps:  d a_k = p_k (dp_k - dot) for visible k, and
            // through M = max_k a_k (autograd routes it to the arg max): dM = -(24 eps / D) dot.  Every bone's entry is
            // written: the pair list of a softmax pass is dense.
            const float d_max = -(float)DANBO_J * kSoftmaxEps * inv_den * dot;
#pragma unroll 4
            for (int k = 0; k < DANBO_J; ++k) {
                float da = 0.f;
                if ((vis >> k) & 1u) {
                    da = expf(a_row[k] - amax) * inv_den * (da_row[k] - dot);
                    if (g_logit_ext) da += g_logit_ext[(size_t)id * DANBO_J + k];
                }
                if (k == amax_at) da += d_max;
                da_row[k] = da;
            }
        }
    }
}

struct AggGrads {             // fp32 accumulators (atomicAdd), shapes of the parameters
    float* w0; float* adjw; float* b0; float* w1; float* b1; float* w2; float* b2;
    float* vol;               // (G,24,240)
    float* axis_scale;        // (24,3)
    float* skts;              // (G,24,4,4) or nullptr: d loss / d world-to-bone matrices (pose optimisation, pose_opt.py:264-339)
};

constexpr int kTileLd = 33;

// column sums of a [32 pairs][32] tile -> lane o gets sum_p T[p][o]
__device__ __forceinline__ float tile_colsum(const float* T, int lane) {
    float s = 0.f;
#pragma unroll
    for (int p = 0; p < 32; ++p) s += T[p * kTileLd + lane];
    return s;
}

// kSoftmax: agg_mode 1 (dense pair lists, blend weight of the pair from the row's masked softmax); the sigmoid
// instantiation carries none of that code.  kWeightGrads = false (pose-only backward, the field is frozen): the
// aggregation net's weight / bias tile sums and atomics and the axis-scale gradient are compiled out; the backward
// through the three layers to each pair's d x, and from there to d vol and d skts, stays.
// kPointGrad (requires !kWeightGrads; the point-gradient backward, danbo_field_agg_bwd_pts): every pair also adds
// sum_k R_k^T A_k^T d t_k over the tree neighbours k of its bone to d_pts[id] (3 per-lane atomics: a warp's 32 pairs
// belong to different rows), d vol / d skts are skipped when their accumulator is NULL, and d t includes the
// derivative of the feature window exp(-2 sum x^6) - the true gradient of the field, where training detaches it.
template <bool kSoftmax, bool kWeightGrads, bool kPointGrad>
__device__ __forceinline__ void
pair_logits_bwd_body(const float* __restrict__ rays, int ray_stride, int S, const float* __restrict__ z,
                     const int* __restrict__ active_ids, const float* __restrict__ pose_skts,
                     const float* __restrict__ pose_vol, int rays_per_pose, int n_poses, const FieldConsts& fc,
                     const PairWork& pw, int pair_capacity, const float* __restrict__ logits,
                     const float* __restrict__ d_logit, const float* __restrict__ d_hbar, const AggGrads& G,
                     const uint32_t* __restrict__ mask, float* __restrict__ d_pts) {
    static_assert(!(kPointGrad && kWeightGrads), "the point-gradient variant forms no weight gradient");
    __shared__ float tiles[4][2][32 * kTileLd];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    float* T1 = tiles[wib][0];
    float* T2 = tiles[wib][1];
    const int* cnt = pw.count();
    int n_chunks = 0;
    for (int j = 0; j < DANBO_J; ++j) n_chunks += (cnt[j] + 31) >> 5;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; c < n_chunks; c += warps) {
        int j = 0, first = 0;
        for (;; ++j) { const int nc = (cnt[j] + 31) >> 5; if (c < first + nc) break; first += nc; }
        const int in_seg = (c - first) * 32 + lane;
        const int at = c * 32 + lane;
        const bool live = in_seg < cnt[j] && at < pair_capacity;
        float px = 0.f, py = 0.f, pz = 0.f, da = 0.f, pj = 0.f;
        int id = 0, pose = 0, row = 0;
        if (live) {
            row = pw.pairs()[at];
            id = active_ids[row];
            const int n = id / S;
            const float* r = rays + (size_t)n * ray_stride;
            const float zz = z[id];
            px = __fadd_rn(r[0], __fmul_rn(r[3], zz));
            py = __fadd_rn(r[1], __fmul_rn(r[4], zz));
            pz = __fadd_rn(r[2], __fmul_rn(r[5], zz));
            pose = n / rays_per_pose; if (pose >= n_poses) pose = n_poses - 1;
            da = d_logit[(size_t)id * DANBO_J + j];
            if (kSoftmax) {
                const uint32_t vis = mask[id];
                if ((vis >> j) & 1u) {
                    float amax, inv_den;
                    softmax_terms(logits + (size_t)id * DANBO_J, vis, amax, inv_den);
                    pj = expf(logits[(size_t)id * DANBO_J + j] - amax) * inv_den;
                }
            } else {
                pj = (1.f / (1.f + expf(-logits[(size_t)id * DANBO_J + j]))) * 1.002f - 0.001f;
            }
        }
        // dense (softmax) pair lists: a pair of an invisible bone that is not the row's arg max carries no gradient
        if (kSoftmax && !__any_sync(0xffffffffu, live && (da != 0.f || pj != 0.f))) continue;
        const float* skt = pose_skts + (size_t)pose * DANBO_J * 16;
        const float* vol = pose_vol + (size_t)pose * DANBO_J * DANBO_VOL;
        // ---- forward recompute: mix -> o1 -> l1 -> o2
        float mix[DANBO_AGG_W];
#pragma unroll
        for (int o = 0; o < DANBO_AGG_W; ++o) mix[o] = 0.f;
        for (uint32_t nb = kNbrMask[j]; nb;) {
            const int k = __ffs(nb) - 1; nb &= nb - 1;
            float x0, x1, x2, h[DANBO_FEAT];
            bone_coords(skt + k * 16, fc.align + k * 16, fc.axis_scale + k * 3, px, py, pz, x0, x1, x2);
            bone_features(vol + k * DANBO_VOL, x0, x1, x2, h);
            const float adj = __ldg(fc.agg_adjw + j * DANBO_J + k) * __ldg(fc.agg_adj + j * DANBO_J + k);
            const float* w = fc.agg_w0 + (size_t)k * DANBO_FEAT * DANBO_AGG_W;
#pragma unroll
            for (int i = 0; i < DANBO_FEAT; ++i) {
                const float hi = h[i] * adj;
#pragma unroll
                for (int o = 0; o < DANBO_AGG_W; ++o) mix[o] = fmaf(hi, __ldg(w + i * DANBO_AGG_W + o), mix[o]);
            }
        }
        float d1[DANBO_AGG_W];                           // l1 -> later delta1
#pragma unroll
        for (int o = 0; o < DANBO_AGG_W; ++o) { mix[o] = fmaxf(mix[o] + __ldg(fc.agg_b0 + o), 0.f); d1[o] = __ldg(fc.agg_b1 + j * DANBO_AGG_W + o); }
        const float* w1 = fc.agg_w1 + (size_t)j * DANBO_AGG_W * DANBO_AGG_W;
#pragma unroll
        for (int i = 0; i < DANBO_AGG_W; ++i)
#pragma unroll
            for (int o = 0; o < DANBO_AGG_W; ++o) d1[o] = fmaf(mix[i], __ldg(w1 + i * DANBO_AGG_W + o), d1[o]);
        // ---- layer 2 backward: a = sum_o relu(l1[o]) W2[j][o] + b2[j]
        if (!live) da = 0.f;
#pragma unroll
        for (int o = 0; o < DANBO_AGG_W; ++o) {
            if (kWeightGrads) T1[lane * kTileLd + o] = da * fmaxf(d1[o], 0.f);          // -> dW2
            d1[o] = d1[o] > 0.f ? da * __ldg(fc.agg_w2 + j * DANBO_AGG_W + o) : 0.f;   // delta1
            if (kWeightGrads) T2[lane * kTileLd + o] = d1[o];
        }
        if (kWeightGrads) {
            __syncwarp();
            atomicAdd(G.w2 + j * DANBO_AGG_W + lane, tile_colsum(T1, lane));
            atomicAdd(G.b1 + j * DANBO_AGG_W + lane, tile_colsum(T2, lane));
            { const float s = warp_sum(da); if (lane == 0) atomicAdd(G.b2 + j, s); }
            __syncwarp();
            // ---- layer 1 backward: dW1[j][i][o] += o1[i] delta1[o];  d o1[i] = sum_o delta1[o] W1[j][i][o]
#pragma unroll
            for (int o = 0; o < DANBO_AGG_W; ++o) T1[lane * kTileLd + o] = mix[o];      // o1 of every pair
            __syncwarp();
            {
                float acc[DANBO_AGG_W];                      // lane = weight row i
#pragma unroll
                for (int o = 0; o < DANBO_AGG_W; ++o) acc[o] = 0.f;
                for (int p = 0; p < 32; ++p) {
                    const float a = T1[p * kTileLd + lane];
#pragma unroll
                    for (int o = 0; o < DANBO_AGG_W; ++o) acc[o] = fmaf(a, T2[p * kTileLd + o], acc[o]);
                }
#pragma unroll
                for (int o = 0; o < DANBO_AGG_W; ++o) atomicAdd(G.w1 + ((size_t)j * DANBO_AGG_W + lane) * DANBO_AGG_W + o, acc[o]);
            }
            __syncwarp();
        }
        float d0[DANBO_AGG_W];                           // delta0 = d o1 * [o1 > 0]
#pragma unroll
        for (int i = 0; i < DANBO_AGG_W; ++i) {
            float s = 0.f;
            // a plain load in the pose-only variant: with no atomics in between, ptxas would otherwise keep all 1 024 W1
            // values of the forward recompute's __ldg loads live for this loop (255 registers, 2.6 KB of spills)
#pragma unroll
            for (int o = 0; o < DANBO_AGG_W; ++o)
                s = fmaf(d1[o], kWeightGrads ? __ldg(w1 + i * DANBO_AGG_W + o) : w1[i * DANBO_AGG_W + o], s);
            d0[i] = mix[i] > 0.f ? s : 0.f;
            if (kWeightGrads) T2[lane * kTileLd + i] = d0[i];
        }
        if (kWeightGrads) {
            __syncwarp();
            atomicAdd(G.b0 + lane, tile_colsum(T2, lane));
            __syncwarp();
        }
        // ---- layer 0 + adjacency mix + feature gather, per tree neighbour
        float gp[3] = {0.f, 0.f, 0.f};                   // kPointGrad: d / d p, summed over the neighbours
        for (uint32_t nb = kNbrMask[j]; nb;) {
            const int k = __ffs(nb) - 1; nb &= nb - 1;
            float x[3], h[DANBO_FEAT];
            bone_coords(skt + k * 16, fc.align + k * 16, fc.axis_scale + k * 3, px, py, pz, x[0], x[1], x[2]);
            bone_features(vol + k * DANBO_VOL, x[0], x[1], x[2], h);
            const float adjw = __ldg(fc.agg_adjw + j * DANBO_J + k), adjm = __ldg(fc.agg_adj + j * DANBO_J + k);
            const float adj = adjw * adjm;
            const float* w = fc.agg_w0 + (size_t)k * DANBO_FEAT * DANBO_AGG_W;
            // d adj = sum_o delta0[o] * (h . W0[k][:, o]);  d h[i] = adj * sum_o delta0[o] W0[k][i][o]
            float dadj = 0.f, dh[DANBO_FEAT];
#pragma unroll
            for (int i = 0; i < DANBO_FEAT; ++i) {
                float s = 0.f;
#pragma unroll
                for (int o = 0; o < DANBO_AGG_W; ++o) s = fmaf(d0[o], __ldg(w + i * DANBO_AGG_W + o), s);
                dadj = fmaf(h[i], s, dadj);
                dh[i] = adj * s;
            }
            if (kWeightGrads) {
                { const float s = warp_sum(live ? dadj : 0.f); if (lane == 0) atomicAdd(G.adjw + j * DANBO_J + k, s * adjm); }
                // dW0[k][i][o] += h[i] * adj * delta0[o]: tiles T1 = h (15 cols), T2 = adj * delta0
#pragma unroll
                for (int i = 0; i < DANBO_FEAT; ++i) T1[lane * kTileLd + i] = live ? h[i] : 0.f;
#pragma unroll
                for (int o = 0; o < DANBO_AGG_W; ++o) T2[lane * kTileLd + o] = adj * d0[o];
                __syncwarp();
                {
                    float acc[DANBO_FEAT];                   // lane = output unit o
#pragma unroll
                    for (int i = 0; i < DANBO_FEAT; ++i) acc[i] = 0.f;
                    for (int p = 0; p < 32; ++p) {
                        const float t = T2[p * kTileLd + lane];
#pragma unroll
                        for (int i = 0; i < DANBO_FEAT; ++i) acc[i] = fmaf(T1[p * kTileLd + i], t, acc[i]);
                    }
#pragma unroll
                    for (int i = 0; i < DANBO_FEAT; ++i) atomicAdd(G.w0 + ((size_t)k * DANBO_FEAT + i) * DANBO_AGG_W + lane, acc[i]);
                }
                __syncwarp();
            }
            if (k == j && live) {                        // direct path: hbar = sum_j p_j h_j
#pragma unroll
                for (int i = 0; i < DANBO_FEAT; ++i) dh[i] = fmaf(pj, d_hbar[(size_t)row * 16 + i], dh[i]);
            }
            // ---- feature gather backward (window detached): taps -> d vol, interpolation weight -> d x -> d axis_scale
            const float a2 = x[0] * x[0], b2 = x[1] * x[1], c2 = x[2] * x[2];
            const float win = expf(-2.f * (a2 * a2 * a2 + b2 * b2 * b2 + c2 * c2 * c2));
            const bool dvol_on = !kPointGrad || G.vol != nullptr;
            float* dvol = dvol_on ? G.vol + ((size_t)pose * DANBO_J + k) * DANBO_VOL : nullptr;
            const float* volk = vol + k * DANBO_VOL;
            float dt[3];                                             // d loss / d t, t = A_k (R_k p + t_k) + a_k = x |s|
            float sw = 0.f;                                          // kPointGrad: sum_c dh[c] * un-windowed h[c]
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const float iy = ((x[a] + 1.f) * (float)DANBO_RES - 1.f) * 0.5f;
                const float fl = floorf(iy);
                const float wt1 = iy - fl, wt0 = 1.f - wt1;
                const int i0 = (int)fl, i1 = i0 + 1;
                const bool ok0 = i0 >= 0 && i0 < DANBO_RES, ok1 = i1 >= 0 && i1 < DANBO_RES;
                float dxa = 0.f;
#pragma unroll
                for (int f = 0; f < 5; ++f) {
                    const float g = dh[f * 3 + a] * win;
                    const int base = f * (DANBO_RES * 3) + a;
                    const float v0 = ok0 ? __ldg(volk + base + i0 * 3) : 0.f;
                    const float v1 = ok1 ? __ldg(volk + base + i1 * 3) : 0.f;
                    if (live && ok0 && dvol_on) atomicAdd(dvol + base + i0 * 3, g * wt0);
                    if (live && ok1 && dvol_on) atomicAdd(dvol + base + i1 * 3, g * wt1);
                    dxa = fmaf(g, v1 - v0, dxa);
                    if (kPointGrad) sw = fmaf(dh[f * 3 + a], v0 * wt0 + v1 * wt1, sw);
                }
                dxa *= 0.5f * (float)DANBO_RES;                      // d iy / d x
                const float sc = __ldg(fc.axis_scale + k * 3 + a);
                if (kWeightGrads) {
                    // x = t / |s|  ->  d x / d s = -x / |s| * sign(s) = -x / s
                    const float ds = warp_sum(live ? -dxa * x[a] / sc : 0.f);
                    if (lane == 0) atomicAdd(G.axis_scale + k * 3 + a, ds);
                }
                dt[a] = live ? dxa / fabsf(sc) : 0.f;
            }
            if (kPointGrad) {
                // the window's own derivative: d win / d x_a = -12 x_a^5 win, times the un-windowed taps of all 15
                // channels (d h[c] / d x_a = h[c] / win * d win / d x_a)
                const float cw = -12.f * win * sw;
#pragma unroll
                for (int a = 0; a < 3; ++a) {
                    const float x2 = x[a] * x[a];
                    if (live) dt[a] += cw * x2 * x2 * x[a] / fabsf(__ldg(fc.axis_scale + k * 3 + a));
                }
            }
            if (kPointGrad || G.skts != nullptr) {
                // ---- d x -> d skts[pose][k] (encoders.py:288-303, :442-444): t = A l + a, l = R p + t_k, so
                // d l = A^T d t and d [R | t_k] = d l (x) [p, 1].  A warp's pairs usually share their pose (rays are
                // image-major): one warp reduction and 12 atomics; mixed warps fall back to per-lane atomics.
                const float* A = fc.align + k * 16;
                float dl[3];
#pragma unroll
                for (int i = 0; i < 3; ++i)
                    dl[i] = fmaf(__ldg(A + 8 + i), dt[2], fmaf(__ldg(A + 4 + i), dt[1], __ldg(A + i) * dt[0]));
                if (kPointGrad) {                                    // d p = R^T d l
                    const float* R = skt + k * 16;
#pragma unroll
                    for (int c = 0; c < 3; ++c)
                        gp[c] = fmaf(__ldg(R + 8 + c), dl[2], fmaf(__ldg(R + 4 + c), dl[1], fmaf(__ldg(R + c), dl[0], gp[c])));
                }
                const uint32_t lm = __ballot_sync(0xffffffffu, live);
                if ((!kPointGrad || G.skts != nullptr) && lm != 0u) {
                    const int pose_ref = __shfl_sync(0xffffffffu, pose, __ffs(lm) - 1);
                    const float pw4[4] = {px, py, pz, 1.f};
                    if (__all_sync(0xffffffffu, !live || pose == pose_ref)) {
                        float* dst = G.skts + ((size_t)pose_ref * DANBO_J + k) * 16;
#pragma unroll
                        for (int i = 0; i < 3; ++i)
#pragma unroll
                            for (int c = 0; c < 4; ++c) {
                                const float v = warp_sum(dl[i] * pw4[c]);          // dl = 0 on dead lanes
                                if (lane == 0) atomicAdd(dst + i * 4 + c, v);
                            }
                    } else if (live) {
                        float* dst = G.skts + ((size_t)pose * DANBO_J + k) * 16;
#pragma unroll
                        for (int i = 0; i < 3; ++i)
#pragma unroll
                            for (int c = 0; c < 4; ++c) atomicAdd(dst + i * 4 + c, dl[i] * pw4[c]);
                    }
                }
            }
        }
        if (kPointGrad && live) {
#pragma unroll
            for (int c = 0; c < 3; ++c) atomicAdd(d_pts + (size_t)id * 3 + c, gp[c]);
        }
    }
}

template <bool kSoftmax, bool kWeightGrads>
__global__ void __launch_bounds__(128)
pair_logits_bwd_kernel(const float* __restrict__ rays, int ray_stride, int S, const float* __restrict__ z,
                       const int* __restrict__ active_ids, const float* __restrict__ pose_skts,
                       const float* __restrict__ pose_vol, int rays_per_pose, int n_poses, FieldConsts fc, PairWork pw,
                       int pair_capacity, const float* __restrict__ logits, const float* __restrict__ d_logit,
                       const float* __restrict__ d_hbar, AggGrads G, const uint32_t* __restrict__ mask) {
    pair_logits_bwd_body<kSoftmax, kWeightGrads, false>(rays, ray_stride, S, z, active_ids, pose_skts, pose_vol,
                                                        rays_per_pose, n_poses, fc, pw, pair_capacity, logits, d_logit,
                                                        d_hbar, G, mask, nullptr);
}

// d_pts (n_rays*S, 3): d / d sample position, added to; G.vol / G.skts may be NULL, the other accumulators are unused
template <bool kSoftmax>
__global__ void __launch_bounds__(128)
pair_logits_bwd_pts_kernel(const float* __restrict__ rays, int ray_stride, int S, const float* __restrict__ z,
                           const int* __restrict__ active_ids, const float* __restrict__ pose_skts,
                           const float* __restrict__ pose_vol, int rays_per_pose, int n_poses, FieldConsts fc,
                           PairWork pw, int pair_capacity, const float* __restrict__ logits,
                           const float* __restrict__ d_logit, const float* __restrict__ d_hbar, AggGrads G,
                           const uint32_t* __restrict__ mask, float* __restrict__ d_pts) {
    pair_logits_bwd_body<kSoftmax, false, true>(rays, ray_stride, S, z, active_ids, pose_skts, pose_vol, rays_per_pose,
                                                n_poses, fc, pw, pair_capacity, logits, d_logit, d_hbar, G, mask, d_pts);
}

}  // namespace danbo

using namespace danbo;

static FieldConsts make_consts_b(const float* const* p) {
    FieldConsts fc;
    fc.align = p[0]; fc.axis_scale = p[1]; fc.agg_w0 = p[2]; fc.agg_adjw = p[3]; fc.agg_adj = p[4];
    fc.agg_b0 = p[5]; fc.agg_w1 = p[6]; fc.agg_b1 = p[7]; fc.agg_w2 = p[8]; fc.agg_b2 = p[9];
    return fc;
}

// grads[10] = { d_w0 (24,15,32), d_adj_w (24,24), d_b0 (32), d_w1 (24,32,32), d_b1 (24,32), d_w2 (24,32), d_b2 (24),
//               d_vol (n_poses,24,240), d_axis_scale (24,3), d_skts (n_poses,24,4,4) or NULL }: fp32 accumulators, added
//               to (zero them first).  d_skts = NULL (poses are constants) skips that gradient.  grads[0..6] and
//               grads[8] all NULL (all or none) select the pose-only variant: no aggregation-net or axis-scale gradient.
// work / pair_capacity: the SAME workspace the forward danbo_field_agg call filled (pair lists are reused).
extern "C" int danbo_field_agg_bwd(const float* rays, int ray_stride, int n_rays, int S, const float* z,
                                   const unsigned int* mask, const int* active_ids, const int* active_count,
                                   int capacity, const float* pose_skts, const float* pose_vol, int rays_per_pose,
                                   int n_poses, const float* const* consts, const float* logits, const float* hbar,
                                   const float* dX, const float* g_logit_ext, float* d_hbar, float* d_logit,
                                   const int* work, int pair_capacity, float* const* grads, int num_sms, int agg_mode,
                                   void* stream) {
    if (capacity <= 0) return 0;
    if (agg_mode < 0 || agg_mode > 1) return -1;
    if (grads == nullptr || grads[7] == nullptr) return -1;
    int n_weight = grads[8] != nullptr;
    for (int i = 0; i < 7; ++i) n_weight += grads[i] != nullptr;
    if (n_weight != 0 && n_weight != 8) return -1;
    const bool wg = n_weight == 8;
    cudaStream_t st = (cudaStream_t)stream;
    const FieldConsts fc = make_consts_b(consts);
    int rblocks = (capacity + 127) / 128;
    if (rblocks > num_sms * 16) rblocks = num_sms * 16;
    field_rows_bwd_kernel<<<rblocks, 128, 0, st>>>(rays, ray_stride, n_rays, S, z, mask, active_ids, active_count,
                                                    capacity, pose_skts, pose_vol, rays_per_pose, n_poses, fc, logits,
                                                    hbar, dX, g_logit_ext, d_hbar, d_logit, agg_mode);
    DANBO_CHECK_LAUNCH();
    AggGrads G{grads[0], grads[1], grads[2], grads[3], grads[4], grads[5], grads[6], grads[7], grads[8], grads[9]};
    PairWork pw{const_cast<int*>(work)};
    int pblocks = (pair_capacity / 32 + 3) / 4;
    if (pblocks > num_sms * 4) pblocks = num_sms * 4;
    auto kern = agg_mode == 1 ? (wg ? pair_logits_bwd_kernel<true, true> : pair_logits_bwd_kernel<true, false>)
                              : (wg ? pair_logits_bwd_kernel<false, true> : pair_logits_bwd_kernel<false, false>);
    kern<<<pblocks, 128, 0, st>>>(rays, ray_stride, S, z, active_ids, pose_skts, pose_vol, rays_per_pose, n_poses, fc, pw,
                                  pair_capacity, logits, d_logit, d_hbar, G, mask);
    DANBO_CHECK_LAUNCH();
    return 0;
}

// The point-gradient backward: field_rows_bwd as above, then the kPointGrad pair kernel.  d_pts (n_rays*S, 3) receives
// d / d p of every sample (added to); d_vol (n_poses,24,240) and d_skts (n_poses,24,4,4) are optional (NULL: skipped).
// The feature window is NOT detached here (see pair_logits_bwd_body), so d_skts is the true derivative, not training's.
extern "C" int danbo_field_agg_bwd_pts(const float* rays, int ray_stride, int n_rays, int S, const float* z,
                                       const unsigned int* mask, const int* active_ids, const int* active_count,
                                       int capacity, const float* pose_skts, const float* pose_vol, int rays_per_pose,
                                       int n_poses, const float* const* consts, const float* logits, const float* hbar,
                                       const float* dX, const float* g_logit_ext, float* d_hbar, float* d_logit,
                                       const int* work, int pair_capacity, float* d_pts, float* d_vol, float* d_skts,
                                       int num_sms, int agg_mode, void* stream) {
    if (capacity <= 0) return 0;
    if (agg_mode < 0 || agg_mode > 1) return -1;
    if (d_pts == nullptr) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    const FieldConsts fc = make_consts_b(consts);
    int rblocks = (capacity + 127) / 128;
    if (rblocks > num_sms * 16) rblocks = num_sms * 16;
    field_rows_bwd_kernel<<<rblocks, 128, 0, st>>>(rays, ray_stride, n_rays, S, z, mask, active_ids, active_count,
                                                    capacity, pose_skts, pose_vol, rays_per_pose, n_poses, fc, logits,
                                                    hbar, dX, g_logit_ext, d_hbar, d_logit, agg_mode);
    DANBO_CHECK_LAUNCH();
    AggGrads G{nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, d_vol, nullptr, d_skts};
    PairWork pw{const_cast<int*>(work)};
    int pblocks = (pair_capacity / 32 + 3) / 4;
    if (pblocks > num_sms * 4) pblocks = num_sms * 4;
    auto kern = agg_mode == 1 ? pair_logits_bwd_pts_kernel<true> : pair_logits_bwd_pts_kernel<false>;
    kern<<<pblocks, 128, 0, st>>>(rays, ray_stride, S, z, active_ids, pose_skts, pose_vol, rays_per_pose, n_poses, fc, pw,
                                  pair_capacity, logits, d_logit, d_hbar, G, mask, d_pts);
    DANBO_CHECK_LAUNCH();
    return 0;
}
