// C1 alpha compositing, R1 importance resampling + sorted merge order, R2 merge of coarse and fine samples.
// Reference: core/networks/nerf.py:281-347 (raw2outputs), core/utils/ray_utils.py:159-203,257-291
// (sample_pdf / isample_from_lineseg), core/raycasters.py:484-514,745-761 (_merge_encodings / merge_samples).
//
// Forward: a group of kL lanes per ray, 32 / kL rays per warp; backward: one warp per ray.  cumprod / cumsum
// accumulate in fp64 like ATen's CPU kernels (acc_type<float>) and round each output to fp32.  16 B raw + 4 B z in,
// 8 B (weight, alpha) out per sample: too few bytes to bind the forward kernels to HBM, they are bound by instruction issue.
#include "common.cuh"
#include "field_common.cuh"
#include <math.h>

namespace danbo {

constexpr int kMaxS = 160;          // longest ray: 96 + 48 = 144 samples
constexpr int kEPL = 5;             // elements per lane at kMaxS
constexpr int kWarpsPerBlock = 4;

struct RaySmem {
    float z[kMaxS];
    float w[kMaxS];
    float cdf[kMaxS];
    float cat[kMaxS];
    float zs[kMaxS];
    int order[kMaxS];
};

__device__ __forceinline__ double warp_excl_prod(double v, int lane) {
    double inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const double u = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc *= u; }
    const double ex = __shfl_up_sync(0xffffffffu, inc, 1);
    return lane == 0 ? 1.0 : ex;
}
__device__ __forceinline__ double warp_excl_sum(double v, int lane) {
    double inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const double u = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += u; }
    const double ex = __shfl_up_sync(0xffffffffu, inc, 1);
    return lane == 0 ? 0.0 : ex;
}

// ---- forward kernels: a group of kL lanes composites one ray, a warp holds 32 / kL rays.  The per-ray work that does
// not grow with S (setup, scans, reductions, the map stores, the merge bookkeeping) is then shared by the rays of a warp
// instead of being repeated by all 32 lanes for every ray.
//
// Sample layout.  The fp32 sums behind the maps (rgb, disp, acc) are defined on a 32-lane layout: virtual lane v holds
// the kEo = ceil(S / 32) samples v*kEo .. v*kEo + kEo - 1, sums them in order, and the 32 partial sums meet in an xor
// butterfly (16, 8, 4, 2, 1).  Lane g of a group holds the virtual lanes g, g + kL, g + 2 kL, ..., so the butterfly levels
// >= kL are lane-local and the rest are shuffles of width kL: the maps come out bit-identical for every kL.
// The fp64 transmittance product is scanned per round of kL virtual lanes; that association differs from a 32-lane scan
// and can move a weight by one fp32 ulp only when the fp64 product lies within 2^-29 (relative) of an fp32 rounding tie.
// The pdf and cdf sums are fp64 sums of fp32 terms no smaller than 1e-5 / total and are exact in any order.
//
// Every lane of a warp stays to the end: a group past the last ray computes on the last ray and stores nothing, so the
// full-warp shuffles of its neighbours stay defined.  Shuffles use width kL, votes and __syncwarp the group's mask.

template <int kL>
__device__ __forceinline__ unsigned group_mask(int lane) {
    return kL == 32 ? 0xffffffffu : ((1u << kL) - 1u) << (lane & ~(kL - 1));
}
template <int kL>
__device__ __forceinline__ double group_incl_prod(double v, int g) {
#pragma unroll
    for (int o = 1; o < kL; o <<= 1) { const double u = __shfl_up_sync(0xffffffffu, v, o, kL); if (g >= o) v *= u; }
    return v;
}
template <int kL>
__device__ __forceinline__ double group_incl_sum(double v, int g) {
#pragma unroll
    for (int o = 1; o < kL; o <<= 1) { const double u = __shfl_up_sync(0xffffffffu, v, o, kL); if (g >= o) v += u; }
    return v;
}
template <int kL, class T>
__device__ __forceinline__ T group_sum(T v) {
#pragma unroll
    for (int o = kL / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o, kL);
    return v;
}

// Composites one ray of S samples (z[0..S), fetch(i) -> raw (rgb, sigma)) on the kL lanes of its group; kEo = ceil(S / 32).
// Writes the weights / alpha rows and the maps when `store`; leaves the weights in w_sm when it is given.
template <int kL, int kEo, class Fetch>
__device__ __forceinline__ void composite_group(const float* z, int S, int g, unsigned gmask, bool store, float norm_d,
                                                float inv_B, const float* __restrict__ noise_row, Fetch fetch, float* w_sm,
                                                float* __restrict__ w_row, float* __restrict__ alpha_row,
                                                float* __restrict__ rgb_out, float* __restrict__ disp_out,
                                                float* __restrict__ acc_out) {
    constexpr int R = 32 / kL;                          // virtual lanes per lane
    float al[R][kEo], cr[R][kEo], cg[R][kEo], cb[R][kEo];
    double lp[R];
#pragma unroll
    for (int j = 0; j < R; ++j) {
        lp[j] = 1.0;
#pragma unroll
        for (int e = 0; e < kEo; ++e) {
            const int i = (j * kL + g) * kEo + e;
            al[j][e] = 0.f; cr[j][e] = cg[j][e] = cb[j][e] = 0.f;
            if (i < S) {
                const float4 raw = fetch(i);
                float d = (i + 1 < S) ? __fsub_rn(z[i + 1], z[i]) : 1e10f;
                d = __fmul_rn(d, norm_d);
                cr[j][e] = (1.f / (1.f + expf(-raw.x))) * 1.002f - 0.001f;
                cg[j][e] = (1.f / (1.f + expf(-raw.y))) * 1.002f - 0.001f;
                cb[j][e] = (1.f / (1.f + expf(-raw.z))) * 1.002f - 0.001f;
                float sg = __fmul_rn(raw.w, inv_B);
                if (noise_row) sg = __fadd_rn(sg, noise_row[i]);
                sg = fmaxf(sg, 0.f);
                al[j][e] = __fsub_rn(1.f, expf(-__fmul_rn(sg, d)));
                lp[j] *= (double)__fadd_rn(__fsub_rn(1.f, al[j][e]), 1e-10f);
            }
        }
    }
    // exclusive product before each virtual lane: a group scan per round, times the product of the rounds before it
    double T[R];
    double carry = 1.0;
#pragma unroll
    for (int j = 0; j < R; ++j) {
        const double inc = group_incl_prod<kL>(lp[j], g);
        const double ex = __shfl_up_sync(0xffffffffu, inc, 1, kL);
        T[j] = carry * (g == 0 ? 1.0 : ex);
        if (j + 1 < R) carry *= __shfl_sync(0xffffffffu, inc, kL - 1, kL);
    }
    float pr[R], pg[R], pb[R], pd[R], pw[R];
#pragma unroll
    for (int j = 0; j < R; ++j) {
        double t = T[j];
        pr[j] = pg[j] = pb[j] = pd[j] = pw[j] = 0.f;
#pragma unroll
        for (int e = 0; e < kEo; ++e) {
            const int i = (j * kL + g) * kEo + e;
            if (i < S) {
                const float w = __fmul_rn(al[j][e], (float)t);
                t *= (double)__fadd_rn(__fsub_rn(1.f, al[j][e]), 1e-10f);
                if (w_sm) w_sm[i] = w;
                if (store) {
                    if (w_row) w_row[i] = w;
                    alpha_row[i] = al[j][e];
                }
                pr[j] = fmaf(w, cr[j][e], pr[j]); pg[j] = fmaf(w, cg[j][e], pg[j]); pb[j] = fmaf(w, cb[j][e], pb[j]);
                pd[j] = fmaf(w, z[i], pd[j]); pw[j] += w;
            }
        }
    }
    // butterfly levels 16 .. kL: virtual lanes j*kL + g and (j + m)*kL + g sit in the same lane
#pragma unroll
    for (int m = R / 2; m > 0; m >>= 1)
#pragma unroll
        for (int j = 0; j < m; ++j) {
            pr[j] += pr[j + m]; pg[j] += pg[j + m]; pb[j] += pb[j + m]; pd[j] += pd[j + m]; pw[j] += pw[j + m];
        }
    const float sr = group_sum<kL>(pr[0]), sg = group_sum<kL>(pg[0]), sb = group_sum<kL>(pb[0]);
    const float sd = group_sum<kL>(pd[0]), sw = group_sum<kL>(pw[0]);
    if (store && g == 0) {
        rgb_out[0] = sr; rgb_out[1] = sg; rgb_out[2] = sb;
        float disp = 1.f / fmaxf(1e-10f, sd / (sw + 1e-10f));
        if (fabsf(sw) <= 1e-8f) disp = 0.f;                         // torch.isclose(sum w, 0) -> disparity 0
        *disp_out = disp;
        *acc_out = fminf(sw, 1.f);
    }
    __syncwarp(gmask);
}

// Coarse pass: composite + inverse-CDF importance sampling + merge order.  Dynamic shared memory: per ray, z[S], w[S],
// cdf[S], and for S_f > 0 the fine samples zs[S_f] with their stable sort (values, indices) when they are out of order.
template <int kL, int kEo>
__global__ void __launch_bounds__(32 * kWarpsPerBlock)
composite_resample_kernel(const float* __restrict__ rays, int ray_stride, int n_rays, int S, int S_f,
                          const float* __restrict__ raw /* (n_rays*S + n_rays, 4); tail = per-ray empty sample */,
                          const uint32_t* __restrict__ mask, const float* __restrict__ z,
                          const float* __restrict__ noise, float inv_B, const float* __restrict__ u_vals /* (S_f) or null */,
                          const float* __restrict__ u_rand /* (n_rays,S_f) or null */,
                          float* __restrict__ weights /* or null */, float* __restrict__ alpha, float* __restrict__ rgb0,
                          float* __restrict__ disp0, float* __restrict__ acc0, float* __restrict__ z_samples,
                          float* __restrict__ z_all, int* __restrict__ order_out, int* __restrict__ inds_out,
                          int smooth /* 1: single_net weights (is_only, ray_utils.py:272-279); 0: the interior weights */) {
    extern __shared__ float dsm[];
    constexpr int kE = (32 / kL) * kEo;                 // samples per lane
    const int lane = threadIdx.x & 31, g = lane & (kL - 1), slot = threadIdx.x / kL;
    const unsigned gmask = group_mask<kL>(lane);
    const int n_slot = blockIdx.x * (blockDim.x / kL) + slot;
    const bool valid = n_slot < n_rays;
    const int n = valid ? n_slot : n_rays - 1;
    float* sz = dsm + (size_t)slot * (3 * S + 3 * S_f);
    float* sw = sz + S;
    float* scdf = sw + S;
    float* szs = scdf + S;
    float* sfz = szs + S_f;
    int* sfi = reinterpret_cast<int*>(sfz + S_f);
    const float* r = rays + (size_t)n * ray_stride;
    const float norm_d = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(r[3], r[3]), __fmul_rn(r[4], r[4])), __fmul_rn(r[5], r[5])));
    for (int i = g; i < S; i += kL) sz[i] = z[(size_t)n * S + i];
    __syncwarp(gmask);
    const float4* raw4 = reinterpret_cast<const float4*>(raw);
    const float4 empty = raw4[(size_t)n_rays * S + n];
    // the raw row is read only for an active sample: DANBO's coarse masks are sparse, and an inactive row would cost 16 B
    auto fetch = [&](int i) { return mask[(size_t)n * S + i] ? raw4[(size_t)n * S + i] : empty; };
    composite_group<kL, kEo>(sz, S, g, gmask, valid, norm_d, inv_B, noise ? noise + (size_t)n * S : nullptr, fetch,
                             S_f > 0 ? sw : nullptr, weights ? weights + (size_t)n * S : nullptr, alpha + (size_t)n * S,
                             rgb0 + (size_t)n * 3, disp0 + n, acc0 + n);
    if (S_f <= 0) return;
    // ---- R1: pdf over the S-2 interior bins, cdf with a leading zero (ray_utils.py:161-164,272-279); lane g holds the
    // contiguous bins g*K .. g*K + K - 1
    const int nb = S - 2;
    const int K = (nb + kL - 1) / kL;                   // <= kE
    float dw[kE];
    double lsum = 0.0;
#pragma unroll
    for (int e = 0; e < kE; ++e) {
        const int k = g * K + e;
        dw[e] = 0.f;
        if (e < K && k < nb) {
            if (smooth) {
                const float a = fmaxf(sw[k], sw[k + 1]), b = fmaxf(sw[k + 1], sw[k + 2]);
                dw[e] = __fadd_rn(__fadd_rn(__fmul_rn(0.5f, __fadd_rn(a, b)), 0.01f), 1e-5f);
            } else {
                dw[e] = __fadd_rn(sw[k + 1], 1e-5f);                        // weights[..., 1:-1] + 1e-5 (sample_pdf)
            }
            lsum += (double)dw[e];
        }
    }
    const float total = (float)group_sum<kL>(lsum);
    double lpdf = 0.0;
#pragma unroll
    for (int e = 0; e < kE; ++e) {
        const int k = g * K + e;
        if (e < K && k < nb) { dw[e] = __fdiv_rn(dw[e], total); lpdf += (double)dw[e]; }
    }
    const double inc = group_incl_sum<kL>(lpdf, g);
    const double ex = __shfl_up_sync(0xffffffffu, inc, 1, kL);
    double run = g == 0 ? 0.0 : ex;
    if (g == 0) scdf[0] = 0.f;
#pragma unroll
    for (int e = 0; e < kE; ++e) {
        const int k = g * K + e;
        if (e < K && k < nb) { run += (double)dw[e]; scdf[k + 1] = (float)run; }
    }
    __syncwarp(gmask);
    const int n_cdf = S - 1;
    for (int j = g; j < S_f; j += kL) {
        const float u = u_rand ? u_rand[(size_t)n * S_f + j] : u_vals[j];
        // searchsorted(cdf, u, right=True) = #{k : cdf[k] <= u}; the cdf is non-decreasing (a running sum of
        // non-negative terms), so the count is the first index with cdf > u: binary search
        int lo = 0, hi = n_cdf;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (scdf[mid] <= u) lo = mid + 1; else hi = mid; }
        const int ind = lo;
        const int below = ind - 1 > 0 ? ind - 1 : 0;
        const int above = ind < n_cdf - 1 ? ind : n_cdf - 1;
        const float cb = scdf[below], ca = scdf[above];
        const float bb = __fmul_rn(.5f, __fadd_rn(sz[below + 1], sz[below]));
        const float ba = __fmul_rn(.5f, __fadd_rn(sz[above + 1], sz[above]));
        float den = __fsub_rn(ca, cb);
        if (den < 1e-5f) den = 1.f;
        const float t = __fdiv_rn(__fsub_rn(u, cb), den);
        const float zsv = __fadd_rn(bb, __fmul_rn(t, __fsub_rn(ba, bb)));
        szs[j] = zsv;
        if (valid) {
            z_samples[(size_t)n * S_f + j] = zsv;
            if (inds_out) inds_out[(size_t)n * S_f + j] = ind;
        }
    }
    __syncwarp(gmask);
    // ---- stable merge of [z ; z_samples] (ties keep concatenation order).  The rank of element i is
    //   #{k : cat[k] < cat[i] or (cat[k] == cat[i] and k < i)}.
    // With z non-decreasing (every sampler's output) and the fine samples stably sorted by (value, index) into fz / fi,
    //   coarse i: i + #{fine < z_i}        fine at sorted position p: #{z <= fz[p]} + p
    // by one binary search each.  Eval draws sorted u, so the fine samples are already in order; train mode draws a
    // random u per ray, and its fine samples are sorted by counting, O(S_f) per sample.  Both checks vote per ray.
    const int St = S + S_f;
    int* out_o = order_out + (size_t)n * St;
    float* out_z = z_all + (size_t)n * St;
    bool z_ok = true, zs_ok = true;
    for (int i = g; i + 1 < S; i += kL) z_ok = z_ok && !(sz[i + 1] < sz[i]);
    for (int j = g; j + 1 < S_f; j += kL) zs_ok = zs_ok && !(szs[j + 1] < szs[j]);
    const unsigned z_bad = __ballot_sync(gmask, !z_ok) & gmask, zs_bad = __ballot_sync(gmask, !zs_ok) & gmask;
    if (z_bad) {                                        // coarse z out of order (no sampler produces it): the plain count
        for (int i = g; i < St; i += kL) {
            const float v = i < S ? sz[i] : szs[i - S];
            int rank = 0;
            for (int k = 0; k < St; ++k) { const float c = k < S ? sz[k] : szs[k - S]; rank += (c < v || (c == v && k < i)) ? 1 : 0; }
            if (valid) { out_o[rank] = i; out_z[rank] = v; }
        }
        return;
    }
    const float* fz = szs;
    const int* fi = nullptr;
    if (zs_bad) {
        for (int j = g; j < S_f; j += kL) {
            const float v = szs[j];
            int p = 0;
            for (int k = 0; k < S_f; ++k) { const float c = szs[k]; p += (c < v || (c == v && k < j)) ? 1 : 0; }
            sfz[p] = v;
            sfi[p] = j;
        }
        __syncwarp(gmask);
        fz = sfz;
        fi = sfi;
    }
    for (int i = g; i < St; i += kL) {
        float v;
        int rank, src;
        if (i < S) {
            v = sz[i];
            int lo = 0, hi = S_f;                               // first fine sample >= v
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (fz[mid] < v) lo = mid + 1; else hi = mid; }
            rank = i + lo;
            src = i;
        } else {
            const int p = i - S;
            v = fz[p];
            int lo = 0, hi = S;                                 // first coarse sample > v
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (sz[mid] <= v) lo = mid + 1; else hi = mid; }
            rank = lo + p;
            src = S + (fi ? fi[p] : p);
        }
        if (valid) { out_o[rank] = src; out_z[rank] = v; }
    }
}

// Fine pass: gather coarse / fine raw by merge order, composite the S_t samples.  No shared memory: z and the merge order
// are read from their rows in global memory.
template <int kL, int kEo>
__global__ void __launch_bounds__(32 * kWarpsPerBlock)
merge_composite_kernel(const float* __restrict__ rays, int ray_stride, int n_rays, int S_c, int S_f,
                       const float* __restrict__ raw0 /* (n_rays*S_c + n_rays, 4) */, const uint32_t* __restrict__ mask0,
                       const float* __restrict__ raw1 /* (n_rays*S_f, 4) */, const uint32_t* __restrict__ mask1,
                       const float* __restrict__ z_all, const int* __restrict__ order, const float* __restrict__ noise,
                       float inv_B, float* __restrict__ weights, float* __restrict__ alpha, float* __restrict__ rgb,
                       float* __restrict__ disp, float* __restrict__ acc, float* __restrict__ raw_merged /* (n,St,4) or null */,
                       const float* __restrict__ confd0, const float* __restrict__ confd1,
                       float* __restrict__ confd_merged /* (n,St,24) or null */, float* __restrict__ invalid_merged /* or null */) {
    const int lane = threadIdx.x & 31, g = lane & (kL - 1), slot = threadIdx.x / kL;
    const unsigned gmask = group_mask<kL>(lane);
    const int n_slot = blockIdx.x * (blockDim.x / kL) + slot;
    const bool valid = n_slot < n_rays;
    const int n = valid ? n_slot : n_rays - 1;
    const int St = S_c + S_f;
    const float* r = rays + (size_t)n * ray_stride;
    const float norm_d = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(r[3], r[3]), __fmul_rn(r[4], r[4])), __fmul_rn(r[5], r[5])));
    const int* ord = order + (size_t)n * St;
    const float4* r0 = reinterpret_cast<const float4*>(raw0);
    const float4* r1 = reinterpret_cast<const float4*>(raw1);
    const float4 empty = r0[(size_t)n_rays * S_c + n];
    auto fetch = [&](int i) {
        const int src = ord[i];
        const bool coarse = src < S_c;
        const size_t sidx = coarse ? (size_t)n * S_c + src : (size_t)n * S_f + src - S_c;
        const uint32_t m = (coarse ? mask0 : mask1)[sidx];  // mask and raw loads issue together; an inactive row is dropped
        const float4 raw = (coarse ? r0 : r1)[sidx];
        const float4 v = m ? raw : empty;
        if (raw_merged && valid) reinterpret_cast<float4*>(raw_merged)[(size_t)n * St + i] = v;
        return v;
    };
    composite_group<kL, kEo>(z_all + (size_t)n * St, St, g, gmask, valid, norm_d, inv_B,
                             noise ? noise + (size_t)n * St : nullptr, fetch, nullptr, weights + (size_t)n * St,
                             alpha + (size_t)n * St, rgb + (size_t)n * 3, disp + n, acc + n);
    if ((confd_merged || invalid_merged) && valid) {       // training outputs (raycasters.py:710-716)
        for (int e = g; e < St * DANBO_J; e += kL) {
            const int i = e / DANBO_J, j = e - i * DANBO_J;
            const int src = ord[i];
            const bool coarse = src < S_c;
            const size_t sidx = coarse ? (size_t)n * S_c + src : (size_t)n * S_f + src - S_c;
            const uint32_t m = coarse ? mask0[sidx] : mask1[sidx];
            const bool vis = (m >> j) & 1u;
            if (invalid_merged) invalid_merged[(size_t)n * St * DANBO_J + e] = vis ? 0.f : 1.f;
            if (confd_merged) confd_merged[(size_t)n * St * DANBO_J + e] = vis ? (coarse ? confd0 : confd1)[sidx * DANBO_J + j] : 0.f;
        }
    }
}

// Fine pass of an eval render with its body-part map: merge_composite_kernel's composite, unchanged, then
//   part_map[n, j] = sum_m w_m p_mj,  p_m = get_agg(logits_m, 1 - visible_m)  (danbo.py:388-415)
// over the merged samples.  Each lane sums w p over the samples whose weights it wrote, in its sample order, into 24
// registers; the group's xor butterfly then adds the lanes' sums in a fixed order (no atomics).  A sample no bone sees
// (mask 0) has p = 0 and is skipped.  Sigmoid passes hold logits only at visible bones, so only those are read; a
// softmax pass holds all 24 of an active row, and its max runs over all of them (field_common.cuh softmax_terms).
template <int kL, int kEo>
__global__ void __launch_bounds__(32 * kWarpsPerBlock)
merge_composite_parts_kernel(const float* __restrict__ rays, int ray_stride, int n_rays, int S_c, int S_f,
                             const float* __restrict__ raw0, const uint32_t* __restrict__ mask0,
                             const float* __restrict__ raw1, const uint32_t* __restrict__ mask1,
                             const float* __restrict__ z_all, const int* __restrict__ order, const float* __restrict__ noise,
                             float inv_B, float* __restrict__ weights, float* __restrict__ alpha, float* __restrict__ rgb,
                             float* __restrict__ disp, float* __restrict__ acc, float* __restrict__ raw_merged,
                             const float* __restrict__ logits0, const float* __restrict__ logits1, int agg_mode,
                             float* __restrict__ part_map /* (n,24) */) {
    const int lane = threadIdx.x & 31, g = lane & (kL - 1), slot = threadIdx.x / kL;
    const unsigned gmask = group_mask<kL>(lane);
    const int n_slot = blockIdx.x * (blockDim.x / kL) + slot;
    const bool valid = n_slot < n_rays;
    const int n = valid ? n_slot : n_rays - 1;
    const int St = S_c + S_f;
    const float* r = rays + (size_t)n * ray_stride;
    const float norm_d = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(r[3], r[3]), __fmul_rn(r[4], r[4])), __fmul_rn(r[5], r[5])));
    const int* ord = order + (size_t)n * St;
    const float4* r0 = reinterpret_cast<const float4*>(raw0);
    const float4* r1 = reinterpret_cast<const float4*>(raw1);
    const float4 empty = r0[(size_t)n_rays * S_c + n];
    auto fetch = [&](int i) {
        const int src = ord[i];
        const bool coarse = src < S_c;
        const size_t sidx = coarse ? (size_t)n * S_c + src : (size_t)n * S_f + src - S_c;
        const uint32_t m = (coarse ? mask0 : mask1)[sidx];
        const float4 raw = (coarse ? r0 : r1)[sidx];
        const float4 v = m ? raw : empty;
        if (raw_merged && valid) reinterpret_cast<float4*>(raw_merged)[(size_t)n * St + i] = v;
        return v;
    };
    float* w_row = weights + (size_t)n * St;
    composite_group<kL, kEo>(z_all + (size_t)n * St, St, g, gmask, valid, norm_d, inv_B,
                             noise ? noise + (size_t)n * St : nullptr, fetch, nullptr, w_row,
                             alpha + (size_t)n * St, rgb + (size_t)n * 3, disp + n, acc + n);
    constexpr int R = 32 / kL;
    float pm[DANBO_J];
#pragma unroll
    for (int j = 0; j < DANBO_J; ++j) pm[j] = 0.f;
    if (valid) {                                        // a group past the last ray wrote no weights: it adds zeros
#pragma unroll
        for (int v = 0; v < R; ++v)
#pragma unroll
            for (int e = 0; e < kEo; ++e) {
                const int i = (v * kL + g) * kEo + e;   // the samples whose weights this lane wrote (composite_group)
                if (i >= St) continue;
                const int src = ord[i];
                const bool coarse = src < S_c;
                const size_t sidx = coarse ? (size_t)n * S_c + src : (size_t)n * S_f + src - S_c;
                const uint32_t m = (coarse ? mask0 : mask1)[sidx];
                if (!m) continue;
                const float w = w_row[i];
                const float* l = (coarse ? logits0 : logits1) + sidx * DANBO_J;
                if (agg_mode == 1) {
                    float amax, inv_den;
                    softmax_terms(l, m, amax, inv_den);
#pragma unroll
                    for (int j = 0; j < DANBO_J; ++j)
                        if ((m >> j) & 1u) pm[j] = fmaf(w, expf(l[j] - amax) * inv_den, pm[j]);
                } else {
#pragma unroll
                    for (int j = 0; j < DANBO_J; ++j)
                        if ((m >> j) & 1u) pm[j] = fmaf(w, (1.f / (1.f + expf(-l[j]))) * 1.002f - 0.001f, pm[j]);
                }
            }
    }
#pragma unroll
    for (int j = 0; j < DANBO_J; ++j) pm[j] = group_sum<kL>(pm[j]);
    if (valid) {
#pragma unroll
        for (int j = 0; j < DANBO_J; ++j)
            if ((j & (kL - 1)) == g) part_map[(size_t)n * DANBO_J + j] = pm[j];
    }
}

}  // namespace danbo

using namespace danbo;

// Lanes per ray of each launcher, indexed by kEo - 1 = ceil(S / 32) - 1.  Each entry is the fastest of 8, 16 and 32 lanes
// on the B200 for that kernel and sample count (scripts/composite_lanes_bench.py, DESIGN §4).
constexpr int kCrLanes[5] = {8, 16, 16, 32, 32};
constexpr int kMcLanes[5] = {8, 16, 32, 32, 32};

extern "C" int danbo_composite_resample(const float* rays, int ray_stride, int n_rays, int S, int S_f, const float* raw,
                                        const unsigned int* mask, const float* z, const float* noise, float inv_B,
                                        const float* u_vals, const float* u_rand, float* weights, float* alpha,
                                        float* rgb0, float* disp0, float* acc0, float* z_samples, float* z_all,
                                        int* order, int* inds, int smooth_weights, void* stream) {
    if (n_rays <= 0) return 0;
    if (S < 3 || S > kMaxS || S_f < 0 || S + S_f > kMaxS) return -1;
    if (S_f > 0 && !u_vals && !u_rand) return -2;
    const size_t smem_per_ray = (size_t)(3 * S + 3 * S_f) * sizeof(float);
#define DANBO_CR_LAUNCH(E) composite_resample_kernel<kCrLanes[E - 1], E>                                              \
        <<<(n_rays + 32 * kWarpsPerBlock / kCrLanes[E - 1] - 1) / (32 * kWarpsPerBlock / kCrLanes[E - 1]),               \
           32 * kWarpsPerBlock, 32 * kWarpsPerBlock / kCrLanes[E - 1] * smem_per_ray, (cudaStream_t)stream>>>(           \
        rays, ray_stride, n_rays, S, S_f, raw, mask, z, noise, inv_B, u_vals, u_rand, weights, alpha, rgb0, disp0, acc0, \
        z_samples, z_all, order, inds, smooth_weights)
    switch ((S + 31) / 32) {                                 // samples per virtual lane: the kernel is specialised on it
        case 1: DANBO_CR_LAUNCH(1); break;
        case 2: DANBO_CR_LAUNCH(2); break;
        case 3: DANBO_CR_LAUNCH(3); break;
        case 4: DANBO_CR_LAUNCH(4); break;
        default: DANBO_CR_LAUNCH(5); break;
    }
#undef DANBO_CR_LAUNCH
    DANBO_CHECK_LAUNCH();
    return 0;
}

extern "C" int danbo_merge_composite(const float* rays, int ray_stride, int n_rays, int S_c, int S_f, const float* raw0,
                                     const unsigned int* mask0, const float* raw1, const unsigned int* mask1,
                                     const float* z_all, const int* order, const float* noise, float inv_B,
                                     float* weights, float* alpha, float* rgb, float* disp, float* acc,
                                     float* raw_merged, const float* confd0, const float* confd1, float* confd_merged,
                                     float* invalid_merged, void* stream) {
    if (n_rays <= 0) return 0;
    if (S_c + S_f > kMaxS) return -1;
#define DANBO_MC_LAUNCH(E) merge_composite_kernel<kMcLanes[E - 1], E>                                                 \
        <<<(n_rays + 32 * kWarpsPerBlock / kMcLanes[E - 1] - 1) / (32 * kWarpsPerBlock / kMcLanes[E - 1]),               \
           32 * kWarpsPerBlock, 0, (cudaStream_t)stream>>>(                                                              \
        rays, ray_stride, n_rays, S_c, S_f, raw0, mask0, raw1, mask1, z_all, order, noise, inv_B, weights, alpha, rgb,  \
        disp, acc, raw_merged, confd0, confd1, confd_merged, invalid_merged)
    switch ((S_c + S_f + 31) / 32) {
        case 1: DANBO_MC_LAUNCH(1); break;
        case 2: DANBO_MC_LAUNCH(2); break;
        case 3: DANBO_MC_LAUNCH(3); break;
        case 4: DANBO_MC_LAUNCH(4); break;
        default: DANBO_MC_LAUNCH(5); break;
    }
#undef DANBO_MC_LAUNCH
    DANBO_CHECK_LAUNCH();
    return 0;
}

extern "C" int danbo_merge_composite_parts(const float* rays, int ray_stride, int n_rays, int S_c, int S_f,
                                           const float* raw0, const unsigned int* mask0, const float* raw1,
                                           const unsigned int* mask1, const float* z_all, const int* order,
                                           const float* noise, float inv_B, float* weights, float* alpha, float* rgb,
                                           float* disp, float* acc, float* raw_merged, const float* confd0,
                                           const float* confd1, int agg_mode, float* part_map, void* stream) {
    if (n_rays <= 0) return 0;
    if (S_c + S_f > kMaxS || !weights || !confd0 || !confd1 || !part_map || agg_mode < 0 || agg_mode > 1) return -1;
#define DANBO_MCP_LAUNCH(E) merge_composite_parts_kernel<kMcLanes[E - 1], E>                                          \
        <<<(n_rays + 32 * kWarpsPerBlock / kMcLanes[E - 1] - 1) / (32 * kWarpsPerBlock / kMcLanes[E - 1]),               \
           32 * kWarpsPerBlock, 0, (cudaStream_t)stream>>>(                                                              \
        rays, ray_stride, n_rays, S_c, S_f, raw0, mask0, raw1, mask1, z_all, order, noise, inv_B, weights, alpha, rgb,  \
        disp, acc, raw_merged, confd0, confd1, agg_mode, part_map)
    switch ((S_c + S_f + 31) / 32) {
        case 1: DANBO_MCP_LAUNCH(1); break;
        case 2: DANBO_MCP_LAUNCH(2); break;
        case 3: DANBO_MCP_LAUNCH(3); break;
        case 4: DANBO_MCP_LAUNCH(4); break;
        default: DANBO_MCP_LAUNCH(5); break;
    }
#undef DANBO_MCP_LAUNCH
    DANBO_CHECK_LAUNCH();
    return 0;
}

// =========================================================================================================
// Backward of C1 (+ R2): gradients of the rendered maps w.r.t. raw.  Autograd of nerf.py:297-347 as it is reached
// from trainer.py:405-409: sources are rgb_map and acc_map (disp_map, alpha and weights carry no gradient), the
// importance samples are detached (ray_utils.py:287), so each ray is independent:
//   w_i = a_i T_i, T_i = prod_{k<i}(1 - a_k + 1e-10)
//   dL/dw_i   = g_rgb . c_i + g_acc [sum w < 1]
//   dL/da_i   = dw_i T_i - (sum_{k>i} dw_k w_k) / (1 - a_i + 1e-10)
//   dL/dsig_i = da_i * dist_i * (1 - a_i) for sigma_i > 0,   dL/dc_i = w_i g_rgb,  c = 1.002 sigmoid(raw) - 0.001
// One warp per ray, forward values recomputed from raw (nothing saved).  Gradients of samples no bone sees are
// summed into the ray's empty entry.
namespace danbo {

template <class Fetch, class Emit>
__device__ __forceinline__ void composite_ray_bwd(RaySmem& sm, int S, int lane, float norm_d, float inv_B,
                                                  const float* __restrict__ noise_row, Fetch fetch, float gr, float gg,
                                                  float gb, float gacc, Emit emit) {
    const int epl = (S + 31) / 32;
    float al[kEPL], sgm[kEPL], dist[kEPL], cr[kEPL], cg[kEPL], cb[kEPL];
    double lp = 1.0;
#pragma unroll
    for (int e = 0; e < kEPL; ++e) {
        const int i = lane * epl + e;
        al[e] = 0.f; sgm[e] = 0.f; dist[e] = 0.f; cr[e] = cg[e] = cb[e] = 0.f;
        if (e < epl && i < S) {
            const float4 raw = fetch(i);
            float d = (i + 1 < S) ? __fsub_rn(sm.z[i + 1], sm.z[i]) : 1e10f;
            d = __fmul_rn(d, norm_d);
            dist[e] = d;
            cr[e] = 1.f / (1.f + expf(-raw.x)); cg[e] = 1.f / (1.f + expf(-raw.y)); cb[e] = 1.f / (1.f + expf(-raw.z));
            float sg = __fmul_rn(raw.w, inv_B);
            if (noise_row) sg = __fadd_rn(sg, noise_row[i]);
            sgm[e] = sg;
            al[e] = __fsub_rn(1.f, expf(-__fmul_rn(fmaxf(sg, 0.f), d)));
            lp *= (double)__fadd_rn(__fsub_rn(1.f, al[e]), 1e-10f);
        }
    }
    double T = warp_excl_prod(lp, lane);
    float w[kEPL], Tf[kEPL], dw[kEPL];
    float wsum = 0.f;
#pragma unroll
    for (int e = 0; e < kEPL; ++e) {
        const int i = lane * epl + e;
        w[e] = 0.f; Tf[e] = 0.f;
        if (e < epl && i < S) {
            Tf[e] = (float)T;
            w[e] = al[e] * Tf[e];
            T *= (double)__fadd_rn(__fsub_rn(1.f, al[e]), 1e-10f);
            wsum += w[e];
        }
    }
    wsum = warp_sum(wsum);
    const float ga = (wsum < 1.f) ? gacc : 0.f;                 // acc = min(sum w, 1)
    // suffix sums of dw_k w_k: lane-local reverse pass + warp suffix scan
    float loc = 0.f;
#pragma unroll
    for (int e = 0; e < kEPL; ++e) {
        const float c0 = cr[e] * 1.002f - 0.001f, c1 = cg[e] * 1.002f - 0.001f, c2 = cb[e] * 1.002f - 0.001f;
        dw[e] = gr * c0 + gg * c1 + gb * c2 + ga;
        loc += dw[e] * w[e];
    }
    float inc = loc;                                            // inclusive suffix over lanes
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const float u = __shfl_down_sync(0xffffffffu, inc, o); if (lane + o < 32) inc += u; }
    float suffix = inc - loc;                                   // sum over lanes > this lane
#pragma unroll
    for (int e = kEPL - 1; e >= 0; --e) {
        const int i = lane * epl + e;
        if (e < epl && i < S) {
            const float om = __fadd_rn(__fsub_rn(1.f, al[e]), 1e-10f);
            const float da = dw[e] * Tf[e] - suffix / om;
            suffix += dw[e] * w[e];
            float4 g;
            g.x = w[e] * gr * 1.002f * cr[e] * (1.f - cr[e]);
            g.y = w[e] * gg * 1.002f * cg[e] * (1.f - cg[e]);
            g.z = w[e] * gb * 1.002f * cb[e] * (1.f - cb[e]);
            g.w = sgm[e] > 0.f ? da * dist[e] * (1.f - al[e]) * inv_B : 0.f;
            emit(i, g);
        }
    }
}

// d raw0 (+)= backward of the coarse composite; d raw0 is (n*S + n, 4), zero-initialised by the caller.
__global__ void __launch_bounds__(32 * kWarpsPerBlock)
composite_bwd_kernel(const float* __restrict__ rays, int ray_stride, int n_rays, int S, const float* __restrict__ raw,
                     const uint32_t* __restrict__ mask, const float* __restrict__ z, const float* __restrict__ noise,
                     float inv_B, const float* __restrict__ g_rgb, const float* __restrict__ g_acc,
                     float* __restrict__ d_raw) {
    __shared__ RaySmem smem[kWarpsPerBlock];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int n = blockIdx.x * kWarpsPerBlock + wib;
    if (n >= n_rays) return;
    RaySmem& sm = smem[wib];
    const float* r = rays + (size_t)n * ray_stride;
    const float norm_d = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(r[3], r[3]), __fmul_rn(r[4], r[4])), __fmul_rn(r[5], r[5])));
    for (int i = lane; i < S; i += 32) sm.z[i] = z[(size_t)n * S + i];
    __syncwarp();
    const float4* raw4 = reinterpret_cast<const float4*>(raw);
    const float4 empty = raw4[(size_t)n_rays * S + n];
    auto fetch = [&](int i) { return mask[(size_t)n * S + i] ? raw4[(size_t)n * S + i] : empty; };
    float4 ge = make_float4(0.f, 0.f, 0.f, 0.f);
    auto emit = [&](int i, float4 g) {
        if (mask[(size_t)n * S + i]) {
            float4* d = reinterpret_cast<float4*>(d_raw) + (size_t)n * S + i;
            float4 o = *d; o.x += g.x; o.y += g.y; o.z += g.z; o.w += g.w; *d = o;
        } else { ge.x += g.x; ge.y += g.y; ge.z += g.z; ge.w += g.w; }
    };
    composite_ray_bwd(sm, S, lane, norm_d, inv_B, noise ? noise + (size_t)n * S : nullptr, fetch,
                      g_rgb[n * 3], g_rgb[n * 3 + 1], g_rgb[n * 3 + 2], g_acc[n], emit);
    ge.x = warp_sum(ge.x); ge.y = warp_sum(ge.y); ge.z = warp_sum(ge.z); ge.w = warp_sum(ge.w);
    if (lane == 0) {
        float4* d = reinterpret_cast<float4*>(d_raw) + (size_t)n_rays * S + n;
        float4 o = *d; o.x += ge.x; o.y += ge.y; o.z += ge.z; o.w += ge.w; *d = o;
    }
}

// backward of the merged composite: scatters to d raw0 (coarse + empty entries) and d raw1 (fine); also routes the
// gradient of the merged blend logits (soft-softmax loss, trainer.py:507-536) back to the two sparse logit buffers.
__global__ void __launch_bounds__(32 * kWarpsPerBlock)
merge_composite_bwd_kernel(const float* __restrict__ rays, int ray_stride, int n_rays, int S_c, int S_f,
                           const float* __restrict__ raw0, const uint32_t* __restrict__ mask0,
                           const float* __restrict__ raw1, const uint32_t* __restrict__ mask1,
                           const float* __restrict__ z_all, const int* __restrict__ order,
                           const float* __restrict__ noise, float inv_B, const float* __restrict__ g_rgb,
                           const float* __restrict__ g_acc, const float* __restrict__ g_confd /* (n,St,24) or null */,
                           float* __restrict__ d_raw0, float* __restrict__ d_raw1,
                           float* __restrict__ d_logit0 /* (n*S_c,24) */, float* __restrict__ d_logit1 /* (n*S_f,24) */) {
    __shared__ RaySmem smem[kWarpsPerBlock];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int n = blockIdx.x * kWarpsPerBlock + wib;
    if (n >= n_rays) return;
    RaySmem& sm = smem[wib];
    const int St = S_c + S_f;
    const float* r = rays + (size_t)n * ray_stride;
    const float norm_d = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(r[3], r[3]), __fmul_rn(r[4], r[4])), __fmul_rn(r[5], r[5])));
    for (int i = lane; i < St; i += 32) { sm.z[i] = z_all[(size_t)n * St + i]; sm.order[i] = order[(size_t)n * St + i]; }
    __syncwarp();
    const float4* r0 = reinterpret_cast<const float4*>(raw0);
    const float4* r1 = reinterpret_cast<const float4*>(raw1);
    const float4 empty = r0[(size_t)n_rays * S_c + n];
    auto fetch = [&](int i) {
        const int src = sm.order[i];
        if (src < S_c) return mask0[(size_t)n * S_c + src] ? r0[(size_t)n * S_c + src] : empty;
        return mask1[(size_t)n * S_f + src - S_c] ? r1[(size_t)n * S_f + src - S_c] : empty;
    };
    float4 ge = make_float4(0.f, 0.f, 0.f, 0.f);
    auto emit = [&](int i, float4 g) {
        const int src = sm.order[i];
        float4* d = nullptr;
        if (src < S_c) { if (mask0[(size_t)n * S_c + src]) d = reinterpret_cast<float4*>(d_raw0) + (size_t)n * S_c + src; }
        else if (mask1[(size_t)n * S_f + src - S_c]) d = reinterpret_cast<float4*>(d_raw1) + (size_t)n * S_f + src - S_c;
        if (d) { float4 o = *d; o.x += g.x; o.y += g.y; o.z += g.z; o.w += g.w; *d = o; }
        else { ge.x += g.x; ge.y += g.y; ge.z += g.z; ge.w += g.w; }
    };
    composite_ray_bwd(sm, St, lane, norm_d, inv_B, noise ? noise + (size_t)n * St : nullptr, fetch,
                      g_rgb[n * 3], g_rgb[n * 3 + 1], g_rgb[n * 3 + 2], g_acc[n], emit);
    ge.x = warp_sum(ge.x); ge.y = warp_sum(ge.y); ge.z = warp_sum(ge.z); ge.w = warp_sum(ge.w);
    if (lane == 0) {
        float4* d = reinterpret_cast<float4*>(d_raw0) + (size_t)n_rays * S_c + n;
        float4 o = *d; o.x += ge.x; o.y += ge.y; o.z += ge.z; o.w += ge.w; *d = o;
    }
    if (g_confd) {
        for (int e = lane; e < St * DANBO_J; e += 32) {
            const int i = e / DANBO_J, j = e - i * DANBO_J;
            const int src = sm.order[i];
            const bool coarse = src < S_c;
            const size_t sidx = coarse ? (size_t)n * S_c + src : (size_t)n * S_f + src - S_c;
            const uint32_t m = coarse ? mask0[sidx] : mask1[sidx];
            if ((m >> j) & 1u) (coarse ? d_logit0 : d_logit1)[sidx * DANBO_J + j] = g_confd[(size_t)n * St * DANBO_J + e];
        }
    }
}

}  // namespace danbo

extern "C" int danbo_composite_bwd(const float* rays, int ray_stride, int n_rays, int S, const float* raw,
                                   const unsigned int* mask, const float* z, const float* noise, float inv_B,
                                   const float* g_rgb, const float* g_acc, float* d_raw, void* stream) {
    if (n_rays <= 0) return 0;
    if (S > danbo::kMaxS) return -1;
    const int G = (n_rays + danbo::kWarpsPerBlock - 1) / danbo::kWarpsPerBlock;
    danbo::composite_bwd_kernel<<<G, 32 * danbo::kWarpsPerBlock, 0, (cudaStream_t)stream>>>(
        rays, ray_stride, n_rays, S, raw, mask, z, noise, inv_B, g_rgb, g_acc, d_raw);
    DANBO_CHECK_LAUNCH();
    return 0;
}

extern "C" int danbo_merge_composite_bwd(const float* rays, int ray_stride, int n_rays, int S_c, int S_f,
                                         const float* raw0, const unsigned int* mask0, const float* raw1,
                                         const unsigned int* mask1, const float* z_all, const int* order,
                                         const float* noise, float inv_B, const float* g_rgb, const float* g_acc,
                                         const float* g_confd, float* d_raw0, float* d_raw1, float* d_logit0,
                                         float* d_logit1, void* stream) {
    if (n_rays <= 0) return 0;
    if (S_c + S_f > danbo::kMaxS) return -1;
    const int G = (n_rays + danbo::kWarpsPerBlock - 1) / danbo::kWarpsPerBlock;
    danbo::merge_composite_bwd_kernel<<<G, 32 * danbo::kWarpsPerBlock, 0, (cudaStream_t)stream>>>(
        rays, ray_stride, n_rays, S_c, S_f, raw0, mask0, raw1, mask1, z_all, order, noise, inv_B, g_rgb, g_acc, g_confd,
        d_raw0, d_raw1, d_logit0, d_logit1);
    DANBO_CHECK_LAUNCH();
    return 0;
}
