// B*: backward of M1 (density/colour MLP) and V1 (per-ray view bias) -- hand-written fp32 kernels, round 1.
//
// Autograd of core/networks/nerf.py:176-209 as reached from trainer.py:573.  The forward tcgen05 kernel saves the bf16
// activation of every layer (train mode); this file turns d raw into d X and parameter gradients:
//   head_bwd        : d raw -> delta of the view layer, d a7 (sigma head), grads of rgb / alpha heads, d ray-bias
//   gemm_dgrad      : D[rows x N] = (A[rows x K] . B[K x N]) (* relu mask) (+ D)          (fp32 SIMT, 128x128x16 tiles)
//   gemm_wgrad      : dW[M x N] += A[rows x M]^T . B[rows x N], split over rows, fp32 atomics
//   colsum          : bias gradients
//   ray_bias_bwd    : grads of views_linears.0[:, 256:], its bias and the frame codes
//   view_root_bwd   : d skts of the root rotation through root-local view directions (perfcap configs, --opt_pose)
// All row counts are device scalars (the active counters), so nothing synchronises with the host.
// Training batches hold ~4e4 active rows, so these are launch/latency bound; the tensor-core (tcgen05) versions are the
// next step once the training step is correct end to end (DESIGN.md §Backward).
#include "common.cuh"
#include <math.h>

namespace danbo {
namespace bwd {

__device__ __forceinline__ float ld_f(const float* p) { return *p; }
__device__ __forceinline__ float ld_f(const __nv_bfloat16* p) { return __bfloat162float(*p); }

constexpr int BM = 128, BN = 128, BK = 16, TM = 8, TN = 8;

// D[m][n] = sum_k A[m][k] * B[k][n]   (A row-major lda, B row-major ldb), m < *rows_ptr.
// Epilogue: v = acc (+ D if accumulate); if mask: v *= (mask[m][n] > 0); D[m][n] = v.
template <typename TA>
__global__ void __launch_bounds__(256)
gemm_dgrad_kernel(const TA* __restrict__ A, int lda, const float* __restrict__ B, int ldb, float* __restrict__ D, int ldd,
                  const int* __restrict__ rows_ptr, int N, int K, int accumulate,
                  const __nv_bfloat16* __restrict__ mask, int ldmask) {
    const int M = *rows_ptr;
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    if (m0 >= M) return;
    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN + 4];
    const int tid = threadIdx.x;
    const int tx = tid % 16, ty = tid / 16;             // 16 x 16 threads, each 8 x 8 outputs
    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;
    for (int k0 = 0; k0 < K; k0 += BK) {
        // A tile: 128 rows x 16 k  -> As[k][m]
        for (int i = tid; i < BM * BK; i += 256) {
            const int m = i / BK, k = i % BK;
            const int gm = m0 + m, gk = k0 + k;
            As[k][m] = (gm < M && gk < K) ? ld_f(A + (size_t)gm * lda + gk) : 0.f;
        }
        for (int i = tid; i < BK * BN; i += 256) {
            const int k = i / BN, n = i % BN;
            const int gk = k0 + k, gn = n0 + n;
            Bs[k][n] = (gk < K && gn < N) ? B[(size_t)gk * ldb + gn] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            float a[TM], b[TN];
#pragma unroll
            for (int i = 0; i < TM; ++i) a[i] = As[k][ty * TM + i];
#pragma unroll
            for (int j = 0; j < TN; ++j) b[j] = Bs[k][tx * TN + j];
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        const int gm = m0 + ty * TM + i;
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            const int gn = n0 + tx * TN + j;
            if (gn >= N) continue;
            float v = acc[i][j];
            if (accumulate) v += D[(size_t)gm * ldd + gn];
            if (mask && !(__bfloat162float(mask[(size_t)gm * ldmask + gn]) > 0.f)) v = 0.f;
            D[(size_t)gm * ldd + gn] = v;
        }
    }
}

// dW[m][n] += sum_r A[r][m] * B[r][n]  over r in this block's row chunk (split-K, atomics).
template <typename TB>
__global__ void __launch_bounds__(256)
gemm_wgrad_kernel(const float* __restrict__ A, int lda, const TB* __restrict__ B, int ldb, float* __restrict__ dW, int ldw,
                  const int* __restrict__ rows_ptr, int M, int N, int rows_per_chunk) {
    const int R = *rows_ptr;
    const int r_begin = blockIdx.z * rows_per_chunk;
    if (r_begin >= R) return;
    const int r_end = min(R, r_begin + rows_per_chunk);
    const int m0 = blockIdx.x * BM, n0 = blockIdx.y * BN;
    __shared__ float As[BK][BM + 4];
    __shared__ float Bs[BK][BN + 4];
    const int tid = threadIdx.x;
    const int tx = tid % 16, ty = tid / 16;
    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;
    for (int r0 = r_begin; r0 < r_end; r0 += BK) {
        for (int i = tid; i < BK * BM; i += 256) {
            const int k = i / BM, m = i % BM;
            const int gr = r0 + k, gm = m0 + m;
            As[k][m] = (gr < r_end && gm < M) ? A[(size_t)gr * lda + gm] : 0.f;
        }
        for (int i = tid; i < BK * BN; i += 256) {
            const int k = i / BN, n = i % BN;
            const int gr = r0 + k, gn = n0 + n;
            Bs[k][n] = (gr < r_end && gn < N) ? ld_f(B + (size_t)gr * ldb + gn) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            float a[TM], b[TN];
#pragma unroll
            for (int i = 0; i < TM; ++i) a[i] = As[k][ty * TM + i];
#pragma unroll
            for (int j = 0; j < TN; ++j) b[j] = Bs[k][tx * TN + j];
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        const int gm = m0 + ty * TM + i;
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            const int gn = n0 + tx * TN + j;
            if (gn < N) atomicAdd(dW + (size_t)gm * ldw + gn, acc[i][j]);
        }
    }
}

// db[n] += sum_r A[r][n]
__global__ void __launch_bounds__(256)
colsum_kernel(const float* __restrict__ A, int lda, float* __restrict__ db, const int* __restrict__ rows_ptr, int N,
              int rows_per_block) {
    const int R = *rows_ptr;
    const int r0 = blockIdx.x * rows_per_block;
    if (r0 >= R) return;
    const int r1 = min(R, r0 + rows_per_block);
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
        float s = 0.f;
        for (int r = r0; r < r1; ++r) s += A[(size_t)r * lda + n];
        atomicAdd(db + n, s);
    }
}

// Heads.  One warp per row.
//   d_raw (per sample id, 4) -> delta9 (rows,128) = (d_rgb . W_rgb) * [g > 0];  d_a7 (rows,256) = d_sigma * w_alpha
//   grads: rgb_linear (3,128)+(3), alpha_linear (256)+(1); d ray_bias[ray] += delta9
// kHeadGrads / kRayBias = false compile those reductions / that output out (pose-only backward: the heads are frozen,
// and d ray_bias is needed only where the view directions depend on the pose).
template <bool kHeadGrads, bool kRayBias>
__global__ void __launch_bounds__(256)
head_bwd_kernel(const float* __restrict__ d_raw, const int* __restrict__ row_sample, const int* __restrict__ row_ray,
                const int* __restrict__ rows_ptr, const __nv_bfloat16* __restrict__ g_save /* (rows,128) */,
                const __nv_bfloat16* __restrict__ a7_save /* (rows,256) */, const float* __restrict__ w_rgb,
                const float* __restrict__ w_alpha, float* __restrict__ delta9, float* __restrict__ d_a7,
                float* __restrict__ d_w_rgb, float* __restrict__ d_b_rgb, float* __restrict__ d_w_alpha,
                float* __restrict__ d_b_alpha, float* __restrict__ d_ray_bias) {
    const int R = *rows_ptr;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    __shared__ float s_wrgb[3][128], s_walpha[256], s_brgb[3], s_balpha;
    if (kHeadGrads) {
        for (int i = threadIdx.x; i < 384; i += 256) s_wrgb[i / 128][i % 128] = 0.f;
        for (int i = threadIdx.x; i < 256; i += 256) s_walpha[i] = 0.f;
        if (threadIdx.x < 3) s_brgb[threadIdx.x] = 0.f;
        if (threadIdx.x == 0) s_balpha = 0.f;
        __syncthreads();
    }
    for (int r = blockIdx.x * 8 + wib; r < R; r += gridDim.x * 8) {
        const float4 g = reinterpret_cast<const float4*>(d_raw)[row_sample[r]];
        const int ray = row_ray[r];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int c = lane + 32 * q;
            const float gv = __bfloat162float(g_save[(size_t)r * 128 + c]);
            const float d = gv > 0.f ? (g.x * w_rgb[c] + g.y * w_rgb[128 + c] + g.z * w_rgb[256 + c]) : 0.f;
            if (delta9) delta9[(size_t)r * 128 + c] = d;
            if (kRayBias) atomicAdd(d_ray_bias + (size_t)ray * 128 + c, d);
            if (kHeadGrads) { atomicAdd(&s_wrgb[0][c], g.x * gv); atomicAdd(&s_wrgb[1][c], g.y * gv); atomicAdd(&s_wrgb[2][c], g.z * gv); }
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int c = lane + 32 * q;
            if (d_a7) d_a7[(size_t)r * 256 + c] = g.w * w_alpha[c];
            if (kHeadGrads) atomicAdd(&s_walpha[c], g.w * __bfloat162float(a7_save[(size_t)r * 256 + c]));
        }
        if (kHeadGrads && lane == 0) { atomicAdd(&s_brgb[0], g.x); atomicAdd(&s_brgb[1], g.y); atomicAdd(&s_brgb[2], g.z); atomicAdd(&s_balpha, g.w); }
    }
    if (!kHeadGrads) return;
    __syncthreads();
    for (int i = threadIdx.x; i < 384; i += 256) atomicAdd(d_w_rgb + i, s_wrgb[i / 128][i % 128]);
    for (int i = threadIdx.x; i < 256; i += 256) atomicAdd(d_w_alpha + i, s_walpha[i]);
    if (threadIdx.x < 3) atomicAdd(d_b_rgb + threadIdx.x, s_brgb[threadIdx.x]);
    if (threadIdx.x == 0) atomicAdd(d_b_alpha, s_balpha);
}

// V1 backward: d_ray_bias (n,128) -> grads of views_linears.0.weight[:, 256:411] (128,411 layout), its bias, and the
// frame codes.  Groups of 16 rays (inputs v recomputed like the forward); a block walks several groups and keeps its
// weight-gradient partial sums in registers (thread = output unit x half of the 155 inputs), so the atomics on the
// shared (128,155) slice happen once per block, not once per group.
__global__ void __launch_bounds__(256)
ray_bias_bwd_kernel(const float* __restrict__ rays, int ray_stride, int n_rays, const int* __restrict__ cam_idx,
                    const float* __restrict__ codes, int n_codes, const float* __restrict__ w_view /* (128,411) */,
                    const float* __restrict__ d_ray_bias, float* __restrict__ d_w_view /* (128,411) */,
                    float* __restrict__ d_b_view, float* __restrict__ d_codes /* (n_codes,128) */) {
    constexpr int RB = 16, VIN = 155, HALF = 78;
    __shared__ float v[VIN][RB];
    __shared__ float db[RB][128];
    __shared__ int s_cam[RB];
    __shared__ float dsum[128];
    __shared__ int one_cam;
    const int o = threadIdx.x & 127, half = threadIdx.x >> 7;
    const int c0 = half * HALF, nc = half == 0 ? HALF : VIN - HALF;
    float acc[HALF];
#pragma unroll
    for (int i = 0; i < HALF; ++i) acc[i] = 0.f;
    float bsum = 0.f;
    const int n_groups = (n_rays + RB - 1) / RB;
    for (int g = blockIdx.x; g < n_groups; g += gridDim.x) {
        const int base = g * RB;
        __syncthreads();                                  // previous group's tiles fully consumed
        for (int i = threadIdx.x; i < RB * VIN; i += blockDim.x) {
            const int rb = i % RB, c = i / RB;
            const int n = base + rb;
            float val = 0.f;
            if (n < n_rays) {
                if (c < 27) {
                    const float* r = rays + (size_t)n * ray_stride + 3;
                    if (c < 3) val = r[c];
                    else { const int q = c - 3, f = q / 6, rem = q - 6 * f; const float x = r[rem % 3] * (float)(1 << f); val = rem < 3 ? sinf(x) : cosf(x); }
                } else {
                    int ci = cam_idx ? cam_idx[n] : 0;
                    ci = ci < 0 ? n_codes : (ci > n_codes - 1 ? n_codes - 1 : ci);
                    val = codes[(size_t)ci * 128 + (c - 27)];
                }
            }
            v[c][rb] = val;
        }
        for (int i = threadIdx.x; i < RB * 128; i += blockDim.x) {
            const int rb = i / 128, oo = i % 128;
            db[rb][oo] = (base + rb < n_rays) ? d_ray_bias[(size_t)(base + rb) * 128 + oo] : 0.f;
        }
        if (threadIdx.x < RB) {
            const int n = base + threadIdx.x;
            int ci = (n < n_rays && cam_idx) ? cam_idx[n] : 0;
            s_cam[threadIdx.x] = (n < n_rays) ? ci : -2;
        }
        __syncthreads();
        float d[RB];
#pragma unroll
        for (int rb = 0; rb < RB; ++rb) { d[rb] = db[rb][o]; bsum += d[rb]; }
#pragma unroll
        for (int i = 0; i < HALF; ++i) {
            if (i < nc) {
                const float4* vr = reinterpret_cast<const float4*>(v[c0 + i]);
#pragma unroll
                for (int q = 0; q < RB / 4; ++q) {
                    const float4 x = vr[q];
                    acc[i] = fmaf(d[4 * q + 0], x.x, acc[i]); acc[i] = fmaf(d[4 * q + 1], x.y, acc[i]);
                    acc[i] = fmaf(d[4 * q + 2], x.z, acc[i]); acc[i] = fmaf(d[4 * q + 3], x.w, acc[i]);
                }
            }
        }
        // frame codes: d code[cam][c'] += sum_o W_v[o][283 + c'] * d_bias[o]   (training: cam >= 0; eval mean code has no grad).
        // Rays arrive image-major, so a group normally has ONE camera: sum its d_bias rows first and do a single
        // 128 x 128 product (the per-ray form is a 2 048-step dependent load/FMA chain per thread: 43 us per group).
        float gsum = 0.f;
#pragma unroll
        for (int rb = 0; rb < RB; ++rb) gsum += (s_cam[rb] >= 0) ? d[rb] : 0.f;
        if (half == 0) dsum[o] = gsum;
        if (threadIdx.x == 0) {
            int c0 = -3; bool same = true;
            for (int rb = 0; rb < RB; ++rb) { const int c = s_cam[rb]; if (c < 0) continue; if (c0 == -3) c0 = c; else if (c != c0) same = false; }
            one_cam = same ? c0 : -4;                   // -3: no ray with a trainable code, -4: mixed
        }
        __syncthreads();
        if (half == 0) {
            const int cp = o;
            if (one_cam >= 0) {
                const int ci = one_cam > n_codes - 1 ? n_codes - 1 : one_cam;
                float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 8
                for (int oo = 0; oo < 128; ++oo) s4[oo & 3] = fmaf(__ldg(w_view + (size_t)oo * 411 + 283 + cp), dsum[oo], s4[oo & 3]);
                atomicAdd(d_codes + (size_t)ci * 128 + cp, (s4[0] + s4[1]) + (s4[2] + s4[3]));
            } else if (one_cam == -4) {
                for (int rb = 0; rb < RB; ++rb) {
                    const int cam = s_cam[rb];
                    if (cam < 0) continue;
                    const int ci = cam > n_codes - 1 ? n_codes - 1 : cam;
                    float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 8
                    for (int oo = 0; oo < 128; ++oo) s4[oo & 3] = fmaf(__ldg(w_view + (size_t)oo * 411 + 283 + cp), db[rb][oo], s4[oo & 3]);
                    atomicAdd(d_codes + (size_t)ci * 128 + cp, (s4[0] + s4[1]) + (s4[2] + s4[3]));
                }
            }
        }
    }
    if (half == 0) atomicAdd(d_b_view + o, bsum);
#pragma unroll
    for (int i = 0; i < HALF; ++i)
        if (i < nc) atomicAdd(d_w_view + (size_t)o * 411 + 256 + c0 + i, acc[i]);
}

// V1 backward to the root rotation (perfcap configs: ray_tr_type=root_local + view_type=relray, pose refinement).  There
// the view branch encodes dn = normalize(m), m = R0 d_ray, R0 = skts[pose, 0, :3, :3] (RootLocalEncoder
// encoders.py:570-578, VecNormEncoder :774-795), and PE(dn) = [dn, sin(2^f dn), cos(2^f dn)]_{f<4} meets columns 256..282
// of W_v.  Per ray:
//   g = W_v[:, 256:283]^T d_ray_bias,   d dn_a = g_a + sum_f 2^f (g_sin,f,a cos(2^f dn_a) - g_cos,f,a sin(2^f dn_a)),
//   d m = (d dn - (dn . d dn) dn) / |m|,   d skts[pose, 0, 0:3, 0:3] += d m (x) d_ray.
// Work layout: 32 rays per block of 4 warps.  The block stages its 32 d_ray_bias rows (float4 loads, a row is 512
// contiguous bytes) and the 128 x 27 weight slice in shared memory.  Then lane = ray and warp w forms the columns
// 7w..7w+6 of g: the d_ray_bias reads are conflict-free (row stride 129) and the weight reads are broadcasts.  Warp
// a < 3 forms d dn_a (four sincos per lane), and warp 0 finishes the per-ray chain.  When all rays of the block share a
// pose (rays are image-major, so almost always) it sums the 9 entries over the block and issues one set of atomics;
// otherwise every ray issues its own.  Three barriers order the phases: staging -> o-loop, gs stores -> the cross-warp gs
// reads (and the reuse of db), d dn -> warp 0.  57 registers, no spills, 36.6 KB of shared memory (-Xptxas -v).
constexpr int VR_RAYS = 32, VR_COLS = 27, VR_GRP = 7;

__global__ void __launch_bounds__(128)
view_root_bwd_kernel(const float* __restrict__ rays, int ray_stride, int n_rays, const float* __restrict__ pose_skts,
                     int rays_per_pose, int n_poses, const float* __restrict__ w_view /* (128,411) */,
                     const float* __restrict__ d_ray_bias /* (n,128) */, float* __restrict__ d_skts) {
    __shared__ float db[VR_RAYS][129];
    __shared__ __align__(16) float ws[4][128][8];          // [warp][o][column 7w + s], slot 7 zero
    __shared__ float gs[VR_RAYS][VR_COLS + 2];              // row stride 29: conflict-free for lane = ray
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int base = blockIdx.x * VR_RAYS;
    const int nr = min(VR_RAYS, n_rays - base);
    for (int i = tid; i < VR_RAYS * 32; i += 128) {
        const int r = i >> 5, q = i & 31;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < nr) v = __ldg(reinterpret_cast<const float4*>(d_ray_bias + (size_t)(base + r) * 128) + q);
        db[r][4 * q + 0] = v.x; db[r][4 * q + 1] = v.y; db[r][4 * q + 2] = v.z; db[r][4 * q + 3] = v.w;
    }
    for (int i = tid; i < 4 * 128 * 8; i += 128) {
        const int w = i >> 10, o = (i >> 3) & 127, s = i & 7, c = w * VR_GRP + s;
        ws[w][o][s] = (s < VR_GRP && c < VR_COLS) ? __ldg(w_view + (size_t)o * 411 + 256 + c) : 0.f;
    }
    __syncthreads();
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int o = 0; o < 128; ++o) {
        const float d = db[lane][o];
        const float4 a = *reinterpret_cast<const float4*>(&ws[warp][o][0]);
        const float4 b = *reinterpret_cast<const float4*>(&ws[warp][o][4]);
        acc[0] = fmaf(a.x, d, acc[0]); acc[1] = fmaf(a.y, d, acc[1]); acc[2] = fmaf(a.z, d, acc[2]);
        acc[3] = fmaf(a.w, d, acc[3]); acc[4] = fmaf(b.x, d, acc[4]); acc[5] = fmaf(b.y, d, acc[5]);
        acc[6] = fmaf(b.z, d, acc[6]);
    }
#pragma unroll
    for (int s = 0; s < VR_GRP; ++s)
        if (warp * VR_GRP + s < VR_COLS) gs[lane][warp * VR_GRP + s] = acc[s];
    // every warp reads columns the other warps wrote, and warps 0-2 overwrite db, which every warp's o-loop reads
    __syncthreads();
    const bool live = lane < nr;
    const int n = base + lane;
    const int pose = live ? min(n / rays_per_pose, n_poses - 1) : 0;
    float dx = 0.f, dy = 0.f, dz = 0.f, nrm = 1.f, dn[3] = {0.f, 0.f, 0.f};
    if (live) {
        const float* r = rays + (size_t)n * ray_stride + 3;
        dx = r[0]; dy = r[1]; dz = r[2];
        const float* R = pose_skts + (size_t)pose * DANBO_J * 16;          // joint 0
        const float m[3] = {fmaf(__ldg(R + 2), dz, fmaf(__ldg(R + 1), dy, __ldg(R + 0) * dx)),
                            fmaf(__ldg(R + 6), dz, fmaf(__ldg(R + 5), dy, __ldg(R + 4) * dx)),
                            fmaf(__ldg(R + 10), dz, fmaf(__ldg(R + 9), dy, __ldg(R + 8) * dx))};
        nrm = fmaxf(sqrtf(m[0] * m[0] + m[1] * m[1] + m[2] * m[2]), 1e-12f);
        dn[0] = m[0] / nrm; dn[1] = m[1] / nrm; dn[2] = m[2] / nrm;
    }
    // d dn_a of ray `lane` by warp a < 3 (4 sincos per lane instead of 12 on one warp)
    if (warp < 3 && live) {
        const int a = warp;
        const float da = warp == 0 ? dn[0] : (warp == 1 ? dn[1] : dn[2]);
        float g = gs[lane][a];
#pragma unroll
        for (int f = 0; f < 4; ++f) {
            const float fr = (float)(1 << f);
            float sn, cs;
            sincosf(da * fr, &sn, &cs);                                  // ray_bias_kernel's sin / cos arguments
            g = fmaf(fr * cs, gs[lane][3 + 6 * f + a], g);
            g = fmaf(-fr * sn, gs[lane][6 + 6 * f + a], g);
        }
        db[lane][a] = g;                                                 // the d_ray_bias tile is consumed
    }
    __syncthreads();
    if (warp != 0) return;
    float out[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) out[i] = 0.f;
    if (live) {
        const float ddn[3] = {db[lane][0], db[lane][1], db[lane][2]};
        const float p = dn[0] * ddn[0] + dn[1] * ddn[1] + dn[2] * ddn[2];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float dm = (ddn[i] - p * dn[i]) / nrm;
            out[3 * i + 0] = dm * dx; out[3 * i + 1] = dm * dy; out[3 * i + 2] = dm * dz;
        }
    }
    const int pose_first = min(base / rays_per_pose, n_poses - 1);
    const int pose_last = min((base + nr - 1) / rays_per_pose, n_poses - 1);
    if (pose_first == pose_last) {
        float* dst = d_skts + (size_t)pose_first * DANBO_J * 16;
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            float v = out[i];
#pragma unroll
            for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
            if (lane == 0) atomicAdd(dst + (i / 3) * 4 + i % 3, v);
        }
    } else if (live) {
        float* dst = d_skts + (size_t)pose * DANBO_J * 16;
#pragma unroll
        for (int i = 0; i < 9; ++i) atomicAdd(dst + (i / 3) * 4 + i % 3, out[i]);
    }
}

}  // namespace bwd
}  // namespace danbo

using namespace danbo;

// D[rows x N] = A[rows x K] . B[K x N]; a_is_bf16 selects the element type of A; mask (bf16, rows x ldmask) optional.
extern "C" int danbo_gemm_dgrad(const void* A, int a_is_bf16, int lda, const float* B, int ldb, float* D, int ldd,
                                const int* rows_dev, int max_rows, int N, int K, int accumulate, const void* mask,
                                int ldmask, void* stream) {
    if (max_rows <= 0) return 0;
    dim3 grid((max_rows + bwd::BM - 1) / bwd::BM, (N + bwd::BN - 1) / bwd::BN);
    if (a_is_bf16)
        bwd::gemm_dgrad_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(
            (const __nv_bfloat16*)A, lda, B, ldb, D, ldd, rows_dev, N, K, accumulate, (const __nv_bfloat16*)mask, ldmask);
    else
        bwd::gemm_dgrad_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(
            (const float*)A, lda, B, ldb, D, ldd, rows_dev, N, K, accumulate, (const __nv_bfloat16*)mask, ldmask);
    DANBO_CHECK_LAUNCH();
    return 0;
}

// dW[M x N] += A[rows x M]^T . B[rows x N]   (A fp32; B bf16 or fp32)
extern "C" int danbo_gemm_wgrad(const float* A, int lda, const void* B, int b_is_bf16, int ldb, float* dW, int ldw,
                                const int* rows_dev, int max_rows, int M, int N, void* stream) {
    if (max_rows <= 0) return 0;
    const int rows_per_chunk = 1024;
    dim3 grid((M + bwd::BM - 1) / bwd::BM, (N + bwd::BN - 1) / bwd::BN, (max_rows + rows_per_chunk - 1) / rows_per_chunk);
    if (b_is_bf16)
        bwd::gemm_wgrad_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(
            A, lda, (const __nv_bfloat16*)B, ldb, dW, ldw, rows_dev, M, N, rows_per_chunk);
    else
        bwd::gemm_wgrad_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(
            A, lda, (const float*)B, ldb, dW, ldw, rows_dev, M, N, rows_per_chunk);
    DANBO_CHECK_LAUNCH();
    return 0;
}

extern "C" int danbo_colsum(const float* A, int lda, float* db, const int* rows_dev, int max_rows, int N, void* stream) {
    if (max_rows <= 0) return 0;
    const int rpb = 256;
    bwd::colsum_kernel<<<(max_rows + rpb - 1) / rpb, 256, 0, (cudaStream_t)stream>>>(A, lda, db, rows_dev, N, rpb);
    DANBO_CHECK_LAUNCH();
    return 0;
}

extern "C" int danbo_mlp_head_bwd(const float* d_raw, const int* row_sample, const int* row_ray, const int* rows_dev,
                                  int max_rows, const void* g_save, const void* a7_save, const float* w_rgb,
                                  const float* w_alpha, float* delta9, float* d_a7, float* d_w_rgb, float* d_b_rgb,
                                  float* d_w_alpha, float* d_b_alpha, float* d_ray_bias, int num_sms, void* stream) {
    if (max_rows <= 0) return 0;
    const int n_head = (d_w_rgb != nullptr) + (d_b_rgb != nullptr) + (d_w_alpha != nullptr) + (d_b_alpha != nullptr);
    if (n_head != 0 && n_head != 4) return -1;
    const bool head = n_head == 4, rb = d_ray_bias != nullptr;
    if (!head && !rb && delta9 == nullptr && d_a7 == nullptr) return 0;      // nothing asked for: no launch
    int blocks = (max_rows + 7) / 8;
    if (blocks > num_sms * 4) blocks = num_sms * 4;
    auto kern = head ? (rb ? bwd::head_bwd_kernel<true, true> : bwd::head_bwd_kernel<true, false>)
                     : (rb ? bwd::head_bwd_kernel<false, true> : bwd::head_bwd_kernel<false, false>);
    kern<<<blocks, 256, 0, (cudaStream_t)stream>>>(
        d_raw, row_sample, row_ray, rows_dev, (const __nv_bfloat16*)g_save, (const __nv_bfloat16*)a7_save, w_rgb, w_alpha,
        delta9, d_a7, d_w_rgb, d_b_rgb, d_w_alpha, d_b_alpha, d_ray_bias);
    DANBO_CHECK_LAUNCH();
    return 0;
}

extern "C" int danbo_ray_bias_bwd(const float* rays, int ray_stride, int n_rays, const int* cam_idx, const float* codes,
                                  int n_codes, const float* w_view, const float* d_ray_bias, float* d_w_view,
                                  float* d_b_view, float* d_codes, void* stream) {
    if (n_rays <= 0) return 0;
    int rb_blocks = (n_rays + 15) / 16;
    if (rb_blocks > 64) rb_blocks = 64 + (rb_blocks - 64) / 8;          // several 16-ray groups per block
    if (rb_blocks > 1184) rb_blocks = 1184;
    bwd::ray_bias_bwd_kernel<<<rb_blocks, 256, 0, (cudaStream_t)stream>>>(
        rays, ray_stride, n_rays, cam_idx, codes, n_codes, w_view, d_ray_bias, d_w_view, d_b_view, d_codes);
    DANBO_CHECK_LAUNCH();
    return 0;
}

extern "C" int danbo_view_root_bwd(const float* rays, int ray_stride, int n_rays, const float* pose_skts,
                                   int rays_per_pose, int n_poses, const float* w_view, const float* d_ray_bias,
                                   float* d_skts, void* stream) {
    if (n_rays <= 0) return 0;
    if (!rays || !pose_skts || !w_view || !d_ray_bias || !d_skts || ray_stride < 6 || rays_per_pose <= 0 || n_poses <= 0)
        return -1;
    if (reinterpret_cast<uintptr_t>(d_ray_bias) & 15) return -1;       // rows are read as float4
    bwd::view_root_bwd_kernel<<<(n_rays + bwd::VR_RAYS - 1) / bwd::VR_RAYS, 128, 0, (cudaStream_t)stream>>>(
        rays, ray_stride, n_rays, pose_skts, rays_per_pose, n_poses, w_view, d_ray_bias, d_skts);
    DANBO_CHECK_LAUNCH();
    return 0;
}

// ------------------------------------------------------------------------------------------------------------
// Adam over ONE flat fp32 arena (all 43 parameter tensors are views of it): the update is a single elementwise
// launch instead of a multi-tensor pass (276 us -> ~10 us for 2.46 M parameters).  torch.optim.Adam's formulas
// (run_nerf.py / raycasters.py:71-78: Adam(lr, betas=(0.9, 0.999)), no weight decay, no amsgrad):
//   m = m + (g - m)(1 - b1);  v = b2 v + (1 - b2) g^2;  p -= (lr / (1 - b1^t)) * m / (sqrt(v) / sqrt(1 - b2^t) + eps)
// step and lr live on the device so a captured CUDA graph sees their current values.
namespace danbo {
namespace bwd {
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                            long long n, const float* __restrict__ lr_dev, float beta1, float beta2, float eps,
                            const float* __restrict__ step_dev) {
    const float t = *step_dev;                               // already incremented for this update
    const float bc1 = 1.f - powf(beta1, t), bc2_sqrt = sqrtf(1.f - powf(beta2, t));
    const float step_size = *lr_dev / bc1;
    const long long n4 = n >> 2;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 pp = reinterpret_cast<float4*>(p)[i], mm = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
        const float4 gg = reinterpret_cast<const float4*>(g)[i];
        float* P = &pp.x; float* M = &mm.x; float* V = &vv.x; const float* G = &gg.x;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            M[k] = M[k] + (G[k] - M[k]) * (1.f - beta1);
            V[k] = V[k] * beta2 + (1.f - beta2) * G[k] * G[k];
            P[k] -= step_size * (M[k] / (sqrtf(V[k]) / bc2_sqrt + eps));
        }
        reinterpret_cast<float4*>(p)[i] = pp; reinterpret_cast<float4*>(m)[i] = mm; reinterpret_cast<float4*>(v)[i] = vv;
    }
    for (long long i = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float gi = g[i];
        const float mi = m[i] + (gi - m[i]) * (1.f - beta1);
        const float vi = v[i] * beta2 + (1.f - beta2) * gi * gi;
        m[i] = mi; v[i] = vi;
        p[i] -= step_size * (mi / (sqrtf(vi) / bc2_sqrt + eps));
    }
}
}  // namespace bwd
}  // namespace danbo

extern "C" int danbo_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n,
                               const float* lr_dev, float beta1, float beta2, float eps, const float* step_dev,
                               int num_sms, void* stream) {
    if (n <= 0) return 0;
    if ((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(grads) | reinterpret_cast<uintptr_t>(exp_avg) |
         reinterpret_cast<uintptr_t>(exp_avg_sq)) & 15) return -1;
    long long blocks = (n / 4 + 255) / 256;
    if (blocks > (long long)num_sms * 8) blocks = (long long)num_sms * 8;
    if (blocks < 1) blocks = 1;
    danbo::bwd::adam_kernel<<<(int)blocks, 256, 0, (cudaStream_t)stream>>>(params, grads, exp_avg, exp_avg_sq, n, lr_dev, beta1,
                                                                          beta2, eps, step_dev);
    DANBO_CHECK_LAUNCH();
    return 0;
}
