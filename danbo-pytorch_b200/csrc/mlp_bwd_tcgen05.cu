// B* for M1 on the tensor cores: fused data-gradient chain + weight-gradient GEMMs (tcgen05 / TMEM / bulk copies).
//
//   dgrad_kernel : one persistent CTA per SM, same structure as the forward kernel (mlp_tcgen05.cu): the delta of every
//                  layer is produced in TMEM as the A operand of the next (transposed-weight) MMA, masked by the saved
//                  activation's relu in the epilogue, and saved as bf16 for the weight gradients.  11 stages per tile:
//                  d feat = d9 Wv ; d7 = (d feat Wf + d sigma w_alpha)[a7>0] ; d6 ; d5 ; dX = d5 W5[:, :195] ; d4 ... d0 ;
//                  dX += d0 W0.
//   transpose_kernel : row-major bf16 [plane][row][256] -> blocks of 64 rows stored as K-major (K = rows) swizzled
//                  operand images, so the weight-gradient MMA (contraction over rows) bulk-copies its operands.
//   wgrad_kernel : dW = delta^T . act with K = rows; CTA = (gemm, output half, K split); fp32 partials, then
//   wgrad_reduce_kernel sums the splits into the parameter-shaped gradient tensors; colsum_planes_kernel = bias grads.
// Reference autograd being replaced: the backward of core/networks/nerf.py:176-209 under trainer.py:573.
#include "tc_common.cuh"

namespace danbo {
namespace mlpb {
using namespace danbo::tc;

constexpr int kStages = 7;                           // ring slots: 84 tiles per row tile = 12 x 7, so the slot and the barrier
                                                     // parity of every tile are compile-time constants of the unrolled schedule
constexpr int kStageBytes = 128 * 64 * 2;
constexpr int kThreads = 320;
constexpr int kNumStagesPerTile = 84;                // weight tiles consumed per 128-row tile
constexpr int kDgradStages = 11;
constexpr uint32_t kAccCol = 0, kActCol = 256;

struct __align__(1024) Smem {
    uint8_t w[kStages][kStageBytes];
    uint8_t stage[8][4096];              // per epilogue warp: [64 features][32 rows] bf16, to write deltas row-transposed
    float w_rgb[3 * 128];
    float w_alpha[256];
    uint64_t w_full[kStages];
    uint64_t w_empty[kStages];
    uint64_t acc_full[2];
    uint64_t act_ready[2];
    uint32_t tmem_base;
};

// stage -> number of 64-wide K chunks, input activation buffer, kind
__host__ __device__ constexpr int st_kchunks(int s) { return s == 0 ? 2 : 4; }
// {0, 1, 0, 1, 0, 0, 1, 0, 1, 0, 1}
__host__ __device__ constexpr int st_inbuf(int s) { return s < 5 ? (s & 1) : ((s - 1) & 1); }
__device__ __forceinline__ bool st_is_x(int s) { return s == 4 || s == 10; }
// row-major activation plane whose relu masks the output of stage s (-1: none)
__device__ __forceinline__ int st_mask_plane(int s) { const int t[kDgradStages] = {-1, 7, 6, 5, -1, 4, 3, 2, 1, 0, -1}; return t[s]; }
// delta plane written by stage s (-1: none); plane 0 = delta9 comes from the prologue
__device__ __forceinline__ int st_delta_plane(int s) { const int t[kDgradStages] = {1, 2, 3, 4, -1, 5, 6, 7, 8, 9, -1}; return t[s]; }

// A warp's 32 rows x 64 features (thread = row, pk = its 64 bf16 values packed in pairs) -> the row-TRANSPOSED image of a
// plane (tr_offset layout, F = 256: blocks of 64 rows, 16-byte units of 8 consecutive rows per feature), which is what
// the weight-gradient MMAs (K = rows) bulk-copy as operands.  Goes through a 4 KB shared-memory block: every thread
// drops its values feature-major, then the warp copies out 16-byte units.  Replaces a separate transpose pass over HBM.
__device__ __forceinline__ void store_transposed(uint32_t stage, int lane, const uint32_t (&pk)[32], uint8_t* __restrict__ plane_t,
                                                 int block64, int rowgroup0, int col0) {
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        const uint32_t a = stage + (uint32_t)((2 * j) * 64 + lane * 2);
        asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"((unsigned short)(pk[j] & 0xffffu)) : "memory");
        asm volatile("st.shared.u16 [%0], %1;" ::"r"(a + 64u), "h"((unsigned short)(pk[j] >> 16)) : "memory");
    }
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int u = lane + 32 * i, f = u >> 2, g = u & 3;
        uint4 v;
        asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                     : "r"(stage + (uint32_t)(f * 64 + g * 16)) : "memory");
        const int gf = col0 + f, rg = rowgroup0 + g;
        *reinterpret_cast<uint4*>(plane_t + (size_t)block64 * (256 * 128) + (gf >> 3) * 1024 + (gf & 7) * 128 + ((rg ^ (gf & 7)) << 4)) = v;
    }
    __syncwarp();
}

// ---- epilogue bodies of the dgrad chain: the stage kind is a template parameter and whatever does not depend on the
// accumulator (relu masks = saved forward activations) is fetched before the wait on the MMA (see mlp_tcgen05.cu).
struct EpiArgs {
    uint64_t* acc_bar; uint32_t phase;
    uint32_t acc, act_out;
    int col0;
    bool valid;
    float g_sigma;
    const float* w_alpha;      // shared memory, at col0
    const uint4* mask;         // forward activation of the layer whose relu gates this delta (row-major bf16), or null
    uint4* delta_out;          // this stage's delta plane (row-major bf16), or null
    uint8_t* delta_t;          // the same plane's row-transposed image, or null
    uint32_t stage; int lane, block64, rowgroup0;
    float* dx;                 // dX row (208 floats)
};

// dX stages: accumulator -> fp32 row (stage 10 adds to what stage 4 stored)
template <bool kAccumulate>
__device__ __forceinline__ void epi_dx(const EpiArgs& E) {
    mbar_wait(E.acc_bar, E.phase);
    tc_fence_after();
    uint32_t v[2][32];
    tmem_ld32(E.acc, v[0]);
    tmem_ld32(E.acc + 32, v[1]);
    tmem_wait_ld();
    if (!E.valid) return;
#pragma unroll
    for (int gq = 0; gq < 2; ++gq)
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int c = E.col0 + 32 * gq + 4 * i;
            if (c < 208) {
                float4 o = make_float4(__uint_as_float(v[gq][4 * i]), __uint_as_float(v[gq][4 * i + 1]),
                                       __uint_as_float(v[gq][4 * i + 2]), __uint_as_float(v[gq][4 * i + 3]));
                float4* p = reinterpret_cast<float4*>(E.dx + c);
                if (kAccumulate) { const float4 old = *p; o.x += old.x; o.y += old.y; o.z += old.z; o.w += old.w; }
                *p = o;
            }
        }
}

// delta stages: accumulator (+ sigma-head term) gated by the saved activation -> bf16 delta in TMEM (next A operand) + HBM
// (kSave: the pose-only variant keeps the delta in TMEM only, no HBM plane and no transposed image)
template <bool kAlpha, bool kMask, bool kSave>
__device__ __forceinline__ void epi_delta(const EpiArgs& E) {
    uint4 m[8];
    if (kMask) {
#pragma unroll
        for (int i = 0; i < 8; ++i) m[i] = E.mask[i];
    }
    mbar_wait(E.acc_bar, E.phase);
    tc_fence_after();
    uint32_t v[2][32];
    tmem_ld32(E.acc, v[0]);
    tmem_ld32(E.acc + 32, v[1]);
    tmem_wait_ld();
    uint32_t pk[32];
#pragma unroll
    for (int gq = 0; gq < 2; ++gq) {
#pragma unroll
        for (int c8 = 0; c8 < 4; ++c8) {
            const uint32_t mw[4] = {m[gq * 4 + c8].x, m[gq * 4 + c8].y, m[gq * 4 + c8].z, m[gq * 4 + c8].w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int e = c8 * 8 + 2 * i;
                float a0 = __uint_as_float(v[gq][e]), a1 = __uint_as_float(v[gq][e + 1]);
                if (kAlpha) {                              // sigma head: d a7 += d sigma * w_alpha
                    a0 = fmaf(E.g_sigma, E.w_alpha[32 * gq + e], a0);
                    a1 = fmaf(E.g_sigma, E.w_alpha[32 * gq + e + 1], a1);
                }
                if (kMask) {
                    if (!(__uint_as_float(mw[i] << 16) > 0.f)) a0 = 0.f;
                    if (!(__uint_as_float(mw[i] & 0xffff0000u) > 0.f)) a1 = 0.f;
                }
                if (!E.valid) { a0 = 0.f; a1 = 0.f; }
                pk[gq * 16 + c8 * 4 + i] = pack_bf16(a0, a1);
            }
        }
        tmem_st16(E.act_out + 16 * gq, *reinterpret_cast<const uint32_t(*)[16]>(&pk[gq * 16]));
        if (kSave && E.delta_out != nullptr) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
                E.delta_out[gq * 4 + i] = make_uint4(pk[gq * 16 + 4 * i], pk[gq * 16 + 4 * i + 1], pk[gq * 16 + 4 * i + 2], pk[gq * 16 + 4 * i + 3]);
        }
    }
    if (kSave && E.delta_t != nullptr) store_transposed(E.stage, E.lane, pk, E.delta_t, E.block64, E.rowgroup0, E.col0);
}

// kSaveDeltas = false: the pose-only variant (no weight gradients follow), whose epilogue writes dX only; delta_save and
// delta_t are not touched.
template <bool kSaveDeltas>
__global__ void __launch_bounds__(kThreads, 1)
dgrad_kernel(const uint8_t* __restrict__ wstream,            // [84][16 KB] transposed-weight tiles (pack_dgrad)
             const float* __restrict__ w_rgb, const float* __restrict__ w_alpha,
             const float* __restrict__ d_raw,                // (*,4) gradient of raw, indexed by sample id
             const int* __restrict__ row_sample, const int* __restrict__ n_rows_ptr,
             const __nv_bfloat16* __restrict__ act_save,     // [9][cap][256] forward activations (row-major)
             const __nv_bfloat16* __restrict__ g_save,       // [cap][128]
             int cap,
             __nv_bfloat16* __restrict__ delta_save,         // [10][cap][256] deltas (row-major, bf16)
             uint8_t* __restrict__ delta_t,                  // [10][blocks of 64 rows][32 KB] the same, row-transposed
             float* __restrict__ dX) {                       // [cap][208]
    extern __shared__ uint8_t smem_raw[];
    Smem& S = *reinterpret_cast<Smem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_rows = *n_rows_ptr;
    const int n_tiles = (n_rows + DANBO_TILE_M - 1) / DANBO_TILE_M;
    for (int i = threadIdx.x; i < 384; i += kThreads) S.w_rgb[i] = w_rgb[i];
    for (int i = threadIdx.x; i < 256; i += kThreads) S.w_alpha[i] = w_alpha[i];
    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&S.w_full[s], 1); mbar_init(&S.w_empty[s], 1); }
        mbar_init(&S.acc_full[0], 1); mbar_init(&S.acc_full[1], 1);
        mbar_init(&S.act_ready[0], 8); mbar_init(&S.act_ready[1], 8);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&S.tmem_base)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = S.tmem_base;

    if (warp == 0) {
        const bool leader = elect_one();
        uint32_t ws = 0, wphase = 0;
        for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
            for (int s = 0; s < kNumStagesPerTile; ++s) {
                mbar_wait(&S.w_empty[ws], wphase ^ 1);
                if (leader) {
                    mbar_expect_tx(&S.w_full[ws], kStageBytes);
                    bulk_g2s(S.w[ws], wstream + (size_t)s * kStageBytes, kStageBytes, &S.w_full[ws]);
                }
                if (++ws == kStages) { ws = 0; wphase ^= 1; }
            }
        }
    } else if (warp == 1) {
        // fully unrolled per-tile schedule (see mlp_tcgen05.cu): runtime ring-slot arithmetic keeps descriptors in vector
        // registers and costs more issue time than the MMAs themselves
        const bool leader = elect_one();
        uint32_t r0 = 0, r1 = 0;
        const uint64_t w_desc0 = make_desc(0) | (uint64_t)((smem_u32(&S.w[0][0]) >> 4) & 0x3FFF);
        for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
#pragma unroll
            for (int s = 0; s < kDgradStages; ++s) {
                mbar_wait(&S.act_ready[0], r0 & 1); ++r0;
                tc_fence_after();
                const uint32_t a_in = tmem + kActCol + 128u * st_inbuf(s);
                const int nkc = st_kchunks(s);
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t d = tmem + kAccCol + 128u * h;
#pragma unroll
                    for (int kc = 0; kc < 4; ++kc) {
                        if (kc >= nkc) continue;
                        if ((h == 0 && kc == 2) || (h == 1 && kc == 0 && nkc <= 2)) { mbar_wait(&S.act_ready[1], r1 & 1); ++r1; }
                        const int tile = s == 0 ? h * 2 + kc : 4 + (s - 1) * 8 + h * 4 + kc;
                        const int slot = tile % kStages;
                        mbar_wait(&S.w_full[slot], (uint32_t)((tile / kStages) & 1));
                        tc_fence_after();
                        const uint64_t bdesc = w_desc0 + (uint64_t)((slot * kStageBytes) >> 4);
                        const uint32_t a_t = a_in + kc * 32;
                        if (leader) {
                            mma_ts(d, a_t, bdesc, kIdesc, kc > 0 ? 1u : 0u);
                            mma_ts(d, a_t + 8, bdesc + 2, kIdesc, 1u);
                            mma_ts(d, a_t + 16, bdesc + 4, kIdesc, 1u);
                            mma_ts(d, a_t + 24, bdesc + 6, kIdesc, 1u);
                            tc_commit(&S.w_empty[slot]);
                            if (kc == nkc - 1) tc_commit(&S.acc_full[h]);
                        }
                        __syncwarp();
                    }
                }
            }
        }
    } else {
        const int q = warp & 3, ch = (warp - 2) >> 2;
        const int row = q * 32 + lane;
        const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
        const uint32_t stage_addr = smem_u32(S.stage[warp - 2]);
        const int n_blk64 = (cap + 63) / 64;
        const size_t plane_t_bytes = (size_t)n_blk64 * (256 * 128);
        uint32_t f0 = 0, f1 = 0;
        for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
            const int grow = t * DANBO_TILE_M + row;
            const bool valid = grow < n_rows;
            const int blk64 = t * 2 + (q >> 1);                  // 64-row block of this warp's rows in the transposed images
            float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
            if (valid) g = reinterpret_cast<const float4*>(d_raw)[row_sample[grow]];
            // ---- prologue: delta9 = (d rgb . W_rgb) * [g > 0] for this thread's 64 of the 128 view-layer units
            {
                uint32_t pk[32];
                const uint4* gs = reinterpret_cast<const uint4*>(g_save + (size_t)(valid ? grow : 0) * 128 + ch * 64);
#pragma unroll
                for (int c8 = 0; c8 < 8; ++c8) {
                    const uint4 gv = gs[c8];
                    const uint32_t gw[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int c = ch * 64 + c8 * 8 + 2 * i;
                        const float g0 = __uint_as_float(gw[i] << 16), g1 = __uint_as_float(gw[i] & 0xffff0000u);
                        float d0 = g.x * S.w_rgb[c] + g.y * S.w_rgb[128 + c] + g.z * S.w_rgb[256 + c];
                        float d1 = g.x * S.w_rgb[c + 1] + g.y * S.w_rgb[128 + c + 1] + g.z * S.w_rgb[256 + c + 1];
                        if (!(g0 > 0.f) || !valid) d0 = 0.f;
                        if (!(g1 > 0.f) || !valid) d1 = 0.f;
                        pk[c8 * 4 + i] = pack_bf16(d0, d1);
                    }
                }
                const uint32_t a0 = tmem + lane_addr + kActCol + 32u * ch;          // buffer 0, packed columns
                tmem_st16(a0, *reinterpret_cast<const uint32_t(*)[16]>(&pk[0]));
                tmem_st16(a0 + 16, *reinterpret_cast<const uint32_t(*)[16]>(&pk[16]));
                if (kSaveDeltas && grow < cap) {
                    uint4* dst = reinterpret_cast<uint4*>(delta_save + (size_t)grow * 256 + ch * 64);
#pragma unroll
                    for (int i = 0; i < 8; ++i) dst[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
                }
                if (kSaveDeltas && delta_t != nullptr && blk64 < n_blk64)
                    store_transposed(stage_addr, lane, pk, delta_t, blk64, (q & 1) * 4, ch * 64);
                tmem_wait_st();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) { mbar_arrive(&S.act_ready[0]); mbar_arrive(&S.act_ready[1]); }
            }
            for (int s = 0; s < kDgradStages; ++s) {
                const int mp = st_mask_plane(s), dp = st_delta_plane(s);
                for (int h = 0; h < 2; ++h) {
                    EpiArgs E;
                    E.acc_bar = &S.acc_full[h];
                    if (h == 0) { E.phase = f0 & 1; ++f0; } else { E.phase = f1 & 1; ++f1; }
                    E.acc = tmem + lane_addr + kAccCol + 128u * h + 64u * ch;
                    E.act_out = tmem + lane_addr + kActCol + 128u * (1 - st_inbuf(s)) + 64u * h + 32u * ch;
                    E.col0 = h * 128 + ch * 64;
                    E.valid = valid;
                    E.g_sigma = g.w;
                    E.w_alpha = S.w_alpha + E.col0;
                    E.mask = mp >= 0 ? reinterpret_cast<const uint4*>(act_save + ((size_t)mp * cap + (valid ? grow : 0)) * 256 + E.col0) : nullptr;
                    E.delta_out = (dp >= 0 && grow < cap) ? reinterpret_cast<uint4*>(delta_save + ((size_t)dp * cap + grow) * 256 + E.col0) : nullptr;
                    E.delta_t = (dp >= 0 && delta_t != nullptr && blk64 < n_blk64) ? delta_t + (size_t)dp * plane_t_bytes : nullptr;
                    E.stage = stage_addr; E.lane = lane; E.block64 = blk64; E.rowgroup0 = (q & 1) * 4;
                    E.dx = dX + (size_t)(valid ? grow : 0) * 208;
                    if (s == 4) epi_dx<false>(E);
                    else if (s == 10) epi_dx<true>(E);
                    else if (s == 0) epi_delta<false, false, kSaveDeltas>(E);
                    else if (s == 1) epi_delta<true, true, kSaveDeltas>(E);
                    else epi_delta<false, true, kSaveDeltas>(E);
                    tmem_wait_st();
                    tc_fence_before();
                    __syncwarp();
                    // the last stage's accumulators are released by the NEXT tile's prologue arrival
                    if (s < kDgradStages - 1 && lane == 0) mbar_arrive(&S.act_ready[h]);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(512u) : "memory");
}

// ---- transposed-weight tile stream for dgrad ---------------------------------------------------------------
struct PackArgs { const float* w[8]; const float* w_feat; const float* w_view; };

// tile index -> (stage, half, kc); stages have 4, 8, 8, ... tiles
__host__ __device__ inline void tile_to_stage(int tile, int& s, int& h, int& kc) {
    if (tile < 4) { s = 0; h = tile / 2; kc = tile % 2; return; }
    tile -= 4;
    s = 1 + tile / 8;
    const int r = tile % 8;
    h = r / 4; kc = r % 4;
}

__global__ void pack_dgrad_kernel(PackArgs a, __nv_bfloat16* __restrict__ wstream) {
    const int total = kNumStagesPerTile * 128 * 64;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int tile = i / (128 * 64), e = i % (128 * 64);
        const int n = e / 64, k = e % 64;
        int s, h, kc;
        tile_to_stage(tile, s, h, kc);
        const int nn = h * 128 + n;               // output column of the stage (an INPUT unit of the layer)
        const int kk = kc * 64 + k;               // contraction index (an OUTPUT unit of the layer)
        float val = 0.f;
        switch (s) {
            case 0: val = a.w_view[(size_t)kk * 411 + nn]; break;                                   // Wv (128,411)[:, :256]
            case 1: val = a.w_feat[(size_t)kk * 256 + nn]; break;
            case 2: val = a.w[7][(size_t)kk * 256 + nn]; break;
            case 3: val = a.w[6][(size_t)kk * 256 + nn]; break;
            case 4: val = nn < DANBO_X_COLS ? a.w[5][(size_t)kk * 451 + nn] : 0.f; break;             // W5[:, :195]
            case 5: val = a.w[5][(size_t)kk * 451 + DANBO_X_COLS + nn]; break;                         // W5[:, 195:]
            case 6: val = a.w[4][(size_t)kk * 256 + nn]; break;
            case 7: val = a.w[3][(size_t)kk * 256 + nn]; break;
            case 8: val = a.w[2][(size_t)kk * 256 + nn]; break;
            case 9: val = a.w[1][(size_t)kk * 256 + nn]; break;
            default: val = nn < DANBO_X_COLS ? a.w[0][(size_t)kk * DANBO_X_COLS + nn] : 0.f; break;  // W0 (256,195)
        }
        wstream[(size_t)tile * (128 * 64) + sw128_offset((uint32_t)n, (uint32_t)k) / 2] = __float2bfloat16_rn(val);
    }
}

// ---- row-major planes -> K-major (K = rows) operand blocks --------------------------------------------------
// in : [planes][cap][ld_in] bf16 row-major (first `width` columns used); out: [planes][n_blocks][256*128 B].
// Rows >= *rows_ptr are written as zeros (they sit in the last 64-row block and must not contribute).
__global__ void __launch_bounds__(256)
transpose_kernel(const __nv_bfloat16* __restrict__ in, int cap, int ld_in, int width, const int* __restrict__ rows_ptr,
                 uint8_t* __restrict__ out, size_t plane_out_bytes) {
    const int R = *rows_ptr;
    const int blk = blockIdx.x, fb = blockIdx.y, plane = blockIdx.z;      // 64-row block, 64-feature block
    if (blk * 64 >= R) return;
    __shared__ __nv_bfloat16 tile[64][72];
    const __nv_bfloat16* src = in + (size_t)plane * cap * ld_in;
    for (int i = threadIdx.x; i < 64 * 8; i += 256) {
        const int r = i / 8, c8 = i % 8;
        const int gr = blk * 64 + r, gc = fb * 64 + c8 * 8;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (gr < R && gc < width) v = *reinterpret_cast<const uint4*>(src + (size_t)gr * ld_in + gc);
        *reinterpret_cast<uint4*>(&tile[r][c8 * 8]) = v;
    }
    __syncthreads();
    uint8_t* dst = out + (size_t)plane * plane_out_bytes + (size_t)blk * (256 * 128);
    for (int i = threadIdx.x; i < 64 * 8; i += 256) {
        const int f = i / 8, rc = i % 8;                                   // feature, 8-row chunk
        __align__(16) __nv_bfloat16 v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = tile[rc * 8 + j][f];
        const uint32_t gf = fb * 64 + f;
        *reinterpret_cast<uint4*>(dst + (gf >> 3) * 1024u + (gf & 7) * 128u + ((rc ^ (gf & 7)) << 4)) = *reinterpret_cast<const uint4*>(v);
    }
}

// ---- weight gradients: dW[item] = delta^T . act, K = rows --------------------------------------------------
struct WgradItem { int a_plane, a_half, b_plane; };       // b_plane: 0..8 = forward activation planes, 9 = X
struct WgradPlan { WgradItem item[21]; int n_items; };

constexpr int kWStages = 4;
struct __align__(1024) WSmem {
    uint8_t a[kWStages][128 * 128];        // [128 out x 64 rows] 16 KB
    uint8_t b[kWStages][256 * 128];        // [256 in x 64 rows] 32 KB
    uint64_t full[kWStages], empty[kWStages], done;
    uint32_t tmem_base;
};
constexpr uint32_t kIdescN256 = (1u << 4) | (1u << 7) | (1u << 10) | ((256u >> 3) << 17) | ((128u >> 4) << 24);

__global__ void __launch_bounds__(192, 1)
wgrad_kernel(WgradPlan plan, const uint8_t* __restrict__ deltaT, size_t delta_plane_bytes, const uint8_t* __restrict__ actT,
             size_t act_plane_bytes, const int* __restrict__ rows_ptr, int n_splits,
             float* __restrict__ partial /* [item][split][128][256] */) {
    extern __shared__ uint8_t smem_raw[];
    WSmem& S = *reinterpret_cast<WSmem*>(smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int item = blockIdx.x / n_splits, split = blockIdx.x % n_splits;
    const int n_blocks = (*rows_ptr + 63) / 64;
    const WgradItem it = plan.item[item];
    if (threadIdx.x == 0) {
        for (int s = 0; s < kWStages; ++s) { mbar_init(&S.full[s], 1); mbar_init(&S.empty[s], 1); }
        mbar_init(&S.done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&S.tmem_base)), "r"(256u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = S.tmem_base;
    const uint8_t* A = deltaT + (size_t)it.a_plane * delta_plane_bytes + (size_t)it.a_half * (128 * 128);
    const uint8_t* B = actT + (size_t)it.b_plane * act_plane_bytes;
    if (warp == 0) {
        const bool leader = elect_one();
        uint32_t st = 0, ph = 0;
        for (int kb = split; kb < n_blocks; kb += n_splits) {
            mbar_wait(&S.empty[st], ph ^ 1);
            if (leader) {
                mbar_expect_tx(&S.full[st], 128 * 128 + 256 * 128);
                bulk_g2s(S.a[st], A + (size_t)kb * (256 * 128), 128 * 128, &S.full[st]);
                bulk_g2s(S.b[st], B + (size_t)kb * (256 * 128), 256 * 128, &S.full[st]);
            }
            if (++st == kWStages) { st = 0; ph ^= 1; }
        }
    } else if (warp == 1) {
        const bool leader = elect_one();
        uint32_t st = 0, ph = 0;
        const uint64_t desc_hi = make_desc(0);
        bool first = true;
        for (int kb = split; kb < n_blocks; kb += n_splits) {
            mbar_wait(&S.full[st], ph);
            tc_fence_after();
            const uint64_t ad = desc_hi | (uint64_t)((smem_u32(S.a[st]) >> 4) & 0x3FFF);
            const uint64_t bd = desc_hi | (uint64_t)((smem_u32(S.b[st]) >> 4) & 0x3FFF);
            if (leader) {
                mma_ss(tmem, ad, bd, kIdescN256, first ? 0u : 1u);
                mma_ss(tmem, ad + 2, bd + 2, kIdescN256, 1u);
                mma_ss(tmem, ad + 4, bd + 4, kIdescN256, 1u);
                mma_ss(tmem, ad + 6, bd + 6, kIdescN256, 1u);
                tc_commit(&S.empty[st]);
            }
            __syncwarp();
            first = false;
            if (++st == kWStages) { st = 0; ph ^= 1; }
        }
        if (leader) tc_commit(&S.done);
        __syncwarp();
    } else {
        // 4 epilogue warps: thread = output row (out unit) of this half, 256 columns (in units)
        const int q = warp & 3;
        const int row = q * 32 + lane;
        float* dst = partial + (((size_t)item * n_splits + split) * 128 + row) * 256;
        const bool any = split < n_blocks;
        if (any) {
            mbar_wait(&S.done, 0);
            tc_fence_after();
        }
#pragma unroll 1
        for (int gq = 0; gq < 8; ++gq) {
            uint32_t v[32];
            if (any) { tmem_ld32(tmem + ((uint32_t)(q * 32) << 16) + 32 * gq, v); tmem_wait_ld(); }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                float4 o = make_float4(0.f, 0.f, 0.f, 0.f);
                if (any) o = make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]), __uint_as_float(v[4 * i + 2]), __uint_as_float(v[4 * i + 3]));
                reinterpret_cast<float4*>(dst + 32 * gq)[i] = o;
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(256u) : "memory");
}

struct ReduceDst { float* ptr; int ld, n_valid, m_rows; };     // destination of an item: rows [a_half*128, +m_rows) of ptr
struct ReducePlan { ReduceDst dst[21]; int a_half[21]; int n_items; };

__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(ReducePlan plan, const float* __restrict__ partial, int n_splits) {
    const int item = blockIdx.y;
    const ReduceDst d = plan.dst[item];
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 128 * 256; i += gridDim.x * blockDim.x) {
        const int r = i / 256, c = i % 256;
        if (r >= d.m_rows || c >= d.n_valid) continue;
        float s = 0.f;
        for (int k = 0; k < n_splits; ++k) s += partial[(((size_t)item * n_splits + k) * 128 + r) * 256 + c];
        d.ptr[(size_t)(plan.a_half[item] * 128 + r) * d.ld + c] += s;
    }
}

// bias gradients: db[plane][c] += sum_rows delta[plane][row][c]    (row-major bf16 planes)
struct BiasPlan { float* db[10]; };
__global__ void __launch_bounds__(256)
colsum_planes_kernel(const __nv_bfloat16* __restrict__ delta, int cap, const int* __restrict__ rows_ptr, BiasPlan plan,
                     int rows_per_block) {
    const int plane = blockIdx.y;
    if (plan.db[plane] == nullptr) return;
    const int R = *rows_ptr;
    const int r0 = blockIdx.x * rows_per_block;
    if (r0 >= R) return;
    const int r1 = min(R, r0 + rows_per_block);
    const int c = threadIdx.x;
    const __nv_bfloat16* src = delta + (size_t)plane * cap * 256;
    float s = 0.f;
    for (int r = r0; r < r1; ++r) s += __bfloat162float(src[(size_t)r * 256 + c]);
    atomicAdd(plan.db[plane] + c, s);
}

}  // namespace mlpb
}  // namespace danbo

using namespace danbo;

extern "C" int danbo_mlp_bwd_workspace(int cap, long long* wstream_bytes, long long* delta_bytes, long long* deltaT_bytes,
                                       long long* actT_bytes, long long* partial_bytes, int* n_splits) {
    const long long blocks = (cap + 63) / 64;
    *wstream_bytes = (long long)mlpb::kNumStagesPerTile * mlpb::kStageBytes;
    *delta_bytes = 10LL * cap * 256 * 2;
    *deltaT_bytes = 10LL * blocks * 256 * 128;
    *actT_bytes = 10LL * blocks * 256 * 128;          // 9 activation planes + X
    *n_splits = 7;
    *partial_bytes = 21LL * (*n_splits) * 128 * 256 * 4;
    return 0;
}

extern "C" int danbo_pack_mlp_dgrad(const float* const* w_pts, const float* w_feat, const float* w_view, void* wstream,
                                    void* stream) {
    mlpb::PackArgs a;
    for (int i = 0; i < 8; ++i) a.w[i] = w_pts[i];
    a.w_feat = w_feat; a.w_view = w_view;
    mlpb::pack_dgrad_kernel<<<296, 256, 0, (cudaStream_t)stream>>>(a, (__nv_bfloat16*)wstream);
    DANBO_CHECK_LAUNCH();
    return 0;
}

template <bool kSaveDeltas>
static int launch_dgrad(const void* wstream_t, const float* w_rgb, const float* w_alpha, const float* d_raw,
                        const int* row_sample, const int* rows_dev, int max_rows, const void* act_save,
                        const void* g_save, int cap, void* delta_save, void* delta_t, float* dX, int num_sms,
                        void* stream) {
    const int smem = (int)sizeof(mlpb::Smem) + 1024;
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(mlpb::dgrad_kernel<kSaveDeltas>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return (int)e;
        attr = true;
    }
    int tiles = (max_rows + DANBO_TILE_M - 1) / DANBO_TILE_M;
    int grid = num_sms < tiles ? num_sms : tiles;
    mlpb::dgrad_kernel<kSaveDeltas><<<grid, mlpb::kThreads, smem, (cudaStream_t)stream>>>(
        (const uint8_t*)wstream_t, w_rgb, w_alpha, d_raw, row_sample, rows_dev, (const __nv_bfloat16*)act_save,
        (const __nv_bfloat16*)g_save, cap, (__nv_bfloat16*)delta_save, (uint8_t*)delta_t, dX);
    DANBO_CHECK_LAUNCH();
    return 0;
}

// Fused data-gradient chain.  delta_save planes: 0 = delta of views_linears.0 (128 wide), 1 = d feature, 2..9 = deltas
// of pts_linears.7..0.  dX (cap,208) fp32 is fully written for valid rows.  delta_save = NULL (then delta_t must be
// NULL too) selects the variant that writes dX only: no weight gradient will read the planes (pose-only backward).
extern "C" int danbo_mlp_dgrad(const void* wstream_t, const float* w_rgb, const float* w_alpha, const float* d_raw,
                               const int* row_sample, const int* rows_dev, int max_rows, const void* act_save,
                               const void* g_save, int cap, void* delta_save, void* delta_t, float* dX, int num_sms,
                               void* stream) {
    if (max_rows <= 0) return 0;
    if (delta_save == nullptr) {
        if (delta_t != nullptr) return -1;
        return launch_dgrad<false>(wstream_t, w_rgb, w_alpha, d_raw, row_sample, rows_dev, max_rows, act_save, g_save,
                                   cap, nullptr, nullptr, dX, num_sms, stream);
    }
    return launch_dgrad<true>(wstream_t, w_rgb, w_alpha, d_raw, row_sample, rows_dev, max_rows, act_save, g_save, cap,
                              delta_save, delta_t, dX, num_sms, stream);
}

// Weight + bias gradients from the saved deltas / activations.
//   act_save [9][cap][256], x_rows [cap][208], delta_save [10][cap][256] (row-major bf16);
//   deltaT / actT / partial: workspaces (danbo_mlp_bwd_workspace).
//   dw[11] = { views_linears.0.weight (128,411), feature_linear.weight, pts_linears.7, .6, .5 (256,451), .4, .3, .2, .1,
//              .0 (256,195) } -- wait order below; db[9] = { feature_linear.bias, pts_linears.7..0 bias }.  Accumulated.
extern "C" int danbo_mlp_wgrad(const void* act_save, const void* x_rows, const void* delta_save, int cap,
                               const int* rows_dev, int max_rows, void* deltaT, int delta_t_ready, void* actT,
                               float* partial, float* const* dw, float* const* db, void* stream) {
    if (max_rows <= 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int blocks = (cap + 63) / 64;
    const size_t plane_bytes = (size_t)blocks * 256 * 128;
    const int used_blocks = (max_rows + 63) / 64;
    // 1. transposes: deltas (10 planes; skipped when danbo_mlp_dgrad wrote deltaT itself), activations (9 planes), X
    if (!delta_t_ready) {
        mlpb::transpose_kernel<<<dim3(used_blocks, 4, 10), 256, 0, st>>>((const __nv_bfloat16*)delta_save, cap, 256, 256, rows_dev,
                                                                          (uint8_t*)deltaT, plane_bytes);
        DANBO_CHECK_LAUNCH();
    }
    mlpb::transpose_kernel<<<dim3(used_blocks, 4, 9), 256, 0, st>>>((const __nv_bfloat16*)act_save, cap, 256, 256, rows_dev,
                                                                     (uint8_t*)actT, plane_bytes);
    DANBO_CHECK_LAUNCH();
    mlpb::transpose_kernel<<<dim3(used_blocks, 4, 1), 256, 0, st>>>((const __nv_bfloat16*)x_rows, cap, 208, 208, rows_dev,
                                                                     (uint8_t*)actT + 9 * plane_bytes, plane_bytes);
    DANBO_CHECK_LAUNCH();
    // 2. the 11 GEMMs as 21 (gemm, output half) items
    //    gemm: A delta plane, B activation plane (9 = X), destination
    struct G { int a, b, dst, col0, nvalid, m; };
    const G gemms[11] = {
        {0, 8, 0, 0, 256, 128},      // views_linears.0.weight[:, :256]   = d9^T feat
        {1, 7, 1, 0, 256, 256},      // feature_linear.weight            = dfeat^T a7
        {2, 6, 2, 0, 256, 256},      // pts_linears.7                    = d7^T a6
        {3, 5, 3, 0, 256, 256},      // pts_linears.6
        {4, 9, 4, 0, 195, 256},      // pts_linears.5[:, :195]           = d5^T X
        {4, 4, 4, 195, 256, 256},    // pts_linears.5[:, 195:]           = d5^T a4
        {5, 3, 5, 0, 256, 256},      // pts_linears.4
        {6, 2, 6, 0, 256, 256},      // pts_linears.3
        {7, 1, 7, 0, 256, 256},      // pts_linears.2
        {8, 0, 8, 0, 256, 256},      // pts_linears.1
        {9, 9, 9, 0, 195, 256},      // pts_linears.0 (256,195)          = d0^T X
    };
    const int ld[10] = {411, 256, 256, 256, 451, 256, 256, 256, 256, 195};
    mlpb::WgradPlan plan;
    mlpb::ReducePlan rplan;
    int n = 0;
    for (int g = 0; g < 11; ++g)
        for (int h = 0; h < gemms[g].m / 128; ++h) {
            plan.item[n] = {gemms[g].a, h, gemms[g].b};
            rplan.dst[n] = {dw[gemms[g].dst] + gemms[g].col0, ld[gemms[g].dst], gemms[g].nvalid, 128};
            rplan.a_half[n] = h;
            ++n;
        }
    plan.n_items = rplan.n_items = n;          // 21
    const int n_splits = 7;
    const int smem = (int)sizeof(mlpb::WSmem) + 1024;
    static bool attr = false;
    if (!attr) {
        cudaError_t e = cudaFuncSetAttribute(mlpb::wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
        if (e != cudaSuccess) return (int)e;
        attr = true;
    }
    mlpb::wgrad_kernel<<<n * n_splits, 192, smem, st>>>(plan, (const uint8_t*)deltaT, plane_bytes, (const uint8_t*)actT,
                                                         plane_bytes, rows_dev, n_splits, partial);
    DANBO_CHECK_LAUNCH();
    mlpb::wgrad_reduce_kernel<<<dim3(32, n), 256, 0, st>>>(rplan, partial, n_splits);
    DANBO_CHECK_LAUNCH();
    // 3. bias gradients: planes 1..9 -> feature_linear.bias, pts_linears.7..0 bias
    mlpb::BiasPlan bp;
    bp.db[0] = nullptr;
    for (int i = 0; i < 9; ++i) bp.db[1 + i] = db[i];
    const int rpb = 128;
    mlpb::colsum_planes_kernel<<<dim3((max_rows + rpb - 1) / rpb, 10), 256, 0, st>>>((const __nv_bfloat16*)delta_save, cap,
                                                                                    rows_dev, bp, rpb);
    DANBO_CHECK_LAUNCH();
    return 0;
}
