// InfoNCE scoring + loss on the tcgen05 tensor cores, forward and backward, score tiles kept on chip.
// Replaces score_function + the loss block of ContrastiveEstimationTrainer.train
// (contrastive_estimation_training.py:12-22, 106-122, 141, 166) and its autograd for the sizes where the
// score GEMM dominates (>= 128 candidates per softmax, E a multiple of 64).  Smaller / regularised cases stay on
// the CUDA-core kernels of infonce.cu, which share the lse layout.
//
// Problems: nprob independent (rows x cols) = (Bp x Bp) score matrices over E:
//   all-steps: nprob = 1, Bp = B*K, prediction row r = (d,k), target column c = (t,k')
//   per-step : nprob = K, Bp = B,   prediction row d, target column t, one problem per step k
// Both operands are packed as K-major bf16 hi/lo planes  X[plane][prob][row][E]  (targets are transposed out of
// their strided (B,E,K) view on the way), fp32-faithful arithmetic = 3 MMAs per product.
//
// Forward (nce_umma_fwd_kernel): CTA = (prob, 128 target columns) loops over all 128-row prediction tiles.
//   D[target c (TMEM lane), prediction r (column)] -- targets sit on M, so the softmax reduction over predictions
//   is a per-THREAD online max / sum-exp over the accumulator row: no shuffles, no partial buffers; two TMEM
//   accumulators overlap the reduction of tile i with the MMAs of tile i+1.
// Backward (nce_umma_bwd_kernel): launched twice with the roles swapped (owner = targets -> dZ, owner =
//   predictions -> dP).  CTA = (prob, 128 owner rows, 256-wide slice of E); per tile of the other operand:
//   S = owner . other^T  ->  G = dL/dS in registers  ->  bf16 hi/lo into a SWIZZLE_128B K-major smem tile  ->
//   acc[owner rows, E slice] += G . other  (other read as MN-major B from the same K-major chunk layout).
//   No atomics, no global score tensor; each output element is written once.
#include "common.cuh"
#include "umma.cuh"

namespace cpc {
using namespace umma;

constexpr int NU_THREADS = 256;
constexpr int NU_TILE = 2 * 128 * 128;            // 32 KB: 128 rows x 64 k, both planes
constexpr int NU_FSTAGES = 3;                     // forward: stages of (A chunk, B chunk)
constexpr int NU_BSTAGES = 2;                     // backward ring

struct NuGeom {
    int B, K, E, all, kind;
    int Bp, nprob, nT, EC;                        // rows per problem, problems, 128-row tiles, 64-wide E chunks
    int passes;                                   // MMA passes per product: 3 = fp32-faithful (hi*hi + hi*lo + lo*hi),
                                                  // 1 = bf16 operand mode (precision = 1: the hi planes only)
    float lambda;
};

static NuGeom nu_geom(const cpc_infonce_params* p) {
    NuGeom g;
    g.B = p->batch; g.K = p->steps; g.E = p->enc; g.all = p->all_steps ? 1 : 0; g.kind = p->score_kind;
    g.Bp = g.all ? g.B * g.K : g.B;
    g.nprob = g.all ? 1 : g.K;
    g.nT = ceil_div(g.Bp, 128);
    g.EC = g.E / 64;
    g.lambda = p->regularization;
    g.passes = p->precision == 0 ? 3 : 1;
    return g;
}

// src element (prob, row, e) at base + prob*sp + row_major*s1 + row_minor*s2 + e*se, row = row_major*minor + row_minor
struct NuSrc { const float* p; long long sp, s1, s2, se; int minor; };

// fp32 (strided) -> bf16 [plane][prob][row][E]; one thread per 8 consecutive e
__global__ void __launch_bounds__(256) nu_pack_kernel(NuSrc src, __nv_bfloat16* __restrict__ out, int nprob, int Bp, int E) {
    const long groups = (long)nprob * Bp * (E >> 3);
    const long plane = (long)nprob * Bp * E;
    for (long gi = (long)blockIdx.x * blockDim.x + threadIdx.x; gi < groups; gi += (long)gridDim.x * blockDim.x) {
        const int e0 = (int)(gi % (E >> 3)) << 3;
        const long pr = gi / (E >> 3);
        const int row = (int)(pr % Bp), prob = (int)(pr / Bp);
        const float* s = src.p + prob * src.sp + (long long)(row / src.minor) * src.s1 + (long long)(row % src.minor) * src.s2;
        __align__(16) __nv_bfloat16 hi[8];
        __align__(16) __nv_bfloat16 lo[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float v = __ldg(s + (long long)(e0 + i) * src.se);
            hi[i] = __float2bfloat16_rn(v);
            lo[i] = __float2bfloat16_rn(v - __bfloat162float(hi[i]));
        }
        const long o = pr * E + e0;
        *reinterpret_cast<uint4*>(out + o) = *reinterpret_cast<const uint4*>(hi);
        *reinterpret_cast<uint4*>(out + plane + o) = *reinterpret_cast<const uint4*>(lo);
    }
}

// softplus(u) = max(u, 0) + log1p(e), sigmoid(u) = (u >= 0 ? 1 : e) / (1 + e) with e = exp(-|u|) in (0, 1]: one ex2, one lg2
// and one reciprocal on the special-function unit per score (the epilogues are bound by it: the libm versions,
// log1pf(expf(u)) and 1 / (1 + expf(-u)), made the softplus sweep 2.3x slower than the linear one).  Relative error
// ~1e-6; log1p switches to its series below 1e-3, where 1 + e would round the information away.
__device__ __forceinline__ float nu_log1p_small(float e) { return e < 1e-3f ? e * fmaf(e, fmaf(e, 0.33333333f, -0.5f), 1.f) : __logf(1.f + e); }
__device__ __forceinline__ float nu_softplus(float u) { return fmaxf(u, 0.f) + nu_log1p_small(__expf(-fabsf(u))); }
__device__ __forceinline__ void nu_softplus_sigmoid(float u, float& sp, float& sg) {
    const float e = __expf(-fabsf(u));
    sp = fmaxf(u, 0.f) + nu_log1p_small(e);
    sg = __fdividef(u >= 0.f ? 1.f : e, 1.f + e);
}

// ---- forward ------------------------------------------------------------------------------------------------
struct __align__(8) NuFwdBarriers {
    uint64_t full[NU_FSTAGES], empty[NU_FSTAGES], acc_full[2], acc_empty[2];
    uint32_t tmem_base;
    float red[4][4];
};

// per-CTA partials: [cta][0] sum over its columns of (lse - diag), [1] max score, [2] sum of scores, [3] regulariser
template <int KIND, bool REG>
__global__ void __launch_bounds__(NU_THREADS, 1) nce_umma_fwd_kernel(const __grid_constant__ CUtensorMap tmap_z,
                                                                    const __grid_constant__ CUtensorMap tmap_p,
                                                                    const NuGeom g, float* __restrict__ lse,
                                                                    float* __restrict__ partials) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    NuFwdBarriers* bars = reinterpret_cast<NuFwdBarriers*>(smem + NU_FSTAGES * 2 * NU_TILE);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int prob = blockIdx.x / g.nT, ct = blockIdx.x - prob * g.nT;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmap_z);
        prefetch_tmap(&tmap_p);
        for (int s = 0; s < NU_FSTAGES; ++s) { mbar_init(&bars->full[s], 1); mbar_init(&bars->empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&bars->acc_full[b], 1); mbar_init(&bars->acc_empty[b], 4); }
        fence_barrier_init();
    }
    if (warp == 2) { tmem_alloc(&bars->tmem_base, 256); tmem_relinquish(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;

    if (warp == 0) {
        if (lane == 0) {
            uint32_t n = 0;
            for (int rt = 0; rt < g.nT; ++rt)
                for (int q = 0; q < g.EC; ++q, ++n) {
                    const int stage = n % NU_FSTAGES;
                    mbar_wait(&bars->empty[stage], ((n / NU_FSTAGES) & 1) ^ 1);
                    mbar_expect_tx(&bars->full[stage], 2 * NU_TILE);
                    uint8_t* st = smem + stage * 2 * NU_TILE;
                    tma_load_4d(st, &tmap_z, &bars->full[stage], q * 64, ct * 128, prob, 0);
                    tma_load_4d(st + NU_TILE, &tmap_p, &bars->full[stage], q * 64, rt * 128, prob, 0);
                }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = make_idesc_bf16(128, 128, 0, 0);
            uint32_t n = 0;
            for (int rt = 0; rt < g.nT; ++rt) {
                const uint32_t buf = rt & 1;
                mbar_wait(&bars->acc_empty[buf], ((rt >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + buf * 128;
                for (int q = 0; q < g.EC; ++q, ++n) {
                    const int stage = n % NU_FSTAGES;
                    mbar_wait(&bars->full[stage], (n / NU_FSTAGES) & 1);
                    tc_fence_after();
                    const uint32_t a0 = smem_u32(smem + stage * 2 * NU_TILE), b0 = a0 + NU_TILE;
#pragma unroll
                    for (int cb = 0; cb < g.passes; ++cb) {                         // (hi,hi) (hi,lo) (lo,hi)
                        const uint32_t a_addr = a0 + (cb == 2 ? 128 * 128 : 0);
                        const uint32_t b_addr = b0 + (cb == 1 ? 128 * 128 : 0);
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            mma_bf16(d_tmem, make_smem_desc(a_addr + k * 32, 16, 1024), make_smem_desc(b_addr + k * 32, 16, 1024),
                                     idesc, (uint32_t)(q | cb | k));
                    }
                    tc_commit(&bars->empty[stage]);
                }
                tc_commit(&bars->acc_full[buf]);
            }
        }
    } else if (warp >= 4) {
        // thread = one target column; online max / sum-exp over every prediction row of the problem
        const int ew = warp & 3;
        const int cl = ew * 32 + lane;
        const int c = ct * 128 + cl;
        const bool col_ok = c < g.Bp;
        float m = -INFINITY, ssum = 0.f, diag = 0.f, vmax = -INFINITY, vsum = 0.f, reg = 0.f, grp = 0.f;
        const float inv_k = 1.f / (float)g.K;
        for (int rt = 0; rt < g.nT; ++rt) {
            const uint32_t buf = rt & 1;
            mbar_wait(&bars->acc_full[buf], (rt >> 1) & 1);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + buf * 128;
            const int n_valid = min(128, g.Bp - rt * 128);                   // prediction rows of this tile inside the problem
            for (int n0 = 0; n0 < 128; n0 += 32) {
                uint32_t raw[32];
                tmem_ld32(taddr + n0, raw);
                tmem_ld_wait();
                if (!col_ok || n0 >= n_valid) continue;
                float v[32];
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float u = __uint_as_float(raw[j]);
                    v[j] = KIND == CPC_SCORE_SOFTPLUS ? nu_softplus(u) : u;
                }
                if (n0 + 32 > n_valid) {                                     // ragged last batch: mask the rows outside
#pragma unroll
                    for (int j = 0; j < 32; ++j) if (n0 + j >= n_valid) v[j] = -INFINITY;
                }
                if (rt == ct && n0 == (cl & 96)) {                           // the tile on the diagonal holds S[c, c]
#pragma unroll
                    for (int j = 0; j < 32; ++j) if (j == (cl & 31)) diag = v[j];
                }
                float bmax = v[0];
#pragma unroll
                for (int j = 1; j < 32; ++j) bmax = fmaxf(bmax, v[j]);
#pragma unroll
                for (int j = 0; j < 32; ++j) vsum += v[j] > -INFINITY ? v[j] : 0.f;
                if (REG) {                                                   // groups of K consecutive rows = one item d
#pragma unroll
                    for (int j = 0; j < 32; ++j)
                        if (n0 + j < n_valid) {
                            grp += v[j];
                            if ((rt * 128 + n0 + j + 1) % g.K == 0) { const float a = grp * inv_k; reg += a * a; grp = 0.f; }
                        }
                }
                vmax = fmaxf(vmax, bmax);
                const float mn = fmaxf(m, bmax);
                float acc = 0.f;
#pragma unroll
                for (int j = 0; j < 32; ++j) acc += __expf(v[j] - mn);              // exp(-inf) = 0 for masked rows
                ssum = ssum * __expf(m - mn) + acc;
                m = mn;
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->acc_empty[buf]);
        }
        float term = 0.f;
        if (col_ok) {
            const float l = m + logf(ssum);
            lse[(size_t)prob * g.Bp + c] = l;
            term = l - diag;
        }
        term = warp_sum(term);
        vmax = warp_max(vmax);
        vsum = warp_sum(vsum);
        reg = warp_sum(reg);
        if (lane == 0) { bars->red[ew][0] = term; bars->red[ew][1] = vmax; bars->red[ew][2] = vsum; bars->red[ew][3] = reg; }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (cl == 0) {
            float* o = partials + (size_t)blockIdx.x * 4;
            o[0] = bars->red[0][0] + bars->red[1][0] + bars->red[2][0] + bars->red[3][0];
            o[1] = fmaxf(fmaxf(bars->red[0][1], bars->red[1][1]), fmaxf(bars->red[2][1], bars->red[3][1]));
            o[2] = bars->red[0][2] + bars->red[1][2] + bars->red[2][2] + bars->red[3][2];
            o[3] = bars->red[0][3] + bars->red[1][3] + bars->red[2][3] + bars->red[3][3];
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, 256); }
}

// out[0] loss, [1] max score, [2] loss without regulariser, [3] mean score
__global__ void __launch_bounds__(256) nce_umma_final_kernel(const float* __restrict__ partials, int ncta, NuGeom g,
                                                            float* __restrict__ out) {
    __shared__ float red[4][8];
    float a = 0.f, mx = -INFINITY, sm = 0.f, rg = 0.f;
    for (int i = threadIdx.x; i < ncta; i += blockDim.x) {
        a += partials[i * 4 + 0];
        mx = fmaxf(mx, partials[i * 4 + 1]);
        sm += partials[i * 4 + 2];
        rg += partials[i * 4 + 3];
    }
    a = warp_sum(a); mx = warp_max(mx); sm = warp_sum(sm); rg = warp_sum(rg);
    if ((threadIdx.x & 31) == 0) {
        red[0][threadIdx.x >> 5] = a; red[1][threadIdx.x >> 5] = mx; red[2][threadIdx.x >> 5] = sm; red[3][threadIdx.x >> 5] = rg;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        a = 0.f; mx = -INFINITY; sm = 0.f; rg = 0.f;
        for (int w = 0; w < 8; ++w) { a += red[0][w]; mx = fmaxf(mx, red[1][w]); sm += red[2][w]; rg += red[3][w]; }
        const double ncols = (double)g.nprob * g.Bp;
        const double nscores = (double)g.nprob * g.Bp * g.Bp;
        const double nreg = g.all ? (double)g.B * g.Bp : (double)g.B * g.B;
        const float loss0 = (float)(a / ncols);
        out[0] = loss0 + g.lambda * (float)(rg / nreg);
        out[1] = mx;
        out[2] = loss0;
        out[3] = (float)(sm / nscores);
    }
}

// ---- backward -----------------------------------------------------------------------------------------------
struct __align__(8) NuBwdBarriers {
    uint64_t full[NU_BSTAGES], empty[NU_BSTAGES], s_full[2], s_empty[2], g_full, g_empty, acc_full;
    uint32_t tmem_base;
    float lse_s[2][128];                          // target lse of the current other-tile, double-buffered by tile parity
};

struct NuBwd {
    NuGeom g;
    int owner_is_target;          // 1: owner rows are targets (output dZ), 0: owner rows are predictions (output dP)
    int n_slices;                 // E / 256 (ceil)
    int n_split;                  // CTAs sharing one (problem, owner tile, E slice): each takes a range of the other operand's
                                  // tiles and adds its partial result atomically (small problems: 16 CTAs -> up to 148)
    const float* lse;             // [prob * Bp + target]
    const float* grad_loss;
    float* out;                   // d_targets (B,E,K) contiguous or d_pred (B,K,E) contiguous
};

template <int KIND>
__global__ void __launch_bounds__(NU_THREADS, 1) nce_umma_bwd_kernel(const __grid_constant__ CUtensorMap tmap_owner,
                                                                    const __grid_constant__ CUtensorMap tmap_other,
                                                                    const NuBwd p) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* ring = smem;                                         // stage: [owner chunk 32 KB][other chunk 32 KB]
    uint8_t* gs = smem + NU_BSTAGES * 2 * NU_TILE;                // G: [plane][K atom (64 other rows)][128 owner rows][128 B]
    NuBwdBarriers* bars = reinterpret_cast<NuBwdBarriers*>(gs + 2 * NU_TILE);
    const NuGeom& g = p.g;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    int w = blockIdx.x;
    const int es = w % p.n_slices; w /= p.n_slices;
    const int sp = w % p.n_split; w /= p.n_split;
    const int ot = w % g.nT;
    const int prob = w / g.nT;
    const int st0 = (int)((long)sp * g.nT / p.n_split), st1 = (int)((long)(sp + 1) * g.nT / p.n_split);   // other tiles of this CTA
    const int n_it = st1 - st0;
    const int e_chunks = min(4, g.EC - es * 4);                   // 64-wide E chunks in this slice

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&tmap_owner);
        prefetch_tmap(&tmap_other);
        for (int s = 0; s < NU_BSTAGES; ++s) { mbar_init(&bars->full[s], 1); mbar_init(&bars->empty[s], 1); }
        for (int b = 0; b < 2; ++b) { mbar_init(&bars->s_full[b], 1); mbar_init(&bars->s_empty[b], 4); }
        mbar_init(&bars->g_full, 4);
        mbar_init(&bars->g_empty, 1);
        mbar_init(&bars->acc_full, 1);
        fence_barrier_init();
    }
    if (warp == 2) { tmem_alloc(&bars->tmem_base, 512); tmem_relinquish(); }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = bars->tmem_base;

    if (warp == 0) {
        if (lane == 0) {
            // order of ring uses (the MMA issuer consumes in the same order): P1(0), then per tile st: P1(st+1), P3(st)
            uint32_t n = 0;
            auto phase1 = [&](int st) {                                      // S = owner . other^T over E
                for (int q = 0; q < g.EC; ++q, ++n) {
                    const int stage = n % NU_BSTAGES;
                    mbar_wait(&bars->empty[stage], ((n / NU_BSTAGES) & 1) ^ 1);
                    mbar_expect_tx(&bars->full[stage], 2 * NU_TILE);
                    uint8_t* sp = ring + stage * 2 * NU_TILE;
                    tma_load_4d(sp, &tmap_owner, &bars->full[stage], q * 64, ot * 128, prob, 0);
                    tma_load_4d(sp + NU_TILE, &tmap_other, &bars->full[stage], q * 64, st * 128, prob, 0);
                }
            };
            if (n_it > 0) phase1(st0);
            for (int st = st0; st < st1; ++st) {
                if (st + 1 < st1) phase1(st + 1);
                for (int a = 0; a < e_chunks; ++a, ++n) {                    // phase 3: other rows, E slice chunk a
                    const int stage = n % NU_BSTAGES;
                    mbar_wait(&bars->empty[stage], ((n / NU_BSTAGES) & 1) ^ 1);
                    mbar_expect_tx(&bars->full[stage], NU_TILE);
                    tma_load_4d(ring + stage * 2 * NU_TILE + NU_TILE, &tmap_other, &bars->full[stage], (es * 4 + a) * 64,
                                st * 128, prob, 0);
                }
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc_s = make_idesc_bf16(128, 128, 0, 0);        // S: both K-major
            const uint32_t idesc_g = make_idesc_bf16(128, 64, 0, 1);         // acc: A = G K-major, B = other MN-major
            const uint32_t gs_addr = smem_u32(gs);
            uint32_t n = 0;
            // S is double-buffered (TMEM columns 0-127 / 128-255): the score GEMM of tile st+1 overlaps the epilogue of st
            auto phase1 = [&](int it) {                                     // it: index inside this CTA's tile range
                const uint32_t buf = it & 1;
                mbar_wait(&bars->s_empty[buf], ((it >> 1) & 1) ^ 1);         // epilogue finished reading this S buffer
                tc_fence_after();
                for (int q = 0; q < g.EC; ++q, ++n) {
                    const int stage = n % NU_BSTAGES;
                    mbar_wait(&bars->full[stage], (n / NU_BSTAGES) & 1);
                    tc_fence_after();
                    const uint32_t a0 = smem_u32(ring + stage * 2 * NU_TILE), b0 = a0 + NU_TILE;
#pragma unroll
                    for (int cb = 0; cb < g.passes; ++cb) {
                        const uint32_t a_addr = a0 + (cb == 2 ? 128 * 128 : 0);
                        const uint32_t b_addr = b0 + (cb == 1 ? 128 * 128 : 0);
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            mma_bf16(tmem_base + buf * 128, make_smem_desc(a_addr + k * 32, 16, 1024),
                                     make_smem_desc(b_addr + k * 32, 16, 1024), idesc_s, (uint32_t)(q | cb | k));
                    }
                    tc_commit(&bars->empty[stage]);
                }
                tc_commit(&bars->s_full[buf]);
            };
            if (n_it > 0) phase1(0);
            for (int it = 0; it < n_it; ++it) {
                if (it + 1 < n_it) phase1(it + 1);
                mbar_wait(&bars->g_full, it & 1);                            // G tile written (and fenced) by the epilogue warps
                tc_fence_after();
                for (int a = 0; a < e_chunks; ++a, ++n) {
                    const int stage = n % NU_BSTAGES;
                    mbar_wait(&bars->full[stage], (n / NU_BSTAGES) & 1);
                    tc_fence_after();
                    const uint32_t b0 = smem_u32(ring + stage * 2 * NU_TILE + NU_TILE);
                    const uint32_t d_tmem = tmem_base + 256 + (uint32_t)a * 64;
#pragma unroll
                    for (int cb = 0; cb < g.passes; ++cb) {                         // (G hi, X hi) (G hi, X lo) (G lo, X hi)
                        const uint32_t ga = gs_addr + (cb == 2 ? NU_TILE : 0);           // lo plane of G
                        const uint32_t ba = b0 + (cb == 1 ? 128 * 128 : 0);
#pragma unroll
                        for (int ks = 0; ks < 8; ++ks) {                     // K = 128 other rows
                            const uint64_t ad = make_smem_desc(ga + (ks >> 2) * (128 * 128) + (ks & 3) * 32, 16, 1024);
                            const uint64_t bd = make_smem_desc(ba + ks * (16 * 128), 64 * 128, 1024);
                            mma_bf16(d_tmem, ad, bd, idesc_g, (uint32_t)(it | cb | ks));
                        }
                    }
                    tc_commit(&bars->empty[stage]);
                }
                tc_commit(&bars->g_empty);
            }
            tc_commit(&bars->acc_full);
        }
    } else if (warp >= 4) {
        const int ew = warp & 3;
        const int rl = ew * 32 + lane;                                       // owner row inside the tile
        const int orow = ot * 128 + rl;
        const bool own_ok = orow < g.Bp;
        const float w_ce = __ldg(p.grad_loss) / ((float)g.nprob * (float)g.Bp);
        const float lse_own = (p.owner_is_target && own_ok) ? __ldg(p.lse + (size_t)prob * g.Bp + orow) : 0.f;
        const uint32_t lane_base = tmem_base + ((uint32_t)(ew * 32) << 16);
        uint8_t* grow = gs + (rl >> 3) * 1024 + (rl & 7) * 128;              // this owner row inside a K atom
        for (int it = 0; it < n_it; ++it) {
            const int st = st0 + it;
            if (!p.owner_is_target) {                                        // lse of the 128 target columns of this tile
                const int c = st * 128 + rl;
                bars->lse_s[it & 1][rl] = c < g.Bp ? __ldg(p.lse + (size_t)prob * g.Bp + c) : 0.f;
            }
            mbar_wait(&bars->s_full[it & 1], (it >> 1) & 1);
            tc_fence_after();
            mbar_wait(&bars->g_empty, (it & 1) ^ 1);                         // previous G tile consumed by the MMAs
            asm volatile("bar.sync 1, 128;" ::: "memory");                  // lse_s visible to all epilogue threads
            const int n_valid = min(128, g.Bp - st * 128);                   // rows of the other operand inside the problem
            const float* lrow = bars->lse_s[it & 1];
            for (int n0 = 0; n0 < 128; n0 += 32) {
                uint32_t raw[32];
                tmem_ld32(lane_base + (uint32_t)((it & 1) * 128 + n0), raw);
                tmem_ld_wait();
                float gv[32];
                float sg[32];                                                 // d softplus / du (softplus scores only)
                if (g.lambda == 0.f) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float u = __uint_as_float(raw[j]);
                        float sc = u;
                        if (KIND == CPC_SCORE_SOFTPLUS) nu_softplus_sigmoid(u, sc, sg[j]);
                        const float l = p.owner_is_target ? lse_own : lrow[n0 + j];
                        gv[j] = w_ce * __expf(sc - l);
                    }
                } else {
                    // all-steps regulariser lambda * mean_{d,t,k'} ((1/K) sum_k S[d,k,t,k'])^2 (:141):
                    // dL/dS[d,k,t,k'] += 2 lambda / (B^2 K^3) * sum_k S[d,k,t,k'].  Prediction rows are ordered (d, k), so the
                    // K-sum runs over K consecutive columns (owner = targets: inside this thread's registers) or over K
                    // consecutive lanes (owner = predictions: warp shuffles); K is a power of two <= 32 (host side).
                    const float w_reg = __ldg(p.grad_loss) * 2.f * g.lambda / ((float)g.B * (float)g.B * (float)g.K * (float)g.K * (float)g.K);
                    float sc[32];
#pragma unroll
                    for (int j = 0; j < 32; ++j) {
                        const float u = __uint_as_float(raw[j]);
                        sc[j] = u;
                        if (KIND == CPC_SCORE_SOFTPLUS) nu_softplus_sigmoid(u, sc[j], sg[j]);
                        const float l = p.owner_is_target ? lse_own : lrow[n0 + j];
                        gv[j] = w_ce * __expf(sc[j] - l);
                    }
                    if (p.owner_is_target) {
#pragma unroll
                        for (int lg = 0; lg < 5; ++lg) {                      // butterfly over the K-aligned column group
                            constexpr int kOne = 1;
                            const int o = kOne << lg;                         // compile-time after unrolling: register indexing
                            if (o < g.K) {
                                float nx[32];
#pragma unroll
                                for (int j = 0; j < 32; ++j) nx[j] = sc[j] + sc[j ^ o];
#pragma unroll
                                for (int j = 0; j < 32; ++j) sc[j] = nx[j];
                            }
                        }
                    } else {
                        for (int o = 1; o < g.K; o <<= 1) {
#pragma unroll
                            for (int j = 0; j < 32; ++j) sc[j] += __shfl_xor_sync(0xffffffffu, sc[j], o);
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 32; ++j) gv[j] = fmaf(w_reg, sc[j], gv[j]);
                }
                if (st == ot && n0 == (rl & 96)) {                           // - w on the diagonal element
#pragma unroll
                    for (int j = 0; j < 32; ++j) if (j == (rl & 31)) gv[j] -= w_ce;
                }
                if (KIND == CPC_SCORE_SOFTPLUS) {
#pragma unroll
                    for (int j = 0; j < 32; ++j) gv[j] *= sg[j];
                }
                if (!own_ok || n0 + 32 > n_valid) {                          // rows outside the problem contribute nothing
#pragma unroll
                    for (int j = 0; j < 32; ++j) if (!own_ok || n0 + j >= n_valid) gv[j] = 0.f;
                }
#pragma unroll
                for (int j8 = 0; j8 < 4; ++j8) {
                    __align__(16) __nv_bfloat16 hi[8];
                    __align__(16) __nv_bfloat16 lo[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        hi[j] = __float2bfloat16_rn(gv[j8 * 8 + j]);
                        lo[j] = __float2bfloat16_rn(gv[j8 * 8 + j] - __bfloat162float(hi[j]));
                    }
                    const int nchunk = n0 / 8 + j8;                          // 16-byte chunk index along K (0..15)
                    uint8_t* dst = grow + (nchunk >> 3) * (128 * 128) + (((nchunk & 7) ^ (rl & 7)) << 4);
                    *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(hi);
                    *reinterpret_cast<uint4*>(dst + NU_TILE) = *reinterpret_cast<const uint4*>(lo);
                }
            }
            tc_fence_before();
            fence_proxy_async();                                             // generic-proxy smem writes -> tensor core
            __syncwarp();
            if (lane == 0) { mbar_arrive(&bars->g_full); mbar_arrive(&bars->s_empty[it & 1]); }
        }
        // flush the accumulator: rows = owner rows, columns = E slice
        mbar_wait(&bars->acc_full, 0);
        tc_fence_after();
        for (int a = 0; a < e_chunks; ++a)
            for (int h = 0; h < 2; ++h) {
                uint32_t raw[32];
                tmem_ld32(lane_base + 256 + (uint32_t)(a * 64 + h * 32), raw);
                tmem_ld_wait();
                if (!own_ok) continue;
                const int e0 = (es * 4 + a) * 64 + h * 32;
                if (p.owner_is_target) {
                    // d_targets (B, E, K) contiguous: target row (t, k') -> ((t*E + e)*K + k')
                    const int t = g.all ? orow / g.K : orow, kk = g.all ? orow - t * g.K : prob;
                    float* o = p.out + ((size_t)t * g.E + e0) * g.K + kk;
                    if (p.n_split > 1) {                                     // partial result: the output was zeroed
#pragma unroll
                        for (int j = 0; j < 32; ++j) atomicAdd(o + (size_t)j * g.K, __uint_as_float(raw[j]));
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; ++j) o[(size_t)j * g.K] = __uint_as_float(raw[j]);
                    }
                } else {
                    // d_pred (B, K, E) contiguous: prediction row (d, k) -> (d*K + k)*E + e
                    const size_t r = g.all ? (size_t)orow : (size_t)orow * g.K + prob;
                    if (p.n_split > 1) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) atomicAdd(p.out + r * g.E + e0 + j, __uint_as_float(raw[j]));
                    } else {
                        float4* o = reinterpret_cast<float4*>(p.out + r * g.E + e0);
#pragma unroll
                        for (int j = 0; j < 8; ++j)
                            o[j] = make_float4(__uint_as_float(raw[4 * j]), __uint_as_float(raw[4 * j + 1]), __uint_as_float(raw[4 * j + 2]),
                                               __uint_as_float(raw[4 * j + 3]));
                    }
                }
            }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) { tc_fence_after(); tmem_dealloc(tmem_base, 512); }
}

// ---- host side ----------------------------------------------------------------------------------------------
// which: 0 forward, 1 backward
bool nce_umma_eligible(const cpc_infonce_params* p, int which) {
    // the kernels below compute dot products only (any other kind would run as linear), and a distance from them would
    // be |p|^2 + |z|^2 - 2 p.z, which cancels for the near pairs the difference kind is about
    if (p->score_kind == CPC_SCORE_DIFFERENCE) return false;
    if (p->enc % 64 != 0 || p->enc < 64 || p->enc > 4096) return false;
    const long bp = p->all_steps ? (long)p->batch * p->steps : p->batch;
    if (bp < 128 || bp > (1 << 24)) return false;                          // tiny problems are latency-bound either way
    // one CTA per 128 owner rows: a single all-steps problem needs >= 8 row tiles to beat
    // the CUDA-core kernel does (measured cross-over, tools/infonce_sweep.py); per-step mode has K problems
    if (p->all_steps && bp < 1024) return false;
    if (p->regularization != 0.f) {
        if (!p->all_steps || 128 % p->steps != 0) return false;            // whole K-groups inside a tile (K a power of two)
        if (which == 1 && p->steps > 32) return false;                     // backward sums K consecutive lanes with shuffles
    }
    return true;
}

static size_t nu_plane_bytes(const NuGeom& g) { return align_up((size_t)2 * g.nprob * g.Bp * g.E * 2, 1024); }

size_t nce_umma_workspace(const cpc_infonce_params* p, int which) {
    if (!nce_umma_eligible(p, which)) return 0;
    const NuGeom g = nu_geom(p);
    return 2 * nu_plane_bytes(g) + (which == 0 ? align_up((size_t)g.nprob * g.nT * 4 * sizeof(float), 256) : 0) + 2048;
}

static int nu_pack_both(const float* pred, const float* targets, const cpc_infonce_params* p, const NuGeom& g,
                        __nv_bfloat16* pp, __nv_bfloat16* zp, cudaStream_t s) {
    NuSrc sp{}, sz{};
    if (g.all) {                        // rows (d,k) / (t,k')
        sp = NuSrc{pred, 0, (long long)g.K * g.E, (long long)g.E, 1, g.K};
        sz = NuSrc{targets, 0, p->tgt_stride_b, p->tgt_stride_k, p->tgt_stride_e, g.K};
    } else {                            // problem k, rows d / t
        sp = NuSrc{pred, (long long)g.E, (long long)g.K * g.E, 0, 1, 1};
        sz = NuSrc{targets, p->tgt_stride_k, p->tgt_stride_b, 0, p->tgt_stride_e, 1};
    }
    const long groups = (long)g.nprob * g.Bp * (g.E / 8);
    int blocks = (int)((groups + 255) / 256);
    if (blocks > 148 * 16) blocks = 148 * 16;
    nu_pack_kernel<<<blocks, 256, 0, s>>>(sp, pp, g.nprob, g.Bp, g.E);
    nu_pack_kernel<<<blocks, 256, 0, s>>>(sz, zp, g.nprob, g.Bp, g.E);
    return cudaGetLastError() == cudaSuccess ? CPC_OK : CPC_ERR_CUDA;
}

static bool nu_tmap(CUtensorMap* t, const void* base, const NuGeom& g) {
    const uint64_t dims[4] = {(uint64_t)g.E, (uint64_t)g.Bp, (uint64_t)g.nprob, 2};
    const uint64_t strides[3] = {(uint64_t)g.E * 2, (uint64_t)g.Bp * g.E * 2, (uint64_t)g.nprob * g.Bp * g.E * 2};
    const uint32_t box[4] = {64, 128, 1, 2};
    return make_tmap_bf16(t, base, 4, dims, strides, box);
}

int nce_umma_fwd(const float* pred, const float* targets, float* out, float* lse, const cpc_infonce_params* p,
                 void* workspace, size_t workspace_bytes, cudaStream_t s) {
    if (!nce_umma_eligible(p, 0)) return CPC_ERR_UNSUPPORTED;
    if (!workspace || workspace_bytes < nce_umma_workspace(p, 0)) return CPC_ERR_WORKSPACE;
    const NuGeom g = nu_geom(p);
    uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 1023) & ~(uintptr_t)1023);
    __nv_bfloat16* pp = reinterpret_cast<__nv_bfloat16*>(ws);
    __nv_bfloat16* zp = reinterpret_cast<__nv_bfloat16*>(ws + nu_plane_bytes(g));
    float* partials = reinterpret_cast<float*>(ws + 2 * nu_plane_bytes(g));
    int st = nu_pack_both(pred, targets, p, g, pp, zp, s);
    if (st != CPC_OK) return st;
    CUtensorMap tz, tp;
    if (!nu_tmap(&tz, zp, g) || !nu_tmap(&tp, pp, g)) return CPC_ERR_CUDA;
    const int smem_bytes = NU_FSTAGES * 2 * NU_TILE + (int)sizeof(NuFwdBarriers) + 1024;
    const int ncta = g.nprob * g.nT;
    auto launch = [&](auto kern) -> int {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes) != cudaSuccess) return CPC_ERR_CUDA;
        kern<<<ncta, NU_THREADS, smem_bytes, s>>>(tz, tp, g, lse, partials);
        return CPC_OK;
    };
    const bool soft = g.kind == CPC_SCORE_SOFTPLUS, reg = g.lambda != 0.f;
    st = soft ? (reg ? launch(nce_umma_fwd_kernel<CPC_SCORE_SOFTPLUS, true>) : launch(nce_umma_fwd_kernel<CPC_SCORE_SOFTPLUS, false>))
              : (reg ? launch(nce_umma_fwd_kernel<CPC_SCORE_LINEAR, true>) : launch(nce_umma_fwd_kernel<CPC_SCORE_LINEAR, false>));
    if (st != CPC_OK) return st;
    CPC_LAUNCH_CHECK();
    nce_umma_final_kernel<<<1, 256, 0, s>>>(partials, ncta, g, out);
    CPC_LAUNCH_CHECK();
    count_launch(4);
    return CPC_OK;
}

int nce_umma_bwd(const float* pred, const float* targets, const float* lse, const float* grad_loss, float* d_pred,
                 float* d_targets, const cpc_infonce_params* p, void* workspace, size_t workspace_bytes, cudaStream_t s) {
    if (!nce_umma_eligible(p, 1)) return CPC_ERR_UNSUPPORTED;
    if (!workspace || workspace_bytes < nce_umma_workspace(p, 1)) return CPC_ERR_WORKSPACE;
    const NuGeom g = nu_geom(p);
    uint8_t* ws = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(workspace) + 1023) & ~(uintptr_t)1023);
    __nv_bfloat16* pp = reinterpret_cast<__nv_bfloat16*>(ws);
    __nv_bfloat16* zp = reinterpret_cast<__nv_bfloat16*>(ws + nu_plane_bytes(g));
    int st = nu_pack_both(pred, targets, p, g, pp, zp, s);
    if (st != CPC_OK) return st;
    CUtensorMap tz, tp;
    if (!nu_tmap(&tz, zp, g) || !nu_tmap(&tp, pp, g)) return CPC_ERR_CUDA;
    const int smem_bytes = NU_BSTAGES * 2 * NU_TILE + 2 * NU_TILE + (int)sizeof(NuBwdBarriers) + 1024;
    NuBwd k{};
    k.g = g; k.lse = lse; k.grad_loss = grad_loss;
    k.n_slices = ceil_div(g.EC, 4);
    // small problems (the native e24 size is 16 CTAs): split the loop over the other operand's tiles across CTAs
    k.n_split = 148 / (g.nprob * g.nT * k.n_slices);
    if (k.n_split > g.nT) k.n_split = g.nT;
    if (k.n_split < 1) k.n_split = 1;
    const int grid = g.nprob * g.nT * k.n_split * k.n_slices;
    if (k.n_split > 1) {
        const size_t n_out = (size_t)g.B * g.K * g.E;
        if (cudaMemsetAsync(d_targets, 0, n_out * sizeof(float), s) != cudaSuccess ||
            cudaMemsetAsync(d_pred, 0, n_out * sizeof(float), s) != cudaSuccess) return CPC_ERR_CUDA;
    }
    auto launch = [&](auto kern) -> int {
        if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes) != cudaSuccess) return CPC_ERR_CUDA;
        k.owner_is_target = 1; k.out = d_targets;
        kern<<<grid, NU_THREADS, smem_bytes, s>>>(tz, tp, k);
        k.owner_is_target = 0; k.out = d_pred;
        kern<<<grid, NU_THREADS, smem_bytes, s>>>(tp, tz, k);
        return CPC_OK;
    };
    st = g.kind == CPC_SCORE_SOFTPLUS ? launch(nce_umma_bwd_kernel<CPC_SCORE_SOFTPLUS>) : launch(nce_umma_bwd_kernel<CPC_SCORE_LINEAR>);
    if (st != CPC_OK) return st;
    CPC_LAUNCH_CHECK();
    count_launch(4);
    return CPC_OK;
}

}  // namespace cpc
