// InfoNCE scoring + loss, forward and backward, with the score tensor kept on chip.
// Replaces score_function + loss block of ContrastiveEstimationTrainer.train
// (contrastive_estimation_training.py:12-22, 106-122, 141, 166) and its autograd.
//
// Notation (SURVEY.md Appendix B): P = pred (B,K,E), Z = targets (B,E,K) strided view.
//   all-steps mode : one problem, rows r=(d,k), columns c=(t,k');  S[r,c] = phi(P[r,:] . Z[t,:,k'])
//   per-step mode  : K problems,  rows d,     columns t;           S_k[d,t] = phi(P[d,k,:] . Z[t,:,k])
// phi is the identity (linear) or softplus; the difference kind scores S = 1 / D with D = |P[r,:] - Z[c,:]|^2, summed
// as squared differences in fp32 (tile_dist), never as |p|^2 + |z|^2 - 2 p.z.
// loss = mean_c (lse_r S[:,c] - S[c,c]) + lambda * mean((mean_k S)^2).  The reference's per-step
// ".view" scramble is a bijection under the mean, so the training loss equals this clean form.
//
// Forward : score tiles (64x64) -> per-(row tile, column) partial (max, sum-exp), diagonal, max,
//           sum, regulariser partials -> combine -> 4 scalars + lse per column.
// Backward: recompute score tiles from P, Z and the saved lse, form G = dL/du on chip, then
//           dP += G Zc and dZc += G^T P with fp32 atomics.  No B*K x B*K tensor ever reaches HBM.
#include "common.cuh"

#include <cstdlib>

namespace cpc {

// infonce_umma.cu: tcgen05 path (>= 128 candidates per softmax, E % 64 == 0)
bool nce_umma_eligible(const cpc_infonce_params* p, int which);
size_t nce_umma_workspace(const cpc_infonce_params* p, int which);
int nce_umma_fwd(const float* pred, const float* targets, float* out, float* lse, const cpc_infonce_params* p,
                 void* workspace, size_t workspace_bytes, cudaStream_t s);
int nce_umma_bwd(const float* pred, const float* targets, const float* lse, const float* grad_loss, float* d_pred,
                 float* d_targets, const cpc_infonce_params* p, void* workspace, size_t workspace_bytes, cudaStream_t s);

// flags & CPC_INFONCE_FLAG_NO_TENSOR keeps everything on the CUDA-core kernels (A/B switch for tests)
static bool nce_tensor_path(const cpc_infonce_params* p, int which) {
    if (p->flags & CPC_INFONCE_FLAG_NO_TENSOR) return false;
    return nce_umma_eligible(p, which);
}

struct NceGeom {
    int B, K, E, all, kind;
    int R, C, nprob, tmr, ncols, nrowtiles;
    long long sb, se, sk;
    float lambda;
};

static int nce_validate(const cpc_infonce_params* p) {
    if (!p) return CPC_ERR_NULL;
    if (p->batch <= 0 || p->steps <= 0 || p->enc <= 0) return CPC_ERR_BAD_SHAPE;
    if (p->steps > TILE) return CPC_ERR_UNSUPPORTED;
    if ((int64_t)p->batch * p->steps > (1 << 30)) return CPC_ERR_BAD_SHAPE;
    if (p->score_kind != CPC_SCORE_LINEAR && p->score_kind != CPC_SCORE_SOFTPLUS && p->score_kind != CPC_SCORE_DIFFERENCE)
        return CPC_ERR_BAD_SHAPE;
    return CPC_OK;
}

static NceGeom nce_geom(const cpc_infonce_params* p) {
    NceGeom g;
    g.B = p->batch; g.K = p->steps; g.E = p->enc; g.all = p->all_steps ? 1 : 0; g.kind = p->score_kind;
    g.sb = p->tgt_stride_b; g.se = p->tgt_stride_e; g.sk = p->tgt_stride_k;
    g.lambda = p->regularization;
    if (g.all) { g.R = g.C = g.B * g.K; g.nprob = 1; g.tmr = (TILE / g.K) * g.K; }
    else       { g.R = g.C = g.B;       g.nprob = g.K; g.tmr = TILE; }
    g.ncols = g.B * g.K;
    g.nrowtiles = ceil_div(g.R, g.tmr);
    return g;
}

// ---- loaders ------------------------------------------------------------------------------------
struct PRows {        // rows: prediction index of the problem; k: e
    static constexpr bool kFast = true;
    const float* p; int R, E; long long base, stride;
    __device__ __forceinline__ float load(int r, int e) const {
        if (r >= R || e >= E) return 0.f;
        return __ldg(p + base + (long long)r * stride + e);
    }
};
struct ZRows {        // rows: target column of the problem; k: e
    static constexpr bool kFast = false;
    const float* z; int C, E, K, all, kfix; long long sb, se, sk;
    __device__ __forceinline__ long long col_base(int c) const {
        if (all) { const int t = c / K; return (long long)t * sb + (long long)(c - t * K) * sk; }
        return (long long)c * sb + (long long)kfix * sk;
    }
    __device__ __forceinline__ float load(int c, int e) const {
        if (c >= C || e >= E) return 0.f;
        return __ldg(z + col_base(c) + (long long)e * se);
    }
};
struct ZByE {         // rows: e; k: local column index (global column = c0 + k)
    static constexpr bool kFast = true;
    ZRows zr; int c0;
    __device__ __forceinline__ float load(int e, int k) const { return zr.load(c0 + k, e); }
};
struct PByE {         // rows: e; k: local row index (global row = r0 + k)
    static constexpr bool kFast = false;
    PRows pr; int r0;
    __device__ __forceinline__ float load(int e, int k) const { return pr.load(r0 + k, e); }
};
struct SmemTile {     // rows/k index a 64x64 tile in shared memory (optionally transposed)
    static constexpr bool kFast = true;
    const float (*g)[TILE + 1]; int transpose;
    __device__ __forceinline__ float load(int r, int k) const { return transpose ? g[k][r] : g[r][k]; }
};

__device__ __forceinline__ float softplus_f(float u) {   // torch F.softplus(beta=1, threshold=20)
    return u > 20.f ? u : log1pf(expf(u));
}
__device__ __forceinline__ float sigmoid_f(float u) { return 1.f / (1.f + expf(-u)); }

// The kernels below are instantiated twice: kDiff = false for the dot-product kinds (linear, softplus: g.kind picks
// phi at run time), kDiff = true for the difference kind, so that neither pays registers for the other's code.
// One problem's 64x64 tile of score arguments: the dot product u, or the squared distance D.
template <bool kDiff, class LA, class LB>
__device__ __forceinline__ void score_tile(const NceGeom& g, const LA& la, const LB& lb, int row0, int col0,
                                           float (&acc)[4][4], TileSmem& sm) {
    if (kDiff) tile_dist(la, lb, row0, col0, 0, g.E, acc, sm);
    else tile_gemm(la, lb, row0, col0, 0, g.E, acc, sm);
}
// Score from the tile value.  D = 0 gives S = +inf, as the reference's 1 / sum(diff ** 2) does: no epsilon.  The loss
// is then NaN (expf(inf - inf) in the column statistics); the reference's is NaN when the coinciding target is the
// prediction's own and +inf when it is another candidate's (torch.logsumexp keeps the +inf).
template <bool kDiff>
__device__ __forceinline__ float score_of(int kind, float a) {
    // hardware reciprocal: the IEEE division's slow-path call made the backward spill; 1/0 = +inf.  Within 2 ulp of
    // 1/D for D in [2^-126, 2^126]; outside (a prediction within ~1e-19 of a target, or |p - z| > 1e19) it flushes to
    // +inf / 0 where IEEE 1/D would still be finite / denormal.
    if (kDiff) return __fdividef(1.f, a);
    return kind == CPC_SCORE_SOFTPLUS ? softplus_f(a) : a;
}

__device__ __forceinline__ PRows make_p(const float* p, const NceGeom& g, int prob) {
    return g.all ? PRows{p, g.R, g.E, 0, g.E} : PRows{p, g.R, g.E, (long long)prob * g.E, (long long)g.K * g.E};
}
__device__ __forceinline__ ZRows make_z(const float* z, const NceGeom& g, int prob) {
    return ZRows{z, g.C, g.E, g.K, g.all, prob, g.sb, g.se, g.sk};
}

__device__ __forceinline__ float half_warp_max(float v) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float half_warp_sum(float v) {
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// block reduce over 256 threads; result valid in thread 0
__device__ __forceinline__ float block_sum(float v, float* red) {
    v = warp_sum(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float r = 0.f;
    if (threadIdx.x < 32) { r = threadIdx.x < 8 ? red[threadIdx.x] : 0.f; r = warp_sum(r); }
    return r;
}
__device__ __forceinline__ float block_max(float v, float* red) {
    v = warp_max(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float r = -INFINITY;
    if (threadIdx.x < 32) { r = threadIdx.x < 8 ? red[threadIdx.x] : -INFINITY; r = warp_max(r); }
    return r;
}

// ---- forward ------------------------------------------------------------------------------------
// grid (col tiles, row tiles, problems).  part_m/part_s: [rowtile][ncols]; diag: [ncols]; cta: [ncta][3] = max,sum,reg.
// Per-step mode: one CTA per (tile, prediction step) -- the K problems used to run one after the other inside a CTA,
// which left the raw-wave configuration (B = 8 ... 64, K = 12: ONE tile) on a single SM for 0.6 - 0.9 ms.  Its
// regulariser couples the problems (mean over k of S_k[d, t]): the CTAs add their scores into rsum (R x C, zeroed by the
// caller) and nce_final_kernel squares the means.
template <bool kDiff>
__global__ void __launch_bounds__(TILE_THREADS) nce_fwd_kernel(const float* __restrict__ P, const float* __restrict__ Z,
                                                              NceGeom g, float* __restrict__ part_m,
                                                              float* __restrict__ part_s, float* __restrict__ diag,
                                                              float* __restrict__ cta, float* __restrict__ rowp_m,
                                                              int* __restrict__ rowp_i, float* __restrict__ rsum) {
    __shared__ TileSmem sm;
    __shared__ float Ss[TILE][TILE + 1];
    __shared__ float red[8];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int col0 = blockIdx.x * TILE, row0 = blockIdx.y * g.tmr;
    float tmax = -INFINITY, tsum = 0.f, reg = 0.f;
    const float inv_k = 1.f / (float)g.K;
    const bool reg_steps = !g.all && g.lambda != 0.f;            // per-step regulariser: through rsum
    {
        const int prob = blockIdx.z;
        float acc[4][4] = {};
        score_tile<kDiff>(g, make_p(P, g, prob), make_z(Z, g, prob), row0, col0, acc, sm);
        float s[4][4];
        bool ok[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int lr = tx * 4 + i, r = row0 + lr, c = col0 + ty * 4 + j;
                ok[i][j] = lr < g.tmr && r < g.R && c < g.C;
                const float v = score_of<kDiff>(g.kind, acc[i][j]);
                s[i][j] = ok[i][j] ? v : -INFINITY;
                if (ok[i][j]) {
                    tmax = fmaxf(tmax, v);
                    tsum += v;
                    if (r == c) diag[prob * g.C + c] = v;
                    if (reg_steps) atomicAdd(rsum + (size_t)r * g.C + c, v);
                }
            }
        // column statistics over this tile's rows
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float m = fmaxf(fmaxf(s[0][j], s[1][j]), fmaxf(s[2][j], s[3][j]));
            m = half_warp_max(m);
            float e = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i) e += ok[i][j] ? expf(s[i][j] - m) : 0.f;
            e = half_warp_sum(e);
            const int c = col0 + ty * 4 + j;
            if (tx == 0 && c < g.C) {
                const size_t o = (size_t)blockIdx.y * g.ncols + (size_t)prob * g.C + c;
                part_m[o] = m;
                part_s[o] = e;
            }
        }
        if (rowp_m != nullptr) {
            // validation accuracy: per row, the best column of this column tile (first maximum wins)
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) Ss[tx * 4 + i][ty * 4 + j] = s[i][j];      // -inf outside the problem
            __syncthreads();
            if (threadIdx.x < TILE) {
                const int lr = threadIdx.x, r = row0 + lr;
                if (lr < g.tmr && r < g.R) {
                    float best = -INFINITY;
                    int arg = 0;
                    for (int cc = 0; cc < TILE; ++cc) {
                        const float v = Ss[lr][cc];
                        if (v > best) { best = v; arg = col0 + cc; }
                    }
                    const size_t o = ((size_t)blockIdx.x * g.nprob + prob) * g.R + r;
                    rowp_m[o] = best;
                    rowp_i[o] = arg;
                }
            }
            __syncthreads();
        }
        if (g.all && g.lambda != 0.f) {
            // regulariser: rows of one item d are K consecutive rows, whole groups live in this tile
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) Ss[tx * 4 + i][ty * 4 + j] = ok[i][j] ? s[i][j] : 0.f;
            __syncthreads();
            const int groups = g.tmr / g.K;
            for (int idx = threadIdx.x; idx < groups * TILE; idx += TILE_THREADS) {
                const int grp = idx / TILE, cc = idx - grp * TILE;
                float a = 0.f;
                for (int k = 0; k < g.K; ++k) a += Ss[grp * g.K + k][cc];
                a *= inv_k;
                reg += a * a;
            }
            __syncthreads();
        }
    }
    const int id = (blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    const float bm = block_max(tmax, red);
    const float bs = block_sum(tsum, red);
    const float br = block_sum(reg, red);
    if (threadIdx.x == 0) { cta[id * 3 + 0] = bm; cta[id * 3 + 1] = bs; cta[id * 3 + 2] = br; }
}

// one thread per column: combine row-tile partials -> lse; block partial of (lse - diag)
__global__ void __launch_bounds__(256) nce_combine_kernel(const float* __restrict__ part_m, const float* __restrict__ part_s,
                                                         const float* __restrict__ diag, float* __restrict__ lse,
                                                         float* __restrict__ blk, int ncols, int nrowtiles) {
    __shared__ float red[8];
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    float term = 0.f;
    if (c < ncols) {
        float m = -INFINITY;
        for (int t = 0; t < nrowtiles; ++t) m = fmaxf(m, part_m[(size_t)t * ncols + c]);
        float s = 0.f;
        for (int t = 0; t < nrowtiles; ++t) s += part_s[(size_t)t * ncols + c] * expf(part_m[(size_t)t * ncols + c] - m);
        const float l = m + logf(s);
        lse[c] = l;
        term = l - diag[c];
    }
    const float b = block_sum(term, red);
    if (threadIdx.x == 0) blk[blockIdx.x] = b;
}

__global__ void __launch_bounds__(256) nce_final_kernel(const float* __restrict__ blk, int nblk, const float* __restrict__ cta,
                                                       int ncta, NceGeom g, float* __restrict__ out,
                                                       const float* __restrict__ rsum) {
    __shared__ float red[8];
    float a = 0.f, mx = -INFINITY, sm = 0.f, rg = 0.f;
    if (rsum != nullptr) {                                        // per-step regulariser: sum over (d, t) of (mean_k S)^2
        const float inv_k = 1.f / (float)g.K;
        for (int i = threadIdx.x; i < g.R * g.C; i += blockDim.x) { const float m = rsum[i] * inv_k; rg += m * m; }
    }
    for (int i = threadIdx.x; i < nblk; i += blockDim.x) a += blk[i];
    for (int i = threadIdx.x; i < ncta; i += blockDim.x) {
        mx = fmaxf(mx, cta[i * 3 + 0]);
        sm += cta[i * 3 + 1];
        rg += cta[i * 3 + 2];
    }
    a = block_sum(a, red);
    mx = block_max(mx, red);
    sm = block_sum(sm, red);
    rg = block_sum(rg, red);
    if (threadIdx.x == 0) {
        const float loss0 = a / (float)g.ncols;
        const double nscores = g.all ? (double)g.R * g.C : (double)g.K * g.B * g.B;
        const double nreg = g.all ? (double)g.B * g.C : (double)g.B * g.B;
        out[0] = loss0 + g.lambda * (float)(rg / nreg);
        out[1] = mx;
        out[2] = loss0;
        out[3] = (float)(sm / nscores);
    }
}

// Validation metrics (contrastive_estimation_training.py:224-247), one block.
//   metrics[0..K)   per-step losses  -mean_b(valid[b, c] - noise[b, c]); in per-step mode noise is the reference's
//                   re-viewed (scrambled) array: noise[b, c] = lse[flat = b*K + c], flat = k*B + t  (Appendix B)
//   metrics[K..2K)  per-step accuracy = #(arg-max over targets hits the own target) / n, n = B*K (all-steps) or B
//   metrics[2K]     mean score
__global__ void __launch_bounds__(256) nce_validate_final_kernel(const float* __restrict__ lse, const float* __restrict__ diag,
                                                                const float* __restrict__ rowp_m,
                                                                const int* __restrict__ rowp_i, int ncoltiles,
                                                                const float* __restrict__ out4, NceGeom g,
                                                                float* __restrict__ metrics) {
    __shared__ float acc_loss[TILE], acc_hit[TILE];
    for (int k = threadIdx.x; k < g.K; k += blockDim.x) { acc_loss[k] = 0.f; acc_hit[k] = 0.f; }
    __syncthreads();
    for (int f = threadIdx.x; f < g.ncols; f += blockDim.x) {
        int kk;
        float term;
        if (g.all) { kk = f % g.K; term = lse[f] - diag[f]; }                     // f = t*K + k'
        else { const int b = f / g.K; kk = f - b * g.K; term = lse[f] - diag[kk * g.B + b]; }
        atomicAdd(&acc_loss[kk], term);
    }
    const int nrows = g.nprob * g.R;
    for (int idx = threadIdx.x; idx < nrows; idx += blockDim.x) {
        const int prob = idx / g.R, r = idx - prob * g.R;
        float best = -INFINITY;
        int arg = -1;
        for (int t = 0; t < ncoltiles; ++t) {
            const size_t o = ((size_t)t * g.nprob + prob) * g.R + r;
            const float v = rowp_m[o];
            if (v > best) { best = v; arg = rowp_i[o]; }
        }
        if (arg == r) atomicAdd(&acc_hit[g.all ? r % g.K : prob], 1.f);
    }
    __syncthreads();
    const float n = g.all ? (float)g.B * (float)g.K : (float)g.B;
    for (int k = threadIdx.x; k < g.K; k += blockDim.x) {
        metrics[k] = acc_loss[k] / (float)g.B;
        metrics[g.K + k] = acc_hit[k] / n;
    }
    if (threadIdx.x == 0) metrics[2 * g.K] = out4[3];
}

// ---- backward -----------------------------------------------------------------------------------
// Per-step regulariser, pass 1: rsum[d, t] += S_k[d, t] for every step k (grid (col tiles, row tiles, K); rsum zeroed).
template <bool kDiff>
__global__ void __launch_bounds__(TILE_THREADS) nce_rsum_kernel(const float* __restrict__ P, const float* __restrict__ Z,
                                                               NceGeom g, float* __restrict__ rsum) {
    __shared__ TileSmem sm;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int col0 = blockIdx.x * TILE, row0 = blockIdx.y * g.tmr;
    const int prob = blockIdx.z;
    float acc[4][4] = {};
    score_tile<kDiff>(g, make_p(P, g, prob), make_z(Z, g, prob), row0, col0, acc, sm);
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int lr = tx * 4 + i, r = row0 + lr, c = col0 + ty * 4 + j;
            if (lr < g.tmr && r < g.R && c < g.C)
                atomicAdd(rsum + (size_t)r * g.C + c, score_of<kDiff>(g.kind, acc[i][j]));
        }
}

// grid (col tiles, row tiles, problems x esplit): a CTA recomputes the score tile of ONE problem and produces the
// gradient columns e = (es + n * esplit) * 64 ... of it (small problems -- one or a few tiles -- are spread over the SMs by
// the problem and by the slice of E; they used to run their K problems and 8 slices one after the other on one SM).
// Difference kind: with H = G * S^2 (dS/dD = -S^2) the tile holds Gs = 2H, and
//   dP[r,:] = -2 sum_c H[r,c] (P[r,:] - Z[c,:]) = (Gs Zc)[r,:] - h_r P[r,:],   h_r  = sum_c Gs[r,c]
//   dZc[c,:] = 2 sum_r H[r,c] (P[r,:] - Z[c,:]) = (Gs^T P)[c,:] - h'_c Z[c,:],  h'_c = sum_r Gs[r,c]
// so the two tile products stay as they are and each CTA adds its tile's share of the rank-1 terms.
template <bool kDiff>
__global__ void __launch_bounds__(TILE_THREADS) nce_bwd_kernel(const float* __restrict__ P, const float* __restrict__ Z,
                                                              const float* __restrict__ lse,
                                                              const float* __restrict__ grad_loss, NceGeom g,
                                                              float* __restrict__ dP, float* __restrict__ dZ,
                                                              const float* __restrict__ rsum, int esplit) {
    __shared__ TileSmem sm;
    __shared__ float Gs[TILE][TILE + 1];
    __shared__ float Sbar[TILE][TILE];         // all-steps regulariser: (group, column); groups = tmr/K <= 64
    __shared__ float hrow[TILE], hcol[TILE];   // difference kind: row / column sums of Gs over this tile
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int col0 = blockIdx.x * TILE, row0 = blockIdx.y * g.tmr;
    const float gl = __ldg(grad_loss);
    const float inv_k = 1.f / (float)g.K;
    const float w_ce = gl / (float)g.ncols;
    const float w_reg = g.all ? gl * g.lambda * 2.f * inv_k / ((float)g.B * (float)g.C)
                              : gl * g.lambda * 2.f * inv_k / ((float)g.B * (float)g.B);
    float sbar[4][4] = {};
    if (!g.all && g.lambda != 0.f) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int lr = tx * 4 + i, r = row0 + lr, c = col0 + ty * 4 + j;
                if (lr < g.tmr && r < g.R && c < g.C) sbar[i][j] = __ldg(rsum + (size_t)r * g.C + c) * inv_k;
            }
    }
    const int prob = blockIdx.z / esplit, es = blockIdx.z - prob * esplit;
    {
        const PRows pr = make_p(P, g, prob);
        const ZRows zr = make_z(Z, g, prob);
        float acc[4][4] = {};
        score_tile<kDiff>(g, pr, zr, row0, col0, acc, sm);
        float s[4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) s[i][j] = score_of<kDiff>(g.kind, acc[i][j]);
        if (g.all && g.lambda != 0.f) {
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const int lr = tx * 4 + i;
                    const bool ok = lr < g.tmr && row0 + lr < g.R && col0 + ty * 4 + j < g.C;
                    Gs[lr][ty * 4 + j] = ok ? s[i][j] : 0.f;
                }
            __syncthreads();
            const int groups = g.tmr / g.K;
            for (int idx = threadIdx.x; idx < groups * TILE; idx += TILE_THREADS) {
                const int grp = idx / TILE, cc = idx - grp * TILE;
                float a = 0.f;
                for (int k = 0; k < g.K; ++k) a += Gs[grp * g.K + k][cc];
                Sbar[grp][cc] = a * inv_k;
            }
            __syncthreads();
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) sbar[i][j] = Sbar[(tx * 4 + i) / g.K < groups ? (tx * 4 + i) / g.K : 0][ty * 4 + j];
            __syncthreads();
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int lr = tx * 4 + i, r = row0 + lr, c = col0 + ty * 4 + j;
                const bool ok = lr < g.tmr && r < g.R && c < g.C;
                float gv = 0.f;
                if (ok) {
                    const float l = __ldg(lse + (size_t)prob * g.C + c);
                    gv = w_ce * (expf(s[i][j] - l) - (r == c ? 1.f : 0.f)) + w_reg * sbar[i][j];
                    if (kDiff) gv *= 2.f * s[i][j] * s[i][j];
                    else if (g.kind == CPC_SCORE_SOFTPLUS) gv *= sigmoid_f(acc[i][j]);
                }
                Gs[lr][ty * 4 + j] = gv;
            }
        __syncthreads();
        if (kDiff) {                                  // entries outside the problem are 0 in Gs
            if (threadIdx.x < TILE) {
                float a = 0.f;
                for (int cc = 0; cc < TILE; ++cc) a += Gs[threadIdx.x][cc];
                hrow[threadIdx.x] = a;
            } else if (threadIdx.x < 2 * TILE) {
                const int cc = threadIdx.x - TILE;
                float a = 0.f;
                for (int rr = 0; rr < TILE; ++rr) a += Gs[rr][cc];
                hcol[cc] = a;
            }
            __syncthreads();
        }
        for (int e0 = es * TILE; e0 < g.E; e0 += esplit * TILE) {
            {   // dP[r, e] += sum_c G[r,c] Zc[c,e]
                float a2[4][4] = {};
                tile_gemm(SmemTile{Gs, 0}, ZByE{zr, col0}, 0, e0, 0, TILE, a2, sm);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int lr = tx * 4 + i, r = row0 + lr;
                    if (lr >= g.tmr || r >= g.R) continue;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int e = e0 + ty * 4 + j;
                        if (e >= g.E) continue;
                        float v = a2[i][j];
                        if (kDiff) v -= hrow[lr] * pr.load(r, e);
                        atomicAdd(dP + pr.base + (long long)r * pr.stride + e, v);
                    }
                }
            }
            {   // dZc[c, e] += sum_r G[r,c] P[r,e]   -> d_targets (B,E,K) contiguous
                float a3[4][4] = {};
                tile_gemm(SmemTile{Gs, 1}, PByE{pr, row0}, 0, e0, 0, TILE, a3, sm);
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int c = col0 + tx * 4 + i;
                    if (c >= g.C) continue;
                    int t, kk;
                    if (g.all) { t = c / g.K; kk = c - t * g.K; } else { t = c; kk = prob; }
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const int e = e0 + ty * 4 + j;
                        if (e >= g.E) continue;
                        float v = a3[i][j];
                        if (kDiff) v -= hcol[tx * 4 + i] * zr.load(c, e);
                        atomicAdd(dZ + ((size_t)t * g.E + e) * g.K + kk, v);
                    }
                }
            }
        }
        __syncthreads();
    }
}

static decltype(&nce_fwd_kernel<false>) nce_fwd_launcher(const NceGeom& g) {
    return g.kind == CPC_SCORE_DIFFERENCE ? nce_fwd_kernel<true> : nce_fwd_kernel<false>;
}

struct NceWs {
    float *part_m, *part_s, *diag, *cta, *blk, *rsum;
    int ncta, nblk;
    size_t bytes;
};
// per-step mode with a regulariser: (R x C) sums over the steps
static size_t nce_rsum_floats(const NceGeom& g) { return (!g.all && g.lambda != 0.f) ? (size_t)g.R * g.C : 0; }
// slices of E per problem in the CUDA-core backward: enough CTAs for the 148 SMs, at most one 64-wide chunk each
static int nce_esplit(const NceGeom& g) {
    const int ctas = ceil_div(g.C, TILE) * g.nrowtiles * g.nprob, chunks = ceil_div(g.E, TILE);
    int e = 148 / ctas;
    if (e > chunks) e = chunks;
    return e < 1 ? 1 : e;
}
static NceWs nce_ws(const NceGeom& g, void* base) {
    NceWs w;
    const int coltiles = ceil_div(g.C, TILE);
    w.ncta = coltiles * g.nrowtiles * g.nprob;
    w.nblk = ceil_div(g.ncols, 256);
    size_t o = 0;
    char* b = reinterpret_cast<char*>(base);
    auto take = [&](size_t n) { float* r = reinterpret_cast<float*>(b + o); o += align_up(n * sizeof(float), 256); return r; };
    w.part_m = take((size_t)g.nrowtiles * g.ncols);
    w.part_s = take((size_t)g.nrowtiles * g.ncols);
    w.diag = take((size_t)g.ncols);
    w.cta = take((size_t)w.ncta * 3);
    w.blk = take((size_t)w.nblk);
    w.rsum = take(nce_rsum_floats(g));
    w.bytes = o;
    return w;
}

}  // namespace cpc

using namespace cpc;

extern "C" size_t cpc_infonce_workspace_bytes(const cpc_infonce_params* p, int which) {
    if (nce_validate(p) != CPC_OK) return 0;
    const NceGeom g = nce_geom(p);
    if (which == 1)
        return nce_umma_eligible(p, 1) ? nce_umma_workspace(p, 1) : align_up(sizeof(float) * nce_rsum_floats(g), 256);
    size_t fwd = nce_ws(g, nullptr).bytes;
    if (which == 0) {
        if (nce_umma_eligible(p, 0) && nce_umma_workspace(p, 0) > fwd) fwd = nce_umma_workspace(p, 0);
        return fwd;
    }
    // validate: forward scratch + lse + 4 scalars + per-(column tile, row) arg-max partials
    const size_t rows = (size_t)ceil_div(g.C, TILE) * g.nprob * g.R;
    return fwd + align_up(sizeof(float) * (size_t)g.ncols, 256) + 256 + 2 * align_up(sizeof(float) * rows, 256);
}

extern "C" int cpc_infonce_fwd(const float* pred, const float* targets, float* out, float* lse,
                               const cpc_infonce_params* p, void* workspace, size_t workspace_bytes, void* stream) {
    int st = nce_validate(p);
    if (st != CPC_OK) return st;
    if (!pred || !targets || !out || !lse) return CPC_ERR_NULL;
    NceGeom g = nce_geom(p);
    NceWs w = nce_ws(g, workspace);
    if (!workspace || workspace_bytes < cpc_infonce_workspace_bytes(p, 0)) return CPC_ERR_WORKSPACE;
    if ((st = check_device()) != CPC_OK) return st;
    cudaStream_t s = (cudaStream_t)stream;
    if (nce_tensor_path(p, 0)) return nce_umma_fwd(pred, targets, out, lse, p, workspace, workspace_bytes, s);
    const size_t n_rsum = nce_rsum_floats(g);
    if (n_rsum && cudaMemsetAsync(w.rsum, 0, sizeof(float) * n_rsum, s) != cudaSuccess) return CPC_ERR_CUDA;
    dim3 grid(ceil_div(g.C, TILE), g.nrowtiles, g.nprob);
    nce_fwd_launcher(g)<<<grid, TILE_THREADS, 0, s>>>(pred, targets, g, w.part_m, w.part_s, w.diag, w.cta, nullptr,
                                                      nullptr, n_rsum ? w.rsum : nullptr);
    CPC_LAUNCH_CHECK();
    nce_combine_kernel<<<w.nblk, 256, 0, s>>>(w.part_m, w.part_s, w.diag, lse, w.blk, g.ncols, g.nrowtiles);
    CPC_LAUNCH_CHECK();
    nce_final_kernel<<<1, 256, 0, s>>>(w.blk, w.nblk, w.cta, w.ncta, g, out, n_rsum ? w.rsum : nullptr);
    CPC_LAUNCH_CHECK();
    count_launch(3);
    return CPC_OK;
}

extern "C" int cpc_infonce_bwd(const float* pred, const float* targets, const float* lse, const float* grad_loss,
                               float* d_pred, float* d_targets, const cpc_infonce_params* p, void* workspace,
                               size_t workspace_bytes, void* stream) {
    int st = nce_validate(p);
    if (st != CPC_OK) return st;
    if (!pred || !targets || !lse || !grad_loss || !d_pred || !d_targets) return CPC_ERR_NULL;
    if ((st = check_device()) != CPC_OK) return st;
    NceGeom g = nce_geom(p);
    cudaStream_t s = (cudaStream_t)stream;
    if (nce_tensor_path(p, 1)) {
        if (!workspace || workspace_bytes < nce_umma_workspace(p, 1)) return CPC_ERR_WORKSPACE;
        return nce_umma_bwd(pred, targets, lse, grad_loss, d_pred, d_targets, p, workspace, workspace_bytes, s);
    }
    const size_t n = sizeof(float) * (size_t)g.B * g.K * g.E;
    if (cudaMemsetAsync(d_pred, 0, n, s) != cudaSuccess) return CPC_ERR_CUDA;
    if (cudaMemsetAsync(d_targets, 0, n, s) != cudaSuccess) return CPC_ERR_CUDA;
    float* rsum = nullptr;
    if (const size_t n_rsum = nce_rsum_floats(g)) {
        if (!workspace || workspace_bytes < sizeof(float) * n_rsum) return CPC_ERR_WORKSPACE;
        rsum = reinterpret_cast<float*>(workspace);
        if (cudaMemsetAsync(rsum, 0, sizeof(float) * n_rsum, s) != cudaSuccess) return CPC_ERR_CUDA;
        auto rsum_kernel = g.kind == CPC_SCORE_DIFFERENCE ? nce_rsum_kernel<true> : nce_rsum_kernel<false>;
        rsum_kernel<<<dim3(ceil_div(g.C, TILE), g.nrowtiles, g.nprob), TILE_THREADS, 0, s>>>(pred, targets, g, rsum);
        CPC_LAUNCH_CHECK();
        count_launch();
    }
    const int esplit = nce_esplit(g);
    dim3 grid(ceil_div(g.C, TILE), g.nrowtiles, g.nprob * esplit);
    auto bwd_kernel = g.kind == CPC_SCORE_DIFFERENCE ? nce_bwd_kernel<true> : nce_bwd_kernel<false>;
    bwd_kernel<<<grid, TILE_THREADS, 0, s>>>(pred, targets, lse, grad_loss, g, d_pred, d_targets, rsum, esplit);
    CPC_LAUNCH_CHECK();
    count_launch();
    return CPC_OK;
}

extern "C" int cpc_infonce_validate(const float* pred, const float* targets, float* metrics,
                                    const cpc_infonce_params* p, void* workspace, size_t workspace_bytes, void* stream) {
    int st = nce_validate(p);
    if (st != CPC_OK) return st;
    if (!pred || !targets || !metrics) return CPC_ERR_NULL;
    const size_t need = cpc_infonce_workspace_bytes(p, 2);
    if (!workspace || workspace_bytes < need) return CPC_ERR_WORKSPACE;
    if ((st = check_device()) != CPC_OK) return st;
    NceGeom g = nce_geom(p);
    g.lambda = 0.f;                                            // validation reports the un-regularised loss
    NceWs w = nce_ws(g, workspace);
    char* base = reinterpret_cast<char*>(workspace) + w.bytes;
    float* lse = reinterpret_cast<float*>(base);
    base += align_up(sizeof(float) * (size_t)g.ncols, 256);
    float* out4 = reinterpret_cast<float*>(base);
    base += 256;
    const int ncoltiles = ceil_div(g.C, TILE);
    const size_t rows = (size_t)ncoltiles * g.nprob * g.R;
    float* rowp_m = reinterpret_cast<float*>(base);
    int* rowp_i = reinterpret_cast<int*>(base + align_up(sizeof(float) * rows, 256));
    cudaStream_t s = (cudaStream_t)stream;
    dim3 grid(ncoltiles, g.nrowtiles, g.nprob);
    nce_fwd_launcher(g)<<<grid, TILE_THREADS, 0, s>>>(pred, targets, g, w.part_m, w.part_s, w.diag, w.cta, rowp_m, rowp_i,
                                                      nullptr);
    CPC_LAUNCH_CHECK();
    nce_combine_kernel<<<w.nblk, 256, 0, s>>>(w.part_m, w.part_s, w.diag, lse, w.blk, g.ncols, g.nrowtiles);
    CPC_LAUNCH_CHECK();
    nce_final_kernel<<<1, 256, 0, s>>>(w.blk, w.nblk, w.cta, w.ncta, g, out4, nullptr);
    CPC_LAUNCH_CHECK();
    nce_validate_final_kernel<<<1, 256, 0, s>>>(lse, w.diag, rowp_m, rowp_i, ncoltiles, out4, g, metrics);
    CPC_LAUNCH_CHECK();
    count_launch(4);
    return CPC_OK;
}
