// Shared device/host helpers for the cpc_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include "../../include/cpc_b200.h"

namespace cpc {

extern std::atomic<uint64_t> g_launches;   // defined in abi.cu
inline void count_launch(int n = 1) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

int check_device();                         // abi.cu: CPC_OK iff current device is sm_100

#define CPC_LAUNCH_CHECK()                                   \
    do {                                                     \
        if (cudaGetLastError() != cudaSuccess) return CPC_ERR_CUDA; \
    } while (0)

// Division by a launch-time constant, exact for 0 <= n < 2^31.
struct FastDiv {
    uint32_t d, m, s;
    __host__ __device__ FastDiv() : d(1), m(1u << 31), s(31) {}
    __host__ __device__ explicit FastDiv(int div) {
        d = (uint32_t)div;
        uint32_t l = 0;
        while ((1ull << l) < d) ++l;
        s = 31 + l;
        m = (uint32_t)(((1ull << s) + d - 1) / d);
    }
    __host__ __device__ __forceinline__ int div(int n) const {
        return (int)(((uint64_t)(uint32_t)n * m) >> s);
    }
    __host__ __device__ __forceinline__ void divmod(int n, int& q, int& r) const {
        q = div(n);
        r = n - q * (int)d;
    }
};

__host__ __device__ __forceinline__ size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }
__host__ __device__ __forceinline__ int ceil_div(int a, int b) { return (a + b - 1) / b; }

// ------------------------------------------------------------------------------------------------
// 64x64 register-tiled fp32 GEMM tile over a K range, operands fetched through functors.
//   acc[i][j] += sum_k A(row0 + tx*4 + i, k) * B(col0 + ty*4 + j, k)
// 256 threads; tx = tid & 15 owns 4 consecutive A rows, ty = tid >> 4 owns 4 consecutive B rows.
// A loader exposes  float load(int row, int k)  (row / k are global indices; out-of-range -> 0) and a
// constexpr bool kFast: true  -> consecutive threads fetch consecutive k of one row (k is the
// contiguous memory axis), false -> consecutive threads fetch consecutive rows at one k.
// ------------------------------------------------------------------------------------------------
constexpr int TILE = 64;
constexpr int TILE_K = 16;
constexpr int TILE_LD = TILE + 4;
constexpr int TILE_THREADS = 256;

struct TileSmem {
    float a[TILE_K][TILE_LD];
    float b[TILE_K][TILE_LD];
};

template <class L>
__device__ __forceinline__ void tile_fill(const L& ld, float (*dst)[TILE_LD], int row0, int k0) {
    const int tid = threadIdx.x;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        int r, kk;
        if (L::kFast) {
            kk = tid & 15;
            r = (tid >> 4) + 16 * i;
        } else {
            r = tid & 63;
            kk = (tid >> 6) + 4 * i;
        }
        dst[kk][r] = ld.load(row0 + r, k0 + kk);
    }
}

template <class LA, class LB>
__device__ __forceinline__ void tile_gemm(const LA& la, const LB& lb, int row0, int col0, int k_begin, int k_end,
                                          float (&acc)[4][4], TileSmem& sm) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    for (int k0 = k_begin; k0 < k_end; k0 += TILE_K) {
        tile_fill(la, sm.a, row0, k0);
        tile_fill(lb, sm.b, col0, k0);
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < TILE_K; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&sm.a[kk][tx * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&sm.b[kk][ty * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w};
            const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
}

// Same tiling, squared distances: acc[i][j] += sum_k (A(row, k) - B(col, k))^2.  The difference is formed before
// squaring, so a near-coincident pair keeps its digits (|a|^2 + |b|^2 - 2 a.b would cancel them).  Out-of-range loads
// are 0 on both sides and add nothing.
template <class LA, class LB>
__device__ __forceinline__ void tile_dist(const LA& la, const LB& lb, int row0, int col0, int k_begin, int k_end,
                                          float (&acc)[4][4], TileSmem& sm) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    for (int k0 = k_begin; k0 < k_end; k0 += TILE_K) {
        tile_fill(la, sm.a, row0, k0);
        tile_fill(lb, sm.b, col0, k0);
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < TILE_K; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&sm.a[kk][tx * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&sm.b[kk][ty * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w};
            const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const float d = av[i] - bv[j];
                    acc[i][j] = fmaf(d, d, acc[i][j]);
                }
        }
        __syncthreads();
    }
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

}  // namespace cpc
