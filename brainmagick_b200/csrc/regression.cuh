// Masked regression losses of the solver's 'l1' and 'mse' objectives (bm/losses.py:11-26, bm/solver.py:76-94):
//   loss = mean over the selected elements of |e - o|^p,   selected = mask.expand_as(estimate),   p = 1 or 2,
// which the reference computes as nn.L1Loss / nn.MSELoss over `estimate[feature_mask]` (a boolean gather, i.e. a
// device->host synchronisation for `nonzero` and two gathered copies per call).  Here: one streaming pass forward, one
// backward, nothing read back by the host.
//
// HBM-bound: forward reads 8 B per element plus the mask, backward reads 8 B and writes 4 B (8 B with the target gradient).
// One warp walks one [T] row of est / out at a time, so every access is coalesced, and the mask row of a [B, 1, T] mask
// (broadcast over F) is found once per row instead of by a division per element.
//
// Selection, not multiplication: an unselected element is never used arithmetically, so a NaN or inf there leaves the loss
// finite and its gradient exactly 0, as with the reference's boolean indexing.  An empty selection gives 0/0 = NaN (nn.MSELoss
// on an empty tensor) and all-zero gradients.
#pragma once
#include "../../include/bm_b200.h"
#include "common.cuh"

namespace bm {

constexpr int REG_THREADS = 256;
constexpr int REG_MAX_BLOCKS = 592;                       // one wave of 4 blocks on each of the B200's 148 SMs
constexpr long long REG_ELEMS_PER_BLOCK = 8192;
constexpr int REG_ILP = 4;                                // row chunks whose loads are in flight before the first use
static_assert(2 * REG_MAX_BLOCKS + 2 == BM_REGRESSION_WS_DOUBLES, "workspace layout");

// workspace (doubles): [0, MAXB) per-block sums | [MAXB, 2 MAXB) per-block counts (u64) | count (double, read by the
// backward) | finalize ticket (u32)
constexpr int REG_WS_COUNT = 2 * REG_MAX_BLOCKS;
constexpr int REG_WS_TICKET = 2 * REG_MAX_BLOCKS + 1;

// The grid is a function of the element count alone, so the partials -- and the fixed-order sum over them -- are the same
// on every call and every device: the loss is bit-identical from call to call.
inline int regression_grid(long long n) {
    long long g = (n + REG_ELEMS_PER_BLOCK - 1) / REG_ELEMS_PER_BLOCK;
    return (int)(g < 1 ? 1 : (g > REG_MAX_BLOCKS ? REG_MAX_BLOCKS : g));
}

// V consecutive elements of one row: a float4 / 4-byte mask word when V == 4 (T % 4 == 0, aligned), else one element.
template <int V>
__device__ __forceinline__ void reg_load(const float* __restrict__ p, int j, float (&v)[V]) {
    if constexpr (V == 4) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(p) + j);
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
    } else {
        v[0] = __ldg(p + j);
    }
}
template <int V>
__device__ __forceinline__ void reg_load_mask(const unsigned char* __restrict__ p, int j, bool (&m)[V]) {
    if constexpr (V == 4) {
        const uchar4 q = __ldg(reinterpret_cast<const uchar4*>(p) + j);
        m[0] = q.x != 0; m[1] = q.y != 0; m[2] = q.z != 0; m[3] = q.w != 0;
    } else {
        m[0] = __ldg(p + j) != 0;
    }
}
template <int V>
__device__ __forceinline__ void reg_store(float* __restrict__ p, int j, const float (&v)[V]) {
    if constexpr (V == 4) {
        reinterpret_cast<float4*>(p)[j] = make_float4(v[0], v[1], v[2], v[3]);
    } else {
        p[j] = v[0];
    }
}

// sum of |e - o|^P (fp64) and count over the selected elements; the last block to finish reduces the per-block partials in
// index order and writes loss[0] = sum / count (fp64, rounded once) and the count for the backward.
template <int P, int V>
__global__ void __launch_bounds__(REG_THREADS, 4) regression_fwd_kernel(
        const float* __restrict__ est, const float* __restrict__ out, const unsigned char* __restrict__ mask, long long rows,
        int F, int full_mask, int T, double* __restrict__ ws, float* __restrict__ loss) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int WPB = REG_THREADS / 32;
    const long long nwarps = (long long)gridDim.x * WPB;
    const int TV = T / V;
    double acc = 0.0;
    unsigned long long cnt = 0;
    for (long long r = (long long)blockIdx.x * WPB + warp; r < rows; r += nwarps) {
        const float* er = est + r * T;
        const float* orow = out + r * T;
        const unsigned char* mr = mask + (full_mask ? r : r / F) * T;
        for (int base = lane; base < TV; base += 32 * REG_ILP) {
            float e[REG_ILP][V], o[REG_ILP][V];
            bool m[REG_ILP][V];
#pragma unroll
            for (int u = 0; u < REG_ILP; ++u) {
                const int j = base + 32 * u;
                if (j < TV) {
                    reg_load_mask<V>(mr, j, m[u]);
                    reg_load<V>(er, j, e[u]);
                    reg_load<V>(orow, j, o[u]);
                } else {
#pragma unroll
                    for (int k = 0; k < V; ++k) m[u][k] = false;
                }
            }
#pragma unroll
            for (int u = 0; u < REG_ILP; ++u) {
#pragma unroll
                for (int k = 0; k < V; ++k) {
                    if (m[u][k]) {
                        const double d = (double)(e[u][k] - o[u][k]);
                        acc += P == 1 ? fabs(d) : d * d;
                        ++cnt;
                    }
                }
            }
        }
    }

    __shared__ double s_sum[WPB];
    __shared__ unsigned long long s_cnt[WPB];
    __shared__ unsigned int s_ticket;
    acc = warp_sum_d(acc);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
    if (lane == 0) { s_sum[warp] = acc; s_cnt[warp] = cnt; }
    __syncthreads();
    unsigned long long* ws_cnt = reinterpret_cast<unsigned long long*>(ws + REG_MAX_BLOCKS);
    if (threadIdx.x == 0) {
        double bs = 0.0;
        unsigned long long bc = 0;
        for (int w = 0; w < WPB; ++w) { bs += s_sum[w]; bc += s_cnt[w]; }
        ws[blockIdx.x] = bs;
        ws_cnt[blockIdx.x] = bc;
        __threadfence();
        s_ticket = atomicAdd(reinterpret_cast<unsigned int*>(ws + REG_WS_TICKET), 1u);
    }
    __syncthreads();
    if (s_ticket != gridDim.x - 1) return;
    __threadfence();
    acc = 0.0;
    cnt = 0;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += REG_THREADS) {
        acc += __ldcg(ws + i);
        cnt += __ldcg(ws_cnt + i);
    }
    acc = warp_sum_d(acc);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
    __syncthreads();
    if (lane == 0) { s_sum[warp] = acc; s_cnt[warp] = cnt; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double total = 0.0;
        unsigned long long n = 0;
        for (int w = 0; w < WPB; ++w) { total += s_sum[w]; n += s_cnt[w]; }
        ws[REG_WS_COUNT] = (double)n;
        loss[0] = (float)(total / (double)n);                 // 0 / 0 = NaN for an empty selection, like the reference
    }
}

// dest = selected ? dL/de : 0 with dL/de = 2 (e - o) gout / count (P = 2) or sign(e - o) gout / count (P = 1; sign(0) = 0,
// NaN stays NaN, as torch.sign); dout = -dest when requested.  gout and count are read on the device.
template <int P, int V>
__global__ void __launch_bounds__(REG_THREADS, 4) regression_bwd_kernel(
        const float* __restrict__ est, const float* __restrict__ out, const unsigned char* __restrict__ mask, long long rows,
        int F, int full_mask, int T, const float* __restrict__ gout, const double* __restrict__ ws, float* __restrict__ dest,
        float* __restrict__ dout) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int WPB = REG_THREADS / 32;
    const long long nwarps = (long long)gridDim.x * WPB;
    const int TV = T / V;
    // one fp64 division rounded once; with the subtraction and the product, three fp32 roundings per element (P = 2)
    const float scale = (float)((P == 2 ? 2.0 : 1.0) * (double)__ldg(gout) / __ldg(ws + REG_WS_COUNT));
    for (long long r = (long long)blockIdx.x * WPB + warp; r < rows; r += nwarps) {
        const float* er = est + r * T;
        const float* orow = out + r * T;
        const unsigned char* mr = mask + (full_mask ? r : r / F) * T;
        float* dr = dest ? dest + r * T : nullptr;
        float* dor = dout ? dout + r * T : nullptr;
        for (int base = lane; base < TV; base += 32 * REG_ILP) {
            float e[REG_ILP][V], o[REG_ILP][V];
            bool m[REG_ILP][V];
#pragma unroll
            for (int u = 0; u < REG_ILP; ++u) {
                const int j = base + 32 * u;
                if (j < TV) {
                    reg_load_mask<V>(mr, j, m[u]);
                    reg_load<V>(er, j, e[u]);
                    reg_load<V>(orow, j, o[u]);
                }
            }
#pragma unroll
            for (int u = 0; u < REG_ILP; ++u) {
                const int j = base + 32 * u;
                if (j >= TV) break;
                float g[V], ng[V];
#pragma unroll
                for (int k = 0; k < V; ++k) {
                    const float d = e[u][k] - o[u][k];
                    float v;
                    if (P == 2) {
                        v = d * scale;
                    } else {
                        const float s = d > 0.f ? 1.f : (d < 0.f ? -1.f : d);     // d == +-0 -> 0, NaN -> NaN
                        v = s * scale;
                    }
                    g[k] = m[u][k] ? v : 0.f;
                    ng[k] = m[u][k] ? -v : 0.f;
                }
                if (dr) reg_store<V>(dr, j, g);
                if (dor) reg_store<V>(dor, j, ng);
            }
        }
    }
}

inline bool reg_aligned(const void* p, unsigned a) { return p == nullptr || (reinterpret_cast<uintptr_t>(p) % a) == 0; }

template <int P>
inline void launch_regression_fwd_p(bool vec, int grid, const float* est, const float* out, const unsigned char* mask,
                                    long long rows, int F, int full, int T, double* ws, float* loss, cudaStream_t st) {
    if (vec)
        regression_fwd_kernel<P, 4><<<grid, REG_THREADS, 0, st>>>(est, out, mask, rows, F, full, T, ws, loss);
    else
        regression_fwd_kernel<P, 1><<<grid, REG_THREADS, 0, st>>>(est, out, mask, rows, F, full, T, ws, loss);
}

template <int P>
inline void launch_regression_bwd_p(bool vec, int grid, const float* est, const float* out, const unsigned char* mask,
                                    long long rows, int F, int full, int T, const float* gout, const double* ws, float* dest,
                                    float* dout, cudaStream_t st) {
    if (vec)
        regression_bwd_kernel<P, 4><<<grid, REG_THREADS, 0, st>>>(est, out, mask, rows, F, full, T, gout, ws, dest, dout);
    else
        regression_bwd_kernel<P, 1><<<grid, REG_THREADS, 0, st>>>(est, out, mask, rows, F, full, T, gout, ws, dest, dout);
}

}  // namespace bm
