// Policy / value heads on CUDA cores (fp32 math).
#pragma once
#include "tc_base.cuh"
#include "tc_reduce.cuh"
#include "categorical.cuh"

namespace b200rl {
using namespace tc;

// ------------------------------------------------------------------ policy/value heads (tiny: CUDA cores, fp32 math)
// A1 = A + 1 head outputs (logits | value), 1 <= A1 <= kMaxHeads.  Head weights live in dynamic shared memory.
constexpr int kMaxHeads = 24;              // (A+1) * 2 KB of head weights must fit the 48 KB default dynamic shared memory
constexpr int kHeadsPartialBlocks = 296;     // row blocks of the head weight gradient (x2 row lanes = partial slabs)
// rows per block of tc_heads_bwd_weight: its dhead rows are staged in (static-limit) shared memory, <= 256 x 32 floats
static inline int64_t heads_rows_per_block(int64_t n) {
    int64_t rpb = (n + kHeadsPartialBlocks - 1) / kHeadsPartialBlocks;
    if (rpb < 16) rpb = 16;
    if (rpb > 256) rpb = 256;
    return rpb;
}

// One row of the heads, computed by one warp: lane a (< A1) returns output a = hid . Wh[a] + bh[a].  Lane l holds hidden
// units [8l, 8l+8) and [256+8l, 256+8l+8) (two 16-byte loads); sW = Wh [A1][512] in shared memory.
__device__ __forceinline__ float heads_row(const bf16* __restrict__ hp, const float* sW, const float* __restrict__ bh, int A1, int lane) {
    float hv[16];
#pragma unroll
    for (int q = 0; q < 2; ++q) {
        const int4 v = ldg16(hp + q * 256 + lane * 8);
        const uint32_t w[4] = {(uint32_t)v.x, (uint32_t)v.y, (uint32_t)v.z, (uint32_t)v.w};
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            hv[q * 8 + 2 * e] = __uint_as_float(w[e] << 16);
            hv[q * 8 + 2 * e + 1] = __uint_as_float(w[e] & 0xFFFF0000u);
        }
    }
    float mine = 0.f;                               // lane a keeps output a
    for (int a = 0; a < A1; ++a) {
        float s = 0.f;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const float4 w0 = *reinterpret_cast<const float4*>(sW + a * 512 + q * 256 + lane * 8);
            const float4 w1 = *reinterpret_cast<const float4*>(sW + a * 512 + q * 256 + lane * 8 + 4);
            s = fmaf(hv[q * 8 + 0], w0.x, s); s = fmaf(hv[q * 8 + 1], w0.y, s);
            s = fmaf(hv[q * 8 + 2], w0.z, s); s = fmaf(hv[q * 8 + 3], w0.w, s);
            s = fmaf(hv[q * 8 + 4], w1.x, s); s = fmaf(hv[q * 8 + 5], w1.y, s);
            s = fmaf(hv[q * 8 + 6], w1.z, s); s = fmaf(hv[q * 8 + 7], w1.w, s);
        }
        s = warp_sum(s);
        if (lane == a) mine = s + bh[a];
    }
    return mine;
}

// out[n][A1] = hidden[n][512](bf16) . Wh[A1][512]^T + bh.  One warp per row: lane l holds hidden units
// [8l, 8l+8) and [256+8l, 256+8l+8) (two 16-byte loads), weights are read as float4 from shared memory.
__global__ void __launch_bounds__(256) tc_heads_fwd(const bf16* __restrict__ hid, const float* __restrict__ Wh,
                                                    const float* __restrict__ bh, int64_t n, int A1, int H,
                                                    float* __restrict__ out) {
    extern __shared__ float sW[];                       // [A1][512]
    for (int i = threadIdx.x; i < A1 * 512; i += blockDim.x) sW[i] = Wh[i];
    __syncthreads();
    const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
    for (int64_t row = (int64_t)blockIdx.x * wpb + (threadIdx.x >> 5); row < n; row += (int64_t)gridDim.x * wpb) {
        const float mine = heads_row(hid + row * 512, sW, bh, A1, lane);
        if (lane < A1) out[row * A1 + lane] = mine;     // one coalesced store per row
    }
}
// Rollout step: heads + Categorical sample in one pass, one warp per row.  The A + 1 outputs are tc_heads_fwd's
// (heads_row), the draw is categorical_sample_kernel's (row_stats + categorical_draw on the same fp32 logits), so action,
// log-probability and value equal the two-kernel chain bit for bit; no [n, A+1] round trip through global memory and no
// entropy (the rollout does not store it).  noise: Exp(1) draws [n, A].
__global__ void __launch_bounds__(256) tc_heads_sample(const bf16* __restrict__ hid, const float* __restrict__ Wh,
                                                       const float* __restrict__ bh, int64_t n, int A,
                                                       const float* __restrict__ noise, int64_t* __restrict__ action,
                                                       float* __restrict__ logprob, float* __restrict__ value) {
    extern __shared__ float sW[];                       // [A1][512]
    __shared__ float sX[8][kMaxHeads];                  // one row of outputs per warp
    const int A1 = A + 1;
    for (int i = threadIdx.x; i < A1 * 512; i += blockDim.x) sW[i] = Wh[i];
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    float* x = sX[wid];
    for (int64_t row = (int64_t)blockIdx.x * wpb + wid; row < n; row += (int64_t)gridDim.x * wpb) {
        const float mine = heads_row(hid + row * 512, sW, bh, A1, lane);
        if (lane < A1) x[lane] = mine;
        __syncwarp();
        if (lane == 0) {
            const RowStats rs = row_stats(x, A);
            const int arg = categorical_draw<false>(x, noise + row * (int64_t)A, A, rs, nullptr);
            action[row] = arg;
            logprob[row] = x[arg] - rs.lse;
            value[row] = x[A];
        }
        __syncwarp();
    }
}
// dhid_pre[n][512] (bf16) = (dhead[n][A1] . Wh[A1][512]) * (hid > 0).  Thread = 8 consecutive hidden units of one
// row (one mask byte in, one 16-byte store out).  Weights are staged transposed, sWt[a][e][group], so the 32 lanes
// of a warp (consecutive groups) hit 32 different banks.
__global__ void __launch_bounds__(256) tc_heads_bwd_data(const float* __restrict__ dhead, const float* __restrict__ Wh,
                                                         const uint8_t* __restrict__ hid_bits, int64_t n, int A1, int H,
                                                         bf16* __restrict__ dhid) {
    extern __shared__ float sWt[];                      // [A1][8][64]
    for (int i = threadIdx.x; i < A1 * 512; i += blockDim.x) {
        const int a = i >> 9, h = i & 511;
        sWt[a * 512 + (h & 7) * 64 + (h >> 3)] = Wh[i];
    }
    __syncthreads();
    const int64_t total = n * 64;                      // 64 groups of 8 per row
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int64_t row = idx >> 6;
        const int g = (int)(idx & 63);
        const uint32_t m = hid_bits[idx];               // bit e: hid[row][8g + e] > 0
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) o[e] = 0.f;
        for (int a = 0; a < A1; ++a) {
            const float d = __ldg(dhead + row * A1 + a);
#pragma unroll
            for (int e = 0; e < 8; ++e) o[e] = fmaf(d, sWt[a * 512 + e * 64 + g], o[e]);
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) if (!((m >> e) & 1u)) o[e] = 0.f;
        int4 w;
        w.x = (int)pack_bf16x2(o[0], o[1]); w.y = (int)pack_bf16x2(o[2], o[3]);
        w.z = (int)pack_bf16x2(o[4], o[5]); w.w = (int)pack_bf16x2(o[6], o[7]);
        *reinterpret_cast<int4*>(dhid + row * 512 + g * 8) = w;
    }
}
// dWh[a][h] = sum_m dhead[m][a] * hid[m][h]; dbh[a] = sum_m dhead[m][a]  (partial slabs per (row block, row lane),
// folded by tc_heads_fold).  Block = 512 threads = 2 row lanes x 256 hidden pairs; the block's dhead rows are staged
// in shared memory once, 8 rows of hidden values are in flight per thread.
template <int MAXA>
__global__ void __launch_bounds__(512) tc_heads_bwd_weight(const float* __restrict__ dhead, const bf16* __restrict__ hid,
                                                           int64_t n, int A1, int H, int64_t rows_per_block,
                                                           float* __restrict__ part) {
    extern __shared__ float sD[];                       // [rows_per_block][A1]
    const int hp = threadIdx.x & 255, rl = threadIdx.x >> 8;
    const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
    int64_t r1 = r0 + rows_per_block;
    if (r1 > n) r1 = n;
    const int nrows = (int)(r1 > r0 ? r1 - r0 : 0);
    for (int i = threadIdx.x; i < nrows * A1; i += blockDim.x) sD[i] = dhead[r0 * A1 + i];
    __syncthreads();
    float acc0[MAXA], acc1[MAXA], bacc[MAXA];
#pragma unroll
    for (int a = 0; a < MAXA; ++a) { acc0[a] = 0.f; acc1[a] = 0.f; bacc[a] = 0.f; }
    const uint32_t* h2 = reinterpret_cast<const uint32_t*>(hid);      // bf16 pairs
    int r = rl;
    for (; r + 14 < nrows; r += 16) {                   // 8 rows (stride 2) in flight
        uint32_t hv[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) hv[u] = __ldg(h2 + (r0 + r + 2 * u) * 256 + hp);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const float x0 = __uint_as_float(hv[u] << 16), x1 = __uint_as_float(hv[u] & 0xFFFF0000u);
            const float* dr = sD + (r + 2 * u) * A1;
#pragma unroll
            for (int a = 0; a < MAXA; ++a) {
                if (a < A1) {
                    const float d = dr[a];
                    acc0[a] = fmaf(d, x0, acc0[a]); acc1[a] = fmaf(d, x1, acc1[a]); bacc[a] += d;
                }
            }
        }
    }
    for (; r < nrows; r += 2) {
        const uint32_t hv = __ldg(h2 + (r0 + r) * 256 + hp);
        const float x0 = __uint_as_float(hv << 16), x1 = __uint_as_float(hv & 0xFFFF0000u);
        const float* dr = sD + r * A1;
#pragma unroll
        for (int a = 0; a < MAXA; ++a) {
            if (a < A1) {
                const float d = dr[a];
                acc0[a] = fmaf(d, x0, acc0[a]); acc1[a] = fmaf(d, x1, acc1[a]); bacc[a] += d;
            }
        }
    }
    float* pb = part + ((int64_t)blockIdx.x * 2 + rl) * A1 * (H + 2);      // slab rows: H weights, bias, pad
#pragma unroll
    for (int a = 0; a < MAXA; ++a) {
        if (a < A1) {
            *reinterpret_cast<float2*>(pb + (int64_t)a * (H + 2) + 2 * hp) = make_float2(acc0[a], acc1[a]);
            if (hp == 0) pb[(int64_t)a * (H + 2) + H] = bacc[a];
        }
    }
}
__global__ void __launch_bounds__(256) tc_heads_fold(const float* __restrict__ part, int nslabs, int A1, int H,
                                                     float* __restrict__ dW, float* __restrict__ db) {
    __shared__ float red[256];
    const int idx = blockIdx.x * 32 + (threadIdx.x & 31);
    const int a = idx / (H + 2), h = idx - a * (H + 2);
    const bool valid = a < A1 && h <= H;                // h == H: bias; h == H + 1: padding
    const float s = zlane_sum(part, (int64_t)A1 * (H + 2), nslabs, idx, valid, red);
    if (!valid || threadIdx.x >= 32) return;
    if (h == H) db[a] = s; else dW[(int64_t)a * H + h] = s;
}

}  // namespace b200rl
