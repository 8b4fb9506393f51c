// conv1 straight from the uint8 rollout (no 16-bit copy of the frames anywhere).
//
// The rollout keeps every frame ONCE as uint8 space-to-depth(4) pixels, 28 224 B per frame (the algorithmic
// minimum; reference: a 14.8 GB fp32 buffer, ppo_atari_envpool.py:203):
//     frames    u8 [img][441 grid rows][64 ch]   row-major    -> forward  (K-major operand rows)
//     frames_t  u8 [img][64 ch][448 grid rows]   channel-major -> weight gradient (lanes = channels, K = rows)
//
// Forward  tc_conv1_i8: integer tensor cores (tcgen05.mma kind::i8, u8 x s8 -> s32, accumulators in TMEM).  The
//   pixels are EXACT (0..255 are integers); the fp32 master weights are split per output channel into two signed
//   8-bit limbs  w ~= s_co * (l1 / 2^7 + l2 / 2^14)  (|error| <= s_co * 2^-15, i.e. 15 bits relative to the row
//   maximum -- tighter than the 8 bits of a bf16 weight), the two limbs are 2 x 32 = 64 GEMM columns, and the
//   epilogue recombines  y = acc1 * s/2^7/255 + acc2 * s/2^14/255 + bias.  Integer accumulation is exact, so the
//   result does not depend on the order of the 256-term dot products.  A 1-byte operand also halves the
//   shared-memory operand traffic that bounded the bf16 kernel (N = 32 is too narrow to amortise the 128-row A tile).
//   Same window scheme as tc_conv_win: one TMA box of 128 + 22 rows per tile, the four 2x2 taps are descriptors
//   shifted by whole 64-byte rows of a SWIZZLE_64B image.
//
// Weight gradient  tc_conv1_wgrad_u8: dW[tap, c, co] = sum_p X[p + off_tap, c] * dY[p, co].  The pixels go
//   uint8 (shared memory, channel-major TMA box) -> fp16 pairs in REGISTERS (one PRMT per two pixels builds
//   1024 + x; the offset is removed once per CTA through the bias partial) -> tensor memory (tcgen05.st), and are
//   consumed as the A operand straight from TMEM (tcgen05.mma with A in TMEM); dY rows are SWIZZLE_64B TMA boxes used
//   as an MN-major B operand with N = 32, loaded at two row offsets (0 and -21) so that one A tile serves all four
//   taps.  No 16-bit image of the frames ever exists in shared or global memory.
#pragma once
#include "tc_base.cuh"
#include <cuda_fp16.h>
#include <cstdlib>
#include "tc_conv_win.cuh"

namespace b200rl {
using namespace tc;

// ------------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// A operand in tensor memory (lane = row m; 32-bit column j holds K elements 2j, 2j+1), B from shared memory
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
        "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
        "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]),
        "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
        "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
        "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_cols(uint32_t taddr, const uint32_t (&v)[32]) { tmem_st32(taddr, v); }
__device__ __forceinline__ void tmem_st_cols(uint32_t taddr, const uint32_t (&v)[16]) { tmem_st16(taddr, v); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

constexpr uint64_t kDescSwizzle64 = 4ull << 61;      // LayoutType::SWIZZLE_64B
// K-major SWIZZLE_64B operand: rows 64 B apart, 8-row atoms 512 B apart (SBO)
__device__ __forceinline__ uint64_t desc_kmajor_sw64(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (32ull << 32) | kDescVersion | kDescSwizzle64;
}
// MN-major SWIZZLE_64B operand with ONE 32-element (64-byte) MN atom: rows = K index, 8-row K groups 512 B apart
__device__ __forceinline__ uint64_t desc_mnmajor_sw64(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | (32ull << 32) | kDescVersion | kDescSwizzle64;
}
// byte offset of 16-byte chunk c (0..3) of row r in a SWIZZLE_64B image (address bits [4,6) ^= bits [7,9))
__device__ __forceinline__ uint32_t img64_off(int r, int c) { return (uint32_t)(r * 64 + ((c ^ ((r >> 1) & 3)) << 4)); }
// u8 x s8 -> s32
__host__ __device__ constexpr uint32_t make_idesc_i8(int M, int N) {
    return (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// A = fp16, B = bf16 or fp16 -> fp32;  b_mn_major = 1: B rows are the K index
__host__ __device__ constexpr uint32_t make_idesc_f16ts(int M, int N, int b_bf16, int b_mn_major) {
    return (1u << 4) | (0u << 7) | ((uint32_t)b_bf16 << 10) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}

// ------------------------------------------------------------------------------------ frame conversion (once per env step)
// uint8 frames [n,4,84,84] (NCHW, as the env delivers them) -> row-major u8 [n,441,64] and channel-major u8 [n,64,448]
// space-to-depth(4) pixels: channel = c*16 + sy*4 + sx of source pixel (4Y+sy, 4X+sx), grid row = Y*21 + X.
// One block per (frame, colour plane c): the 84x84 plane is staged in shared memory (coalesced 16-byte reads).
__global__ void __launch_bounds__(256) tc_frames_to_s2d_u8(const uint8_t* __restrict__ obs, const int64_t* __restrict__ rows, int64_t n,
                                                           uint8_t* __restrict__ out_rm, uint8_t* __restrict__ out_cm) {
    __shared__ __align__(16) uint8_t plane[7056];
    const int64_t i = blockIdx.x >> 2;
    const int c = blockIdx.x & 3;
    const int64_t img = rows ? rows[i] : i;
    const int4* src = reinterpret_cast<const int4*>(obs + img * 28224 + c * 7056);
    for (int t = threadIdx.x; t < 441; t += 256) reinterpret_cast<int4*>(plane)[t] = __ldg(src + t);
    __syncthreads();
    // row-major: 16 bytes (4 rows of 4 pixels) per grid position
    for (int pos = threadIdx.x; pos < 441; pos += 256) {
        const int Y = pos / 21, X = pos - Y * 21;
        const uint8_t* p = plane + (Y * 4) * 84 + X * 4;
        int4 v;
        v.x = *reinterpret_cast<const int*>(p); v.y = *reinterpret_cast<const int*>(p + 84);
        v.z = *reinterpret_cast<const int*>(p + 168); v.w = *reinterpret_cast<const int*>(p + 252);
        *reinterpret_cast<int4*>(out_rm + (i * 441 + pos) * 64 + c * 16) = v;
    }
    // channel-major: channel (sy, sx) of this plane, 4 consecutive grid rows per 32-bit store (448-byte rows, zero tail)
    for (int t = threadIdx.x; t < 16 * 112; t += 256) {
        const int ch = t / 112, q = t - ch * 112;
        const int sy = ch >> 2, sx = ch & 3;
        uint32_t w = 0;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const int pos = q * 4 + e;
            if (pos < 441) {
                const int Y = pos / 21, X = pos - Y * 21;
                w |= (uint32_t)plane[(Y * 4 + sy) * 84 + X * 4 + sx] << (8 * e);
            }
        }
        *reinterpret_cast<uint32_t*>(out_cm + (i * 64 + c * 16 + ch) * 448 + q * 4) = w;
    }
}

// ------------------------------------------------------------------------------------ conv1 weight limbs
// w[co][c][ky][kx] (fp32) -> s8 limbs L[(limb, co)][tap (a,b)][c*16 + sy*4 + sx] with ky = 4a+sy, kx = 4b+sx, and the
// per-column output scales sc[limb*32 + co] = s_co / 2^(7*(limb+1)) / 255 (the /255 of ppo_atari_envpool.py:144).
__global__ void __launch_bounds__(256) tc_pack_conv1_i8(const float* __restrict__ w, int8_t* __restrict__ limbs, float* __restrict__ sc) {
    __shared__ float red[32];
    const int co = blockIdx.x, idx = threadIdx.x;                  // idx = (c, ky, kx)
    const float v = w[co * 256 + idx];
    float m = fabsf(v);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((idx & 31) == 0) red[idx >> 5] = m;
    __syncthreads();
    float mx = red[0];
#pragma unroll
    for (int k = 1; k < 8; ++k) mx = fmaxf(mx, red[k]);
    const float s = mx > 0.f ? mx * (128.0f / 127.0f) : 1.0f;
    const float u = v / s * 128.0f;                                // |u| <= 127
    float l1 = rintf(u);
    l1 = fminf(fmaxf(l1, -127.f), 127.f);
    float l2 = rintf((u - l1) * 128.0f);
    l2 = fminf(fmaxf(l2, -127.f), 127.f);
    const int kx = idx & 7, ky = (idx >> 3) & 7, c = idx >> 6;
    const int a = ky >> 2, sy = ky & 3, b = kx >> 2, sx = kx & 3;
    const int k = (a * 2 + b) * 64 + c * 16 + sy * 4 + sx;
    limbs[co * 256 + k] = (int8_t)l1;
    limbs[(32 + co) * 256 + k] = (int8_t)l2;
    if (idx == 0) {
        sc[co] = s / 128.0f / 255.0f;
        sc[32 + co] = s / 16384.0f / 255.0f;
    }
}

// ------------------------------------------------------------------------------------ conv1 forward (kind::i8)
struct Conv1U8Params {
    const int64_t* rows;     // optional image gather (minibatch rows of the rollout)
    int n;                   // images in this launch
    int64_t n_images;        // images addressable through `rows`
    const int8_t* limbs;     // [64][256] s8 (tc_pack_conv1_i8)
    const float* sc;         // [64] column scales
    const float* bias;       // [32]
    bf16* out;               // act1 as 2x2 cells [n,100,128]
    uint32_t* mask_out;      // act1 > 0 bits: [n,100 cells] x 4 words
};

// Pair rows: TMA delivers one shared-memory row (<= 128 B) per request at ~5.5 cycles per request and SM -- the rate at
// which 128-byte rows saturate HBM -- so a box of 64-byte rows moves half the bytes in the same time (measured: the first
// version of this kernel, boxes of 152 x 64 B, sat at 44 % DRAM with its MMA issuer waiting on the TMA barrier).  The
// row-major image [441][64 B] is therefore read as 221 rows of 128 B = PAIRS of grid positions (2q, 2q+1): one box of
// 139 pair rows per 256 output positions.  GEMM rows are pair rows; the even and the odd position of each pair get their own
// accumulator, and a tap (dy, dx) of position p = 2q + e is the 64-byte half ((e + dx + dy) & 1) of pair row
// q + (e + 21 dy + dx) / 2 -- a K-major SWIZZLE_128B descriptor shifted by whole rows plus a 64-byte K offset.
// Epilogue arithmetic of conv1 on the integer tensor cores, shared by tc_conv1_i8 and the fused rollout tower
// (tc_rollout_tower.cuh): one output position's 32 channels from its two limb accumulators.
// y = (128 acc1 + acc2) * (s / 2^14 / 255) + bias: the limb recombination is exact in int32 (|128 acc1| < 2^31).
// Returns the ReLU mask bits (y > 0); pk = the 32 ReLU'd bf16 outputs, packed in pairs.
__device__ __forceinline__ uint32_t conv1_i8_epilogue(const uint32_t (&a1)[32], const uint32_t (&a2)[32], const float* s_sc,
                                                      const float* s_bias, uint32_t (&pk)[16]) {
    uint32_t bits = 0u;
#pragma unroll
    for (int c4 = 0; c4 < 32; c4 += 4) {
        const float4 sc = *reinterpret_cast<const float4*>(s_sc + c4);
        const float4 bi = *reinterpret_cast<const float4*>(s_bias + c4);
        const float f0 = fmaf((float)((int)a1[c4] * 128 + (int)a2[c4]), sc.x, bi.x);
        const float f1 = fmaf((float)((int)a1[c4 + 1] * 128 + (int)a2[c4 + 1]), sc.y, bi.y);
        const float f2 = fmaf((float)((int)a1[c4 + 2] * 128 + (int)a2[c4 + 2]), sc.z, bi.z);
        const float f3 = fmaf((float)((int)a1[c4 + 3] * 128 + (int)a2[c4 + 3]), sc.w, bi.w);
        bits |= (f0 > 0.f ? 1u : 0u) << c4;
        bits |= (f1 > 0.f ? 1u : 0u) << (c4 + 1);
        bits |= (f2 > 0.f ? 1u : 0u) << (c4 + 2);
        bits |= (f3 > 0.f ? 1u : 0u) << (c4 + 3);
        pk[c4 >> 1] = pack_bf16x2_relu(f0, f1);
        pk[(c4 >> 1) + 1] = pack_bf16x2_relu(f2, f3);
    }
    return bits;
}

constexpr bool kConv1I8Direct256 = true;
template <int STAGES, int DBG>
__global__ void __launch_bounds__(kConvWinThreads, 1) tc_conv1_i8(const __grid_constant__ CUtensorMap tmA, const Conv1U8Params p, int total_tiles) {
    constexpr int BN = 64, WR = 144, NTAPS = 4;
    constexpr int STAGE_BYTES = WR * 128;           // 18432 = 18 x 1024
    constexpr int B_CHUNK = BN * 64;                // one tap of the limb image: 64 rows x 64 B (SWIZZLE_64B)
    constexpr int NT = 4;                           // tiles in flight in TMEM (see conv_win_acc_bufs)
    constexpr uint32_t TMEM_COLS = 2 * NT * BN;     // accumulator 2 (q % NT) + e: tile q, e = 0 even / 1 odd positions
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t full_bar[STAGES], empty_bar[STAGES], tfull_bar[2 * NT], tempty_bar[2 * NT];
    __shared__ uint32_t tmem_base_smem;
    __shared__ __align__(16) float s_sc[32], s_bias[32];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int tid = threadIdx.x, warp = tid >> 5;
    uint8_t* sW = smem;                             // 4 taps x 4096 B
    uint8_t* sRing = smem + NTAPS * B_CHUNK;        // 16384: 1024-aligned
    uint8_t* sStage = sRing + (size_t)STAGES * STAGE_BYTES;     // 16 epilogue warps x (32 rows x 64 B + 32 row offsets)

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < 2 * NT; ++a) { mbar_init(&tfull_bar[a], 1); mbar_init(&tempty_bar[a], 4); }
        fence_barrier_init();
        tma_prefetch_desc(&tmA);
    }
    if (warp == 1) tmem_alloc(&tmem_base_smem, TMEM_COLS);
    for (int idx = tid; idx < NTAPS * BN * 4; idx += blockDim.x) {          // 16-byte chunks of the limb image
        const int c16 = idx & 3;
        const int t = (idx >> 2) & 3;
        const int r = idx >> 4;
        *reinterpret_cast<int4*>(sW + t * B_CHUNK + img64_off(r, c16)) = ldg16(p.limbs + r * 256 + t * 64 + c16 * 16);
    }
    if (tid < 32) { s_sc[tid] = p.sc[32 + tid]; s_bias[tid] = p.bias[tid]; }      // sc[32 + co] = s_co / 2^14 / 255
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_d = tmem_base_smem;
    // a tile = 128 pair rows = 256 grid positions; 2 tiles per image (441 positions used)
    const int tile_begin = (int)(((int64_t)total_tiles * blockIdx.x) / gridDim.x);
    const int tile_end = (int)(((int64_t)total_tiles * (blockIdx.x + 1)) / gridDim.x);

    if (warp == 0) {
        // ======================= TMA producer: one [139 (144) pair rows x 128 B] box of one image per tile; the image
        // coordinate is the minibatch gather, fetched one tile ahead
        if (tid == 0) {
            uint32_t q = 0;
            int z_next = 0;
            if (tile_begin < tile_end) {
                const int img = tile_begin >> 1;
                z_next = p.rows ? (int)__ldg(p.rows + img) : img;
            }
            for (int tile = tile_begin; tile < tile_end; ++tile, ++q) {
                const uint32_t s = q % STAGES;
                const int z = z_next;
                if (tile + 1 < tile_end) {
                    const int img = (tile + 1) >> 1;
                    z_next = p.rows ? (int)__ldg(p.rows + img) : img;
                }
                if (q >= (uint32_t)STAGES) mbar_wait(&empty_bar[s], ((q / STAGES) - 1) & 1);
                if (DBG & 2) { mbar_arrive(&full_bar[s]); continue; }
                mbar_arrive_expect_tx(&full_bar[s], (uint32_t)STAGE_BYTES);
                tma_load_3d(smem_u32(sRing + (size_t)s * STAGE_BYTES), &tmA, 0, (tile & 1) * 128, z, &full_bar[s]);
            }
        }
    } else if (warp == 1) {
        // ======================= MMA issuer (warp-uniform loop, one elected lane): per tile and parity 4 taps x 2 K-steps of
        // 32 bytes.  A: K-major SWIZZLE_128B pair rows (row shift + 64-byte half); B: K-major SWIZZLE_64B limb rows.
        const bool leader = elect_one();
        constexpr uint32_t idesc = make_idesc_i8(128, BN);
        const uint64_t a_hi = desc_kmajor(0) & 0xFFFFFFFF00000000ull;
        const uint32_t a_flags = (uint32_t)(desc_kmajor(0) & 0xFFFFFFFFull);
        const uint64_t b_hi = desc_kmajor_sw64(0) & 0xFFFFFFFF00000000ull;
        const uint32_t b_flags = (uint32_t)(desc_kmajor_sw64(0) & 0xFFFFFFFFull);
        const uint32_t w_lo = ((smem_u32(sW) & 0x3FFFFu) >> 4) | b_flags;
        // tap t = (dy, dx): position offset 21 dy + dx; for parity e the operand is half (e + off) & 1 of pair row + (e + off) >> 1
        constexpr int off[4] = {0, 1, 21, 22};
        uint32_t q = 0;
        for (int tile = tile_begin; tile < tile_end; ++tile, ++q) {
            const uint32_t s = q % STAGES;
            mbar_wait(&full_bar[s], (q / STAGES) & 1);
            const uint32_t win_lo = ((smem_u32(sRing + (size_t)s * STAGE_BYTES) & 0x3FFFFu) >> 4) | a_flags;
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const uint32_t acc = 2 * (q % NT) + e;
                if (q >= (uint32_t)NT) mbar_wait(&tempty_bar[acc], ((q / NT) - 1) & 1);
                tc_fence_after_sync();
                if (leader) {
                    const uint32_t d_addr = tmem_d + acc * BN;
#pragma unroll
                    for (int t = 0; t < NTAPS; ++t) {
                        if (DBG & 4) break;
                        const int po = e + off[t];
                        const uint32_t a_lo = win_lo + (uint32_t)((po >> 1) * 8 + (po & 1) * 4);      // rows of 128 B, halves of 64 B
                        const uint32_t b_lo = w_lo + (uint32_t)((t * B_CHUNK) >> 4);
#pragma unroll
                        for (int kk = 0; kk < 2; ++kk)
                            umma_i8(d_addr, a_hi | (uint64_t)(a_lo + 2 * kk), b_hi | (uint64_t)(b_lo + 2 * kk), idesc,
                                    (t | kk) != 0 ? 1u : 0u);
                    }
                    if (e == 1) umma_commit(&empty_bar[s]);
                    umma_commit(&tfull_bar[acc]);
                }
                __syncwarp();
            }
        }
    } else {
        // ======================= epilogue: warps 2-17 = four groups of four (one warp per TMEM lane quadrant); group
        // (e, tp) drains the accumulator of parity e of the tiles of parity tp: lane = pair row q, output position p = 2q + e.
        // (Four groups: see tc_conv_win.cuh -- the epilogue's dependent instruction chain is the tile period otherwise.)
        const int ew = warp & 3;
        const int grp = (warp - 2) >> 2;
        const int e = grp & 1, tp = grp >> 1;
        const int lrow = ew * 32 + (tid & 31);
        const uint32_t lane_base = tmem_d + ((uint32_t)(ew * 32) << 16);
        for (int tile = tile_begin + tp; tile < tile_end; tile += 2) {
            const uint32_t k = (uint32_t)(tile - tile_begin);
            const uint32_t acc = 2 * (k % NT) + e;
            const uint32_t lane_addr = lane_base + acc * BN;
            const int i = tile >> 1;
            const int rem = 2 * (((tile & 1) << 7) + lrow) + e;
            const int Y = (rem * 3121) >> 16, X = rem - Y * 21;          // rem / 21 for rem < 512
            const bool valid = rem < 441 && Y < 20 && X < 20;
            const int64_t cell = ((int64_t)i * 10 + (Y >> 1)) * 10 + (X >> 1);
            const int cls = (Y & 1) * 2 + (X & 1);
            mbar_wait(&tfull_bar[acc], (k / NT) & 1);
            tc_fence_after_sync();
            uint32_t a1[32], a2[32];
            if (DBG & 8) {
#pragma unroll
                for (int c4 = 0; c4 < 32; ++c4) { a1[c4] = (uint32_t)(tile + c4); a2[c4] = (uint32_t)(lrow * c4); }
            } else {
                tmem_ld32(lane_addr, a1);
                tmem_ld32(lane_addr + 32, a2);
                tmem_ld_wait();
            }
            tc_fence_before_sync();
            __syncwarp();
            if ((tid & 31) == 0) mbar_arrive(&tempty_bar[acc]);            // accumulator drained
            uint32_t pk[16];
            const uint32_t bits = conv1_i8_epilogue(a1, a2, s_sc, s_bias, pk);
            if (valid && !(DBG & 1)) p.mask_out[cell * 4 + cls] = bits;
            // Stores: a lane owns one output row (64 B at its own 2x2-cell address), so a direct 16-byte store instruction of
            // the warp touches 32 different lines = 32 L1 wavefronts -- measured, the epilogue's global stores took more of
            // the L1 data pipe than the MMAs' operand reads.  The rows go through a per-warp staging tile instead (XOR
            // swizzle: conflict-free both ways), and 4 consecutive lanes write one row's 64 bytes: 8 lines per instruction.
            if (kConv1I8Direct256) {
                // two 256-bit stores per row instead of the staging round trip (two warp syncs, 8 shared-memory instructions)
                if (valid && !(DBG & 1)) {
                    uint8_t* dst = reinterpret_cast<uint8_t*>(p.out) + (cell * 4 + cls) * 64;
                    st_global_256(dst, make_int4((int)pk[0], (int)pk[1], (int)pk[2], (int)pk[3]), make_int4((int)pk[4], (int)pk[5], (int)pk[6], (int)pk[7]));
                    st_global_256(dst + 32, make_int4((int)pk[8], (int)pk[9], (int)pk[10], (int)pk[11]),
                                  make_int4((int)pk[12], (int)pk[13], (int)pk[14], (int)pk[15]));
                }
                continue;
            }
            uint8_t* stg = sStage + (size_t)(warp - 2) * 2304;
            const int lane = tid & 31;
            {
                const uint32_t f = (uint32_t)(lane >> 1) & 3u;
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    *reinterpret_cast<int4*>(stg + lane * 64 + ((((uint32_t)c) ^ f) << 4)) =
                        make_int4((int)pk[4 * c], (int)pk[4 * c + 1], (int)pk[4 * c + 2], (int)pk[4 * c + 3]);
                reinterpret_cast<int*>(stg + 2048)[lane] = valid ? (int)(cell * 4 + cls) : -1;      // 64-byte units of act1
            }
            __syncwarp();
#pragma unroll
            for (int i2 = 0; i2 < 4; ++i2) {
                const int R = (lane >> 2) + 8 * i2, c = lane & 3;
                const int unit = reinterpret_cast<const int*>(stg + 2048)[R];
                const int4 v = *reinterpret_cast<const int4*>(stg + R * 64 + ((((uint32_t)c) ^ ((uint32_t)(R >> 1) & 3u)) << 4));
                if (unit >= 0 && !(DBG & 1)) *reinterpret_cast<int4*>(reinterpret_cast<uint8_t*>(p.out) + (int64_t)unit * 64 + c * 16) = v;
            }
            __syncwarp();
        }
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_d, TMEM_COLS);
}

// ------------------------------------------------------------------------------------ conv1 weight gradient (uint8 frames -> TMEM)
// dW[tap, c, co] = sum_p X[p + off_tap, c] * dY[p, co] over the grid positions p of an image, off = {0, 1, 21, 22}
// (taps (dy, dx) of the 2x2 window on the 21-wide grid).  Written over k = p + s_b with s_b = {0, 21}:
//       D_b[(h, c), co] = sum_k X[k + h, c] * dY[k - s_b, co],    tap = 2 b + h.
//   A  (tensor memory, 128 lanes x 64 columns per step of 128 grid rows k): lanes 0-63 hold channel c of the pixel
//       stream X[k], lanes 64-127 the same stream one pixel later (h = 1).  ONE tile per step serves all four taps.
//   B  (shared memory, MN-major SWIZZLE_64B, N = 32): the dY rows of the step, rows [k0, k0 + 128) for b = 0 and rows
//       [k0 - 21, k0 + 107) for b = 1.  The stages form one contiguous ring, so the b = 1 operand is the same tile with its
//       descriptor start moved 21 rows back into the previous stage (the swizzle is a function of the address bits:
//       tools/experiments/umma_mnshift_test.cu); stage 0 is preceded by a 24-row pad that receives the previous rows by a
//       second small TMA box.  Negative rows and rows >= 441 are zero-filled by the TMA unit: images are independent and
//       occupy 512-row slots, and a CTA owns whole images.
//   X  : channel-major frames [img][64 ch][448 rows] u8, staged in blocks of 128 positions (SWIZZLE_128B boxes of 64 full
//        lines; 16-byte reads of 32 consecutive channel rows are bank-conflict free through the swizzle).  The h = 1 stream
//        needs one pixel of the next block.
//   dY : d(act1) on the 21x21 grid, fp16 [img][441][32] scaled by 2^12 (written by conv2's data gradient with a
//        saturating conversion); rows of invalid positions (x = 20 or y = 20) are zero.
//   Sixteen convert warps (two sets alternating steps; lane quadrant = warp % 4, K half) read their channel's bytes with 16-byte loads, expand
//   uint8 -> fp16 with one PRMT per two pixels (bytes (x, 0x64) = fp16 1024 + x; the offset is taken out again through the
//   bias partial) -- the h = 1 warps first funnel-shift by one byte -- and tcgen05.st 32 columns into tensor memory.
//   Two issuer warps (one per tap group b) run tcgen05.mma with A in TMEM; four more warps accumulate the bias gradient
//   (column sums of dY) from the staged tiles and drain the accumulators at the end.  Partial tiles go to
//   ws[cta][256][64] / wsb[cta][64] (first 32 columns used; row = tap * 64 + c) and are folded in fixed order by tc_fold_win.
//
// Round-2 history: the first version kept the shift on the A side (four tap tiles = 128 TMEM columns per step, written by
// the convert warps as two shifted copies) with three A buffers.  Stage knock-outs (tools/conv1_knockout.py, compile-time
// instantiations) showed 1150 cycles per step against an HBM floor of 625: 540 cycles of pure barrier hand-shake
// (convert -> issuer -> tcgen05.commit -> convert, only three steps in flight), 330 of conversion ALU and 150 of
// tcgen05.st/ld.shared, added up rather than overlapped.  Moving the shift to the B side halves the conversions and the
// tensor-memory writes and leaves room for six A buffers.
struct Conv1WgradU8Params {
    const int64_t* rows;       // optional image gather (minibatch rows of the rollout)
    int n;                     // images of the minibatch
    int64_t rows_per_cta;      // multiple of 512 grid rows = whole images (M = n * 512)
    float* ws;
    float* wsb;
};
// X blocks (8 KB: 64 channels x 128 positions) and dY steps (8 KB) in flight: 210 KB per SM; the gather reads need ~3 us
// of loads in flight to cover their latency.
constexpr int kC1WXStages = 12, kC1WYStages = 14;
constexpr int kC1WBlock = 64 * 128, kC1WYBytes = 128 * 64, kC1WYPadRows = 24, kC1WYPad = kC1WYPadRows * 64;
constexpr int kC1WShift = 21;                     // grid rows between the two tap groups
constexpr float kDact1Scale = 4096.0f;

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}
// 2 NH pixels (NH / 2 words starting at byte offset B of W[0]) -> NH fp16 pairs H with value 1024 + x (bytes (x, 0x64) are the
// fp16 1024 + x exactly); the 1024 is NOT removed here: sum_k (1024 + x) dY = dW + 1024 sum_k dY, and sum_k dY is the bias
// partial the same CTA computes anyway, so the drain subtracts 1024 x it (fp32; the offset costs < 1e-5 relative accuracy).
template <int B, int NH>
__device__ __forceinline__ void u8_to_f16_biased(const uint32_t* W, uint32_t (&H)[NH]) {
#pragma unroll
    for (int j = 0; j < NH / 2; ++j) {
        uint32_t x = W[j];
        if (B == 1) x = prmt(W[j], W[j + 1], 0x4321u);
        if (B == 2) x = prmt(W[j], W[j + 1], 0x5432u);
        if (B == 3) x = prmt(W[j], W[j + 1], 0x6543u);
        H[2 * j] = prmt(x, 0x64646464u, 0x5140u);
        H[2 * j + 1] = prmt(x, 0x64646464u, 0x7362u);
    }
}
constexpr float kU8Bias = 1024.0f;

constexpr int kC1WConvWarps = 16;                // two sets of eight: set s converts the steps it = s (mod 2)
constexpr int kC1WThreads = (4 + kC1WConvWarps + 4 + 2) * 32;     // + two more MMA issuer warps
// DBG (stage knock-outs, tools/conv1_knockout.py): 1 = no uint8 -> fp16 conversion, 2 = no TMA, 4 = no MMAs, 8 = no bias
// sums, 16 = no tcgen05.st, 32 = no shared-memory loads; results are then garbage by construction.  The product is DBG = 0.
template <int DBG>
__global__ void __launch_bounds__(kC1WThreads, 1) tc_conv1_wgrad_u8(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmY,
                                                                  const __grid_constant__ CUtensorMap tmYpad, const Conv1WgradU8Params p) {
    constexpr int XS = kC1WXStages, YS = kC1WYStages;
    constexpr int NA = 6;                                 // A-operand buffers in TMEM (64 columns each)
    constexpr uint32_t TMEM_COLS = 512, COL_D = 0, COL_A = 128;         // 4 accumulator tiles of 32 columns; COL_A + NA * 64 = 512
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t xfull[XS], xempty[XS], yfull[YS], yempty[YS], a_full[NA], a_empty[NA], done_bar;
    __shared__ uint32_t tmem_base_smem;
    __shared__ float sRed[32 * 32], sBias[32];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sX = smem;                                 // XS blocks of 8 KB
    uint8_t* sYpad = smem + (size_t)XS * kC1WBlock;     // 24 rows in front of stage 0 (the ring's wrap-around halo)
    uint8_t* sYb = sYpad + kC1WYPad;                    // YS stages of 8 KB, contiguous
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) {
        // one arrival per warp GROUP (a set of eight convert warps, the four dY warps): the groups synchronise internally
        // with named barriers and one thread talks to the mbarriers
        for (int s = 0; s < XS; ++s) { mbar_init(&xfull[s], 1); mbar_init(&xempty[s], 2); }
        for (int s = 0; s < YS; ++s) { mbar_init(&yfull[s], 1); mbar_init(&yempty[s], 2 + 1); }
        for (int b = 0; b < NA; ++b) { mbar_init(&a_full[b], 1); mbar_init(&a_empty[b], 2); }
        mbar_init(&done_bar, 4);
        fence_barrier_init();
        tma_prefetch_desc(&tmX);
        tma_prefetch_desc(&tmY);
        tma_prefetch_desc(&tmYpad);
    }
    if (warp == 3) tmem_alloc(&tmem_base_smem, TMEM_COLS);
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem0 = tmem_base_smem;
    const int64_t M = (int64_t)p.n * 512;
    const int64_t m_begin = (int64_t)blockIdx.x * p.rows_per_cta;
    int64_t m_end = m_begin + p.rows_per_cta;
    if (m_end > M) m_end = M;
    const int nsteps = m_end > m_begin ? (int)((m_end - m_begin) >> 7) : 0;
    const int64_t g0 = m_begin >> 7;                       // first global step (4 steps per image)

    if (warp == 0) {
        // ======================= TMA producer 1: X block k (k = 0 .. nsteps, the last one only feeds the one-pixel halo).
        // Two producer threads: one thread's step is a serial chain too (gather index, mbarrier wait ~90 cycles, expect_tx,
        // bulk-tensor issue); with X and dY in one thread it was the step period once the convert warps alternated.
        if (lane == 0 && nsteps > 0) {
            auto image_of = [&](int64_t g) -> int {
                int64_t img = g >> 2;
                if (img >= p.n) img = p.n - 1;             // the halo block after the very last step: any mapped block will do
                return p.rows ? (int)__ldg(p.rows + img) : (int)img;
            };
            // the gather index is fetched one IMAGE (four steps) ahead: a load per step sat on this thread's critical path
            int z = image_of(g0), z_next = image_of(g0 + 4);        // g0 is image-aligned (whole images per CTA)
            for (int k = 0; k <= nsteps; ++k) {
                const int64_t g = g0 + k;
                if (k > 0 && (g & 3) == 0) { z = z_next; z_next = image_of(g + 4); }
                const int xs = k % XS;
                if (k >= XS) mbar_wait(&xempty[xs], ((k / XS) - 1) & 1);
                if (DBG & 2) mbar_arrive(&xfull[xs]);
                else {
                    mbar_arrive_expect_tx(&xfull[xs], (uint32_t)kC1WBlock);
                    tma_load_3d(smem_u32(sX + (size_t)xs * kC1WBlock), &tmX, (int)(g & 3) * 128, 0, z, &xfull[xs]);
                }
            }
        }
    } else if (warp == 3) {
        // ======================= TMA producer 2: the dY rows of step k.  The tail of stage s is read by step k + 1 (b = 1), so
        // stage s is reloaded (step k + YS) once step k + 1 has been consumed: the ring is YS - 1 steps deep.
        if (lane == 0) {
            for (int k = 0; k < nsteps; ++k) {
                const int64_t g = g0 + k;
                const int ys = k % YS;
                // stage ys was read by step k - YS (its own rows, both tap groups) and by step k - YS + 1 (its tail, b = 1): the
                // two steps belong to different issuer warps (step parity), so BOTH must have been consumed before the reload
                if (k >= YS) mbar_wait2(&yempty[ys], ((k / YS) - 1) & 1, &yempty[(k + 1) % YS], ((k - YS + 1) / YS) & 1);
                if (DBG & 2) mbar_arrive(&yfull[ys]);
                else {
                    mbar_arrive_expect_tx(&yfull[ys], (uint32_t)(kC1WYBytes + (ys == 0 ? kC1WYPad : 0)));
                    tma_load_3d(smem_u32(sYb + (size_t)ys * kC1WYBytes), &tmY, 0, (int)(g & 3) * 128, (int)(g >> 2), &yfull[ys]);
                    if (ys == 0) tma_load_3d(smem_u32(sYpad), &tmYpad, 0, (int)(g & 3) * 128 - kC1WYPadRows, (int)(g >> 2), &yfull[ys]);
                }
            }
        }
        __syncwarp();
    } else if (warp == 1 || warp == 2 || warp >= 4 + kC1WConvWarps + 4) {
        // ======================= MMA issuers: tap group b, step parity par; 8 K-steps of 16 rows per step, A from TMEM.
        // An issuer's step is a serial chain as well (two mbarrier waits, eight descriptor/issue sequences, two commits:
        // ~480 cycles, the kernel's period with every stage knocked out), so each tap group has two issuers that alternate
        // steps into their OWN accumulator tiles (summed in the drain: the accumulation order stays fixed).
        const int b = warp <= 2 ? warp - 1 : warp - (4 + kC1WConvWarps + 4);
        const int par = warp <= 2 ? 0 : 1;
        const bool leader = elect_one();
        constexpr uint32_t idesc = make_idesc_f16ts(128, 32, 0, 1);
        const uint64_t desc_hi = desc_mnmajor_sw64(0) & 0xFFFFFFFF00000000ull;
        const uint32_t desc_lo_flags = (uint32_t)(desc_mnmajor_sw64(0) & 0xFFFFFFFFull);
        const uint32_t d_col = tmem0 + COL_D + (uint32_t)((par * 2 + b) * 32);
        for (int it = par; it < nsteps; it += 2) {
            const int ys = it % YS, buf = it % NA;
            // The b = 1 operand starts 21 rows back, inside the PREVIOUS stage (or the halo in front of stage 0, which arrives
            // with stage 0's own transaction count).  That stage belongs to step it - 1, whose bulk copy is tracked by a
            // barrier only the other parity's issuers wait on -- and bulk copies issued in order may COMPLETE out of order.
            // Without this wait the tail could be read before its copy had landed: stale rows, and on the first pass over the
            // ring never-written shared memory (non-finite fp16 bit patterns -> NaN gradients for the dy = 1 taps, seen once
            // in ~20 bench iterations).  All polls of the step go out together.
            {
                const bool need_prev = (b == 1) && ys != 0;
                const int ps = need_prev ? ys - 1 : ys;
                const uint32_t pph = need_prev ? (uint32_t)(((it - 1) / YS) & 1) : (uint32_t)((it / YS) & 1);
                const bool p_ok = mbar_try_wait(&yfull[ps], pph);
                mbar_wait2(&yfull[ys], (it / YS) & 1, &a_full[buf], (it / NA) & 1);
                if (!p_ok) mbar_wait(&yfull[ps], pph);
            }
            tc_fence_after_sync();
            if (leader) {
                const uint32_t y_lo = ((smem_u32(sYb + (size_t)ys * kC1WYBytes - (size_t)(b * kC1WShift * 64)) & 0x3FFFFu) >> 4) | desc_lo_flags;
                const uint32_t a_col = tmem0 + COL_A + (uint32_t)(buf * 64);
#pragma unroll
                for (int kk = 0; kk < 8; ++kk) {
                    if (DBG & 4) break;
                    umma_f16_ts(d_col, a_col + 8 * kk, desc_hi | (uint64_t)(y_lo + 64 * kk), idesc, (it != par || kk != 0) ? 1u : 0u);
                }
                umma_commit(&yempty[ys]);
                umma_commit(&a_empty[buf]);
            }
            __syncwarp();
        }
        if (leader) umma_commit(&done_bar);
        __syncwarp();
    } else if (warp >= 4 && warp < 4 + kC1WConvWarps) {
        // ======================= convert warps: uint8 channel rows -> fp16 pairs -> tensor memory.
        // A warp's step is a serial chain -- three mbarrier waits (~90 cycles each even when already complete), the 16-byte
        // loads, ~50 PRMTs, tcgen05.st + wait::st, two arrives: ~1000 cycles, and with one set of eight warps that chain WAS
        // the step period (knock-outs: 520 cycles per step with every stage switched off).  Two sets alternate steps.
        const int q = warp & 3, kh = ((warp - 4) >> 2) & 1, set = (warp - 4) >> 3;
        const int h = q >> 1;                               // pixel stream: X[k] (lanes 0-63) or X[k + 1] (lanes 64-127)
        const int c = (q & 1) * 32 + lane;
        const uint32_t lane_base = tmem0 + COL_A + ((uint32_t)(q * 32) << 16) + (uint32_t)(kh * 32);
        const int chunk0 = kh * 4;                          // first 16-byte chunk of this K half (64 pixels)
        constexpr int NCH = 5;                              // + one chunk for the h = 1 stream's last pixel
        const uint32_t row_off = (uint32_t)c * 128u, sw = (uint32_t)(c & 7);
        const bool set_leader = ((warp - 4) & 7) == 0;
        for (int it = set; it < nsteps; it += 2) {
            const int xm = it % XS, xh = (it + 1) % XS, buf = it % NA;
            if (set_leader) {                                  // all three polls of the step go out together
                const bool a_free = it < NA || mbar_try_wait(&a_empty[buf], ((it / NA) - 1) & 1);
                mbar_wait2(&xfull[xm], (it / XS) & 1, &xfull[xh], ((it + 1) / XS) & 1);
                if (!a_free) mbar_wait(&a_empty[buf], ((it / NA) - 1) & 1);
            }
            if (set == 0) asm volatile("bar.sync 2, 256;" ::: "memory"); else asm volatile("bar.sync 3, 256;" ::: "memory");
            const uint8_t* bm = sX + (size_t)xm * kC1WBlock + row_off;
            const uint8_t* bh = sX + (size_t)xh * kC1WBlock + row_off;
            uint32_t W[4 * NCH];
#pragma unroll
            for (int v = 0; v < NCH; ++v) {
                if (DBG & 32) { W[4 * v] = W[4 * v + 1] = W[4 * v + 2] = W[4 * v + 3] = (uint32_t)(it + v); continue; }
                const int ci = chunk0 + v;
                const uint8_t* src = (ci < 8 ? bm : bh) + ((((uint32_t)ci & 7u) ^ sw) << 4);
                const int4 t = *reinterpret_cast<const int4*>(src);
                W[4 * v] = (uint32_t)t.x; W[4 * v + 1] = (uint32_t)t.y; W[4 * v + 2] = (uint32_t)t.z; W[4 * v + 3] = (uint32_t)t.w;
            }
            uint32_t H[32];
            if (DBG & 1) {
#pragma unroll
                for (int m = 0; m < 32; ++m) H[m] = W[m % (4 * NCH)];
            } else if (h == 0) u8_to_f16_biased<0, 32>(W, H); else u8_to_f16_biased<1, 32>(W, H);
            tc_fence_after_sync();
            if (!(DBG & 16)) tmem_st32(lane_base + (uint32_t)(buf * 64), H);
            else if (H[0] == 0x12345u && H[31] == 0x54321u) mbar_arrive(&a_full[buf]);     // keep the values alive
            tmem_st_wait();
            tc_fence_before_sync();
            if (set == 0) asm volatile("bar.sync 2, 256;" ::: "memory"); else asm volatile("bar.sync 3, 256;" ::: "memory");
            // block k is read as the main block of step k and as the halo of step k - 1 (the other set): two arrivals release
            // it; block 0 has no halo reader, so its main readers arrive twice
            if (set_leader && lane == 0) {
                mbar_arrive(&xempty[xm]);
                if (it == 0) mbar_arrive(&xempty[xm]);
                mbar_arrive(&xempty[xh]);
                mbar_arrive(&a_full[buf]);
            }
        }
    } else if (warp >= 4 + kC1WConvWarps && warp < 4 + kC1WConvWarps + 4) {
        // ======================= dY warps: bias gradient = column sums of dY from the staged tiles (fp32, fixed order)
        const int tb = tid - (4 + kC1WConvWarps) * 32;
        const int rq = tb >> 2, c16 = tb & 3;
        float bsum[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) bsum[e] = 0.f;
        for (int it = 0; it < nsteps; ++it) {
            const int ys = it % YS;
            if (tb < 32) mbar_wait(&yfull[ys], (it / YS) & 1);
            asm volatile("bar.sync 1, 128;" ::: "memory");
            const uint8_t* sY = sYb + (size_t)ys * kC1WYBytes;          // the step's own rows
#pragma unroll
            for (int ps = 0; ps < 4; ++ps) {
                if (DBG & 8) break;
                const int rr = ps * 32 + rq;
                const int4 v = *reinterpret_cast<const int4*>(sY + img64_off(rr, c16));
                const uint32_t w[4] = {(uint32_t)v.x, (uint32_t)v.y, (uint32_t)v.z, (uint32_t)v.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&w[e]));
                    bsum[2 * e] += f.x;
                    bsum[2 * e + 1] += f.y;
                }
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (tb == 0) mbar_arrive(&yempty[ys]);
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) sRed[rq * 32 + c16 * 8 + e] = bsum[e];
        asm volatile("bar.sync 1, 128;" ::: "memory");
        if (tb < 32) {
            float t = 0.f;
#pragma unroll
            for (int l = 0; l < 32; ++l) t += sRed[l * 32 + tb];
            p.wsb[(int64_t)blockIdx.x * 64 + tb] = t;
            // what the 1024 offset of every pixel added to each (tap, c) row: the CTA owns whole images, so the rows of the
            // b = 1 operand (shifted by 21, zero outside the image) sum to the same value as the rows of the b = 0 operand
            sBias[tb] = t * kU8Bias;
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        // drain the two accumulator tiles
        if (nsteps > 0) {
            mbar_wait(&done_bar, 0);
            tc_fence_after_sync();
        }
        const int lrow = (warp & 3) * 32 + lane;
        float* wsc = p.ws + (int64_t)blockIdx.x * 256 * 64;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const uint32_t taddr = tmem0 + COL_D + (uint32_t)(j * 32) + ((uint32_t)((warp & 3) * 32) << 16);
            float4* dst = reinterpret_cast<float4*>(wsc + (int64_t)(j * 128 + lrow) * 64);
#pragma unroll
            for (int hc = 0; hc < 2; ++hc) {                     // 16 columns at a time (register budget of the 832-thread CTA)
                uint32_t v[16], v2[16];
#pragma unroll
                for (int e = 0; e < 16; ++e) v[e] = v2[e] = 0u;
                if (nsteps > 0) tmem_ld16(taddr + hc * 16, v);
                if (nsteps > 1) tmem_ld16(taddr + 64 + hc * 16, v2);     // the odd steps' accumulator of the same tap group
                if (nsteps > 0) tmem_ld_wait();
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int c0 = hc * 16 + 4 * e;
                    dst[hc * 4 + e] = make_float4(__uint_as_float(v[4 * e]) + __uint_as_float(v2[4 * e]) - sBias[c0],
                                                  __uint_as_float(v[4 * e + 1]) + __uint_as_float(v2[4 * e + 1]) - sBias[c0 + 1],
                                                  __uint_as_float(v[4 * e + 2]) + __uint_as_float(v2[4 * e + 2]) - sBias[c0 + 2],
                                                  __uint_as_float(v[4 * e + 3]) + __uint_as_float(v2[4 * e + 3]) - sBias[c0 + 3]);
                }
            }
        }
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 3) tmem_dealloc(tmem0, TMEM_COLS);
}

static int launch_conv1_wgrad_u8(const Conv1WgradU8Params& p, const void* frames_cm, int64_t n_images, const void* dact1_f16, int ctas,
                                 cudaStream_t s, const char* what) {
    const size_t smem = (size_t)kC1WXStages * kC1WBlock + kC1WYPad + (size_t)kC1WYStages * kC1WYBytes + 1024;
    int rc;
    if (p.rows_per_cta % 512 != 0) return fail(B200RL_ERR_INVALID_ARGUMENT, "%s: a CTA must own whole images (512 grid rows)", what);
    CUtensorMap tmX, tmY, tmYpad;
    memset(&tmX, 0, sizeof(tmX)); memset(&tmY, 0, sizeof(tmY)); memset(&tmYpad, 0, sizeof(tmYpad));
    // frames [img][64 ch][448 positions] u8: box = [64 ch][128 positions], SWIZZLE_128B; dY [img][441 rows][32 co] fp16 = 64-byte
    // rows: box [128 rows][64 B], SWIZZLE_64B
    if ((rc = make_tmap_3d_u8(&tmX, frames_cm, n_images, 64, 448, 448, 64, 128, what))) return rc;
    if ((rc = make_tmap_3d_u8(&tmY, dact1_f16, p.n, 441, 64, 64, 128, 64, what))) return rc;
    if ((rc = make_tmap_3d_u8(&tmYpad, dact1_f16, p.n, 441, 64, 64, kC1WYPadRows, 64, what))) return rc;
    // stage knock-outs (tools/conv1_knockout.py) are separate instantiations: flags tested at run time inside the convert
    // loop cost the product kernel 20 % (measured)
    static const int dbg = getenv("B200RL_DBG_CONV1W") ? atoi(getenv("B200RL_DBG_CONV1W")) : 0;
#define B200RL_C1W_CASE(D)                                                                  \
    case D: {                                                                               \
        static SmemAttrCache attr;                                                          \
        if ((rc = attr.ensure(tc_conv1_wgrad_u8<D>, smem, what))) return rc;                \
        tc_conv1_wgrad_u8<D><<<ctas, kC1WThreads, smem, s>>>(tmX, tmY, tmYpad, p);                  \
        break;                                                                              \
    }
    switch (dbg) {
        B200RL_C1W_CASE(0) B200RL_C1W_CASE(1) B200RL_C1W_CASE(2) B200RL_C1W_CASE(4) B200RL_C1W_CASE(8) B200RL_C1W_CASE(16)
        B200RL_C1W_CASE(32) B200RL_C1W_CASE(15) B200RL_C1W_CASE(63)
        default: return fail(B200RL_ERR_INVALID_ARGUMENT, "%s: no knock-out instantiation %d", what, dbg);
    }
#undef B200RL_C1W_CASE
    return check_launch(what);
}

constexpr int kConv1I8Stages = 8;
static int launch_conv1_i8(const Conv1U8Params& p, const void* frames_rm, cudaStream_t s, const char* what) {
    constexpr int STAGES = kConv1I8Stages;
    const size_t smem = (size_t)4 * 64 * 64 + (size_t)STAGES * 144 * 128 + 16 * 2304 + 1024;
    const int total = p.n * 2;                     // 2 tiles of 128 pair rows (256 grid positions) per image (441 used)
    static const int dbg = getenv("B200RL_DBG_CONV1") ? atoi(getenv("B200RL_DBG_CONV1")) : 0;
    int grid = num_sms();
    if (grid > total) grid = total;
    CUtensorMap tmA;
    memset(&tmA, 0, sizeof(tmA));
    // the row-major image [441][64 B] viewed as 221 pair rows of 128 B (image stride 28 224 B = 220.5 rows: the second
    // half of row 220 belongs to the next image and only ever feeds invalid positions); SWIZZLE_128B boxes of 144 rows
    int rc = make_tmap_pairs_u8(&tmA, frames_rm, p.n_images, what);
    if (rc) return rc;
#define B200RL_C1F_CASE(D)                                                                  \
    case D: {                                                                               \
        static SmemAttrCache attr;                                                          \
        if ((rc = attr.ensure(tc_conv1_i8<STAGES, D>, smem, what))) return rc;              \
        tc_conv1_i8<STAGES, D><<<grid, kConvWinThreads, smem, s>>>(tmA, p, total);          \
        break;                                                                              \
    }
    switch (dbg) {
        B200RL_C1F_CASE(0) B200RL_C1F_CASE(1) B200RL_C1F_CASE(2) B200RL_C1F_CASE(4) B200RL_C1F_CASE(3) B200RL_C1F_CASE(6)
        B200RL_C1F_CASE(7) B200RL_C1F_CASE(8) B200RL_C1F_CASE(12) B200RL_C1F_CASE(15)
        default: return fail(B200RL_ERR_INVALID_ARGUMENT, "%s: no knock-out instantiation %d", what, dbg);
    }
#undef B200RL_C1F_CASE
    return check_launch(what);
}

}  // namespace b200rl
