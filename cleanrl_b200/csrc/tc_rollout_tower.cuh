// Rollout conv tower: conv1 -> conv2 -> conv3 of the bf16 NatureCNN for one env step, one persistent kernel.
//
// The rollout evaluates the policy once per env step at n = 1024 (or a group / chunk of it).  As three kernels, every
// conv paid its own fixed cost (barrier set-up, TMEM allocation, staging its weights, filling and draining a pipeline of
// 3-7 tiles per CTA) and act1 / act2 made a round trip through HBM that nothing else reads: the update recomputes its own
// activations.  Here each CTA takes a contiguous range of whole images and runs the three convolutions per image with
// act1 and act2 held only in shared memory; act3 (bf16 [n,49,64], dense) goes to the workspace the fc GEMM reads.  No
// ReLU masks are written (no backward pass reads the rollout's activations).
//
// Same instructions, same bits: conv1 issues tc_conv1_i8's kind::i8 MMAs (pair rows, even / odd accumulators, two limbs),
// conv2 / conv3 the bf16 MMAs of tc_conv_win<64,2,..,4> / <64,1,..,9> in the same tap / chunk / K order, and the
// epilogues call the same arithmetic (conv1_i8_epilogue, win_scale_bias32, win_pack_relu32).  Which tile covers an output
// row does not change its bits, so act3 equals the three-kernel chain's exactly.
//
// Input, by template parameter:
//   RAW = true   uint8 NCHW frames [n,4,84,84].  Four converter warps build the space-to-depth pixels in registers, write
//                both rollout orientations (row-major [n,441,64], channel-major [n,64,448] with rows 441..447 zero, what
//                tc_frames_to_s2d_u8 writes) and the frame's pair rows into shared memory for conv1.  Image i+1's bytes are
//                loaded while image i computes.
//   RAW = false  the row-major slot is already written (frame-stack delta upload): one TMA box of 224 pair rows per image.
//
// Warp roles (576 threads): 0 = conv2 / conv3 MMA issuer, 1 = conv1 MMA issuer, 2-9 = conv1 epilogue (two groups of four
// warps, one per 128-pair-row tile), 10-13 = conv2 + conv3 epilogues, 14-17 = frame producer (RAW: converters; else one
// TMA thread).  The two issuers commit to their own barriers; tcgen05.commit tracks the issuing thread's MMAs only.
#pragma once
#include "tc_base.cuh"
#include "tc_conv_win.cuh"
#include "tc_conv1_u8.cuh"

namespace b200rl {
using namespace tc;

struct TowerParams {
    const uint8_t* frames;   // RAW: uint8 [n,4,84,84]
    uint8_t* slot_rm;        // RAW: written [n,441,64]; else read through the tensor map
    uint8_t* slot_cm;        // RAW: written [n,64,448]
    int n;
    const int8_t* limbs;     // conv1 limbs [64][256] s8 (tc_pack_conv1_i8)
    const float* sc;         // conv1 column scales [64]
    const float* b1;         // conv1 bias [32]
    const bf16* w2;          // conv2 packed [64][4 taps * 128]
    const float* b2;
    const bf16* w3;          // conv3 packed [64][9 taps * 64]
    const float* b3;
    bf16* act3;              // [n,49,64]
};

// Shared-memory layout (offsets from the 1024-aligned base; every operand image starts on a 1024-byte boundary, which the
// SWIZZLE_128B / SWIZZLE_64B address patterns require).  Windows are sized to what VALID outputs read:
//   conv1's largest valid tap reaches pair row 220, conv2's cell row 88 + 11 = 99, conv3's row 60 + 20 = 80.
// The row-shifted descriptors of the discarded rows (tile rows past the image) read further, and those reads must stay
// inside the allocation, so the buffers are ordered such that each overrun lands in the next one:
//   frame (224 rows) -> tile 1 reads pair rows up to 128 + 127 + 11 = 266: 42 rows into act1;
//   act1 column image 1 (104 rows) -> rows up to 127 + 11 = 138: 35 rows into act2;
//   act2 (88 rows) -> rows up to 127 + 20 = 147: 60 rows (7.5 KB) into the conv1 limbs (16 KB) that follow.
// What they read there only ever reaches discarded rows.
constexpr int kTwFrameRows = 224, kTwAct1Rows = 104, kTwAct2Rows = 88;
constexpr int kTwFrame = 0;
constexpr int kTwAct1 = kTwFrame + kTwFrameRows * 128;            // 2 column images (channels 0-63, 64-127) of the 10x10 cells
constexpr int kTwAct1Img = kTwAct1Rows * 128;
constexpr int kTwAct2 = kTwAct1 + 2 * kTwAct1Img;                  // [81 (88) rows][64 ch]
constexpr int kTwW1 = kTwAct2 + kTwAct2Rows * 128;                 // conv1 limbs: 4 taps x 64 rows x 64 B (SWIZZLE_64B)
constexpr int kTwW2 = kTwW1 + 4 * 4096;                            // conv2: 8 chunks x 64 rows x 128 B
constexpr int kTwW3 = kTwW2 + 8 * 8192;                            // conv3: 9 chunks x 64 rows x 128 B
constexpr int kTwSmemBytes = kTwW3 + 9 * 8192;
constexpr size_t kTwSmemAlloc = (size_t)kTwSmemBytes + 1024;
static_assert(kTwAct1 % 1024 == 0 && kTwAct1Img % 1024 == 0 && kTwAct2 % 1024 == 0 && kTwW1 % 1024 == 0 && kTwW2 % 1024 == 0 &&
              kTwW3 % 1024 == 0, "operand images must be 1024-byte aligned");
static_assert(266 * 128 + 128 <= kTwAct1 + kTwAct1Img, "conv1 overrun must stay inside act1");
static_assert(kTwAct1 + kTwAct1Img + 139 * 128 <= kTwAct2 + kTwAct2Rows * 128, "conv2 overrun must stay inside act2");
static_assert(kTwAct2 + 148 * 128 <= kTwW2, "conv3 overrun must stay inside the conv1 limbs");
static_assert(kTwSmemAlloc <= 227 * 1024, "tower exceeds the 227 KB of shared memory per block");
constexpr int kTwThreads = 18 * 32;
// TMEM columns: conv1 accumulators (tile, parity) x 64 at 0..255, conv2 at 256, conv3 at 320
constexpr uint32_t kTwTmemCols = 512, kTwAcc2 = 256, kTwAcc3 = 320;

template <bool RAW>
__global__ void __launch_bounds__(kTwThreads, 1) tc_rollout_tower(const __grid_constant__ CUtensorMap tmF, const TowerParams p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t fr_full, fr_empty, acc1_full, acc1_empty, a1_full, a1_empty, acc2_full, acc2_empty, a2_full, a2_empty,
        acc3_full, acc3_empty;
    __shared__ uint32_t tmem_base_smem;
    __shared__ __align__(16) float s_sc[32], s_bias[32];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint8_t* sFrame = smem + kTwFrame;
    uint8_t* sAct1 = smem + kTwAct1;
    uint8_t* sAct2 = smem + kTwAct2;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    if (tid == 0) {
        mbar_init(&fr_full, 1); mbar_init(&fr_empty, 1);
        mbar_init(&acc1_full, 1); mbar_init(&acc1_empty, 8);
        mbar_init(&a1_full, 8); mbar_init(&a1_empty, 1);
        mbar_init(&acc2_full, 1); mbar_init(&acc2_empty, 4);
        mbar_init(&a2_full, 4); mbar_init(&a2_empty, 1);
        mbar_init(&acc3_full, 1); mbar_init(&acc3_empty, 4);
        fence_barrier_init();
        if (!RAW) tma_prefetch_desc(&tmF);
    }
    if (warp == 1) tmem_alloc(&tmem_base_smem, kTwTmemCols);
    // resident weights: conv1 limbs (tc_conv1_i8's image), conv2 / conv3 (tc_conv_win's chunk images).  9 728 16-byte chunks,
    // 17 per thread: the loads of a batch are issued together (one L2 round trip per batch instead of one per chunk)
    {
        constexpr int kC1 = 4 * 64 * 4, kC2 = 8 * 64 * 8, kC3 = 9 * 64 * 8, kAll = kC1 + kC2 + kC3, kBatch = 8;
        for (int base = 0; base < kAll; base += kBatch * kTwThreads) {
            int4 v[kBatch];
            uint32_t dst[kBatch];
#pragma unroll
            for (int u = 0; u < kBatch; ++u) {
                const int idx = base + u * kTwThreads + tid;
                dst[u] = 0xFFFFFFFFu;
                if (idx < kC1) {
                    const int c16 = idx & 3, t = (idx >> 2) & 3, r = idx >> 4;
                    dst[u] = kTwW1 + t * 4096 + img64_off(r, c16);
                    v[u] = ldg16(p.limbs + r * 256 + t * 64 + c16 * 16);
                } else if (idx < kC1 + kC2) {
                    const int i = idx - kC1, c16 = i & 7, t = i >> 3, r = t % 64, j = t / 64;
                    dst[u] = kTwW2 + j * 8192 + img_off(r, c16);
                    v[u] = ldg16(p.w2 + (int64_t)r * 512 + j * 64 + c16 * 8);
                } else if (idx < kAll) {
                    const int i = idx - kC1 - kC2, c16 = i & 7, t = i >> 3, r = t % 64, j = t / 64;
                    dst[u] = kTwW3 + j * 8192 + img_off(r, c16);
                    v[u] = ldg16(p.w3 + (int64_t)r * 576 + j * 64 + c16 * 8);
                }
            }
#pragma unroll
            for (int u = 0; u < kBatch; ++u)
                if (dst[u] != 0xFFFFFFFFu) *reinterpret_cast<int4*>(smem + dst[u]) = v[u];
        }
    }
    // frame rows 221..223 and the second half of pair row 220 (position 441) are never written by the converters
    if (RAW)
        for (int idx = tid; idx < 4 * 8; idx += blockDim.x) {
            const int r = 220 + (idx >> 3), c16 = idx & 7;
            if (r > 220 || c16 >= 4) *reinterpret_cast<int4*>(sFrame + img_off(r, c16)) = make_int4(0, 0, 0, 0);
        }
    if (tid < 32) { s_sc[tid] = p.sc[32 + tid]; s_bias[tid] = p.b1[tid]; }
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem = tmem_base_smem;
    const int img0 = (int)(((int64_t)p.n * blockIdx.x) / gridDim.x);
    const int cnt = (int)(((int64_t)p.n * (blockIdx.x + 1)) / gridDim.x) - img0;

    if (warp == 1) {
        // ======================= conv1 issuer: per image, tile tp (pair rows 128 tp ..) x parity e, 4 taps x 2 K-steps
        const bool leader = elect_one();
        constexpr uint32_t idesc = make_idesc_i8(128, 64);
        const uint64_t a_hi = desc_kmajor(0) & 0xFFFFFFFF00000000ull;
        const uint32_t a_flags = (uint32_t)(desc_kmajor(0) & 0xFFFFFFFFull);
        const uint64_t b_hi = desc_kmajor_sw64(0) & 0xFFFFFFFF00000000ull;
        const uint32_t b_flags = (uint32_t)(desc_kmajor_sw64(0) & 0xFFFFFFFFull);
        const uint32_t w_lo = ((smem_u32(smem + kTwW1) & 0x3FFFFu) >> 4) | b_flags;
        constexpr int off[4] = {0, 1, 21, 22};
        for (int k = 0; k < cnt; ++k) {
            mbar_wait(&fr_full, k & 1);
            if (k > 0) mbar_wait(&acc1_empty, (k - 1) & 1);
            tc_fence_after_sync();
            if (leader) {
#pragma unroll
                for (int tp = 0; tp < 2; ++tp) {
                    const uint32_t win_lo = ((smem_u32(sFrame + tp * 128 * 128) & 0x3FFFFu) >> 4) | a_flags;
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const uint32_t d_addr = tmem + (uint32_t)(2 * tp + e) * 64;
#pragma unroll
                        for (int t = 0; t < 4; ++t) {
                            const int po = e + off[t];
                            const uint32_t a_lo = win_lo + (uint32_t)((po >> 1) * 8 + (po & 1) * 4);
                            const uint32_t b_lo = w_lo + (uint32_t)((t * 4096) >> 4);
#pragma unroll
                            for (int kk = 0; kk < 2; ++kk)
                                umma_i8(d_addr, a_hi | (uint64_t)(a_lo + 2 * kk), b_hi | (uint64_t)(b_lo + 2 * kk), idesc,
                                        (t | kk) != 0 ? 1u : 0u);
                        }
                    }
                }
                umma_commit(&fr_empty);
                umma_commit(&acc1_full);
            }
            __syncwarp();
        }
    } else if (warp == 0) {
        // ======================= conv2 / conv3 issuer (tc_conv_win's loop: taps, then column chunks, then K-steps of 16)
        const bool leader = elect_one();
        constexpr uint32_t idesc = make_idesc(128, 64, 0, 0);
        const uint64_t desc_hi = desc_kmajor(0) & 0xFFFFFFFF00000000ull;
        const uint32_t flags = (uint32_t)(desc_kmajor(0) & 0xFFFFFFFFull);
        const uint32_t a1_lo = ((smem_u32(sAct1) & 0x3FFFFu) >> 4) | flags;
        const uint32_t a2_lo = ((smem_u32(sAct2) & 0x3FFFFu) >> 4) | flags;
        const uint32_t w2_lo = ((smem_u32(smem + kTwW2) & 0x3FFFFu) >> 4) | flags;
        const uint32_t w3_lo = ((smem_u32(smem + kTwW3) & 0x3FFFFu) >> 4) | flags;
        constexpr int sh2[4] = {0, 1, 10, 11};
        for (int k = 0; k < cnt; ++k) {
            mbar_wait(&a1_full, k & 1);
            if (k > 0) mbar_wait(&acc2_empty, (k - 1) & 1);
            tc_fence_after_sync();
            if (leader) {
#pragma unroll
                for (int t = 0; t < 4; ++t) {
#pragma unroll
                    for (int c = 0; c < 2; ++c) {
                        const uint32_t a_lo = a1_lo + (uint32_t)((c * kTwAct1Img) >> 4) + (uint32_t)sh2[t] * 8u;
                        const uint32_t b_lo = w2_lo + (uint32_t)(((t * 2 + c) * 8192) >> 4);
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk)
                            umma_bf16(tmem + kTwAcc2, desc_hi | (uint64_t)(a_lo + 2 * kk), desc_hi | (uint64_t)(b_lo + 2 * kk), idesc,
                                      (t | c | kk) != 0 ? 1u : 0u);
                    }
                }
                umma_commit(&a1_empty);
                umma_commit(&acc2_full);
            }
            __syncwarp();
            mbar_wait(&a2_full, k & 1);
            if (k > 0) mbar_wait(&acc3_empty, (k - 1) & 1);
            tc_fence_after_sync();
            if (leader) {
#pragma unroll
                for (int t = 0; t < 9; ++t) {
                    const uint32_t a_lo = a2_lo + (uint32_t)((t / 3) * 9 + (t % 3)) * 8u;
                    const uint32_t b_lo = w3_lo + (uint32_t)((t * 8192) >> 4);
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        umma_bf16(tmem + kTwAcc3, desc_hi | (uint64_t)(a_lo + 2 * kk), desc_hi | (uint64_t)(b_lo + 2 * kk), idesc,
                                  (t | kk) != 0 ? 1u : 0u);
                }
                umma_commit(&a2_empty);
                umma_commit(&acc3_full);
            }
            __syncwarp();
        }
    } else if (warp < 10) {
        // ======================= conv1 epilogue: group tp drains the two parity accumulators of tile tp; lane = pair row
        const int ew = warp & 3, tp = (warp - 2) >> 2;
        const int lrow = ew * 32 + lane;
        const uint32_t lane_base = tmem + ((uint32_t)(ew * 32) << 16);
        for (int k = 0; k < cnt; ++k) {
            mbar_wait(&acc1_full, k & 1);
            if (k > 0) mbar_wait(&a1_empty, (k - 1) & 1);       // conv2 of the previous image has read act1
            tc_fence_after_sync();
#pragma unroll 1
            for (int e = 0; e < 2; ++e) {
                uint32_t a1[32], a2[32];
                const uint32_t lane_addr = lane_base + (uint32_t)(2 * tp + e) * 64;
                tmem_ld32(lane_addr, a1);
                tmem_ld32(lane_addr + 32, a2);
                tmem_ld_wait();
                if (e == 1) {
                    tc_fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc1_empty);
                }
                const int rem = 2 * ((tp << 7) + lrow) + e;
                const int Y = (rem * 3121) >> 16, X = rem - Y * 21;          // rem / 21 for rem < 512
                if (rem < 441 && Y < 20 && X < 20) {
                    uint32_t pk[16];
                    conv1_i8_epilogue(a1, a2, s_sc, s_bias, pk);
                    // act1 as 2x2 cells: position (Y, X) -> cell row, channels cls*32 .. of the 128 = column image cls / 2,
                    // 16-byte chunks (cls & 1) * 4 .. + 3 of the row
                    const int cell = (Y >> 1) * 10 + (X >> 1), cls = (Y & 1) * 2 + (X & 1);
                    uint8_t* row = sAct1 + (cls >> 1) * kTwAct1Img;
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        *reinterpret_cast<int4*>(row + img_off(cell, (cls & 1) * 4 + j)) =
                            make_int4((int)pk[4 * j], (int)pk[4 * j + 1], (int)pk[4 * j + 2], (int)pk[4 * j + 3]);
                }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&a1_full);
        }
    } else if (warp < 14) {
        // ======================= conv2 epilogue -> act2 (shared), conv3 epilogue -> act3 (global); lane = grid row
        const int ew = warp & 3;
        const int m = ew * 32 + lane;
        const uint32_t lane_addr = tmem + ((uint32_t)(ew * 32) << 16);
        const int Y2 = m / 10, X2 = m - Y2 * 10;
        const bool v2 = m < 100 && Y2 < 9 && X2 < 9;
        const int Y3 = m / 9, X3 = m - Y3 * 9;
        const bool v3 = m < 81 && Y3 < 7 && X3 < 7;
        for (int k = 0; k < cnt; ++k) {
            mbar_wait(&acc2_full, k & 1);
            if (k > 0) mbar_wait(&a2_empty, (k - 1) & 1);       // conv3 of the previous image has read act2
            tc_fence_after_sync();
#pragma unroll 1
            for (int g = 0; g < 2; ++g) {
                uint32_t v[32];
                tmem_ld32(lane_addr + kTwAcc2 + g * 32, v);
                tmem_ld_wait();
                if (g == 1) {
                    tc_fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc2_empty);
                }
                if (!v2) continue;
                win_scale_bias32(v, p.b2 + g * 32, 1.0f);
                int4 w[4];
                win_pack_relu32(v, w);
                const int r = Y2 * 9 + X2;
#pragma unroll
                for (int j = 0; j < 4; ++j) *reinterpret_cast<int4*>(sAct2 + img_off(r, g * 4 + j)) = w[j];
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(&a2_full);
            mbar_wait(&acc3_full, k & 1);
            tc_fence_after_sync();
            const int64_t img = img0 + k;
#pragma unroll 1
            for (int g = 0; g < 2; ++g) {
                uint32_t v[32];
                tmem_ld32(lane_addr + kTwAcc3 + g * 32, v);
                tmem_ld_wait();
                if (g == 1) {
                    tc_fence_before_sync();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc3_empty);
                }
                if (!v3) continue;
                win_scale_bias32(v, p.b3 + g * 32, 1.0f);
                int4 w[4];
                win_pack_relu32(v, w);
                bf16* dst = p.act3 + ((img * 7 + Y3) * 7 + X3) * 64 + g * 32;
                st_global_256(dst, w[0], w[1]);
                st_global_256(dst + 16, w[2], w[3]);
            }
        }
    } else if (RAW) {
        // ======================= converters (warps 14-17): item = (4 consecutive grid positions q4, colour plane c).  One
        // item is 16 source words (4 positions x 4 pixel rows of 4 bytes) = four 16-byte row-major chunks, and, transposed
        // as 4x4 bytes per pixel row, the 16 channel-major words (channel c*16 + sy*4 + sx, positions 4 q4 .. 4 q4 + 3).
        const int ct = tid - 14 * 32;                            // 0..127
        constexpr int kItems = 112 * 4, kPer = kItems / 128 + 1;  // 448 items, <= 4 per thread
        for (int k = 0; k < cnt; ++k) {
            const int64_t img = img0 + k;
            const uint8_t* src = p.frames + img * 28224;
            uint32_t W[kPer][16];
#pragma unroll
            for (int j = 0; j < kPer; ++j) {
                const int it = ct + 128 * j;
                const int c = it & 3, q4 = it >> 2;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int pos = q4 * 4 + e;
                    const int Y = (pos * 3121) >> 16, X = pos - Y * 21;
                    const bool ok = it < kItems && pos < 441;
                    const uint32_t* w = reinterpret_cast<const uint32_t*>(src + c * 7056 + (Y * 4) * 84 + X * 4);
#pragma unroll
                    for (int sy = 0; sy < 4; ++sy) W[j][e * 4 + sy] = ok ? __ldg(w + sy * 21) : 0u;
                }
            }
#pragma unroll
            for (int j = 0; j < kPer; ++j) {
                const int it = ct + 128 * j;
                if (it >= kItems) continue;
                const int c = it & 3, q4 = it >> 2;
                // channel-major: word (sy, sx) = byte sx of pixel row sy of the 4 positions
                uint32_t* cm = reinterpret_cast<uint32_t*>(p.slot_cm + (img * 64 + c * 16) * 448) + q4;
#pragma unroll
                for (int sy = 0; sy < 4; ++sy) {
                    const uint32_t lo = prmt(W[j][sy], W[j][4 + sy], 0x5140u), hi = prmt(W[j][8 + sy], W[j][12 + sy], 0x5140u);
                    const uint32_t lo2 = prmt(W[j][sy], W[j][4 + sy], 0x7362u), hi2 = prmt(W[j][8 + sy], W[j][12 + sy], 0x7362u);
                    cm[(sy * 4 + 0) * 112] = prmt(lo, hi, 0x5410u);
                    cm[(sy * 4 + 1) * 112] = prmt(lo, hi, 0x7632u);
                    cm[(sy * 4 + 2) * 112] = prmt(lo2, hi2, 0x5410u);
                    cm[(sy * 4 + 3) * 112] = prmt(lo2, hi2, 0x7632u);
                }
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int pos = q4 * 4 + e;
                    if (pos >= 441) continue;
                    *reinterpret_cast<int4*>(p.slot_rm + (img * 441 + pos) * 64 + c * 16) =
                        make_int4((int)W[j][e * 4], (int)W[j][e * 4 + 1], (int)W[j][e * 4 + 2], (int)W[j][e * 4 + 3]);
                }
            }
            if (k > 0) mbar_wait(&fr_empty, (k - 1) & 1);         // conv1 of the previous image has read the frame
#pragma unroll
            for (int j = 0; j < kPer; ++j) {
                const int it = ct + 128 * j;
                if (it >= kItems) continue;
                const int c = it & 3, q4 = it >> 2;
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int pos = q4 * 4 + e;
                    if (pos >= 441) continue;
                    const int q = pos >> 1;
                    *reinterpret_cast<int4*>(sFrame + img_off(q, (pos & 1) * 4 + c)) =
                        make_int4((int)W[j][e * 4], (int)W[j][e * 4 + 1], (int)W[j][e * 4 + 2], (int)W[j][e * 4 + 3]);
                }
            }
            fence_proxy_async_smem();
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (ct == 0) mbar_arrive(&fr_full);
        }
    } else if (warp == 14) {
        // ======================= TMA producer: the stored slot's 221 pair rows (+3 zero-filled) per image
        if (lane == 0) {
            for (int k = 0; k < cnt; ++k) {
                if (k > 0) mbar_wait(&fr_empty, (k - 1) & 1);
                mbar_arrive_expect_tx(&fr_full, (uint32_t)(kTwFrameRows * 128));
                tma_load_3d(smem_u32(sFrame), &tmF, 0, 0, img0 + k, &fr_full);
            }
        }
        __syncwarp();
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, kTwTmemCols);
}

static int launch_rollout_tower(const TowerParams& p, cudaStream_t s, const char* what) {
    int grid = num_sms();
    if (grid > p.n) grid = p.n;
    CUtensorMap tmF;
    memset(&tmF, 0, sizeof(tmF));
    int rc;
    if (p.frames) {
        static SmemAttrCache attr;
        if ((rc = attr.ensure(tc_rollout_tower<true>, kTwSmemAlloc, what))) return rc;
        tc_rollout_tower<true><<<grid, kTwThreads, kTwSmemAlloc, s>>>(tmF, p);
    } else {
        if ((rc = make_tmap_pairs_u8(&tmF, p.slot_rm, p.n, what, kTwFrameRows))) return rc;
        static SmemAttrCache attr;
        if ((rc = attr.ensure(tc_rollout_tower<false>, kTwSmemAlloc, what))) return rc;
        tc_rollout_tower<false><<<grid, kTwThreads, kTwSmemAlloc, s>>>(tmF, p);
    }
    return check_launch(what);
}

}  // namespace b200rl
