// tcgen05 "window" convolution kernel + launcher (see net_tc.cu for the layer plan).
#pragma once
#include "tc_base.cuh"

namespace b200rl {
using namespace tc;

// ------------------------------------------------------------------ kernel 1c: "window" convolution
// Stride-1 convolutions over activations stored as a LINEAR pixel grid [n*G rows, CPR*64 channels]
// (G = Hp*Wp grid positions per image).  GEMM rows enumerate grid positions, so tap (dy,dx) of a row is
// simply the row `dy*Wp+dx` further down: the CTA stages ONE window of 128+maxshift rows per tile and
// every tap is a tcgen05 operand descriptor whose start address is shifted by whole 128-byte rows
// (the SWIZZLE_128B pattern is a function of the shared-memory address bits, so any row shift is legal:
// tools/experiments/umma_shift_test.cu).  Each activation row is therefore read from L2 once per tile
// instead of once per tap, and the producers do no im2col index arithmetic at all.  Grid positions whose
// window would leave the image (X >= vW or Y >= vH) are computed but not stored.
enum { WOUT_DENSE = 0, WOUT_S2D2 = 1, WOUT_DACT2 = 2, WOUT_DACT1 = 3 };
struct WinParams {
    const bf16* A;           // [n*G, CPR*64]
    const int64_t* rows;     // optional image gather (conv1 reads the rollout through mb_inds)
    int64_t M;               // n*G
    int n, G, Wp;
    // image-aligned tiling (conv1): every image owns 2^tpi_shift tiles of 128 grid rows (rows >= G are padding),
    // so a window never spans two images and the minibatch gather is just the TMA box's image coordinate.
    // 0 = tiles walk the linear grid [n*G] (activations produced by this library, always contiguous).
    int tpi_shift;
    int64_t n_images;        // images addressable through `rows` (size of the tensor map's outer dimension)
    int ntaps;
    int shift[16];           // dy*Wp + dx per tap (non-negative)
    int WR;                  // window rows: 128 + max shift, rounded up to 8
    const bf16* Bw;          // packed weights [N][ntaps*CPR*64]
    int N;
    int vH, vW;              // valid outputs: Y < vH && X < vW
    int out_mode;
    bf16* out;               // primary output
    bf16* out2;              // WOUT_DACT2: padded 11x11 copy
    // ReLU masks travel as BITS (1 = the forward activation was > 0), one 32-bit word per 32 channels, in the row
    // order of the tensor they describe: 16x fewer bytes than re-reading the bf16 activation
    const uint32_t* mask_bits;   // input mask (data-gradient kernels): words of the row this thread writes
    uint32_t* mask_out;          // output mask (forward kernels with relu)
    const float* bias;
    float scale;
    int relu;
    int out_f16;             // store fp16 (saturating) instead of bf16: d(act1) feeding the uint8 conv1 weight gradient
};

__device__ __forceinline__ uint32_t pack_f16x2_sat(float lo, float hi) {
    uint32_t d;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}

// Epilogue arithmetic of the forward window convolutions, shared by tc_conv_win and the fused rollout tower
// (tc_rollout_tower.cuh): 32 fp32 accumulators of one row -> acc * scale + bias (bias: 32 floats, global memory) ...
__device__ __forceinline__ void win_scale_bias32(uint32_t (&v)[32], const float* bias, float scale) {
    const float4* bp = reinterpret_cast<const float4*>(bias);
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        const float4 bv = __ldg(bp + e);
        v[4 * e] = __float_as_uint(fmaf(__uint_as_float(v[4 * e]), scale, bv.x));
        v[4 * e + 1] = __float_as_uint(fmaf(__uint_as_float(v[4 * e + 1]), scale, bv.y));
        v[4 * e + 2] = __float_as_uint(fmaf(__uint_as_float(v[4 * e + 2]), scale, bv.z));
        v[4 * e + 3] = __float_as_uint(fmaf(__uint_as_float(v[4 * e + 3]), scale, bv.w));
    }
}
// ... -> ReLU folded into the bf16 conversion, 64 bytes of output row.
__device__ __forceinline__ void win_pack_relu32(const uint32_t (&v)[32], int4 (&w)[4]) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        w[e].x = (int)pack_bf16x2_relu(__uint_as_float(v[8 * e]), __uint_as_float(v[8 * e + 1]));
        w[e].y = (int)pack_bf16x2_relu(__uint_as_float(v[8 * e + 2]), __uint_as_float(v[8 * e + 3]));
        w[e].z = (int)pack_bf16x2_relu(__uint_as_float(v[8 * e + 4]), __uint_as_float(v[8 * e + 5]));
        w[e].w = (int)pack_bf16x2_relu(__uint_as_float(v[8 * e + 6]), __uint_as_float(v[8 * e + 7]));
    }
}

// Thread roles (576 threads): warp 0 = TMA producer; warp 1 = MMA issuer; warps 2-17 = FOUR epilogue groups of four warps
// (one warp per TMEM lane quadrant).  Group h owns accumulator buffer h and drains tiles h, h + 4, ...
// Why four groups: an epilogue warp runs a ~250-500 instruction dependent chain per tile (tcgen05.ld, scale/bias, ReLU
// mask, bf16 packing, stores); with two groups every scheduler held two such warps and ncu showed 0.2-0.4 instructions per
// cycle and scheduler with the tensor pipe at 25-45 % -- the epilogue's LATENCY was the tile period.  Four warps per scheduler
// hide it.  Measured and dropped: a second MMA-issuer warp (no gain: the issuing thread is not the limit).
constexpr int kConvWinThreads = 576;                     // the widest instance (4 groups); see conv_win_groups
// N = 128 tiles (conv2 data gradient) keep two groups: their epilogue holds 4 x 32 accumulator columns per row and was
// measured 10 % slower with four groups (register pressure at 576 threads); the narrower kernels gain 0-12 %.
__host__ __device__ constexpr int conv_win_groups(int BN) { return BN >= 128 ? 2 : 4; }
__host__ __device__ constexpr int conv_win_threads(int BN) { return 64 + conv_win_groups(BN) * 128; }
__host__ __device__ constexpr int conv_win_acc_bufs(int BN) { return BN <= 128 ? 4 : 2; }
template <int BN, int CPR, int STAGES, int NTAPS>
__global__ void __launch_bounds__(conv_win_threads(BN), 1) tc_conv_win(const __grid_constant__ CUtensorMap tmA, const WinParams p,
                                                      int total_tiles) {
    constexpr int B_CHUNK = BN * 128;
    constexpr int NB = conv_win_acc_bufs(BN);
    constexpr int NG = conv_win_groups(BN);
    static_assert(NB % NG == 0, "every epilogue group owns NB / NG accumulator buffers");
    constexpr uint32_t TMEM_COLS = (NB * BN) < 32 ? 32 : NB * BN;
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint64_t full_bar[STAGES], empty_bar[STAGES], tfull_bar[NB], tempty_bar[NB];
    __shared__ uint32_t tmem_base_smem;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int tid = threadIdx.x, warp = tid >> 5;
    const int nchunks = p.ntaps * CPR;
    const int K = nchunks * 64;
    const int IMG = p.WR * 128;                 // one 64-channel column image of the window
    const int STAGE_BYTES = IMG * CPR;
    uint8_t* sW = smem;
    uint8_t* sRing = smem + (size_t)nchunks * B_CHUNK;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
        for (int a = 0; a < NB; ++a) { mbar_init(&tfull_bar[a], 1); mbar_init(&tempty_bar[a], 4); }
        fence_barrier_init();
        tma_prefetch_desc(&tmA);
    }
    if (warp == 1) tmem_alloc(&tmem_base_smem, TMEM_COLS);
    for (int idx = tid; idx < nchunks * BN * 8; idx += blockDim.x) {
        const int c16 = idx & 7;
        int t = idx >> 3;
        const int r = t % BN; const int j = t / BN;
        int4 v = make_int4(0, 0, 0, 0);
        if (r < p.N) v = ldg16(p.Bw + (int64_t)r * K + j * 64 + c16 * 8);
        *reinterpret_cast<int4*>(sW + (size_t)j * B_CHUNK + img_off(r, c16)) = v;
    }
    fence_proxy_async_smem();
    tc_fence_before_sync();
    __syncthreads();
    tc_fence_after_sync();
    const uint32_t tmem_d = tmem_base_smem;
    // each CTA walks a CONTIGUOUS range of tiles: with the minibatch gather every image (3-4 tiles) is then
    // touched by one SM only (TLB / L2 locality), and the image indices of tile+1 can be prefetched
    const int tile_begin = (int)(((int64_t)total_tiles * blockIdx.x) / gridDim.x);
    const int tile_end = (int)(((int64_t)total_tiles * (blockIdx.x + 1)) / gridDim.x);

    if (warp == 0) {
        // ======================= TMA producer: the window is one rectangular box per 64-channel column chunk ====
        if (tid == 0) {
            uint32_t q = 0;
            const int tmask = (1 << p.tpi_shift) - 1;
            // image-aligned mode: the box's image coordinate is the (optional) minibatch gather; the index of the
            // NEXT tile's image is fetched one tile ahead so the dependent load never delays a TMA issue
            int z_next = 0;
            if (p.tpi_shift && tile_begin < tile_end) {
                const int img = tile_begin >> p.tpi_shift;
                z_next = p.rows ? (int)__ldg(p.rows + img) : img;
            }
            for (int tile = tile_begin; tile < tile_end; ++tile, ++q) {
                const uint32_t s = q % STAGES;
                const int z = z_next;
                if (p.tpi_shift && tile + 1 < tile_end) {
                    const int img = (tile + 1) >> p.tpi_shift;
                    z_next = p.rows ? (int)__ldg(p.rows + img) : img;
                }
                if (q >= (uint32_t)STAGES) mbar_wait(&empty_bar[s], ((q / STAGES) - 1) & 1);
                const uint32_t dst = smem_u32(sRing + (size_t)s * STAGE_BYTES);
                mbar_arrive_expect_tx(&full_bar[s], (uint32_t)STAGE_BYTES);
                if (p.tpi_shift) {
#pragma unroll
                    for (int c = 0; c < CPR; ++c) tma_load_3d(dst + c * IMG, &tmA, c * 64, (tile & tmask) * 128, z, &full_bar[s]);
                } else {
#pragma unroll
                    for (int c = 0; c < CPR; ++c) tma_load_2d(dst + c * IMG, &tmA, c * 64, tile * 128, &full_bar[s]);
                }
            }
        }
    } else if (warp == 1) {
        // ======================= MMA issuer: the WHOLE warp walks the tile loop (uniform control flow keeps the
        // descriptor arithmetic in uniform registers), one elected lane issues.  Descriptors differ from a per-stage /
        // per-tap base only in their 14-bit start-address field, so each MMA costs two 32-bit adds.
        const bool leader = elect_one();
        constexpr uint32_t idesc = make_idesc(128, BN, 0, 0);
        const uint64_t desc_hi = desc_kmajor(0) & 0xFFFFFFFF00000000ull;
        const uint32_t desc_lo_flags = (uint32_t)(desc_kmajor(0) & 0xFFFFFFFFull);       // LBO field
        const uint32_t w_lo = ((smem_u32(sW) & 0x3FFFFu) >> 4) | desc_lo_flags;
        for (uint32_t q = 0; (int)q < tile_end - tile_begin; ++q) {
            const uint32_t acc = q % NB, s = q % STAGES;
            if (q >= (uint32_t)NB) mbar_wait(&tempty_bar[acc], ((q / NB) - 1) & 1);
            mbar_wait(&full_bar[s], (q / STAGES) & 1);
            tc_fence_after_sync();
            if (leader) {
                const uint32_t d_addr = tmem_d + acc * BN;
                const uint32_t win_lo = ((smem_u32(sRing + (size_t)s * STAGE_BYTES) & 0x3FFFFu) >> 4) | desc_lo_flags;
#pragma unroll
                for (int t = 0; t < NTAPS; ++t) {
#pragma unroll
                    for (int c = 0; c < CPR; ++c) {
                        const uint32_t a_lo = win_lo + (uint32_t)((c * IMG) >> 4) + (uint32_t)p.shift[t] * 8u;
                        const uint32_t b_lo = w_lo + (uint32_t)(((t * CPR + c) * B_CHUNK) >> 4);
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk)
                            umma_bf16(d_addr, desc_hi | (uint64_t)(a_lo + 2 * kk), desc_hi | (uint64_t)(b_lo + 2 * kk), idesc,
                                      (t | c | kk) != 0 ? 1u : 0u);
                    }
                }
                umma_commit(&empty_bar[s]);
                umma_commit(&tfull_bar[acc]);
            }
            __syncwarp();
        }
    } else {
        // ======================= epilogue: warps 2-17 = two groups of four (one warp per TMEM lane quadrant).
        // Group h owns accumulator buffer h, i.e. every other tile of the CTA's range, and handles ALL BN columns
        // of its rows: the row -> (image, Y, X) -> output offset arithmetic is paid once per tile and thread, and
        // is incremental (a tile step is 256 grid rows; Y = rem / Wp by multiply-shift, exact for G*Wp < 65536).
        const int ew = warp & 3;
        const int h = (warp - 2) >> 2;                       // epilogue group 0..3
        const int lrow = ew * 32 + (tid & 31);
        const uint32_t mW = (65536u + (uint32_t)p.Wp - 1u) / (uint32_t)p.Wp;
        constexpr int TSTEP = NG * 128;                      // grid rows between two tiles of one group
        const int step_i = TSTEP / p.G, step_rem = TSTEP % p.G;
        int64_t r = ((int64_t)tile_begin + h) * 128 + lrow;      // linear-grid mode state (unused when image-aligned)
        int i_lin = (int)(r / p.G);
        int rem_lin = (int)(r - (int64_t)i_lin * p.G);
        const int tmask = (1 << p.tpi_shift) - 1;
        const uint32_t lane_base = tmem_d + ((uint32_t)(ew * 32) << 16);
        constexpr int NW = BN / 32;                          // 32-column groups = mask words per row
        uint32_t k = 0;                                      // tiles this group has drained
        for (int tile = tile_begin + h; tile < tile_end; tile += NG, ++k) {
            const uint32_t acc = (uint32_t)(tile - tile_begin) % NB;           // group h drains buffers h, h + NG, ...
            const uint32_t lane_addr = lane_base + acc * BN;
            int i = i_lin, rem = rem_lin;
            bool inside = r < p.M;
            if (p.tpi_shift) {                               // image-aligned tiles: rows >= G of an image are padding
                i = tile >> p.tpi_shift;
                rem = ((tile & tmask) << 7) + lrow;
                inside = rem < p.G;
            }
            const int Y = (int)(((uint32_t)rem * mW) >> 16), X = rem - Y * p.Wp;
            const bool valid = inside && (Y < p.vH) && (X < p.vW);
            int64_t o1 = 0, o2 = 0, ob = 0;
            if (p.out_mode == WOUT_DENSE) {
                const int64_t orow = ((int64_t)i * p.vH + Y) * p.vW + X;
                o1 = orow * p.N; ob = orow * (p.N >> 5);
            } else if (p.out_mode == WOUT_S2D2) {
                const int64_t cell = ((int64_t)i * 10 + (Y >> 1)) * 10 + (X >> 1);
                const int cls = (Y & 1) * 2 + (X & 1);
                o1 = cell * 128 + cls * 32; ob = cell * 4 + cls;
            } else if (p.out_mode == WOUT_DACT2) {
                o1 = ((int64_t)i * 100 + Y * 10 + X) * 64;                 // 10-grid linear (conv2 wgrad)
                o2 = ((int64_t)i * 121 + (Y + 1) * 11 + (X + 1)) * 64;     // zero-padded 11x11 (conv2 dgrad)
                ob = ((int64_t)i * 81 + Y * 9 + X) * 2;                    // act2 mask words
            } else {
                ob = ((int64_t)i * 100 + Y * 10 + X) * 4;                  // act1 (2x2 cells) mask words
            }
            // the row's mask words are requested BEFORE waiting for the accumulator (latency overlaps the MMAs)
            uint32_t mb[NW];
#pragma unroll
            for (int g = 0; g < NW; ++g) mb[g] = 0xFFFFFFFFu;
            if (p.mask_bits != nullptr && valid) {
                if (NW == 4) {
                    const int4 t = ldg16(p.mask_bits + ob);
                    mb[0] = (uint32_t)t.x; mb[1 % NW] = (uint32_t)t.y; mb[2 % NW] = (uint32_t)t.z; mb[3 % NW] = (uint32_t)t.w;
                } else if (NW == 2) {
                    const uint2 t = __ldg(reinterpret_cast<const uint2*>(p.mask_bits + ob));
                    mb[0] = t.x; mb[1 % NW] = t.y;
                } else {
                    mb[0] = __ldg(p.mask_bits + ob);
                }
            }
            mbar_wait(&tfull_bar[acc], ((uint32_t)(tile - tile_begin) / NB) & 1);
            tc_fence_after_sync();
#pragma unroll
            for (int g = 0; g < NW; ++g) {
                uint32_t v[32];
                tmem_ld32(lane_addr + g * 32, v);
                tmem_ld_wait();
                if (g == NW - 1) {             // accumulator drained: hand the buffer back before the global stores
                    tc_fence_before_sync();
                    __syncwarp();
                    if ((tid & 31) == 0) mbar_arrive(&tempty_bar[acc]);
                }
                if (!valid || g * 32 >= p.N) continue;
                if (p.bias) {
                    win_scale_bias32(v, p.bias + g * 32, p.scale);
                } else {
#pragma unroll
                    for (int e = 0; e < 32; ++e) v[e] = __float_as_uint(__uint_as_float(v[e]) * p.scale);
                }
                if (p.relu) {
                    uint32_t bits = 0u;
#pragma unroll
                    for (int e = 0; e < 32; ++e) {
                        const float f = __uint_as_float(v[e]);
                        bits |= (f > 0.f ? 1u : 0u) << e;           // the clamp itself is folded into the bf16 conversion below
                    }
                    if (p.mask_out) p.mask_out[ob + g] = bits;
                }
                if (p.mask_bits) {
#pragma unroll
                    for (int e = 0; e < 32; ++e) if (!((mb[g] >> e) & 1u)) v[e] = 0u;
                }
                int4 w[4];
                if (p.out_f16) {
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        w[e].x = (int)pack_f16x2_sat(__uint_as_float(v[8 * e]), __uint_as_float(v[8 * e + 1]));
                        w[e].y = (int)pack_f16x2_sat(__uint_as_float(v[8 * e + 2]), __uint_as_float(v[8 * e + 3]));
                        w[e].z = (int)pack_f16x2_sat(__uint_as_float(v[8 * e + 4]), __uint_as_float(v[8 * e + 5]));
                        w[e].w = (int)pack_f16x2_sat(__uint_as_float(v[8 * e + 6]), __uint_as_float(v[8 * e + 7]));
                    }
                } else if (p.relu) {
                    win_pack_relu32(v, w);
                } else {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    w[e].x = (int)pack_bf16x2(__uint_as_float(v[8 * e]), __uint_as_float(v[8 * e + 1]));
                    w[e].y = (int)pack_bf16x2(__uint_as_float(v[8 * e + 2]), __uint_as_float(v[8 * e + 3]));
                    w[e].z = (int)pack_bf16x2(__uint_as_float(v[8 * e + 4]), __uint_as_float(v[8 * e + 5]));
                    w[e].w = (int)pack_bf16x2(__uint_as_float(v[8 * e + 6]), __uint_as_float(v[8 * e + 7]));
                }
                }
                // Stores: a lane owns one output row, so every store instruction of the warp touches 32 different lines = 32 L1
                // wavefronts; on the N = 128 conv2 data gradient they were ~70 % of the tile period.  256-bit stores halve
                // the instructions (conv2 data gradient 338 -> 288 us, conv3 data gradient 308 -> 256, conv2 forward -5 %).
                // Measured against it: coalescing through a shared-memory tile (4 or 8 lanes per row) -- conv3 data gradient 263,
                // conv2 forward equal, conv3 forward +5 %, conv2 data gradient +18..23 % (extra warp syncs in a latency-bound
                // epilogue) -- so the direct form stays.
                bf16* dst;
                if (p.out_mode == WOUT_DACT1) {
                    // column group g = (py,px) of the cell -> input pixel (2Y+py, 2X+px) of the 21-grid, 32 channels
                    dst = p.out + ((int64_t)i * 441 + (2 * Y + (g >> 1)) * 21 + 2 * X + (g & 1)) * 32;
                } else {
                    dst = p.out + o1 + g * 32;
                }
                st_global_256(dst, w[0], w[1]);
                st_global_256(dst + 16, w[2], w[3]);
                if (p.out_mode == WOUT_DACT2) {
                    bf16* dst2 = p.out2 + o2 + g * 32;
                    st_global_256(dst2, w[0], w[1]);
                    st_global_256(dst2 + 16, w[2], w[3]);
                }
            }
            r += TSTEP; i_lin += step_i; rem_lin += step_rem;
            if (rem_lin >= p.G) { rem_lin -= p.G; ++i_lin; }
        }
    }
    tc_fence_before_sync();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_d, TMEM_COLS);
}

template <int BN, int CPR, int STAGES, int NTAPS>
static int launch_conv_win(const WinParams& p, cudaStream_t s, const char* what) {
    if (p.ntaps != NTAPS) return fail(B200RL_ERR_INVALID_ARGUMENT, "%s: %d taps, kernel instance has %d", what, p.ntaps, NTAPS);
    const size_t smem = (size_t)p.ntaps * CPR * BN * 128 + (size_t)STAGES * p.WR * 128 * CPR + 1024;
    static SmemAttrCache attr;
    if (int rc = attr.ensure(tc_conv_win<BN, CPR, STAGES, NTAPS>, smem, what)) return rc;
    if ((int64_t)p.G * p.Wp >= 65536 || p.G < 1 || p.N % 32 != 0)
        return fail(B200RL_ERR_INVALID_ARGUMENT, "%s: grid %d x width %d outside the epilogue's multiply-shift range, or N %% 32 != 0", what, p.G, p.Wp);
    if (p.rows && !p.tpi_shift) return fail(B200RL_ERR_INVALID_ARGUMENT, "%s: the image gather needs image-aligned tiling", what);
    if (p.tpi_shift && (128 << p.tpi_shift) < p.G) return fail(B200RL_ERR_INVALID_ARGUMENT, "%s: tiles per image too small", what);
    const int total = p.tpi_shift ? (int)((int64_t)p.n << p.tpi_shift) : (int)ceil_div(p.M, 128);
    int grid = num_sms();
    if (grid > total) grid = total;
    CUtensorMap tmA;
    memset(&tmA, 0, sizeof(tmA));
    int rc;
    // the window is a TMA box [WR rows x 64 channels] per column chunk: of the linear grid, or of one image
    if (p.tpi_shift) rc = make_tmap_3d(&tmA, p.A, p.n_images, p.G, (int64_t)CPR * 64, p.WR, what);
    else rc = make_tmap_2d(&tmA, p.A, p.M, (int64_t)CPR * 64, p.WR, what);
    if (rc) return rc;
    tc_conv_win<BN, CPR, STAGES, NTAPS><<<grid, conv_win_threads(BN), smem, s>>>(tmA, p, total);
    return check_launch(what);
}

}  // namespace b200rl
