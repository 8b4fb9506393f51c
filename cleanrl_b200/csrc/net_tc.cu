// NatureCNN on the 5th-gen tensor cores (tcgen05.mma, accumulators in TMEM), bf16 operands,
// fp32 accumulation.  Reference network: cleanrl/ppo_atari_envpool.py:123-139.
//
// Data layout in HBM (all activations are LINEAR PIXEL GRIDS: row = grid position, 128 bytes = 64 channels)
//   frames   bf16 [n, 21x21, 64]   space-to-depth(4) of the uint8 frames: channel = c*16 + sy*4 + sx of source
//                                  pixel (4Y+sy, 4X+sx); written once per env step (tc_frames_to_s2d), 0..255 is
//                                  exact in bf16 and the /255 of ppo_atari_envpool.py:144 is applied to the fp32
//                                  accumulator.  conv1 (8x8 s4) = 2x2 stride-1 conv on this grid.
//   act1     bf16 [n, 10x10, 128]  conv1 output as 2x2 cells (space-to-depth(2)): conv2 (4x4 s2) = 2x2 stride-1.
//   act2     bf16 [n,  9x9,  64]   act3 bf16 [n, 7x7, 64]   hidden bf16 [n, 512]
//   gradients of act3 / act2 are written twice by their producer: on the consumer-weight-gradient's grid
//   (zeros at positions that are not valid outputs) and zero-padded for the data-gradient's "full" correlation;
//   d(act1) lives on the 21x21 grid with 32 channels.  Never-written positions rely on a zero-initialised
//   workspace.  The minibatch gather b_obs[mb_inds] (ppo.py:250, 3.7 GB fp32 per minibatch in the reference)
//   is an image-index indirection inside the conv1 kernels.
//
// Kernels
//   tc_conv_win<BN,CPR,STAGES,NTAPS>   stride-1 "window" convolution (conv1/2/3 forward, conv3/conv2 data-gradient):
//       GEMM rows enumerate grid positions, so tap (dy,dx) of row r is row r + dy*Wp + dx.  A persistent CTA
//       stages ONE window of 128+maxshift rows per tile as a TMA box (cp.async.bulk.tensor; for conv1 a 3-D box
//       whose image coordinate is the minibatch gather) and every tap is a UMMA descriptor whose start address is
//       shifted by whole 128-byte rows (legal for SWIZZLE_128B: the pattern is a function of the smem address
//       bits; tools/experiments/umma_shift_test.cu).  Weights stay resident in smem.  Warp 0 = TMA producer, warp 1 issues tcgen05.mma
//       (warp-uniform loop, elected lane); warps 2-9 = two epilogue groups that own alternate tiles and drain
//       double-buffered accumulators; ReLU masks are exchanged between forward and backward as bits.
//   tc_wgrad_win                 conv weight gradients: dW^T[(tap,c), co] = sum_r X[r+shift_tap, c] * dY[r, co]; the same
//       row images are read as MN-major operands (rows = reduction index), taps again by row shifts; the bias
//       gradient (column sums of dY) is accumulated by the four dY warps from the staged tiles.
//   tc_gemm_tma<BN,STAGES>       fc forward / data-gradient: both operands are TMA boxes of row-major matrices.
//   tc_wgrad_tma                 fc weight gradient (MN-major views of TMA-loaded dhid / act3 row boxes).
//   tc_heads_*                   the A+1 head outputs in fp32 on CUDA cores (tc_heads_sample: + the rollout's sampler).
//   tc_rollout_tower<RAW>        rollout step: conv1 -> conv2 -> conv3 per image with act1 / act2 in shared memory.
#include <cuda.h>            // CUtensorMap types only; the encoder is resolved at run time (no libcuda link)
#include "tc_base.cuh"
#include "tc_conv_win.cuh"
#include "tc_conv1_u8.cuh"
#include "tc_gemm_tma.cuh"
#include "tc_wgrad_win.cuh"
#include "tc_reduce.cuh"
#include "tc_aux.cuh"
#include "tc_heads.cuh"
#include "tc_rollout_tower.cuh"

// =====================================================================================
// Host side: NatureCNN plan over the kernels above (C-ABI entry points, include/b200rl.h)
// =====================================================================================
namespace b200rl {

struct NatureLayout {
    int A;
    // flat fp32 parameter offsets (libb200rl order: trunk, then both head weights, then both head biases)
    int64_t c1w, c1b, c2w, c2b, c3w, c3b, fcw, fcb, hw, hb, total;
    // packed bf16 operand offsets (elements)
    int64_t w1f, w2f, w2dg, w3f, w3dg, wfcf, wfcdg, w1l, w1sc, packed_total;
    explicit NatureLayout(int A_) : A(A_) {
        int64_t o = 0;
        c1w = o; o += 32 * 4 * 8 * 8;  c1b = o; o += 32;
        c2w = o; o += 64 * 32 * 4 * 4; c2b = o; o += 64;
        c3w = o; o += 64 * 64 * 3 * 3; c3b = o; o += 64;
        fcw = o; o += 512 * 3136;      fcb = o; o += 512;
        hw = o;  o += (int64_t)(A + 1) * 512;
        hb = o;  o += A + 1;
        total = o;
        int64_t q = 0;
        w1f = q; q += 32 * 256;
        w2f = q; q += 64 * 512;
        w2dg = q; q += 4 * 32 * 256;
        w3f = q; q += 64 * 576;
        w3dg = q; q += 64 * 576;
        wfcf = q; q += 512 * 3136;
        wfcdg = q; q += 3136 * 512;
        w1l = q; q += 64 * 256 / 2;          // conv1 weight limbs: s8 [64][256] (16 KB)
        w1sc = q; q += 64 * 2;               // conv1 column scales: f32 [64]
        packed_total = q;
    }
};

struct NatureActs {   // bf16 element offsets inside the (zero-initialised) activation workspace for batch n
    int64_t x0, act1, act2, act3, hid, dhid, dact3a, dact3b, dact2a, dact2b, dact1, m1, m2, m3, m4, total;
    explicit NatureActs(int64_t n, bool with_x0 = true) {
        int64_t o = 0;
        x0 = o; if (with_x0) o += n * 28224;     // space-to-depth frames [n,441,64] (only for uint8 input)
        act1 = o; o += n * 12800;                // conv1 out as 2x2 cells   [n,100,128]
        act2 = o; o += n * 5184;                 // conv2 out               [n, 81, 64]
        act3 = o; o += n * 3136;                 // conv3 out               [n, 49, 64]
        hid = o;  o += n * 512;
        dhid = o; o += n * 512;
        dact3a = o; o += n * 5184;               // d(act3) on the 9x9 linear grid (zeros outside 7x7)
        dact3b = o; o += n * 7744;               // d(act3) zero-padded to 11x11 (interior at +2,+2)
        dact2a = o; o += n * 6400;               // d(act2) on the 10x10 linear grid (zeros at row/col 9)
        dact2b = o; o += n * 7744;               // d(act2) zero-padded to 11x11 (interior at +1,+1)
        dact1 = o; o += n * 14112;               // d(act1) on the 21x21 linear grid, 32 channels
        // ReLU masks as bits (uint32 words; offsets stay in bf16 elements = 2 words per 4 elements)
        auto pad8 = [](int64_t v) { return (v + 7) & ~int64_t(7); };
        m1 = o; o += pad8(n * 100 * 4 * 2);      // act1 > 0: [n,100 cells] x 4 words (128 channels)
        m2 = o; o += pad8(n * 81 * 2 * 2);       // act2 > 0: [n,81] x 2 words
        m3 = o; o += pad8(n * 49 * 2 * 2);       // act3 > 0: [n,49] x 2 words (= dense [n,3136] / 32)
        m4 = o; o += pad8(n * 16 * 2);           // hid  > 0: [n] x 16 words
        total = o;
    }
};

static void gemm_rowmajor(KGemmParams& p, const bf16* x, int64_t n, int nchunks) {   // x [n, 64*nchunks]
    memset(&p, 0, sizeof(p));
    p.scale = 1.f;
    p.A = x; p.M = n; p.nchunks = nchunks;
}


// ---- window-convolution descriptions of the three conv layers
static void win_defaults(WinParams& p) { memset(&p, 0, sizeof(p)); p.scale = 1.f; }
static int round8(int v) { return (v + 7) & ~7; }
static void win_conv1(WinParams& p, const bf16* x0, const int64_t* rows, int64_t n) {     // 2x2 taps on the 21x21 s2d grid
    p.A = x0; p.rows = rows; p.n = (int)n; p.G = 441; p.Wp = 21; p.M = n * 441;
    p.tpi_shift = 2;                             // 4 tiles of 128 grid rows per image (441 used)
    p.n_images = rows ? (int64_t)1 << 24 : n;    // gather indices are the caller's contract (never range-checked)
    p.ntaps = 4; p.shift[0] = 0; p.shift[1] = 1; p.shift[2] = 21; p.shift[3] = 22; p.WR = round8(128 + 22);
}
static void win_conv2(WinParams& p, const bf16* act1, int64_t n) {                         // 2x2 taps on the 10x10 cell grid
    p.A = act1; p.n = (int)n; p.G = 100; p.Wp = 10; p.M = n * 100;
    p.ntaps = 4; p.shift[0] = 0; p.shift[1] = 1; p.shift[2] = 10; p.shift[3] = 11; p.WR = round8(128 + 11);
}
static void win_conv3(WinParams& p, const bf16* act2, int64_t n) {                         // 3x3 taps on the 9x9 grid
    p.A = act2; p.n = (int)n; p.G = 81; p.Wp = 9; p.M = n * 81;
    p.ntaps = 9; for (int ky = 0; ky < 3; ++ky) for (int kx = 0; kx < 3; ++kx) p.shift[ky * 3 + kx] = ky * 9 + kx;
    p.WR = round8(128 + 20);
}
static void wgw_defaults(WGradWinParams& w) { memset(&w, 0, sizeof(w)); }

static int64_t round_up(int64_t a, int64_t b) { return ceil_div(a, b) * b; }

struct WPlan { int64_t rows_per_cta; int splits; };
static WPlan wgrad_plan(int64_t M, int target_ctas, int quantum = 32) {
    WPlan w;
    w.rows_per_cta = round_up(ceil_div(M, target_ctas), quantum);
    if (w.rows_per_cta < quantum) w.rows_per_cta = quantum;
    w.splits = (int)ceil_div(M, w.rows_per_cta);
    if (w.splits < 1) w.splits = 1;
    return w;
}
static const int kC1Ctas = 296, kC2Ctas = 148, kC3Ctas = 148, kFcSplits = 8;

static int launch_wgrad_win(const WGradWinParams& p, int ctas, cudaStream_t s, const char* what) {
    const size_t smem = (size_t)kWgradWinStages * ((size_t)p.WRX * 128 * p.cpr + 128 * 128) + 4096 + 1024;
    static SmemAttrCache attr;
    if (int rc0 = attr.ensure(tc_wgrad_win, smem, what)) return rc0;
    CUtensorMap tmX, tmY;
    memset(&tmX, 0, sizeof(tmX)); memset(&tmY, 0, sizeof(tmY));
    // TMA when rows are contiguous, dY rows are exactly 128 bytes and every CTA owns whole 128-row steps
    // all-TMA when dY rows are exactly 128 bytes; image-aligned steps (3-D TMA for X, cp.async for dY) otherwise
    const int use_tma = p.tpi_shift ? 0 : 1;
    if (p.rows_per_cta % 128 != 0) return fail(B200RL_ERR_INVALID_ARGUMENT, "%s: rows per CTA must be a multiple of 128", what);
    int rc;
    if (use_tma) {
        if (p.rows || p.ldy != 64 || p.ncolsY != 64)
            return fail(B200RL_ERR_INVALID_ARGUMENT, "%s: linear-grid mode needs contiguous rows and 64-channel dY", what);
        if ((rc = make_tmap_2d(&tmX, p.X, p.M, (int64_t)p.cpr * 64, p.WRX, what))) return rc;
        if ((rc = make_tmap_2d(&tmY, p.Y, p.M, 64, 128, what))) return rc;
    } else {
        if ((128 << p.tpi_shift) < p.G) return fail(B200RL_ERR_INVALID_ARGUMENT, "%s: steps per image too small", what);
        if ((rc = make_tmap_3d(&tmX, p.X, p.n_images, p.G, (int64_t)p.cpr * 64, p.WRX, what))) return rc;
    }
    tc_wgrad_win<<<ctas, kWgradWinThreads, smem, s>>>(tmX, tmY, p, use_tma);
    return check_launch(what);
}

static int colsum(const bf16* Y, int64_t M, int ld, int ncols, float* part, float* db, cudaStream_t s) {
    int64_t rpb = ceil_div(M, 148 * 3);
    if (rpb < 64) rpb = 64;
    const int nb = (int)ceil_div(M, rpb);
    tc_colsum_partial<<<nb, 256, 0, s>>>(Y, M, ld, ncols, rpb, part);
    tc_colsum_final<<<(unsigned)ceil_div(ncols, 32), 256, 0, s>>>(part, nb, ncols, db);
    return check_launch("colsum", 2);
}
static size_t colsum_ws(int64_t M, int ncols) {
    int64_t rpb = ceil_div(M, 148 * 3);
    if (rpb < 64) rpb = 64;
    return (size_t)ceil_div(M, rpb) * ncols * sizeof(float);
}

}  // namespace b200rl

using namespace b200rl;

extern "C" int64_t b200rl_naturecnn_param_count(int A) { return A >= 1 ? NatureLayout(A).total : -1; }
extern "C" int64_t b200rl_naturecnn_grad_tail_offset(int A) { return A >= 1 ? NatureLayout(A).fcw : -1; }
extern "C" size_t b200rl_naturecnn_bf16_packed_bytes(int A) { return A >= 1 ? (size_t)NatureLayout(A).packed_total * 2 : 0; }
extern "C" size_t b200rl_naturecnn_bf16_acts_bytes(int64_t n, int obs_format) {
    return n >= 0 ? (size_t)NatureActs(n, obs_format == B200RL_OBS_U8_NCHW).total * 2 + 256 : 0;
}

extern "C" int b200rl_frames_to_s2d_bf16(const uint8_t* obs, const int64_t* rows, int64_t n, void* out, void* stream) {
    B200RL_REQUIRE(n >= 0, "frames_to_s2d: negative n");
    if (n == 0) return B200RL_OK;
    B200RL_REQUIRE(obs && out, "frames_to_s2d: null pointer");
    B200RL_REQUIRE(aligned(obs, 4) && aligned(out, 16), "frames_to_s2d: misaligned buffer");
    cudaStream_t s = (cudaStream_t)stream;
    ProfScope ps(s, "frames_to_s2d", 0, (double)n * 28224 * 3);
    tc_frames_to_s2d<<<(unsigned)ceil_div(n * 1764, 256), 256, 0, s>>>(obs, rows, n, reinterpret_cast<bf16*>(out));
    return check_launch("frames_to_s2d");
}

extern "C" int b200rl_frames_to_s2d_u8(const uint8_t* obs, const int64_t* rows, int64_t n, uint8_t* out_rm, uint8_t* out_cm, void* stream) {
    B200RL_REQUIRE(n >= 0, "frames_to_s2d_u8: negative n");
    if (n == 0) return B200RL_OK;
    B200RL_REQUIRE(obs && out_rm && out_cm, "frames_to_s2d_u8: null pointer");
    B200RL_REQUIRE(aligned(obs, 16) && aligned(out_rm, 16) && aligned(out_cm, 16), "frames_to_s2d_u8: misaligned buffer");
    B200RL_REQUIRE(n <= (int64_t)1 << 28, "frames_to_s2d_u8: n too large");
    cudaStream_t s = (cudaStream_t)stream;
    ProfScope ps(s, "frames_to_s2d", 0, (double)n * (28224 + 28224 + 28672));
    tc_frames_to_s2d_u8<<<(unsigned)(n * 4), 256, 0, s>>>(obs, rows, n, out_rm, out_cm);
    return check_launch("frames_to_s2d_u8");
}

extern "C" size_t b200rl_naturecnn_bf16_workspace_bytes(int64_t n, int A) {
    if (n < 1 || A < 1) return 0;
    size_t a = 0;
    auto mx = [&](size_t v) { if (v > a) a = v; };
    mx((size_t)wgrad_plan(n * 512, kC1Ctas, 128).splits * 256 * 64 * 4);
    mx((size_t)wgrad_plan(n * 100, kC2Ctas, 128).splits * 512 * 64 * 4);
    mx((size_t)wgrad_plan(n * 81, kC3Ctas, 128).splits * 640 * 64 * 4);
    mx((size_t)wgrad_plan(n, kFcSplits, 64).splits * 512 * (13 * 256) * 4);
    size_t b = 0;
    auto mb = [&](size_t v) { if (v > b) b = v; };
    mb(colsum_ws(n * 441, 32)); mb(colsum_ws(n * 100, 64)); mb(colsum_ws(n * 81, 64)); mb(colsum_ws(n, 512));
    mb((size_t)2 * ceil_div(n, heads_rows_per_block(n)) * (A + 1) * 514 * 4);
    return a + b + 512;
}

extern "C" int b200rl_naturecnn_bf16_pack(const float* params, int A, void* packed, void* stream) {
    B200RL_REQUIRE(params && packed && A >= 1 && A < kMaxHeads, "naturecnn_pack: bad arguments (A must be in [1,23])");
    B200RL_REQUIRE(aligned(packed, 16), "naturecnn_pack: packed buffer must be 16-B aligned");
    const NatureLayout L(A);
    bf16* P = reinterpret_cast<bf16*>(packed);
    cudaStream_t s = (cudaStream_t)stream;
    ProfScope ps(s, "pack_weights", 0, (double)L.total * 4 + (double)L.packed_total * 2);
    tc_pack_conv1_s2d<<<32, 256, 0, s>>>(params + L.c1w, P + L.w1f);
    tc_pack_conv1_i8<<<32, 256, 0, s>>>(params + L.c1w, reinterpret_cast<int8_t*>(P + L.w1l), reinterpret_cast<float*>(P + L.w1sc));
    tc_pack_conv2_cells<<<128, 256, 0, s>>>(params + L.c2w, P + L.w2f);
    tc_pack_conv_s2_classes<<<(unsigned)ceil_div(32768, 256), 256, 0, s>>>(params + L.c2w, 64, 32, P + L.w2dg);
    tc_pack_conv<<<(unsigned)ceil_div(36864, 256), 256, 0, s>>>(params + L.c3w, 64, 64, 3, 3, 0, P + L.w3f, P + L.w3dg);
    tc_pack_fc<<<dim3(512 / 8, 49 / 7), 256, 0, s>>>(params + L.fcw, 512, 49, P + L.wfcf, P + L.wfcdg);
    return check_launch("naturecnn_pack", 6);
}

extern "C" int b200rl_naturecnn_bf16_forward(const void* obs, int obs_format, const int64_t* rows, int64_t n, int A,
                                             const float* params, const void* packed, void* acts,
                                             float* head_out, void* stream) {
    B200RL_REQUIRE(n >= 0, "naturecnn_forward: negative n");
    if (n == 0) return B200RL_OK;
    B200RL_REQUIRE(obs && params && packed && acts && head_out, "naturecnn_forward: null pointer");
    B200RL_REQUIRE(A >= 1 && A < kMaxHeads, "naturecnn_forward: A=%d outside [1,23]", A);
    B200RL_REQUIRE(obs_format == B200RL_OBS_U8_NCHW || obs_format == B200RL_OBS_S2D_BF16 || obs_format == B200RL_OBS_S2D_U8,
                   "naturecnn_forward: bad obs_format %d", obs_format);
    B200RL_REQUIRE(aligned(obs, 16) && aligned(acts, 16) && aligned(packed, 16), "naturecnn_forward: misaligned buffer");
    B200RL_REQUIRE(n <= (int64_t)1 << 22, "naturecnn_forward: n too large");
    const NatureLayout L(A);
    const NatureActs Q(n, obs_format == B200RL_OBS_U8_NCHW);
    const bf16* P = reinterpret_cast<const bf16*>(packed);
    bf16* act = reinterpret_cast<bf16*>(acts);
    cudaStream_t s = (cudaStream_t)stream;
    int rc;
    KGemmParams p;
    WinParams wp;
    // conv1: 2x2 window conv on space-to-depth frames -> act1 as 2x2 cells [n,10,10,128]
    const bf16* x0 = reinterpret_cast<const bf16*>(obs);
    const int64_t* x0rows = rows;
    if (obs_format == B200RL_OBS_U8_NCHW) {
        if ((rc = b200rl_frames_to_s2d_bf16(reinterpret_cast<const uint8_t*>(obs), rows, n, act + Q.x0, stream))) return rc;
        x0 = act + Q.x0; x0rows = nullptr;
    }
    if (obs_format == B200RL_OBS_S2D_U8) {
        // uint8 space-to-depth frames straight into the integer tensor cores (tc_conv1_u8.cuh)
        Conv1U8Params cp;
        memset(&cp, 0, sizeof(cp));
        cp.rows = rows; cp.n = (int)n; cp.n_images = rows ? (int64_t)1 << 24 : n;
        cp.limbs = reinterpret_cast<const int8_t*>(P + L.w1l); cp.sc = reinterpret_cast<const float*>(P + L.w1sc);
        cp.bias = params + L.c1b; cp.out = act + Q.act1; cp.mask_out = reinterpret_cast<uint32_t*>(act + Q.m1);
        ProfScope ps(s, "conv1_fwd", 2.0 * n * 400 * 32 * 256, (double)n * (28224 + 12800 * 2 + 1600));
        if ((rc = launch_conv1_i8(cp, obs, s, "naturecnn/conv1_i8"))) return rc;
    } else {
    win_defaults(wp); win_conv1(wp, x0, x0rows, n);
    wp.Bw = P + L.w1f; wp.N = 32; wp.vH = 20; wp.vW = 20; wp.out_mode = WOUT_S2D2; wp.out = act + Q.act1;
    wp.bias = params + L.c1b; wp.scale = 1.0f / 255.0f; wp.relu = 1; wp.mask_out = reinterpret_cast<uint32_t*>(act + Q.m1);
    { ProfScope ps(s, "conv1_fwd", 2.0 * n * 400 * 32 * 256, (double)n * ((28224 + 12800) * 2 + 1600));
      if ((rc = launch_conv_win<32, 1, 9, 4>(wp, s, "naturecnn/conv1"))) return rc; }
    }
    // conv2: 2x2 window conv on the 128-channel cells -> act2 [n,9,9,64]
    win_defaults(wp); win_conv2(wp, act + Q.act1, n);
    wp.Bw = P + L.w2f; wp.N = 64; wp.vH = 9; wp.vW = 9; wp.out_mode = WOUT_DENSE; wp.out = act + Q.act2;
    wp.bias = params + L.c2b; wp.relu = 1; wp.mask_out = reinterpret_cast<uint32_t*>(act + Q.m2);
    { ProfScope ps(s, "conv2_fwd", 2.0 * n * 81 * 64 * 512, (double)n * ((12800 + 5184) * 2 + 648));
      if ((rc = launch_conv_win<64, 2, 4, 4>(wp, s, "naturecnn/conv2"))) return rc; }
    // conv3: 3x3 window conv -> act3 [n,7,7,64]
    win_defaults(wp); win_conv3(wp, act + Q.act2, n);
    wp.Bw = P + L.w3f; wp.N = 64; wp.vH = 7; wp.vW = 7; wp.out_mode = WOUT_DENSE; wp.out = act + Q.act3;
    wp.bias = params + L.c3b; wp.relu = 1; wp.mask_out = reinterpret_cast<uint32_t*>(act + Q.m3);
    { ProfScope ps(s, "conv3_fwd", 2.0 * n * 49 * 64 * 576, (double)n * ((5184 + 3136) * 2 + 392));
      if ((rc = launch_conv_win<64, 1, 6, 9>(wp, s, "naturecnn/conv3"))) return rc; }
    // fc -> hidden [n,512]
    gemm_rowmajor(p, act + Q.act3, n, 49);
    p.Bw = P + L.wfcf; p.N = 512; p.out = act + Q.hid; p.ldo = 512; p.bias = params + L.fcb; p.relu = 1;
    p.mask_out = reinterpret_cast<uint32_t*>(act + Q.m4);
    { ProfScope ps(s, "fc_fwd", 2.0 * n * 512 * 3136, (double)n * (3136 + 512) * 2 + 512.0 * 3136 * 2);
      // small batches (rollout step): narrower N tiles => 4x more CTAs for the same work
      if (n <= 8192) { if ((rc = launch_gemm_tma<64, 8>(p, s, "naturecnn/fc"))) return rc; }
      else if ((rc = launch_gemm_tma<256, 4>(p, s, "naturecnn/fc"))) return rc; }
    // heads (fp32 math on CUDA cores): head_out [n, A+1] = [logits | value]
    { ProfScope ps(s, "heads_fwd", 2.0 * n * 512 * (A + 1), (double)n * (1024 + 4 * (A + 1)));
      int hb = (int)ceil_div(n, 8); if (hb > num_sms() * 8) hb = num_sms() * 8;
      tc_heads_fwd<<<hb, 256, (size_t)(A + 1) * 2048, s>>>(act + Q.hid, params + L.hw, params + L.hb, n, A + 1, 512, head_out); }
    return check_launch("naturecnn/heads");
}

extern "C" int b200rl_naturecnn_bf16_rollout_step(const uint8_t* frames, uint8_t* slot_rm, uint8_t* slot_cm, int64_t n, int A,
                                                  const float* params, const void* packed, void* acts, const float* noise,
                                                  int64_t* action, float* logprob, float* value, void* stream) {
    B200RL_REQUIRE(n >= 0, "naturecnn_rollout_step: negative n");
    if (n == 0) return B200RL_OK;
    B200RL_REQUIRE(slot_rm && params && packed && acts && noise && action && logprob && value, "naturecnn_rollout_step: null pointer");
    B200RL_REQUIRE(!frames || slot_cm, "naturecnn_rollout_step: raw frames need the channel-major slot");
    B200RL_REQUIRE(A >= 1 && A < kMaxHeads, "naturecnn_rollout_step: A=%d outside [1,23]", A);
    B200RL_REQUIRE(aligned(slot_rm, 16) && aligned(acts, 16) && aligned(packed, 16) && (!frames || (aligned(frames, 16) && aligned(slot_cm, 16))),
                   "naturecnn_rollout_step: misaligned buffer");
    B200RL_REQUIRE(n <= (int64_t)1 << 22, "naturecnn_rollout_step: n too large");
    const NatureLayout L(A);
    const NatureActs Q(n, false);              // the workspace of a uint8 space-to-depth forward (format 2)
    const bf16* P = reinterpret_cast<const bf16*>(packed);
    bf16* act = reinterpret_cast<bf16*>(acts);
    cudaStream_t s = (cudaStream_t)stream;
    int rc;
    TowerParams tp;
    memset(&tp, 0, sizeof(tp));
    tp.frames = frames; tp.slot_rm = slot_rm; tp.slot_cm = slot_cm; tp.n = (int)n;
    tp.limbs = reinterpret_cast<const int8_t*>(P + L.w1l); tp.sc = reinterpret_cast<const float*>(P + L.w1sc); tp.b1 = params + L.c1b;
    tp.w2 = P + L.w2f; tp.b2 = params + L.c2b; tp.w3 = P + L.w3f; tp.b3 = params + L.c3b; tp.act3 = act + Q.act3;
    { ProfScope ps(s, "rollout_tower", 2.0 * n * (400 * 32 * 256 + 81 * 64 * 512 + 49 * 64 * 576),
                   (double)n * ((frames ? 28224 * 2 + 28672 : 28224) + 3136 * 2));
      if ((rc = launch_rollout_tower(tp, s, "naturecnn/rollout_tower"))) return rc; }
    // fc -> hidden [n,512]: the training forward's GEMM (bit-exact with it)
    KGemmParams p;
    gemm_rowmajor(p, act + Q.act3, n, 49);
    p.Bw = P + L.wfcf; p.N = 512; p.out = act + Q.hid; p.ldo = 512; p.bias = params + L.fcb; p.relu = 1;
    { ProfScope ps(s, "fc_fwd", 2.0 * n * 512 * 3136, (double)n * (3136 + 512) * 2 + 512.0 * 3136 * 2);
      if (n <= 8192) { if ((rc = launch_gemm_tma<64, 8>(p, s, "naturecnn/fc"))) return rc; }
      else if ((rc = launch_gemm_tma<256, 4>(p, s, "naturecnn/fc"))) return rc; }
    { ProfScope ps(s, "rollout_heads_sample", 2.0 * n * 512 * (A + 1), (double)n * (1024 + 4 * A + 20));
      int hb = (int)ceil_div(n, 8); if (hb > num_sms() * 8) hb = num_sms() * 8;
      tc_heads_sample<<<hb, 256, (size_t)(A + 1) * 2048, s>>>(act + Q.hid, params + L.hw, params + L.hb, n, A, noise, action, logprob, value); }
    return check_launch("naturecnn/heads_sample");
}

extern "C" int b200rl_naturecnn_bf16_backward(const void* obs, const void* obs_aux, int obs_format, const int64_t* rows, int64_t n, int A,
                                              const float* params, const void* packed, void* acts,
                                              const float* dhead, float* grads,
                                              void* workspace, size_t workspace_bytes, void* tail_ready_event, void* stream) {
    B200RL_REQUIRE(n >= 1, "naturecnn_backward: n must be >= 1");
    B200RL_REQUIRE(obs && params && packed && acts && dhead && grads && workspace, "naturecnn_backward: null pointer");
    B200RL_REQUIRE(A >= 1 && A < kMaxHeads, "naturecnn_backward: A=%d outside [1,23]", A);
    B200RL_REQUIRE(aligned(workspace, 16), "naturecnn_backward: workspace misaligned");
    const size_t need = b200rl_naturecnn_bf16_workspace_bytes(n, A);
    if (workspace_bytes < need) return fail(B200RL_ERR_WORKSPACE, "naturecnn_backward: workspace %zu < %zu", workspace_bytes, need);
    B200RL_REQUIRE(obs_format == B200RL_OBS_U8_NCHW || obs_format == B200RL_OBS_S2D_BF16 || obs_format == B200RL_OBS_S2D_U8,
                   "naturecnn_backward: bad obs_format %d", obs_format);
    B200RL_REQUIRE(obs_format != B200RL_OBS_S2D_U8 || (obs_aux && aligned(obs_aux, 16)), "naturecnn_backward: the uint8 rollout needs obs_aux");
    const NatureLayout L(A);
    const NatureActs Q(n, obs_format == B200RL_OBS_U8_NCHW);
    const bf16* P = reinterpret_cast<const bf16*>(packed);
    bf16* act = reinterpret_cast<bf16*>(acts);
    cudaStream_t s = (cudaStream_t)stream;
    // uint8 input: forward left the space-to-depth frames of this minibatch in the workspace
    const bf16* x0 = obs_format == B200RL_OBS_U8_NCHW ? act + Q.x0 : reinterpret_cast<const bf16*>(obs);   // unused for S2D_U8
    const int64_t* x0rows = obs_format == B200RL_OBS_U8_NCHW ? nullptr : rows;
    // workspace split: [wgrad partials | small partials]
    size_t big = 0;
    {
        auto mx = [&](size_t v) { if (v > big) big = v; };
        mx((size_t)wgrad_plan(n * 512, kC1Ctas, 128).splits * 256 * 64 * 4);
        mx((size_t)wgrad_plan(n * 100, kC2Ctas, 128).splits * 512 * 64 * 4);
        mx((size_t)wgrad_plan(n * 81, kC3Ctas, 128).splits * 640 * 64 * 4);
        mx((size_t)wgrad_plan(n, kFcSplits, 64).splits * 512 * (13 * 256) * 4);
        big = (big + 255) & ~(size_t)255;
    }
    float* wsbig = reinterpret_cast<float*>(workspace);
    float* wssmall = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + big);
    int rc;
    const int A1 = A + 1;
    // ---- heads: dW, db, then dhid_pre = (dhead . Wh) * (hid > 0)
    {
        const int64_t rpb = heads_rows_per_block(n);
        const int nb = (int)ceil_div(n, rpb);
        ProfScope ps(s, "heads_bwd", 4.0 * n * 512 * A1, (double)n * (2048 + 64 + 8 * A1));
        const size_t sd = (size_t)rpb * A1 * sizeof(float);
        if (A1 <= 8) tc_heads_bwd_weight<8><<<nb, 512, sd, s>>>(dhead, act + Q.hid, n, A1, 512, rpb, wssmall);
        else tc_heads_bwd_weight<kMaxHeads><<<nb, 512, sd, s>>>(dhead, act + Q.hid, n, A1, 512, rpb, wssmall);
        tc_heads_fold<<<(unsigned)ceil_div(A1 * 514, 32), 256, 0, s>>>(wssmall, 2 * nb, A1, 512, grads + L.hw, grads + L.hb);
        int db_blocks = (int)ceil_div(n * 64, 256); if (db_blocks > num_sms() * 8) db_blocks = num_sms() * 8;
        tc_heads_bwd_data<<<db_blocks, 256, (size_t)A1 * 2048, s>>>(dhead, params + L.hw, reinterpret_cast<const uint8_t*>(act + Q.m4), n, A1, 512, act + Q.dhid);
        if ((rc = check_launch("naturecnn/heads_bwd", 3))) return rc;
    }
    KGemmParams p;
    // ---- fc: dW[o][c*49+p] = sum_m dhid[m][o] * act3[m][p*64+c]
    {
        const WPlan pl = wgrad_plan(n, kFcSplits, 64);
        { ProfScope ps(s, "fc_wgrad", 2.0 * n * 512 * 3136, (double)n * (3136 + 512) * 2 + 512.0 * 3136 * 4);
          CUtensorMap tmX, tmY;
          if ((rc = make_tmap_2d(&tmX, act + Q.dhid, n, 512, 64, "naturecnn/fc_wgrad"))) return rc;
          if ((rc = make_tmap_2d(&tmY, act + Q.act3, n, 3136, 64, "naturecnn/fc_wgrad"))) return rc;
          const size_t smem = (size_t)4 * (2 + 4) * 64 * 128 + 1024;
          static SmemAttrCache attr;
          if ((rc = attr.ensure(tc_wgrad_tma, smem, "naturecnn/fc_wgrad"))) return rc;
          tc_wgrad_tma<<<dim3(pl.splits, 4, 13), 160, smem, s>>>(tmX, tmY, n, pl.rows_per_cta, 2, 4, wsbig);
          if ((rc = check_launch("naturecnn/fc_wgrad"))) return rc; }
        { ProfScope ps(s, "wgrad_fold_bias", 0, 0);
          note_launches(1); tc_fold_fc<<<(unsigned)ceil_div((int64_t)512 * 3136, 256), 256, 0, s>>>(wsbig, pl.splits, 512, 13 * 256, 512, 3136, 64, 49, 1.f, grads + L.fcw);
          if ((rc = colsum(act + Q.dhid, n, 512, 512, wssmall, grads + L.fcb, s))) return rc; }
        // grads[fcw .. total) (fc weight + bias, both heads) are final: the caller may start exchanging them now
        if (tail_ready_event) {
            cudaError_t e = cudaEventRecord(reinterpret_cast<cudaEvent_t>(tail_ready_event), s);
            if (e != cudaSuccess) return fail(B200RL_ERR_CUDA, "naturecnn_backward: cudaEventRecord: %s", cudaGetErrorString(e));
        }
        // dact3_pre = (dhid . Wfc) * (act3 > 0), written on the 9x9 linear grid and the zero-padded 11x11 grid
        gemm_rowmajor(p, act + Q.dhid, n, 8);
        p.Bw = P + L.wfcdg; p.N = 3136; p.out = act + Q.dact3a; p.out2 = act + Q.dact3b; p.dual_dact3 = 1;
        p.ldo = 3136; p.mask_bits = reinterpret_cast<const uint32_t*>(act + Q.m3);
        { ProfScope ps(s, "fc_dgrad", 2.0 * n * 512 * 3136, (double)n * ((3136 + 512) * 2 + 392) + 512.0 * 3136 * 2);
          if ((rc = launch_gemm_tma<256, 4>(p, s, "naturecnn/fc_dgrad"))) return rc; }
    }
    WGradWinParams gw;
    WinParams wp;
    FoldWin fw;
    // ---- conv3: dW from act2 windows x dact3 (9x9 grid), then dact2 = full correlation of padded dact3 with W3
    {
        wgw_defaults(gw);
        gw.X = act + Q.act2; gw.M = n * 81; gw.n = (int)n; gw.G = 81; gw.cpr = 1; gw.nslots = 10; gw.WRX = round8(128 + 20);
        for (int t = 0; t < 9; ++t) gw.shift[t] = (t / 3) * 9 + (t % 3);
        const int st[10] = {0, 1, 2, 3, 4, 5, 6, 7, 7, 8};      // slot 8 duplicates tap 7 so that tap 8 has a partner
        for (int k = 0; k < 10; ++k) { gw.slot_tap[k] = st[k]; gw.slot_cc[k] = 0; }
        gw.Y = act + Q.dact3a; gw.ldy = 64; gw.ncolsY = 64;
        const WPlan pl = wgrad_plan(n * 81, kC3Ctas, 128);
        gw.rows_per_cta = pl.rows_per_cta; gw.ws = wsbig; gw.wsb = wssmall;
        { ProfScope ps(s, "conv3_wgrad", 2.0 * n * 49 * 64 * 576, (double)n * (5184 + 5184) * 2);
          if ((rc = launch_wgrad_win(gw, pl.splits, s, "naturecnn/conv3_wgrad"))) return rc; }
        memset(&fw, 0, sizeof(fw));
        fw.layer = 3; fw.S = pl.splits; fw.nslots = 10; fw.Cout = 64; fw.scale = 1.f; fw.bscale = 1.f;
        for (int k = 0; k < 10; ++k) { fw.slot_tap[k] = st[k]; fw.slot_skip[k] = (k == 8); }
        { ProfScope ps(s, "wgrad_fold_bias", 0, 0);
          fw.wsb = wssmall; fw.db = grads + L.c3b;
          tc_fold_win<<<(unsigned)ceil_div(640 * 64 + 64, 32), 256, 0, s>>>(wsbig, fw, grads + L.c3w);
          if ((rc = check_launch("naturecnn/conv3_fold"))) return rc; }
        win_defaults(wp);
        wp.A = act + Q.dact3b; wp.n = (int)n; wp.G = 121; wp.Wp = 11; wp.M = n * 121; wp.ntaps = 9;
        for (int ky = 0; ky < 3; ++ky) for (int kx = 0; kx < 3; ++kx) wp.shift[ky * 3 + kx] = (2 - ky) * 11 + (2 - kx);
        wp.WR = round8(128 + 24);
        wp.Bw = P + L.w3dg; wp.N = 64; wp.vH = 9; wp.vW = 9; wp.out_mode = WOUT_DACT2;
        wp.out = act + Q.dact2a; wp.out2 = act + Q.dact2b; wp.mask_bits = reinterpret_cast<const uint32_t*>(act + Q.m2);
        { ProfScope ps(s, "conv3_dgrad", 2.0 * n * 81 * 64 * 576, (double)n * ((7744 + 6400 + 7744) * 2 + 648));
          if ((rc = launch_conv_win<64, 1, 6, 9>(wp, s, "naturecnn/conv3_dgrad"))) return rc; }
    }
    // ---- conv2: dW from act1 cell windows x dact2 (10x10 grid); dact1 = one N=128 GEMM over the 4 stride-parity
    //      classes (the 4 channel groups of a cell)
    {
        wgw_defaults(gw);
        gw.X = act + Q.act1; gw.M = n * 100; gw.n = (int)n; gw.G = 100; gw.cpr = 2; gw.nslots = 8; gw.WRX = round8(128 + 11);
        gw.shift[0] = 0; gw.shift[1] = 1; gw.shift[2] = 10; gw.shift[3] = 11;
        for (int k = 0; k < 8; ++k) { gw.slot_tap[k] = k >> 1; gw.slot_cc[k] = k & 1; }
        gw.Y = act + Q.dact2a; gw.ldy = 64; gw.ncolsY = 64;
        const WPlan pl = wgrad_plan(n * 100, kC2Ctas, 128);
        gw.rows_per_cta = pl.rows_per_cta; gw.ws = wsbig; gw.wsb = wssmall;
        { ProfScope ps(s, "conv2_wgrad", 2.0 * n * 81 * 64 * 512, (double)n * (12800 + 6400) * 2);
          if ((rc = launch_wgrad_win(gw, pl.splits, s, "naturecnn/conv2_wgrad"))) return rc; }
        memset(&fw, 0, sizeof(fw));
        fw.layer = 2; fw.S = pl.splits; fw.nslots = 8; fw.Cout = 64; fw.scale = 1.f; fw.bscale = 1.f;
        for (int k = 0; k < 8; ++k) { fw.slot_tap[k] = k >> 1; fw.slot_cc[k] = k & 1; }
        { ProfScope ps(s, "wgrad_fold_bias", 0, 0);
          fw.wsb = wssmall; fw.db = grads + L.c2b;
          tc_fold_win<<<(unsigned)ceil_div(512 * 64 + 64, 32), 256, 0, s>>>(wsbig, fw, grads + L.c2w);
          if ((rc = check_launch("naturecnn/conv2_fold"))) return rc; }
        win_defaults(wp);
        wp.A = act + Q.dact2b; wp.n = (int)n; wp.G = 121; wp.Wp = 11; wp.M = n * 121; wp.ntaps = 4;
        for (int a = 0; a < 2; ++a) for (int b = 0; b < 2; ++b) wp.shift[a * 2 + b] = (1 - a) * 11 + (1 - b);
        wp.WR = round8(128 + 12);
        wp.Bw = P + L.w2dg; wp.N = 128; wp.vH = 10; wp.vW = 10; wp.out_mode = WOUT_DACT1;
        wp.out = act + Q.dact1; wp.mask_bits = reinterpret_cast<const uint32_t*>(act + Q.m1);
        if (obs_format == B200RL_OBS_S2D_U8) { wp.out_f16 = 1; wp.scale = kDact1Scale; }     // fp16 x 2^12 for the TMEM-fed conv1 wgrad
        { ProfScope ps(s, "conv2_dgrad", 2.0 * n * 400 * 32 * 256, (double)n * ((7744 + 14112) * 2 + 1600));
          if ((rc = launch_conv_win<128, 1, 6, 4>(wp, s, "naturecnn/conv2_dgrad"))) return rc; }
    }
    // ---- conv1 (no data gradient: the input is the observation)
    if (obs_format == B200RL_OBS_S2D_U8) {
        // uint8 channel-major frames -> fp16 in registers -> tensor memory (tc_conv1_u8.cuh); 1 CTA per SM (512 TMEM columns)
        Conv1WgradU8Params cw;
        memset(&cw, 0, sizeof(cw));
        const WPlan pl = wgrad_plan(n * 512, kC2Ctas, 512);          // whole images per CTA
        cw.rows = rows; cw.n = (int)n; cw.rows_per_cta = pl.rows_per_cta; cw.ws = wsbig; cw.wsb = wssmall;
        { ProfScope ps(s, "conv1_wgrad", 2.0 * n * 400 * 32 * 256, (double)n * (28672 + 14112 * 2));
          if ((rc = launch_conv1_wgrad_u8(cw, obs_aux, rows ? (int64_t)1 << 24 : n, act + Q.dact1, pl.splits, s, "naturecnn/conv1_wgrad_u8"))) return rc; }
        memset(&fw, 0, sizeof(fw));
        fw.layer = 1; fw.S = pl.splits; fw.nslots = 4; fw.Cout = 32; fw.scale = 1.0f / 255.0f / kDact1Scale; fw.bscale = 1.0f / kDact1Scale;
        const int st1[4] = {0, 1, 2, 3};               // ws rows: tile b, lane m -> tap 2 b + (m >> 6)
        for (int k = 0; k < 4; ++k) fw.slot_tap[k] = st1[k];
        { ProfScope ps(s, "wgrad_fold_bias", 0, 0);
          fw.wsb = wssmall; fw.db = grads + L.c1b;
          tc_fold_win<<<(unsigned)ceil_div(256 * 32 + 32, 32), 256, 0, s>>>(wsbig, fw, grads + L.c1w);
          if ((rc = check_launch("naturecnn/conv1_fold"))) return rc; }
    } else {
        wgw_defaults(gw);
        gw.X = x0; gw.rows = x0rows; gw.M = n * 512; gw.n = (int)n; gw.G = 441; gw.cpr = 1; gw.nslots = 4; gw.WRX = round8(128 + 22);
        gw.tpi_shift = 2; gw.n_images = x0rows ? (int64_t)1 << 24 : n;       // 4 steps of 128 grid rows per image
        gw.shift[0] = 0; gw.shift[1] = 1; gw.shift[2] = 21; gw.shift[3] = 22;
        for (int k = 0; k < 4; ++k) { gw.slot_tap[k] = k; gw.slot_cc[k] = 0; }
        gw.Y = act + Q.dact1; gw.ldy = 32; gw.ncolsY = 32;
        const WPlan pl = wgrad_plan(n * 512, kC1Ctas, 128);
        gw.rows_per_cta = pl.rows_per_cta; gw.ws = wsbig; gw.wsb = wssmall;
        { ProfScope ps(s, "conv1_wgrad", 2.0 * n * 400 * 32 * 256, (double)n * (28224 + 14112) * 2);
          if ((rc = launch_wgrad_win(gw, pl.splits, s, "naturecnn/conv1_wgrad"))) return rc; }
        memset(&fw, 0, sizeof(fw));
        fw.layer = 1; fw.S = pl.splits; fw.nslots = 4; fw.Cout = 32; fw.scale = 1.0f / 255.0f; fw.bscale = 1.f;
        for (int k = 0; k < 4; ++k) fw.slot_tap[k] = k;
        { ProfScope ps(s, "wgrad_fold_bias", 0, 0);
          fw.wsb = wssmall; fw.db = grads + L.c1b;
          tc_fold_win<<<(unsigned)ceil_div(256 * 32 + 32, 32), 256, 0, s>>>(wsbig, fw, grads + L.c1w);
          if ((rc = check_launch("naturecnn/conv1_fold"))) return rc; }
    }
    return B200RL_OK;
}
