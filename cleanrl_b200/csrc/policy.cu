// Categorical policy head: rollout-side sampling epilogue and the fused PPO
// minibatch loss (+ gradients wrt logits/value).
//
// Both kernels are one-thread-per-sample over tiny rows (A <= 64 logits), i.e.
// pure HBM/latency-bound elementwise work: rows are 4*A bytes, read once;
// per-sample scalars are gathered through mb_inds (random 4-B reads served
// by L2; the flat batch tensors are 512 KB each at N=1024,T=128).
// Algorithmic bytes per sample (loss): 4*A (logits) + 4 (value) + 8 (index)
// + 8+4*4 (action + 4 scalars) + 4*A + 4 (grads out) = 44 + 8*A.
#include "common.cuh"
#include "categorical.cuh"
#include <cfloat>

namespace b200rl {

constexpr int kMaxA = 64;

__global__ void __launch_bounds__(128) categorical_sample_kernel(
    const float* __restrict__ logits, int64_t ld, const float* __restrict__ noise,
    const float* __restrict__ value_in, int64_t ldv, int64_t n, int A,
    int64_t* __restrict__ action, float* __restrict__ logprob, float* __restrict__ entropy,
    float* __restrict__ value_out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* x = logits + i * ld;
    const float* q = noise + i * (int64_t)A;
    const RowStats rs = row_stats(x, A);
    float ent;
    const int arg = categorical_draw<true>(x, q, A, rs, &ent);
    action[i] = arg;
    logprob[i] = x[arg] - rs.lse;
    if (entropy) entropy[i] = -ent;
    if (value_out && value_in) value_out[i] = value_in[i * ldv];
}

// log_prob / entropy of GIVEN actions (Agent.get_action_and_value(x, action), ppo.py:121-126)
__global__ void __launch_bounds__(128) categorical_eval_kernel(
    const float* __restrict__ logits, int64_t ld, const int64_t* __restrict__ action, int64_t n, int A,
    float* __restrict__ logprob, float* __restrict__ entropy) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* x = logits + i * ld;
    const RowStats rs = row_stats(x, A);
    float ent = 0.f;
    for (int k = 0; k < A; ++k) {
        const float nl = x[k] - rs.lse;
        ent += fmaxf(nl, -FLT_MAX) * (expf(nl - rs.m2) / rs.s2);
    }
    int a = (int)action[i];
    a = a < 0 ? 0 : (a >= A ? A - 1 : a);
    logprob[i] = x[a] - rs.lse;
    if (entropy) entropy[i] = -ent;
}

// ---- advantage statistics of the gathered minibatch (single block, 2 passes).
// Loads are issued 8 at a time per thread (independent index -> value chains in flight), but every thread still
// accumulates its strided elements in ascending order, so the result does not depend on the batching.
__device__ __forceinline__ float adv_pass(const float* __restrict__ b_adv, const int64_t* __restrict__ inds, int64_t M,
                                          float mean, bool squared) {
    float s = 0.f;
    const int64_t step = blockDim.x;
    int64_t i = threadIdx.x;
    for (; i + 7 * step < M; i += 8 * step) {
        int64_t j[8];
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) j[u] = inds ? __ldg(inds + i + u * step) : i + u * step;
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = __ldg(b_adv + j[u]);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const float d = v[u] - mean;
            s += squared ? d * d : v[u];
        }
    }
    for (; i < M; i += step) {
        const float v = b_adv[inds ? inds[i] : i];
        const float d = v - mean;
        s += squared ? d * d : v;
    }
    return s;
}
__global__ void __launch_bounds__(1024) adv_stats_kernel(
    const float* __restrict__ b_adv, const int64_t* __restrict__ inds, int64_t M, float* __restrict__ out2) {
    __shared__ float red[32];
    const float mean = block_sum(adv_pass(b_adv, inds, M, 0.f, false), red) / (float)M;
    const float ss = block_sum(adv_pass(b_adv, inds, M, mean, true), red);
    if (threadIdx.x == 0) {
        out2[0] = mean;
        out2[1] = sqrtf(ss / (float)(M - 1));  // unbiased, torch.std default
    }
}

constexpr int kLossThreads = 256;
constexpr int kNumStats = 7;

struct LossParams {
    const float* logits; int64_t ld;
    const float* value; int64_t ldv;
    const int64_t* inds;
    const int64_t* b_actions;
    const float* b_logprobs; const float* b_adv; const float* b_ret; const float* b_val;
    int64_t M; int A;
    float clip, ent_coef, vf_coef;
    int norm_adv, clip_vloss;
    float* dlogits; int64_t ldd;
    float* dvalue; int64_t lddv;
    float* stats;
    const float* adv_stats;   // [2] mean, std
    float* partials;          // [gridDim.x][kNumStats]
    unsigned int* ticket;
};

__global__ void __launch_bounds__(kLossThreads) ppo_loss_kernel(LossParams P) {
    __shared__ float red[32];
    __shared__ bool is_last;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    float acc[kNumStats];
#pragma unroll
    for (int k = 0; k < kNumStats; ++k) acc[k] = 0.f;
    if (i < P.M) {
        const int64_t j = P.inds ? P.inds[i] : i;
        const float* x = P.logits + i * P.ld;
        const int A = P.A;
        const int a = (int)P.b_actions[j];
        const RowStats rs = row_stats(x, A);
        float ent = 0.f;
        for (int k = 0; k < A; ++k) {
            const float nl = x[k] - rs.lse;
            const float p = expf(nl - rs.m2) / rs.s2;
            ent += fmaxf(nl, -FLT_MAX) * p;
        }
        ent = -ent;
        const float newlogprob = x[a] - rs.lse;
        const float logratio = newlogprob - P.b_logprobs[j];
        const float ratio = expf(logratio);
        float adv = P.b_adv[j];
        if (P.norm_adv) adv = (adv - P.adv_stats[0]) / (P.adv_stats[1] + 1e-8f);
        const float lo = 1.f - P.clip, hi = 1.f + P.clip;
        const float rc = fminf(fmaxf(ratio, lo), hi);
        const float pg1 = -adv * ratio, pg2 = -adv * rc;
        const float pg = fmaxf(pg1, pg2);
        const float nv = P.value[i * P.ldv];
        const float R = P.b_ret[j], V = P.b_val[j];
        float vterm, gv;
        const float du = nv - R;
        const float vu = du * du;
        if (P.clip_vloss) {
            const float d = nv - V;
            const float vcl = V + fminf(fmaxf(d, -P.clip), P.clip);
            const float dc = vcl - R;
            const float vc = dc * dc;
            vterm = fmaxf(vu, vc);
            const float gu = 2.f * du;
            const float gc = (d >= -P.clip && d <= P.clip) ? 2.f * dc : 0.f;
            gv = (vu > vc) ? gu : ((vc > vu) ? gc : 0.5f * (gu + gc));
        } else {
            vterm = vu;
            gv = 2.f * du;
        }
        acc[0] = pg;
        acc[1] = vterm;
        acc[2] = ent;
        acc[3] = -logratio;
        acc[4] = (ratio - 1.f) - logratio;
        acc[5] = (fabsf(ratio - 1.0f) > P.clip) ? 1.f : 0.f;
        // gradients (torch autograd rules: max splits ties, clamp passes through inclusively)
        const float invM = 1.0f / (float)P.M;
        const float inrange = (ratio >= lo && ratio <= hi) ? 1.f : 0.f;
        float g_ratio = 0.f;
        if (pg1 > pg2) g_ratio = -adv;
        else if (pg1 == pg2) g_ratio = 0.5f * (-adv) * (1.f + inrange);
        const float g_lp = g_ratio * ratio * invM;
        const float g_ent = -P.ent_coef * invM;
        float* dl = P.dlogits + i * P.ldd;
        for (int k = 0; k < A; ++k) {
            const float nl = x[k] - rs.lse;
            const float p = expf(nl - rs.m2) / rs.s2;
            const float onehot = (k == a) ? 1.f : 0.f;
            dl[k] = g_lp * (onehot - p) + g_ent * (-p * (nl + ent));
        }
        P.dvalue[i * P.lddv] = P.vf_coef * 0.5f * invM * gv;
    }
    // ---- deterministic two-level reduction of the 6 sums
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const float s = block_sum(acc[k], red);
        if (threadIdx.x == 0) P.partials[(int64_t)blockIdx.x * kNumStats + k] = s;
    }
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned t = atomicAdd(P.ticket, 1u);
        is_last = (t == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    float tot[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        float s = 0.f;
        for (unsigned b = threadIdx.x; b < gridDim.x; b += blockDim.x)
            s += __ldcg(P.partials + (int64_t)b * kNumStats + k);
        tot[k] = block_sum(s, red);
    }
    if (threadIdx.x == 0) {
        const float invM = 1.0f / (float)P.M;
        const float pg_loss = tot[0] * invM;
        const float v_loss = 0.5f * (tot[1] * invM);
        const float ent_loss = tot[2] * invM;
        P.stats[0] = pg_loss;
        P.stats[1] = v_loss;
        P.stats[2] = ent_loss;
        P.stats[3] = tot[3] * invM;
        P.stats[4] = tot[4] * invM;
        P.stats[5] = tot[5] * invM;
        P.stats[6] = pg_loss - P.ent_coef * ent_loss + v_loss * P.vf_coef;
        P.stats[7] = P.norm_adv ? P.adv_stats[0] : 0.f;
        P.stats[8] = P.norm_adv ? P.adv_stats[1] : 1.f;
        *P.ticket = 0;  // re-arm for the next launch (graph replay safe)
    }
}


// ================================================================== diagonal Gaussian policy
// (cleanrl/ppo_continuous_action.py:134-141: Normal(mean, exp(logstd)), log_prob(a).sum(1), entropy().sum(1))
constexpr int kMaxD = 32;
constexpr float kLogSqrt2Pi = 0.9189385332046727f;   // math.log(math.sqrt(2*math.pi)) of torch/distributions/normal.py

__device__ __forceinline__ void gaussian_row(const float* __restrict__ mean, const float* __restrict__ logstd,
                                             const float* __restrict__ a, int D, float& logprob, float& entropy) {
    float lp = 0.f, ent = 0.f;
    for (int d = 0; d < D; ++d) {
        const float std = expf(logstd[d]);
        const float var = std * std;
        const float ls = logf(std);
        const float diff = a[d] - mean[d];
        lp += -(diff * diff) / (2.f * var) - ls - kLogSqrt2Pi;
        ent += 0.5f + kLogSqrt2Pi + ls;
    }
    logprob = lp;
    entropy = ent;
}

__global__ void __launch_bounds__(128) gaussian_sample_kernel(
    const float* __restrict__ mean, int64_t ld, const float* __restrict__ logstd, const float* __restrict__ noise,
    const float* __restrict__ value_in, int64_t ldv, int64_t n, int D,
    float* __restrict__ action, float* __restrict__ logprob, float* __restrict__ entropy, float* __restrict__ value_out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* m = mean + i * ld;
    float* a = action + i * D;
    for (int d = 0; d < D; ++d)   // torch.normal(mean, std): randn.mul_(std).add_(mean), separately rounded
        a[d] = __fadd_rn(__fmul_rn(noise[i * D + d], expf(logstd[d])), m[d]);
    float lp, ent;
    gaussian_row(m, logstd, a, D, lp, ent);
    logprob[i] = lp;
    if (entropy) entropy[i] = ent;
    if (value_out && value_in) value_out[i] = value_in[i * ldv];
}

__global__ void __launch_bounds__(128) gaussian_eval_kernel(
    const float* __restrict__ mean, int64_t ld, const float* __restrict__ logstd, const float* __restrict__ action,
    int64_t n, int D, float* __restrict__ logprob, float* __restrict__ entropy) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float lp, ent;
    gaussian_row(mean + i * ld, logstd, action + i * D, D, lp, ent);
    logprob[i] = lp;
    if (entropy) entropy[i] = ent;
}

struct GLossParams {
    const float* mean; int64_t ld;
    const float* logstd;
    const float* value; int64_t ldv;
    const int64_t* inds;
    const float* b_actions;      // [B, D]
    const float* b_logprobs; const float* b_adv; const float* b_ret; const float* b_val;
    int64_t M; int D;
    float clip, ent_coef, vf_coef;
    int norm_adv, clip_vloss;
    float* dmean; int64_t ldd;
    float* dlogstd;              // [D]
    float* dvalue; int64_t lddv;
    float* stats;
    const float* adv_stats;
    float* partials;             // [gridDim.x][kNumStats + kMaxD]
    unsigned int* ticket;
};

__global__ void __launch_bounds__(kLossThreads) ppo_loss_gaussian_kernel(GLossParams P) {
    __shared__ float red[32];
    __shared__ bool is_last;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int D = P.D;
    float acc[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) acc[k] = 0.f;
    float g_lp = 0.f;
    const float* m = nullptr;
    const float* a = nullptr;
    if (i < P.M) {
        const int64_t j = P.inds ? P.inds[i] : i;
        m = P.mean + i * P.ld;
        a = P.b_actions + j * D;
        float newlogprob, ent;
        gaussian_row(m, P.logstd, a, D, newlogprob, ent);
        const float logratio = newlogprob - P.b_logprobs[j];
        const float ratio = expf(logratio);
        float adv = P.b_adv[j];
        if (P.norm_adv) adv = (adv - P.adv_stats[0]) / (P.adv_stats[1] + 1e-8f);
        const float lo = 1.f - P.clip, hi = 1.f + P.clip;
        const float rc = fminf(fmaxf(ratio, lo), hi);
        const float pg1 = -adv * ratio, pg2 = -adv * rc;
        const float nv = P.value[i * P.ldv];
        const float R = P.b_ret[j], V = P.b_val[j];
        float vterm, gv;
        const float du = nv - R;
        const float vu = du * du;
        if (P.clip_vloss) {
            const float d = nv - V;
            const float vcl = V + fminf(fmaxf(d, -P.clip), P.clip);
            const float dc = vcl - R;
            const float vc = dc * dc;
            vterm = fmaxf(vu, vc);
            const float gu = 2.f * du;
            const float gc = (d >= -P.clip && d <= P.clip) ? 2.f * dc : 0.f;
            gv = (vu > vc) ? gu : ((vc > vu) ? gc : 0.5f * (gu + gc));
        } else {
            vterm = vu;
            gv = 2.f * du;
        }
        acc[0] = fmaxf(pg1, pg2);
        acc[1] = vterm;
        acc[2] = ent;
        acc[3] = -logratio;
        acc[4] = (ratio - 1.f) - logratio;
        acc[5] = (fabsf(ratio - 1.0f) > P.clip) ? 1.f : 0.f;
        const float invM = 1.0f / (float)P.M;
        const float inrange = (ratio >= lo && ratio <= hi) ? 1.f : 0.f;
        float g_ratio = 0.f;
        if (pg1 > pg2) g_ratio = -adv;
        else if (pg1 == pg2) g_ratio = 0.5f * (-adv) * (1.f + inrange);
        g_lp = g_ratio * ratio * invM;
        float* dm = P.dmean + i * P.ldd;
        for (int d = 0; d < D; ++d) {
            const float std = expf(P.logstd[d]);
            dm[d] = g_lp * (a[d] - m[d]) / (std * std);
        }
        P.dvalue[i * P.lddv] = P.vf_coef * 0.5f * invM * gv;
    }
    float* pb = P.partials + (int64_t)blockIdx.x * (kNumStats + kMaxD);
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        const float s = block_sum(acc[k], red);
        if (threadIdx.x == 0) pb[k] = s;
    }
    for (int d = 0; d < D; ++d) {   // d logprob / d logstd_d = (a-mean)^2 / var - 1
        float t = 0.f;
        if (i < P.M) {
            const float std = expf(P.logstd[d]);
            const float diff = a[d] - m[d];
            t = g_lp * (diff * diff / (std * std) - 1.f);
        }
        const float s = block_sum(t, red);
        if (threadIdx.x == 0) pb[kNumStats + d] = s;
    }
    if (threadIdx.x == 0) {
        __threadfence();
        is_last = (atomicAdd(P.ticket, 1u) == gridDim.x - 1);
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    float tot[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) {
        float s = 0.f;
        for (unsigned b = threadIdx.x; b < gridDim.x; b += blockDim.x) s += __ldcg(P.partials + (int64_t)b * (kNumStats + kMaxD) + k);
        tot[k] = block_sum(s, red);
    }
    for (int d = 0; d < D; ++d) {
        float s = 0.f;
        for (unsigned b = threadIdx.x; b < gridDim.x; b += blockDim.x) s += __ldcg(P.partials + (int64_t)b * (kNumStats + kMaxD) + kNumStats + d);
        const float t = block_sum(s, red);
        // entropy bonus: d(-ent_coef * mean(sum_d entropy_d)) / d logstd_d = -ent_coef
        if (threadIdx.x == 0) P.dlogstd[d] = t - P.ent_coef;
    }
    if (threadIdx.x == 0) {
        const float invM = 1.0f / (float)P.M;
        const float pg_loss = tot[0] * invM;
        const float v_loss = 0.5f * (tot[1] * invM);
        const float ent_loss = tot[2] * invM;
        P.stats[0] = pg_loss; P.stats[1] = v_loss; P.stats[2] = ent_loss;
        P.stats[3] = tot[3] * invM; P.stats[4] = tot[4] * invM; P.stats[5] = tot[5] * invM;
        P.stats[6] = pg_loss - P.ent_coef * ent_loss + v_loss * P.vf_coef;
        P.stats[7] = P.norm_adv ? P.adv_stats[0] : 0.f;
        P.stats[8] = P.norm_adv ? P.adv_stats[1] : 1.f;
        *P.ticket = 0;
    }
}

}  // namespace b200rl

extern "C" int b200rl_categorical_sample_f32(const float* logits, int64_t ld_logits, const float* noise,
                                             const float* value_in, int64_t ld_value,
                                             int64_t n, int A,
                                             int64_t* action, float* logprob, float* entropy, float* value_out,
                                             void* stream) {
    using namespace b200rl;
    B200RL_REQUIRE(n >= 0, "categorical_sample: negative n");
    if (n == 0) return B200RL_OK;
    B200RL_REQUIRE(A >= 1 && A <= kMaxA, "categorical_sample: A=%d outside [1,%d]", A, kMaxA);
    B200RL_REQUIRE(logits && noise && action && logprob, "categorical_sample: null pointer");
    B200RL_REQUIRE(ld_logits >= A, "categorical_sample: ld_logits < A");
    const unsigned blocks = (unsigned)ceil_div(n, 128);
    ProfScope ps((cudaStream_t)stream, "categorical_sample", 0, (double)n * (8.0 * A + 24));
    categorical_sample_kernel<<<blocks, 128, 0, (cudaStream_t)stream>>>(
        logits, ld_logits, noise, value_in, ld_value, n, A, action, logprob, entropy, value_out);
    return check_launch("categorical_sample");
}

extern "C" int b200rl_categorical_eval_f32(const float* logits, int64_t ld_logits, const int64_t* action,
                                           int64_t n, int A, float* logprob, float* entropy, void* stream) {
    using namespace b200rl;
    B200RL_REQUIRE(n >= 0, "categorical_eval: negative n");
    if (n == 0) return B200RL_OK;
    B200RL_REQUIRE(A >= 1 && A <= kMaxA, "categorical_eval: A=%d outside [1,%d]", A, kMaxA);
    B200RL_REQUIRE(logits && action && logprob, "categorical_eval: null pointer");
    B200RL_REQUIRE(ld_logits >= A, "categorical_eval: ld_logits < A");
    categorical_eval_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(
        logits, ld_logits, action, n, A, logprob, entropy);
    return check_launch("categorical_eval");
}

extern "C" size_t b200rl_ppo_loss_workspace_bytes(int64_t M) {
    using namespace b200rl;
    if (M < 0) return 0;
    const int64_t blocks = ceil_div(M > 0 ? M : 1, kLossThreads);
    // [0,16): adv stats (2 f32) ; [16,32): ticket ; then partials
    return 32 + (size_t)blocks * kNumStats * sizeof(float);
}

extern "C" int b200rl_ppo_loss_f32(const float* new_logits, int64_t ld_logits,
                                   const float* new_value, int64_t ld_value,
                                   const int64_t* mb_inds,
                                   const int64_t* b_actions, const float* b_logprobs,
                                   const float* b_advantages, const float* b_returns, const float* b_values,
                                   int64_t M, int A,
                                   double clip_coef, double ent_coef, double vf_coef,
                                   int norm_adv, int clip_vloss,
                                   float* dlogits, int64_t ld_dlogits, float* dvalue, int64_t ld_dvalue,
                                   float* stats, void* workspace, size_t workspace_bytes, void* stream) {
    using namespace b200rl;
    B200RL_REQUIRE(M >= 1, "ppo_loss: M must be >= 1 (got %lld)", (long long)M);
    B200RL_REQUIRE(!norm_adv || M >= 2, "ppo_loss: norm_adv needs M >= 2 (unbiased std)");
    B200RL_REQUIRE(A >= 1 && A <= kMaxA, "ppo_loss: A=%d outside [1,%d]", A, kMaxA);
    B200RL_REQUIRE(new_logits && new_value && b_actions && b_logprobs && b_advantages && b_returns && b_values,
                   "ppo_loss: null input pointer");
    B200RL_REQUIRE(dlogits && dvalue && stats, "ppo_loss: null output pointer");
    B200RL_REQUIRE(ld_logits >= A && ld_dlogits >= A && ld_value >= 1 && ld_dvalue >= 1, "ppo_loss: bad strides");
    B200RL_REQUIRE(workspace && aligned(workspace, 16), "ppo_loss: workspace null or not 16-B aligned");
    if (workspace_bytes < b200rl_ppo_loss_workspace_bytes(M))
        return fail(B200RL_ERR_WORKSPACE, "ppo_loss: workspace %zu < %zu bytes", workspace_bytes,
                    b200rl_ppo_loss_workspace_bytes(M));
    cudaStream_t s = (cudaStream_t)stream;
    float* adv_stats = reinterpret_cast<float*>(workspace);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(reinterpret_cast<char*>(workspace) + 16);
    float* partials = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + 32);
    ProfScope ps(s, "ppo_loss", 0, (double)M * (44.0 + 8.0 * A));
    cudaError_t e = cudaMemsetAsync(ticket, 0, sizeof(unsigned int), s);
    if (e != cudaSuccess) return fail(B200RL_ERR_CUDA, "ppo_loss: memset: %s", cudaGetErrorString(e));
    if (norm_adv) { note_launches(1); adv_stats_kernel<<<1, 1024, 0, s>>>(b_advantages, mb_inds, M, adv_stats); }
    LossParams P;
    P.logits = new_logits; P.ld = ld_logits; P.value = new_value; P.ldv = ld_value;
    P.inds = mb_inds; P.b_actions = b_actions; P.b_logprobs = b_logprobs; P.b_adv = b_advantages;
    P.b_ret = b_returns; P.b_val = b_values; P.M = M; P.A = A;
    P.clip = (float)clip_coef; P.ent_coef = (float)ent_coef; P.vf_coef = (float)vf_coef;
    P.norm_adv = norm_adv; P.clip_vloss = clip_vloss;
    P.dlogits = dlogits; P.ldd = ld_dlogits; P.dvalue = dvalue; P.lddv = ld_dvalue;
    P.stats = stats; P.adv_stats = adv_stats; P.partials = partials; P.ticket = ticket;
    const unsigned blocks = (unsigned)ceil_div(M, kLossThreads);
    ppo_loss_kernel<<<blocks, kLossThreads, 0, s>>>(P);
    return check_launch("ppo_loss");
}

extern "C" int b200rl_gaussian_sample_f32(const float* mean, int64_t ld_mean, const float* logstd, const float* noise,
                                          const float* value_in, int64_t ld_value, int64_t n, int D,
                                          float* action, float* logprob, float* entropy, float* value_out, void* stream) {
    using namespace b200rl;
    B200RL_REQUIRE(n >= 0, "gaussian_sample: negative n");
    if (n == 0) return B200RL_OK;
    B200RL_REQUIRE(D >= 1 && D <= kMaxD, "gaussian_sample: D=%d outside [1,%d]", D, kMaxD);
    B200RL_REQUIRE(mean && logstd && noise && action && logprob, "gaussian_sample: null pointer");
    B200RL_REQUIRE(ld_mean >= D, "gaussian_sample: ld_mean < D");
    ProfScope ps((cudaStream_t)stream, "gaussian_sample", 0, (double)n * (12.0 * D + 16));
    gaussian_sample_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(
        mean, ld_mean, logstd, noise, value_in, ld_value, n, D, action, logprob, entropy, value_out);
    return check_launch("gaussian_sample");
}

extern "C" int b200rl_gaussian_eval_f32(const float* mean, int64_t ld_mean, const float* logstd, const float* action,
                                        int64_t n, int D, float* logprob, float* entropy, void* stream) {
    using namespace b200rl;
    B200RL_REQUIRE(n >= 0, "gaussian_eval: negative n");
    if (n == 0) return B200RL_OK;
    B200RL_REQUIRE(D >= 1 && D <= kMaxD, "gaussian_eval: D=%d outside [1,%d]", D, kMaxD);
    B200RL_REQUIRE(mean && logstd && action && logprob, "gaussian_eval: null pointer");
    B200RL_REQUIRE(ld_mean >= D, "gaussian_eval: ld_mean < D");
    gaussian_eval_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(mean, ld_mean, logstd, action, n, D, logprob, entropy);
    return check_launch("gaussian_eval");
}

extern "C" size_t b200rl_ppo_loss_gaussian_workspace_bytes(int64_t M) {
    using namespace b200rl;
    if (M < 0) return 0;
    return 32 + (size_t)ceil_div(M > 0 ? M : 1, kLossThreads) * (kNumStats + kMaxD) * sizeof(float);
}

extern "C" int b200rl_ppo_loss_gaussian_f32(const float* new_mean, int64_t ld_mean, const float* logstd,
                                            const float* new_value, int64_t ld_value, const int64_t* mb_inds,
                                            const float* b_actions, const float* b_logprobs,
                                            const float* b_advantages, const float* b_returns, const float* b_values,
                                            int64_t M, int D, double clip_coef, double ent_coef, double vf_coef,
                                            int norm_adv, int clip_vloss,
                                            float* dmean, int64_t ld_dmean, float* dlogstd, float* dvalue, int64_t ld_dvalue,
                                            float* stats, void* workspace, size_t workspace_bytes, void* stream) {
    using namespace b200rl;
    B200RL_REQUIRE(M >= 1, "ppo_loss_gaussian: M must be >= 1");
    B200RL_REQUIRE(!norm_adv || M >= 2, "ppo_loss_gaussian: norm_adv needs M >= 2");
    B200RL_REQUIRE(D >= 1 && D <= kMaxD, "ppo_loss_gaussian: D=%d outside [1,%d]", D, kMaxD);
    B200RL_REQUIRE(new_mean && logstd && new_value && b_actions && b_logprobs && b_advantages && b_returns && b_values,
                   "ppo_loss_gaussian: null input pointer");
    B200RL_REQUIRE(dmean && dlogstd && dvalue && stats, "ppo_loss_gaussian: null output pointer");
    B200RL_REQUIRE(ld_mean >= D && ld_dmean >= D && ld_value >= 1 && ld_dvalue >= 1, "ppo_loss_gaussian: bad strides");
    B200RL_REQUIRE(workspace && aligned(workspace, 16), "ppo_loss_gaussian: workspace null or misaligned");
    if (workspace_bytes < b200rl_ppo_loss_gaussian_workspace_bytes(M))
        return fail(B200RL_ERR_WORKSPACE, "ppo_loss_gaussian: workspace %zu < %zu bytes", workspace_bytes,
                    b200rl_ppo_loss_gaussian_workspace_bytes(M));
    cudaStream_t s = (cudaStream_t)stream;
    float* adv_stats = reinterpret_cast<float*>(workspace);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(reinterpret_cast<char*>(workspace) + 16);
    float* partials = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + 32);
    ProfScope ps(s, "ppo_loss_gaussian", 0, (double)M * (48.0 + 12.0 * D));
    cudaError_t e = cudaMemsetAsync(ticket, 0, sizeof(unsigned int), s);
    if (e != cudaSuccess) return fail(B200RL_ERR_CUDA, "ppo_loss_gaussian: memset: %s", cudaGetErrorString(e));
    if (norm_adv) { note_launches(1); adv_stats_kernel<<<1, 1024, 0, s>>>(b_advantages, mb_inds, M, adv_stats); }
    GLossParams P;
    P.mean = new_mean; P.ld = ld_mean; P.logstd = logstd; P.value = new_value; P.ldv = ld_value; P.inds = mb_inds;
    P.b_actions = b_actions; P.b_logprobs = b_logprobs; P.b_adv = b_advantages; P.b_ret = b_returns; P.b_val = b_values;
    P.M = M; P.D = D; P.clip = (float)clip_coef; P.ent_coef = (float)ent_coef; P.vf_coef = (float)vf_coef;
    P.norm_adv = norm_adv; P.clip_vloss = clip_vloss;
    P.dmean = dmean; P.ldd = ld_dmean; P.dlogstd = dlogstd; P.dvalue = dvalue; P.lddv = ld_dvalue;
    P.stats = stats; P.adv_stats = adv_stats; P.partials = partials; P.ticket = ticket;
    ppo_loss_gaussian_kernel<<<(unsigned)ceil_div(M, kLossThreads), kLossThreads, 0, s>>>(P);
    return check_launch("ppo_loss_gaussian");
}
