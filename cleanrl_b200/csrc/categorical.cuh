// Categorical distribution arithmetic shared by the samplers (policy.cu, the fused heads+sampler of tc_heads.cuh) and the
// loss kernels of policy.cu.
#pragma once
#include <cuda_runtime.h>
#include <cfloat>

namespace b200rl {

// Normalised logits / probs of one row exactly as torch builds them:
//   lse = log(sum exp(x - max)) + max ; nl = x - lse            (Categorical ctor)
//   p   = exp(nl - max(nl)) / sum exp(nl - max(nl))              (softmax of nl)
struct RowStats {
    float lse;   // logsumexp of raw logits
    float m2;    // max of normalised logits
    float s2;    // sum exp(nl - m2)
};

__device__ __forceinline__ RowStats row_stats(const float* __restrict__ x, int A) {
    float m = -INFINITY;
    for (int k = 0; k < A; ++k) m = fmaxf(m, x[k]);
    const float mm = (fabsf(m) == INFINITY) ? 0.f : m;
    float s = 0.f;
    for (int k = 0; k < A; ++k) s += expf(x[k] - mm);
    RowStats r;
    r.lse = logf(s) + mm;
    float m2 = -INFINITY;
    for (int k = 0; k < A; ++k) m2 = fmaxf(m2, x[k] - r.lse);
    float s2 = 0.f;
    for (int k = 0; k < A; ++k) s2 += expf((x[k] - r.lse) - m2);
    r.m2 = m2;
    r.s2 = s2;
    return r;
}

// Gumbel-free exact sampling with Exp(1) noise q: argmax_k p_k / q_k (strict > keeps the first maximum, as torch's
// argmax).  ENT: also return the entropy sum_k nl_k p_k (negated by the caller).
template <bool ENT>
__device__ __forceinline__ int categorical_draw(const float* __restrict__ x, const float* __restrict__ q, int A, const RowStats& rs,
                                                float* ent_out) {
    float best = -INFINITY, ent = 0.f;
    int arg = 0;
    for (int k = 0; k < A; ++k) {
        const float nl = x[k] - rs.lse;
        const float p = expf(nl - rs.m2) / rs.s2;
        const float sc = p / q[k];
        if (sc > best) { best = sc; arg = k; }  // strict > keeps the first maximum (torch argmax)
        if (ENT) ent += fmaxf(nl, -FLT_MAX) * p;
    }
    if (ENT) *ent_out = ent;
    return arg;
}

}  // namespace b200rl
