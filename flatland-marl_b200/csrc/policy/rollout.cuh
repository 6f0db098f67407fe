// rollout.cuh — what a PPO rollout needs beyond the forward pass (include/flatland_policy_b200.h):
//   masked_choice   the soft choice of plfActor.py:27-44 for one agent and a given uniform, with the log-probability of the
//                   chosen action; k_choose (fixed uniform) and k_sample (seeded Philox uniform) both call it
//   k_sample        fl_policy_sample_actions: one thread per agent, counter-based draws (no generator state to keep)
//   k_gae           fl_policy_gae: one warp per environment, lanes reduce the agents' rewards, lane 0 runs the backward
//                   recurrence in float64
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace rollout {

// Philox4x32-10 (Salmon et al., SC'11; the Random123 constants): counter c, key k -> four 32-bit words in c.
__device__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; r++) {
        const uint32_t lo0 = 0xD2511F53u * c[0], hi0 = __umulhi(0xD2511F53u, c[0]);
        const uint32_t lo1 = 0xCD9E8D57u * c[2], hi1 = __umulhi(0xCD9E8D57u, c[2]);
        const uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}

// The uniform of agent i of global environment g at `step` (header comment of fl_policy_sample_actions): 53 bits, [0, 1).
__device__ __forceinline__ double uniform53(uint64_t seed, uint64_t step, uint32_t g, uint32_t i) {
    uint32_t c[4] = {(uint32_t)step, (uint32_t)(step >> 32), g, i};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    return ((double)(c[0] >> 5) * 67108864.0 + (double)(c[1] >> 6)) / 9007199254740992.0;
}

// np.random.choice(valid, p=softmax(logits[valid])) with its one uniform u: the first valid action whose normalised
// cumulative probability exceeds u; no valid action -> 0.  *log_prob (when given): fp32 masked log-softmax of the chosen
// action from the same exponentials, 0 when no action is valid.
__device__ __forceinline__ uint8_t masked_choice(const float *__restrict__ logits, const uint8_t *__restrict__ valid, double u,
                                                 float *log_prob) {
    float x[5];
    int idx[5], cnt = 0;
    for (int j = 0; j < 5; j++)
        if (valid[j]) { x[cnt] = logits[j]; idx[cnt++] = j; }
    if (cnt == 0) {
        if (log_prob) *log_prob = 0.0f;
        return 0;
    }
    float mx = x[0];
    for (int j = 1; j < cnt; j++) mx = fmaxf(mx, x[j]);
    float ex[5], sum = 0.0f;
    for (int j = 0; j < cnt; j++) { ex[j] = expf(x[j] - mx); sum += ex[j]; }
    double cdf[5], run = 0.0;
    for (int j = 0; j < cnt; j++) { run += (double)(ex[j] / sum); cdf[j] = run; }
    int pick = cnt - 1;
    for (int j = 0; j < cnt; j++)
        if (cdf[j] / run > u) { pick = j; break; }
    if (log_prob) *log_prob = (x[pick] - mx) - logf(sum);
    return (uint8_t)idx[pick];
}

// logits / valid / actions / log_probs: [E][N][5] / [E][N][5] / [E][N] / [E][N], one thread per agent.
__global__ void k_sample(const float *__restrict__ logits, const uint8_t *__restrict__ valid, long long E, long long N,
                         long long env_offset, uint64_t seed, uint64_t step, uint8_t *__restrict__ actions,
                         float *__restrict__ log_probs) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= E * N) return;
    const long long e = t / N, i = t - e * N;
    const double u = uniform53(seed, step, (uint32_t)(env_offset + e), (uint32_t)i);
    float lp;
    actions[t] = masked_choice(logits + t * 5, valid + t * 5, u, &lp);
    log_probs[t] = lp;
}

// GAE over a [T+1]-row buffer (fl_policy_gae): warp w of the grid handles environment e = w.  The agents' rewards of a row
// are summed exactly (int64), their mean is the reward the critic (a mean over agents) predicts.
__global__ void k_gae(const int32_t *__restrict__ rewards, const uint8_t *__restrict__ dones, const float *__restrict__ values,
                      const uint8_t *__restrict__ acted, long long T, long long E, long long N, double gamma, double lam,
                      float *__restrict__ adv, float *__restrict__ ret) {
    const long long e = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (e >= E) return;
    double a_next = 0.0;
    for (long long k = T - 1; k >= 0; k--) {
        const int32_t *r = rewards + ((k + 1) * E + e) * N;
        long long s = 0;
        for (long long i = lane; i < N; i += 32) s += r[i];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, d);
        if (lane == 0) {
            const long long ke = k * E + e;
            double a = 0.0, rt = 0.0;
            if (acted[ke]) {
                const double live = dones[((k + 1) * E + e) * (N + 1) + N] ? 0.0 : 1.0;
                const double v = (double)values[ke];
                // rounded operations (no FMA contraction): the same float64 bits as a plain left-to-right evaluation
                const double delta = __dsub_rn(__dadd_rn((double)s / (double)N, __dmul_rn(__dmul_rn(gamma, (double)values[ke + E]), live)), v);
                a = __dadd_rn(delta, __dmul_rn(__dmul_rn(__dmul_rn(gamma, lam), live), a_next));
                rt = __dadd_rn(a, v);
            }
            adv[ke] = (float)a;
            ret[ke] = (float)rt;
            a_next = a;
        }
    }
}

}  // namespace rollout
