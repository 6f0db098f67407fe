// policy_f32.cuh — the policy forward pass in the reference's own arithmetic: fp32 operands, fp32 accumulation, exact
// erf-GELU / sigmoid / tanh, no folded or rescaled weights (fl_policy_forward_f32).
//
// The tensor-core path of policy.cu multiplies in bf16; its logits agree with the reference network to about 1e-2,
// which is enough to choose the same action almost always but is not the reference's arithmetic.  This path is: every
// product of solution/nn/net_tree.py / TreeLSTM.py is evaluated as torch evaluates it on the CPU — fp32 FMA on the CUDA
// cores — so that logits and values agree with the reference to summation-order rounding (about 1e-6) and the chosen
// actions are the reference's.  It costs what fp32 on CUDA cores costs (about 10x the tensor-core path) and exists for
// callers that need the reference's numbers, and as the yardstick of the bf16 path.
//
// Structure: one tiled SGEMM kernel (64 x 64 x 16 tiles, 4 x 4 outputs per thread, gathered rows, two concatenated A
// sources) for every matrix product; the Tree-LSTM runs level by level over per-level node lists built on the device
// (k_tl_*, policy_f32_grad.cuh), with small element-wise kernels for the gates (TreeLSTM.py:59-154); attention is one warp
// per (query, head).  The kernels are launched by ppograph::run (policy.cu), the one launch sequence of this forward and of
// the training forward.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace f32path {

constexpr int T_H = 128;        // tree embedding / hidden size
constexpr int NODES = 31;
constexpr int NF = 12;
constexpr int MAX_LEVELS = 11;

// ---- SGEMM: C[m][n] = act(sum_k A(m, k) * W[n][k] + bias[n]), m < M (M read from *d_M when d_M != nullptr) -------------
// A(m, k) = a1[row1(m) * lda1 + k] for k < K1, a2[m * lda2 + k - K1] for K1 <= k < K1 + K2; row1(m) = idx1 ? idx1[m] : m.
struct GemmArgs {
    const float *a1; const int32_t *idx1; long long lda1; int K1;
    const float *a2; long long lda2; int K2;
    const float *w; const float *bias; float *c; long long ldc;
    long long M; const int32_t *d_M; int N; int act;      // act: 0 none, 1 GELU(erf)
    float *pre;                                           // when set: the value before the activation, at c's offsets (training forward)
};

__device__ __forceinline__ float gelu_erf(float x) { return x * 0.5f * (1.0f + erff(x * 0.70710678118654752440f)); }
__device__ __forceinline__ float sigmoid_f(float x) { return 1.0f / (1.0f + expf(-x)); }

__global__ void __launch_bounds__(256) k_gemm_f32(GemmArgs g) {
    __shared__ float sa[16][64 + 4], sw[16][64 + 4];
    const long long M = g.d_M ? (long long)*g.d_M : g.M;
    const long long m0 = (long long)blockIdx.x * 64;
    if (m0 >= M) return;
    const int n0 = blockIdx.y * 64, K = g.K1 + g.K2, tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;               // outputs: rows ty*4.., cols tx*4..
    float acc[4][4] = {};
    // loader mapping: 256 threads load a 64 x 16 tile: row = tid / 4, four consecutive k = (tid & 3) * 4
    const int lr = tid >> 2, lk = (tid & 3) * 4;
    const long long am = m0 + lr;
    long long arow1 = -1;
    if (am < M) arow1 = g.idx1 ? (long long)g.idx1[am] : am;
    const int wn = n0 + lr;
    for (int k0 = 0; k0 < K; k0 += 16) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int k = k0 + lk + u;
            float av = 0.0f, wv = 0.0f;
            if (am < M && k < K) av = k < g.K1 ? g.a1[arow1 * g.lda1 + k] : g.a2[am * g.lda2 + (k - g.K1)];
            if (wn < g.N && k < K) wv = g.w[(long long)wn * K + k];
            sa[lk + u][lr] = av;
            sw[lk + u][lr] = wv;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; kk++) {
            float a[4], w[4];
#pragma unroll
            for (int i = 0; i < 4; i++) { a[i] = sa[kk][ty * 4 + i]; w[i] = sw[kk][tx * 4 + i]; }
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const long long m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int n = n0 + tx * 4 + j;
            if (n >= g.N) continue;
            float v = acc[i][j] + (g.bias ? g.bias[n] : 0.0f);
            if (g.pre) g.pre[m * g.ldc + n] = v;
            if (g.act == 1) v = gelu_erf(v);
            g.c[m * g.ldc + n] = v;
        }
    }
}

// ---- Tree-LSTM --------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float clean(float f) { return (isinf(f) && f > 0.0f) ? -1.0f : f; }   // eval_env.py:76

// leaves (node_order == 0): iou = W_iou x + b; c = sigmoid(i) tanh(u); h = sigmoid(o) tanh(c)   (TreeLSTM.py:96-111 with no children)
__global__ void k_tree_leaves(const float *__restrict__ forest, const int32_t *__restrict__ node_order, long long n_nodes,
                              const float *__restrict__ wiou, const float *__restrict__ biou, float *__restrict__ h, float *__restrict__ c) {
    const long long node = blockIdx.x;
    if (node >= n_nodes || node_order[node] != 0) return;
    __shared__ float x[NF];
    if (threadIdx.x < NF) x[threadIdx.x] = clean(forest[node * NF + threadIdx.x]);
    __syncthreads();
    const int j = threadIdx.x;                               // 128 threads
    float g[3];
#pragma unroll
    for (int q = 0; q < 3; q++) {
        float a = 0.0f;
        for (int k = 0; k < NF; k++) a = fmaf(x[k], wiou[(q * T_H + j) * NF + k], a);
        g[q] = a + biou[q * T_H + j];
    }
    const float cn = sigmoid_f(g[0]) * tanhf(g[2]);
    c[node * T_H + j] = cn;
    h[node * T_H + j] = sigmoid_f(g[1]) * tanhf(cn);
}

// gather lists of one level: child node of every (parent m, k) and the merge row (first child) of every parent
__global__ void k_level_rows(const int32_t *__restrict__ list, const int32_t *__restrict__ d_M, const int8_t *__restrict__ child_base,
                             int32_t *__restrict__ merge_row, int32_t *__restrict__ child_row) {
    const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= *d_M) return;
    const int32_t node = list[m];
    const int32_t first = node - node % NODES + child_base[node];
    merge_row[m] = first;
    for (int k = 0; k < 3; k++) child_row[3 * m + k] = first + k;
}

// forget gates: fc[m][k*128 + j] = sigmoid(W_f x_m + b_f + U_f h_child)[j] * c_child[j]   (TreeLSTM.py:125-139)
__global__ void k_forget(const float *__restrict__ fraw, const int32_t *__restrict__ list, const int32_t *__restrict__ child_row,
                         const int32_t *__restrict__ d_M, const float *__restrict__ forest, const float *__restrict__ wf,
                         const float *__restrict__ bf, const float *__restrict__ c, float *__restrict__ fc) {
    const long long m = blockIdx.x;
    if (m >= *d_M) return;
    __shared__ float x[NF];
    const int32_t node = list[m];
    if (threadIdx.x < NF) x[threadIdx.x] = clean(forest[(long long)node * NF + threadIdx.x]);
    __syncthreads();
    const int j = threadIdx.x & 127, k = threadIdx.x >> 7;   // 384 threads: child k, unit j
    float a = 0.0f;
    for (int q = 0; q < NF; q++) a = fmaf(x[q], wf[j * NF + q], a);
    const float f = sigmoid_f((a + bf[j]) + fraw[(3 * m + k) * T_H + j]);
    fc[m * (3 * T_H) + k * T_H + j] = f * c[(long long)child_row[3 * m + k] * T_H + j];
}

// inner nodes: iou = (W_iou x + b) + U_iou merge; c = sigmoid(i) tanh(u) + (W_c fc + b_c); h = sigmoid(o) tanh(c)
__global__ void k_inner(const float *__restrict__ iou_raw, const float *__restrict__ craw, const int32_t *__restrict__ list,
                        const int32_t *__restrict__ d_M, const float *__restrict__ forest, const float *__restrict__ wiou,
                        const float *__restrict__ biou, const float *__restrict__ bc, float *__restrict__ h, float *__restrict__ c) {
    const long long m = blockIdx.x;
    if (m >= *d_M) return;
    __shared__ float x[NF];
    const int32_t node = list[m];
    if (threadIdx.x < NF) x[threadIdx.x] = clean(forest[(long long)node * NF + threadIdx.x]);
    __syncthreads();
    const int j = threadIdx.x;                               // 128 threads
    float g[3];
#pragma unroll
    for (int q = 0; q < 3; q++) {
        float a = 0.0f;
        for (int k = 0; k < NF; k++) a = fmaf(x[k], wiou[(q * T_H + j) * NF + k], a);
        g[q] = (a + biou[q * T_H + j]) + iou_raw[m * (3 * T_H) + q * T_H + j];
    }
    const float cn = sigmoid_f(g[0]) * tanhf(g[2]) + (craw[m * T_H + j] + bc[j]);
    c[(long long)node * T_H + j] = cn;
    h[(long long)node * T_H + j] = sigmoid_f(g[1]) * tanhf(cn);
}

// emb[:, 128:256] = h of the root node; cat buffers
__global__ void k_copy_cols(const float *__restrict__ src, long long lds, float *__restrict__ dst, long long ldd, long long rows, int cols) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * cols) return;
    const long long r = i / cols;
    const int cc = (int)(i - r * cols);
    dst[r * ldd + cc] = src[r * lds + cc];
}

// nn.MultiheadAttention over the agents of one environment (net_tree.py:20-32): one warp per (agent, head), 64 dims = 2 per
// lane; softmax with the running maximum; qkv [T][768] = q | k | v, out [T][ldo] columns head*64..; lse (when set, training
// forward): [T][4] log-sum-exp of the scores, from which the backward recomputes the probabilities
__global__ void k_attention(const float *__restrict__ qkv, float *__restrict__ out, long long ldo, long long n_env, int N,
                            float *__restrict__ lse) {
    const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (wid >= n_env * N * 4) return;
    const int head = (int)(wid & 3);
    const long long agent = wid >> 2, env = agent / N;
    const float scale = 0.125f;                               // 1 / sqrt(64)
    const float *q = qkv + agent * 768 + head * 64;
    const float q0 = q[lane] * scale, q1 = q[lane + 32] * scale;
    float mx = -INFINITY, den = 0.0f, o0 = 0.0f, o1 = 0.0f;
    for (int j = 0; j < N; j++) {
        const float *kp = qkv + (env * N + j) * 768 + 256 + head * 64;
        float s = q0 * kp[lane] + q1 * kp[lane + 32];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
        const float nm = fmaxf(mx, s), corr = expf(mx - nm), p = expf(s - nm);
        const float *vp = kp + 256;
        den = den * corr + p;
        o0 = o0 * corr + p * vp[lane];
        o1 = o1 * corr + p * vp[lane + 32];
        mx = nm;
    }
    out[agent * ldo + head * 64 + lane] = o0 / den;
    out[agent * ldo + head * 64 + lane + 32] = o1 / den;
    if (lse && lane == 0) lse[agent * 4 + head] = mx + logf(den);
}

// last layers: logits[a][0..4] = actor_net.4(y_actor[a]); value[env] = mean_a critic_net.4(y_critic[a])
__global__ void k_heads_final(const float *__restrict__ ya, const float *__restrict__ yc, const float *__restrict__ wa, const float *__restrict__ ba,
                              const float *__restrict__ wc, const float *__restrict__ bc, float *__restrict__ logits, float *__restrict__ value, int N) {
    const long long env = blockIdx.x;
    extern __shared__ float sv[];                               // [N] critic outputs
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int a = warp; a < N; a += nw) {
        const long long row = env * N + a;
        float acc[6];
#pragma unroll
        for (int o = 0; o < 6; o++) {
            const float *w = o < 5 ? wa + o * 128 : wc;
            const float *y = o < 5 ? ya + row * 128 : yc + row * 128;
            float s = 0.0f;
            for (int k = lane; k < 128; k += 32) s = fmaf(y[k], w[k], s);
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, d);
            acc[o] = s;
        }
        if (lane < 5) logits[row * 5 + lane] = acc[lane] + ba[lane];
        if (lane == 0) sv[a] = acc[5] + bc[0];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.0f;
        for (int a = 0; a < N; a++) s += sv[a];
        value[env] = s / (float)N;
    }
}

}  // namespace f32path
