// policy_f32_grad.cuh — the PPO loss of the fp32 network and its gradients with respect to every parameter
// (fl_policy_ppo_grad_f32, include/flatland_policy_b200.h).  Everything runs in fp32 on the CUDA cores.
//
// Training forward: the kernels of policy_f32.cuh launched by ppograph::run (policy.cu), which is also fl_policy_forward_f32,
// so logits and values are bit-identical to it.  For training every level and layer writes its own slice of the workspace,
// the GEMMs also store their pre-activations (GemmArgs::pre) and attention its log-sum-exp per (agent, head); the forward
// alone carves a smaller layout without them (carve, train = false).  The level lists are built in a fixed order (tree
// order, then node order; k_tl_*) with no atomics, because the weight gradients reduce over their rows.
//
// Loss: k_ppo_count (|S| and the number of acted rows; int64 integer atomics, exact in any order and across shards),
// k_ppo_loss (one CTA per environment row: log pi with masked_choice's arithmetic, clipped surrogate, entropy, value term,
// d loss / d logits and d loss / d critic output), k_ppo_stats (one CTA, fixed-order reduction of the per-row sums).  The
// loss and the statistics divide by the denominators in PpoArgs::gcnt: the call's own counts, or the counts of the whole
// minibatch when the rows are one shard of it (fl_policy_ppo_grad_shard_*).  The loss options (FlPpoOptions,
// fl_policy_ppo_grad_ex_*) run in k_ppo_loss<true>: advantages normalised by the float64 moments in PpoArgs::gmom (the
// minibatch's, or these rows' from k_ppo_moments, one CTA in a fixed order) and the clipped value term; k_ppo_loss<false> is
// the plain loss.
//
// Backward: k_gemm_dx (dX = dY W, optional gathered output rows, added term, accumulation and GELU' epilogue), k_gemm_dw +
// k_dw_reduce (dW = dY^T X and db over fixed row chunks into partial buffers, then summed in chunk order), k_attn_bwd_q /
// k_attn_bwd_kv (one warp per (query, head) and per (key, head), P recomputed from the log-sum-exp), k_inner_bwd /
// k_forget_bwd (Tree-LSTM gates, from the deepest level down to the leaves; every child has one parent, so child rows are
// written without atomics).  No floating-point atomics: two calls with the same inputs give the same bytes.
#pragma once
#include "policy_f32.cuh"

namespace f32grad {
using namespace f32path;

constexpr int MAX_CHUNKS = 128;   // row chunks of one weight-gradient reduction (bounds the partial buffer)
constexpr int MIN_CHUNK = 64;     // fewest rows per chunk
constexpr int SCAN = 1024;        // trees per block of the level-list scan
constexpr int DW_MAX = 768 * 257; // largest N x (K + 1) of a weight gradient (in_proj with its bias)

__device__ __forceinline__ float gelu_grad(float x) {
    return 0.5f * (1.0f + erff(x * 0.70710678118654752440f)) + x * 0.39894228040143267794f * expf(-0.5f * x * x);
}

// ---- level lists in a fixed order --------------------------------------------------------------------------------------
// per tree: first child of every node (adjacency rows of one parent are consecutive, child of row r is r + 1:
// TreeLSTM.py:118-119) and the number of nodes of every level 0..10 -> tcnt[lv][t]
__global__ void k_tl_count(const int32_t *__restrict__ adj, const int32_t *__restrict__ node_order, long long T,
                           int8_t *__restrict__ child_base, int32_t *__restrict__ tcnt) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    int8_t cb[f32path::NODES];
    for (int n = 0; n < f32path::NODES; n++) cb[n] = -1;
    for (int r = f32path::NODES - 2; r >= 0; r--) {
        const int p = adj[(t * (f32path::NODES - 1) + r) * 3];
        if (p >= 0 && p < f32path::NODES) cb[p] = (int8_t)(r + 1);    // descending r: ends on the first row of the parent
    }
    int cnt[MAX_LEVELS];
    for (int l = 0; l < MAX_LEVELS; l++) cnt[l] = 0;
    for (int n = 0; n < f32path::NODES; n++) {
        child_base[t * f32path::NODES + n] = cb[n];
        const int lv = node_order[t * f32path::NODES + n];
        if (lv >= 0 && lv < MAX_LEVELS) cnt[lv]++;
    }
    for (int l = 0; l < MAX_LEVELS; l++) tcnt[l * T + t] = cnt[l];
}

// grid (blocks of SCAN trees, level): exclusive prefix of tcnt inside the block -> tpos, block total -> btot[lv][blk]
__global__ void __launch_bounds__(SCAN) k_tl_scan(const int32_t *__restrict__ tcnt, long long T, int nblk, int32_t *__restrict__ tpos,
                                                  int32_t *__restrict__ btot) {
    __shared__ int wsum[32];
    const int lv = blockIdx.y, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long t = (long long)blockIdx.x * SCAN + threadIdx.x;
    const int v = t < T ? tcnt[lv * T + t] : 0;
    int x = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int y = __shfl_up_sync(0xFFFFFFFFu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    if (warp == 0) {
        int y = wsum[lane];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int z = __shfl_up_sync(0xFFFFFFFFu, y, d);
            if (lane >= d) y += z;
        }
        wsum[lane] = y;
    }
    __syncthreads();
    if (t < T) tpos[lv * T + t] = x - v + (warp ? wsum[warp - 1] : 0);
    if (threadIdx.x == SCAN - 1) btot[lv * nblk + blockIdx.x] = wsum[31];
}

// one CTA: block totals -> block offsets (in place), counts[lv] = nodes of level lv, counts[16 + lv] = list offset of level lv
__global__ void k_tl_tops(int32_t *__restrict__ btot, int nblk, int32_t *__restrict__ counts) {
    const int lv = threadIdx.x;
    if (lv < MAX_LEVELS) {
        int run = 0;
        for (int b = 0; b < nblk; b++) {
            const int v = btot[lv * nblk + b];
            btot[lv * nblk + b] = run;
            run += v;
        }
        counts[lv] = run;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int off = 0;
        for (int l = 0; l <= MAX_LEVELS; l++) {
            counts[16 + l] = off;
            if (l < MAX_LEVELS) off += counts[l];
        }
    }
}

// one thread per tree: its nodes of every level, in node order, at their list positions
__global__ void k_tl_fill(const int32_t *__restrict__ node_order, long long T, int nblk, const int32_t *__restrict__ tpos,
                          const int32_t *__restrict__ boff, const int32_t *__restrict__ counts, int32_t *__restrict__ lists) {
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= T) return;
    const int blk = (int)(t / SCAN);
    int pos[MAX_LEVELS];
    for (int l = 0; l < MAX_LEVELS; l++) pos[l] = counts[16 + l] + boff[l * nblk + blk] + tpos[l * T + t];
    for (int n = 0; n < f32path::NODES; n++) {
        const int lv = node_order[t * f32path::NODES + n];
        if (lv >= 0 && lv < MAX_LEVELS) lists[pos[lv]++] = (int32_t)(t * f32path::NODES + n);
    }
}

// node features with +inf replaced (eval_env.py:76), the X operand of W_iou's and W_f's gradients
__global__ void k_clean(const float *__restrict__ forest, float *__restrict__ x, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) x[i] = clean(forest[i]);
}

// ---- dense backward ----------------------------------------------------------------------------------------------------
// C[row(m)][k] = gelu'(pre[m][k]) * (sum_n A[m][n] W[n][k] + add[m][k] + C_old[row(m)][k]), row(m) = cidx ? cidx[m] : m;
// every term but the product optional.  64 x 64 x 16 tiles as k_gemm_f32; the reduction runs over W's rows.
struct DxArgs {
    const float *a; long long lda; int Nn;            // A [M][Nn]
    const float *w; long long ldw; int K;             // W [Nn][ldw], columns 0..K-1
    float *c; const int32_t *cidx; long long ldc;
    const float *add; long long ldadd; int accum;
    const float *pre; long long ldpre;
    long long M;
};

__global__ void __launch_bounds__(256) k_gemm_dx(DxArgs g) {
    __shared__ float sa[16][64 + 4], sw[16][64 + 4];
    const long long m0 = (long long)blockIdx.x * 64;
    const int k0 = blockIdx.y * 64, tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    float acc[4][4] = {};
    const int lr = tid >> 2, ln = (tid & 3) * 4;              // A loader: row, four consecutive n
    const int wr = tid >> 4, wc = (tid & 15) * 4;             // W loader: n, four consecutive k
    const long long am = m0 + lr;
    for (int n0 = 0; n0 < g.Nn; n0 += 16) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int n = n0 + ln + u;
            sa[ln + u][lr] = (am < g.M && n < g.Nn) ? g.a[am * g.lda + n] : 0.0f;
            const int wn = n0 + wr, wk = k0 + wc + u;
            sw[wr][wc + u] = (wn < g.Nn && wk < g.K) ? g.w[(long long)wn * g.ldw + wk] : 0.0f;
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
        if (m >= g.M) continue;
        const long long row = g.cidx ? (long long)g.cidx[m] : m;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int k = k0 + tx * 4 + j;
            if (k >= g.K) continue;
            float v = acc[i][j];
            if (g.add) v += g.add[m * g.ldadd + k];
            if (g.accum) v += g.c[row * g.ldc + k];
            if (g.pre) v *= gelu_grad(g.pre[m * g.ldpre + k]);
            g.c[row * g.ldc + k] = v;
        }
    }
}

// partial[z][n][k] = sum over rows m of chunk z of dY[m][n] X(m, k); X(m, k) = x1[row1(m)][k] (k < K1), x2[m][k - K1]
// (K1 <= k < K1 + K2), 1 (k == K1 + K2, when bias: the bias gradient)
struct DwArgs {
    const float *dy; long long ldy; int N;
    const float *x1; const int32_t *idx1; long long ldx1; int K1;
    const float *x2; long long ldx2; int K2;
    int bias;
    long long M, chunk;
    float *part;
};

__global__ void __launch_bounds__(256) k_gemm_dw(DwArgs g) {
    __shared__ float sy[16][64 + 4], sx[16][64 + 4];
    const int n0 = blockIdx.x * 64, k0 = blockIdx.y * 64, tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int Kp = g.K1 + g.K2 + g.bias;
    const long long r0 = (long long)blockIdx.z * g.chunk, r1 = min(g.M, r0 + g.chunk);
    float acc[4][4] = {};
    const int lr = tid >> 4, lc = (tid & 15) * 4;
    for (long long m = r0; m < r1; m += 16) {
        const long long mm = m + lr;
        const bool ok = mm < r1;
        const long long row1 = ok ? (g.idx1 ? (long long)g.idx1[mm] : mm) : 0;
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int n = n0 + lc + u, k = k0 + lc + u;
            sy[lr][lc + u] = (ok && n < g.N) ? g.dy[mm * g.ldy + n] : 0.0f;
            float xv = 0.0f;
            if (ok && k < Kp) xv = k < g.K1 ? g.x1[row1 * g.ldx1 + k] : (k < g.K1 + g.K2 ? g.x2[mm * g.ldx2 + (k - g.K1)] : 1.0f);
            sx[lr][lc + u] = xv;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; kk++) {
            float y[4], x[4];
#pragma unroll
            for (int i = 0; i < 4; i++) { y[i] = sy[kk][ty * 4 + i]; x[i] = sx[kk][tx * 4 + i]; }
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 4; j++) acc[i][j] = fmaf(y[i], x[j], acc[i][j]);
        }
        __syncthreads();
    }
    float *out = g.part + (long long)blockIdx.z * g.N * Kp;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const int n = n0 + ty * 4 + i;
        if (n >= g.N) continue;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int k = k0 + tx * 4 + j;
            if (k < Kp) out[(long long)n * Kp + k] = acc[i][j];
        }
    }
}

// dW[n][k] (row stride K) and db[n] (column K of the partials, when db) = sum of the nch partials in chunk order; 0 when nch = 0
__global__ void k_dw_reduce(const float *__restrict__ part, int nch, int N, int K, int bias, float *__restrict__ dw, float *__restrict__ db) {
    const int Kp = K + bias;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)N * Kp) return;
    float s = 0.0f;
    for (int c = 0; c < nch; c++) s += part[(long long)c * N * Kp + i];
    const int n = (int)(i / Kp), k = (int)(i - (long long)n * Kp);
    if (k < K) dw[(long long)n * K + k] = s;
    else db[n] = s;
}

// dst[r][c] = src[r][c] * gelu'(pre[r][c]), c < cols
__global__ void k_gelu_bwd(const float *__restrict__ src, long long lds, const float *__restrict__ pre, long long ldp,
                           float *__restrict__ dst, long long ldd, long long rows, int cols) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * cols) return;
    const long long r = i / cols;
    const int cc = (int)(i - r * cols);
    dst[r * ldd + cc] = src[r * lds + cc] * gelu_grad(pre[r * ldp + cc]);
}

// ---- attention backward (k_attention's softmax, P = exp(s - lse)) ------------------------------------------------------
// one warp per (query i, head): D_i = dO_i . O_i -> Dq[i][head]; dq_i = scale * sum_j P_ij (dO_i . v_j - D_i) k_j
__global__ void k_attn_bwd_q(const float *__restrict__ qkv, const float *__restrict__ o, const float *__restrict__ dout,
                             const float *__restrict__ lse, float *__restrict__ dqkv, float *__restrict__ Dq, long long n_env, int N) {
    const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (wid >= n_env * N * 4) return;
    const int head = (int)(wid & 3);
    const long long agent = wid >> 2, env = agent / N;
    const float scale = 0.125f;
    const float *q = qkv + agent * 768 + head * 64;
    const float q0 = q[lane] * scale, q1 = q[lane + 32] * scale;
    const float do0 = dout[agent * 256 + head * 64 + lane], do1 = dout[agent * 256 + head * 64 + lane + 32];
    float D = do0 * o[agent * 256 + head * 64 + lane] + do1 * o[agent * 256 + head * 64 + lane + 32];
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) D += __shfl_xor_sync(0xFFFFFFFFu, D, d);
    const float L = lse[agent * 4 + head];
    float dq0 = 0.0f, dq1 = 0.0f;
    for (int j = 0; j < N; j++) {
        const float *kp = qkv + (env * N + j) * 768 + 256 + head * 64, *vp = kp + 256;
        const float k0 = kp[lane], k1 = kp[lane + 32];
        float s = q0 * k0 + q1 * k1, dp = do0 * vp[lane] + do1 * vp[lane + 32];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            s += __shfl_xor_sync(0xFFFFFFFFu, s, d);
            dp += __shfl_xor_sync(0xFFFFFFFFu, dp, d);
        }
        const float ds = expf(s - L) * (dp - D);
        dq0 = fmaf(ds, k0, dq0);
        dq1 = fmaf(ds, k1, dq1);
    }
    dqkv[agent * 768 + head * 64 + lane] = dq0 * scale;
    dqkv[agent * 768 + head * 64 + lane + 32] = dq1 * scale;
    if (lane == 0) Dq[agent * 4 + head] = D;
}

// one warp per (key j, head): dv_j = sum_i P_ij dO_i, dk_j = scale * sum_i P_ij (dO_i . v_j - D_i) q_i
__global__ void k_attn_bwd_kv(const float *__restrict__ qkv, const float *__restrict__ dout, const float *__restrict__ lse,
                              const float *__restrict__ Dq, float *__restrict__ dqkv, long long n_env, int N) {
    const long long wid = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (wid >= n_env * N * 4) return;
    const int head = (int)(wid & 3);
    const long long agent = wid >> 2, env = agent / N;
    const float scale = 0.125f;
    const float *kp = qkv + agent * 768 + 256 + head * 64, *vp = kp + 256;
    const float k0 = kp[lane], k1 = kp[lane + 32], v0 = vp[lane], v1 = vp[lane + 32];
    float dk0 = 0.0f, dk1 = 0.0f, dv0 = 0.0f, dv1 = 0.0f;
    for (int i = 0; i < N; i++) {
        const long long qi = env * N + i;
        const float *q = qkv + qi * 768 + head * 64;
        const float q0 = q[lane] * scale, q1 = q[lane + 32] * scale;
        const float do0 = dout[qi * 256 + head * 64 + lane], do1 = dout[qi * 256 + head * 64 + lane + 32];
        float s = q0 * k0 + q1 * k1, dp = do0 * v0 + do1 * v1;
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            s += __shfl_xor_sync(0xFFFFFFFFu, s, d);
            dp += __shfl_xor_sync(0xFFFFFFFFu, dp, d);
        }
        const float p = expf(s - lse[qi * 4 + head]), ds = p * (dp - Dq[qi * 4 + head]);
        dv0 = fmaf(p, do0, dv0);
        dv1 = fmaf(p, do1, dv1);
        dk0 = fmaf(ds, q0, dk0);
        dk1 = fmaf(ds, q1, dk1);
    }
    dqkv[agent * 768 + 256 + head * 64 + lane] = dk0;
    dqkv[agent * 768 + 256 + head * 64 + lane + 32] = dk1;
    dqkv[agent * 768 + 512 + head * 64 + lane] = dv0;
    dqkv[agent * 768 + 512 + head * 64 + lane + 32] = dv1;
}

// ---- Tree-LSTM backward ------------------------------------------------------------------------------------------------
// nodes of one level (list[m]), k_inner / k_tree_leaves recomputed: g = (W_iou x + b) [+ iou_raw]; c, dh, dc of the node ->
// dG[m] = d(i, o, u pre-activations) and, for inner nodes, dC[m] = d(c) (= d(W_c fc + b_c)); leaves pass iou_raw = dC = null
__global__ void k_inner_bwd(const float *__restrict__ iou_raw, const int32_t *__restrict__ list, const float *__restrict__ xcl,
                            const float *__restrict__ wiou, const float *__restrict__ biou, const float *__restrict__ c,
                            const float *__restrict__ dh, const float *__restrict__ dc, float *__restrict__ dG, float *__restrict__ dC) {
    const long long m = blockIdx.x;
    __shared__ float x[NF];
    const int32_t node = list[m];
    if (threadIdx.x < NF) x[threadIdx.x] = xcl[(long long)node * NF + threadIdx.x];
    __syncthreads();
    const int j = threadIdx.x;
    float g[3];
#pragma unroll
    for (int q = 0; q < 3; q++) {
        float a = 0.0f;
        for (int k = 0; k < NF; k++) a = fmaf(x[k], wiou[(q * T_H + j) * NF + k], a);
        g[q] = iou_raw ? (a + biou[q * T_H + j]) + iou_raw[m * (3 * T_H) + q * T_H + j] : a + biou[q * T_H + j];
    }
    const float si = sigmoid_f(g[0]), so = sigmoid_f(g[1]), tu = tanhf(g[2]);
    const float tc = tanhf(c[(long long)node * T_H + j]), dhv = dh[(long long)node * T_H + j];
    const float dcc = dc[(long long)node * T_H + j] + dhv * so * (1.0f - tc * tc);
    dG[m * (3 * T_H) + j] = dcc * tu * si * (1.0f - si);
    dG[m * (3 * T_H) + T_H + j] = dhv * tc * so * (1.0f - so);
    dG[m * (3 * T_H) + 2 * T_H + j] = dcc * si * (1.0f - tu * tu);
    if (dC) dC[m * T_H + j] = dcc;
}

// forget gates of one level (k_forget recomputed: f = sigmoid((W_f x_parent + b_f) + U_f h_child)); dfc = d(f * c_child) ->
// dc of the child (written: it has one parent), dF[3m + k] = d(f pre-activation), dFs[m] = sum over the three children (the
// operand of W_f is the parent's features)
__global__ void k_forget_bwd(const float *__restrict__ fraw, const int32_t *__restrict__ list, const int32_t *__restrict__ child_row,
                             const float *__restrict__ xcl, const float *__restrict__ wf, const float *__restrict__ bf,
                             const float *__restrict__ c, const float *__restrict__ dfc, float *__restrict__ dc, float *__restrict__ dF,
                             float *__restrict__ dFs) {
    const long long m = blockIdx.x;
    __shared__ float x[NF], sdf[3][T_H];
    const int32_t node = list[m];
    if (threadIdx.x < NF) x[threadIdx.x] = xcl[(long long)node * NF + threadIdx.x];
    __syncthreads();
    const int j = threadIdx.x & 127, k = threadIdx.x >> 7;
    float a = 0.0f;
    for (int q = 0; q < NF; q++) a = fmaf(x[q], wf[j * NF + q], a);
    const float f = sigmoid_f((a + bf[j]) + fraw[(3 * m + k) * T_H + j]);
    const long long crow = child_row[3 * m + k];
    const float d = dfc[m * (3 * T_H) + k * T_H + j];
    dc[crow * T_H + j] = d * f;
    const float df = d * c[crow * T_H + j] * f * (1.0f - f);
    dF[(3 * m + k) * T_H + j] = df;
    sdf[k][j] = df;
    __syncthreads();
    if (k == 0) dFs[m * T_H + j] = (sdf[0][j] + sdf[1][j]) + sdf[2][j];
}

// ---- PPO loss ----------------------------------------------------------------------------------------------------------
struct PpoArgs {
    const float *logits, *value, *old_lp, *adv, *ret;
    const uint8_t *valid, *actions, *acted;
    long long E; int N;
    float eps, vf, ent;
    unsigned long long *cnt;            // [0] |S|, [1] acted rows of these rows (k_ppo_count; zeroed before it)
    float *dlogits, *dcrit, *rowstats;  // [T][5], [T], [E][5]
    const long long *gcnt;              // the denominators: [0] |S|, [1] acted rows of the whole minibatch (cnt for one shard)
    // options (k_ppo_loss<true> only): vf_clip > 0 clips the value term around old_values [E]; norm_adv normalises A by the
    // minibatch moments gmom = [sum_S A, sum_S A^2] (float64) with the denominator sigma + adv_eps
    const float *old_values; const double *gmom;
    float vf_clip, adv_eps; int norm_adv;
};

__device__ __forceinline__ int block_sum_i(int v, int *sh) {
    for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, d);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    int s = 0;
    for (int w = 0; w < (int)(blockDim.x >> 5); w++) s += sh[w];
    return s;
}

__global__ void k_ppo_count(PpoArgs p) {
    __shared__ int sh[32];
    const long long e = blockIdx.x;
    if (!p.acted[e]) return;
    int n = 0;
    for (int i = threadIdx.x; i < p.N; i += blockDim.x) {
        const uint8_t *v = p.valid + (e * p.N + i) * 5;
        n += (v[0] | v[1] | v[2] | v[3] | v[4]) ? 1 : 0;
    }
    n = block_sum_i(n, sh);
    if (threadIdx.x == 0) {
        if (n) atomicAdd(&p.cnt[0], (unsigned long long)n);
        atomicAdd(&p.cnt[1], 1ull);
    }
}

// one CTA (1024 threads): out = [sum_S A, sum_S A^2] in float64, each acted row's A counted once per agent of S.  Warp w takes
// rows w, w + 32, ... in order (|S| of a row: an integer warp sum), then thread 0 adds the 32 warp sums in warp order: the
// same bytes for the same inputs.
__global__ void __launch_bounds__(1024) k_ppo_moments(PpoArgs p, double *__restrict__ out) {
    __shared__ double sh[2][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double s1 = 0.0, s2 = 0.0;
    for (long long e = warp; e < p.E; e += 32) {
        if (!p.acted[e]) continue;
        int n = 0;
        for (int i = lane; i < p.N; i += 32) {
            const uint8_t *v = p.valid + (e * p.N + i) * 5;
            n += (v[0] | v[1] | v[2] | v[3] | v[4]) ? 1 : 0;
        }
        for (int d = 16; d > 0; d >>= 1) n += __shfl_xor_sync(0xFFFFFFFFu, n, d);
        const double a = (double)p.adv[e];
        s1 += (double)n * a;
        s2 += (double)n * (a * a);
    }
    if (lane == 0) { sh[0][warp] = s1; sh[1][warp] = s2; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double t1 = 0.0, t2 = 0.0;
        for (int w = 0; w < 32; w++) { t1 += sh[0][w]; t2 += sh[1][w]; }
        out[0] = t1;
        out[1] = t2;
    }
}

// one CTA (128 threads) per environment row; rowstats[e] = sums over the row's agents in S of (policy term, entropy,
// logp_old - logp_new, |r - 1| > eps) and the value term (V - R)^2 (0 for rows with acted = 0).  OPT (PpoArgs options):
// A is normalised by the minibatch moments and the value term is max((V - R)^2, (V_clip - R)^2); without it the kernel is
// the plain loss, arithmetic unchanged.
template <bool OPT>
__global__ void __launch_bounds__(128) k_ppo_loss(PpoArgs p) {
    __shared__ float sh[4][128];
    const long long e = blockIdx.x;
    const long long nS = p.gcnt[0], nR = p.gcnt[1];
    const bool acted = p.acted[e] != 0;
    const float invS = nS > 0 ? 1.0f / (float)nS : 0.0f;
    float A = p.adv[e], dV = (acted && nR > 0) ? p.vf * 2.0f * (p.value[e] - p.ret[e]) / (float)nR : 0.0f;
    float vterm = (p.value[e] - p.ret[e]) * (p.value[e] - p.ret[e]);
    if (OPT) {
        if (p.norm_adv) {   // (A - mu) / (sigma + adv_eps) in float64, sigma the unbiased deviation over S; 0 when that is 0
            const double n = (double)nS, s = p.gmom[0], q = p.gmom[1];
            const double mu = nS > 0 ? s / n : 0.0;
            const double var = nS > 1 ? fmax(0.0, (q - s * s / n) / (n - 1.0)) : 0.0;
            const double den = sqrt(var) + (double)p.adv_eps;
            A = den > 0.0 ? (float)(((double)A - mu) / den) : 0.0f;
        }
        if (p.vf_clip > 0.0f) {   // V_clip = V_old + clip(V - V_old, -c, c); the unclipped square wins ties (dV as above)
            const float V = p.value[e], R = p.ret[e], Vo = p.old_values[e], c = p.vf_clip, dvo = V - Vo;
            const float Vc = dvo > c ? Vo + c : (dvo < -c ? Vo - c : V);
            const float uc = (Vc - R) * (Vc - R);
            if (uc > vterm) { vterm = uc; dV = 0.0f; }
        }
    }
    float acc[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    for (int i = threadIdx.x; i < p.N; i += blockDim.x) {
        const long long t = e * p.N + i;
        const float *x = p.logits + t * 5;
        const uint8_t *va = p.valid + t * 5;
        float dl[5] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
        p.dcrit[t] = dV / (float)p.N;
        int cnt = 0;
        float mx = 0.0f;
        for (int j = 0; j < 5; j++)
            if (va[j]) { mx = cnt ? fmaxf(mx, x[j]) : x[j]; cnt++; }
        if (acted && cnt > 0) {
            // masked_choice's arithmetic: exponentials in action order, (x_a - max) - log(sum)
            float ex[5], sum = 0.0f;
            for (int j = 0; j < 5; j++)
                if (va[j]) { ex[j] = expf(x[j] - mx); sum += ex[j]; }
            const float ls = logf(sum);
            const int a = p.actions[t] < 5 ? p.actions[t] : 4;    // actions are 0..4 (header); keeps the read in the row
            const float lp = (x[a] - mx) - ls, lpo = p.old_lp[t];
            const float r = expf(lp - lpo), s1 = r * A, s2 = fminf(fmaxf(r, 1.0f - p.eps), 1.0f + p.eps) * A;
            const float gpol = s1 <= s2 ? -A * r : 0.0f;       // d(-min(s1, s2)) / d logp_new; the gradient flows through r A on ties
            float H = 0.0f, pj[5], lpj[5];
            for (int j = 0; j < 5; j++)
                if (va[j]) { pj[j] = ex[j] / sum; lpj[j] = (x[j] - mx) - ls; H -= pj[j] * lpj[j]; }
            for (int j = 0; j < 5; j++)
                if (va[j]) dl[j] = invS * (gpol * ((j == a ? 1.0f : 0.0f) - pj[j]) + p.ent * pj[j] * (lpj[j] + H));
            acc[0] += -fminf(s1, s2);
            acc[1] += H;
            acc[2] += lpo - lp;
            acc[3] += fabsf(r - 1.0f) > p.eps ? 1.0f : 0.0f;
        }
        for (int j = 0; j < 5; j++) p.dlogits[t * 5 + j] = dl[j];
    }
    for (int q = 0; q < 4; q++) sh[q][threadIdx.x] = acc[q];
    __syncthreads();
    for (int s = 64; s > 0; s >>= 1) {
        if (threadIdx.x < s)
            for (int q = 0; q < 4; q++) sh[q][threadIdx.x] += sh[q][threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        for (int q = 0; q < 4; q++) p.rowstats[e * 5 + q] = sh[q][0];
        p.rowstats[e * 5 + 4] = acted ? vterm : 0.0f;
    }
}

// one CTA of 256 threads: stats = (policy, value, entropy, approx KL, clip fraction, |S|, acted rows, total loss); the sums
// over these rows divided by the minibatch's counts gcnt, and the counts cnt of these rows
__global__ void __launch_bounds__(256) k_ppo_stats(const float *__restrict__ rowstats, long long E,
                                                   const unsigned long long *__restrict__ cnt, const long long *__restrict__ gcnt,
                                                   float vf, float ent, float *__restrict__ stats) {
    __shared__ float sh[5][256];
    float acc[5] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    for (long long e = threadIdx.x; e < E; e += 256)
        for (int q = 0; q < 5; q++) acc[q] += rowstats[e * 5 + q];
    for (int q = 0; q < 5; q++) sh[q][threadIdx.x] = acc[q];
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (threadIdx.x < s)
            for (int q = 0; q < 5; q++) sh[q][threadIdx.x] += sh[q][threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const bool hS = gcnt[0] > 0, hR = gcnt[1] > 0;
        const float nS = (float)gcnt[0], nR = (float)gcnt[1];
        const float pol = hS ? sh[0][0] / nS : 0.0f, entm = hS ? sh[1][0] / nS : 0.0f;
        const float val = hR ? sh[4][0] / nR : 0.0f;
        stats[0] = pol;
        stats[1] = val;
        stats[2] = entm;
        stats[3] = hS ? sh[2][0] / nS : 0.0f;
        stats[4] = hS ? sh[3][0] / nS : 0.0f;
        stats[5] = (float)cnt[0];
        stats[6] = (float)cnt[1];
        stats[7] = pol - ent * entm + vf * val;
    }
}

// ---- workspace ---------------------------------------------------------------------------------------------------------
struct Wg {
    float *h, *c, *xcl, *iou, *fraw, *fc, *craw;
    int8_t *child_base; int32_t *tcnt, *tpos, *btot, *counts, *lists, *merge_row, *child_row;
    float *ap[4], *aa[3], *emb, *qkv[3], *att[3], *cat[3], *mpre[3], *xs[3], *lse[3];
    float *y1p[2], *y1[2], *y2p[2], *y2[2];                  // actor, critic
    float *dlogits, *dcrit, *rowstats, *dz, *dy1, *dy2, *dcat, *datt, *dqkv, *dx[2], *Dq;
    float *dh, *dc, *dG, *dC, *dFC, *dF, *dFs, *part;
    long long cap; int nblk;
};

inline int n_chunks(long long M) {
    if (M <= 0) return 0;
    const long long n = (M + MIN_CHUNK - 1) / MIN_CHUNK;
    return (int)(n < MAX_CHUNKS ? n : MAX_CHUNKS);
}

// train: the training forward, the loss and the backward.  Otherwise the forward alone (fl_policy_forward_f32): the
// pointers only the backward reads (xcl, ap, mpre, lse, y1p, y2p, d*, part) stay null, and a dense buffer is shared once
// the forward has read it for the last time (aa[2] = aa[0]; one qkv, att and cat for the three layers; xs ping-pongs; one
// y1 for both heads; y2 stays per head, k_heads_final reads both).
inline size_t carve(Wg &w, unsigned char *base, long long T, bool train) {
    w = Wg{};
    size_t off = 0;
    auto take = [&](size_t bytes) { unsigned char *p = base ? base + off : nullptr; off = (off + bytes + 255) & ~(size_t)255; return p; };
    auto f = [&](long long n) { return (float *)take((size_t)n * 4); };
    const long long nodes = T * f32path::NODES, cap = T * 10;     // at most 10 inner nodes per 31-node ternary tree
    w.cap = cap;
    w.nblk = (int)((T + SCAN - 1) / SCAN);
    w.h = f(nodes * T_H); w.c = f(nodes * T_H);
    if (train) w.xcl = f(nodes * NF);
    w.iou = f(cap * 384); w.fraw = f(cap * 384); w.fc = f(cap * 384); w.craw = f(cap * 128);
    w.child_base = (int8_t *)take(nodes);
    w.tcnt = (int32_t *)take(MAX_LEVELS * T * 4); w.tpos = (int32_t *)take(MAX_LEVELS * T * 4);
    w.btot = (int32_t *)take((size_t)MAX_LEVELS * w.nblk * 4); w.counts = (int32_t *)take(64 * 4);
    w.lists = (int32_t *)take(nodes * 4); w.merge_row = (int32_t *)take(cap * 4); w.child_row = (int32_t *)take(cap * 3 * 4);
    if (train)
        for (int i = 0; i < 4; i++) w.ap[i] = f(T * 256);
    for (int i = 0; i < 3; i++) w.aa[i] = train || i < 2 ? f(T * 256) : w.aa[0];
    w.emb = f(T * 256);
    for (int l = 0; l < 3; l++) {
        const bool own = train || l == 0;
        w.qkv[l] = own ? f(T * 768) : w.qkv[0]; w.att[l] = own ? f(T * 256) : w.att[0]; w.cat[l] = own ? f(T * 512) : w.cat[0];
        if (train) w.mpre[l] = f(T * 256);
        w.xs[l] = train || l < 2 ? f(T * 256) : w.xs[0];
        if (train) w.lse[l] = f(T * 4);
    }
    for (int h = 0; h < 2; h++) {
        if (train) w.y1p[h] = f(T * 256);
        w.y1[h] = train || h == 0 ? f(T * 256) : w.y1[0];
        if (train) w.y2p[h] = f(T * 128);
        w.y2[h] = f(T * 128);
    }
    if (!train) return off;
    w.dlogits = f(T * 5); w.dcrit = f(T); w.rowstats = f(T * 5);                    // E <= T rows
    w.dz = f(T * 512); w.dy1 = f(T * 256); w.dy2 = f(T * 128); w.dcat = f(T * 512); w.datt = f(T * 256); w.dqkv = f(T * 768);
    w.dx[0] = f(T * 256); w.dx[1] = f(T * 256); w.Dq = f(T * 4);
    w.dh = f(nodes * T_H); w.dc = f(nodes * T_H); w.dG = f(nodes * 384);
    w.dC = f(cap * 128); w.dFC = f(cap * 384); w.dF = f(cap * 384); w.dFs = f(cap * 128);
    w.part = f((long long)n_chunks(nodes) * DW_MAX);        // the longest reduction has at most `nodes` rows
    return off;
}

}  // namespace f32grad
