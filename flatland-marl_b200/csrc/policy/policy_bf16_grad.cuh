// policy_bf16_grad.cuh — the tensor-core products of fl_policy_ppo_grad_bf16 (include/flatland_policy_b200.h): the forward
// X W^T, the input gradient dY W and the weight gradient dY^T X of the 20 large weight matrices, with bf16 operands (fp32
// values rounded to nearest even) and fp32 accumulation in tensor memory (tcgen05.mma kind::f16, M = N = 128 per CTA).
//
// One kernel, k_tc_gemm<KIND>, serves all three products.  Every operand is fp32 in the workspace (or the caller's
// parameters); the CTA's 256 threads load it, round it to bf16 and store it in the K-major, 128-byte-swizzled layout of
// desc_sw128 while staging.  A product whose reduction runs along the memory rows of an operand (W in dY W, both operands
// of dY^T X) is transposed by the same stores, so every MMA sees two K-major operands and the instruction descriptor is
// idesc_bf16.  Staging is double-buffered over 64-wide reduction slabs: the loads of slab s overlap the MMAs of slab s - 1.
//
// Operand sources are those of the fp32 kernels: rows gathered through an index (children's h, the merge row), a second
// source concatenated along the reduction (the heads' cat(emb, x)), widths that are no multiple of 4 (agent_attr's 83
// features: scalar loads, zero padding).  The epilogue reads the accumulator through shared memory so that global stores
// are row-contiguous, and applies, in the fp32 kernels' order: + bias, + add, + the old output (accumulation), the stored
// pre-activation, GELU(erf), the GELU' multiply, scattered output rows.  The weight gradient runs over fixed row chunks
// (blockIdx.z) into fp32 partials that f32grad::k_dw_reduce sums in chunk order; the bias column of the partials is the
// fp32 sum of the unrounded dY over the chunk's rows (k_db_part).  No floating-point atomics.
#pragma once
#include "policy_f32_grad.cuh"
#include "umma.cuh"

namespace bf16grad {
using namespace umma;

constexpr int TC_THREADS = 256;
constexpr int TC_TILE = 128 * 128;                  // bytes of one 128-row x 64-element bf16 operand tile
constexpr int TC_SMEM = 1024 + 4 * TC_TILE + 64;    // alignment slack, two stages of (A, B) tiles, barriers and TMEM slot
constexpr int TC_PITCH = 33;                        // epilogue staging: 32 rows x 32 columns per warp
constexpr int DW_MIN_CHUNK = 512;                   // fewest rows per weight-gradient chunk (the fp32 path's is 64)

enum { TC_FWD = 0, TC_DX = 1, TC_DW = 2 };

// A matrix view S(r, j) with two parts concatenated along j:
//   S(r, j) = p1[row1(r) * ld1 + j] (j < k1), p2[r * ld2 + j - k1] (k1 <= j < k1 + k2), 0 beyond or for r >= rows,
//   row1(r) = idx ? idx[r] : r.
struct Src {
    const float *p1; const int32_t *idx; long long ld1; int k1;
    const float *p2; long long ld2; int k2;
    long long rows;
    int vec;                                        // p1, p2, ld1, ld2, k1 and k2 all multiples of 4 floats: float4 loads
};

// C[row(m)][n] = epilogue(sum_j A(m, j) B(n, j)), m < rows, n < cols, row(m) = cidx ? cidx[m] : m
struct Epi {
    float *c; const int32_t *cidx; long long ldc; long long rows; int cols;
    const float *bias;                              // + bias[n]
    const float *add; long long ldadd;              // + add[m][n]
    int accum;                                      // + C[row(m)][n]
    float *pre;                                     // the value before the activation -> pre[m * ldc + n]
    int act;                                        // 1: GELU(erf)
    const float *gpre; long long ldgpre;            // * gelu'(gpre[m][n])
};

// KIND  A(m, j)              B(n, j)              reduction
// FWD   a.S(m, j)            b.S(n, j) (= W)      j < red
// DX    a.S(m, j) (= dY)     b.S(j, n) (= W^T)    j < red (W's rows)
// DW    a.S(j, m) (= dY^T)   b.S(j, n) (= X^T)    j in chunk blockIdx.z: [z chunk, min(red, (z + 1) chunk))
struct TcArgs {
    Src a, b;
    long long red, chunk;
    Epi e;
    long long zstride;                              // DW: output offset of chunk z (partials [z][N][K + 1])
};

__device__ __forceinline__ float src_at(const Src &s, long long r, long long j) {
    if (r >= s.rows) return 0.0f;
    if (j < s.k1) return s.p1[(s.idx ? (long long)s.idx[r] : r) * s.ld1 + j];
    if (j < s.k1 + s.k2) return s.p2[r * s.ld2 + (j - s.k1)];
    return 0.0f;
}

__device__ __forceinline__ float4 src_at4(const Src &s, long long r, long long j) {   // vec: j % 4 == 0
    if (r >= s.rows || j >= s.k1 + s.k2) return make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    const float *p = j < s.k1 ? s.p1 + (s.idx ? (long long)s.idx[r] : r) * s.ld1 + j : s.p2 + r * s.ld2 + (j - s.k1);
    return __ldg(reinterpret_cast<const float4 *>(p));
}

// 8 consecutive reduction elements of one tile row, rounded to bf16 and packed: one 16-byte chunk of the swizzled row
struct Chunks { uint32_t v[16]; };

// Tile row i (0..127) of the 128 x 64 slab: S row i0 + i, columns j0 .. j0 + 63, bound jend.  Thread t packs the chunks
// (i, c) = (t / 8 + 32 q, t % 8), q = 0..3.
__device__ __forceinline__ void load_rows(const Src &s, long long i0, long long j0, long long jend, Chunks &out) {
    const int t = threadIdx.x, c = t & 7;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const long long r = i0 + (t >> 3) + 32 * q, j = j0 + 8 * c;
        float f[8];
        if (s.vec && j + 8 <= jend) {
            const float4 x = src_at4(s, r, j), y = src_at4(s, r, j + 4);
            f[0] = x.x; f[1] = x.y; f[2] = x.z; f[3] = x.w; f[4] = y.x; f[5] = y.y; f[6] = y.z; f[7] = y.w;
        } else {
#pragma unroll
            for (int u = 0; u < 8; u++) f[u] = j + u < jend ? src_at(s, r, j + u) : 0.0f;
        }
#pragma unroll
        for (int u = 0; u < 4; u++) out.v[4 * q + u] = pack_bf16(f[2 * u], f[2 * u + 1]);
    }
}
__device__ __forceinline__ void store_rows(uint32_t tile, const Chunks &in) {
    const int t = threadIdx.x, c = t & 7;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const int i = (t >> 3) + 32 * q;
        st_shared_v4(tile + (uint32_t)i * 128u + (uint32_t)((c ^ (i & 7)) << 4), in.v[4 * q], in.v[4 * q + 1], in.v[4 * q + 2], in.v[4 * q + 3]);
    }
}

// Tile row i is S column i0 + i, the reduction runs over S rows j0 .. j0 + 63 (bound jend).  Thread t packs the chunks of
// tile rows 4 (t % 32) .. + 3 at reduction block c = t / 32: eight S rows, four columns each.
__device__ __forceinline__ void load_cols(const Src &s, long long i0, long long j0, long long jend, Chunks &out) {
    const int t = threadIdx.x, ib = 4 * (t & 31), c = t >> 5;
    float f[8][4];
#pragma unroll
    for (int u = 0; u < 8; u++) {
        const long long r = j0 + 8 * c + u, col = i0 + ib;
        if (r >= jend) {
            f[u][0] = f[u][1] = f[u][2] = f[u][3] = 0.0f;
        } else if (s.vec) {
            const float4 x = src_at4(s, r, col);
            f[u][0] = x.x; f[u][1] = x.y; f[u][2] = x.z; f[u][3] = x.w;
        } else {
#pragma unroll
            for (int w = 0; w < 4; w++) f[u][w] = src_at(s, r, col + w);
        }
    }
#pragma unroll
    for (int w = 0; w < 4; w++)
#pragma unroll
        for (int u = 0; u < 4; u++) out.v[4 * w + u] = pack_bf16(f[2 * u][w], f[2 * u + 1][w]);
}
__device__ __forceinline__ void store_cols(uint32_t tile, const Chunks &in) {
    const int t = threadIdx.x, ib = 4 * (t & 31), c = t >> 5;
#pragma unroll
    for (int w = 0; w < 4; w++) {
        const int i = ib + w;
        st_shared_v4(tile + (uint32_t)i * 128u + (uint32_t)((c ^ (i & 7)) << 4), in.v[4 * w], in.v[4 * w + 1], in.v[4 * w + 2], in.v[4 * w + 3]);
    }
}

template <int KIND>
__global__ void __launch_bounds__(TC_THREADS, 2) k_tc_gemm(TcArgs g) {
    extern __shared__ unsigned char smem_raw[];
    unsigned char *smem = (unsigned char *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t *bar = (uint64_t *)(smem + 4 * TC_TILE);               // [0], [1]: stage free (MMA commit)
    uint32_t *tmem_slot = (uint32_t *)(bar + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long i0 = (long long)blockIdx.x * 128, n0 = (long long)blockIdx.y * 128;
    long long jlo = 0, jend = g.red;
    if (KIND == TC_DW) {
        jlo = (long long)blockIdx.z * g.chunk;
        jend = min(g.red, jlo + g.chunk);
    }
    if (warp == 0) {
        if (lane == 0) { mbar_init(&bar[0], 1); mbar_init(&bar[1], 1); mbar_init_fence(); }
        __syncwarp();
        tmem_alloc(tmem_slot, 128);
    }
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    const uint32_t sbase = smem_u32(smem);
    const uint32_t idesc = idesc_bf16(128, 128);
    const int ns = (int)((jend - jlo + 63) / 64);
    for (int s = 0; s < ns; s++) {
        const long long j0 = jlo + 64LL * s;
        Chunks ca, cb;
        if (KIND == TC_DW) load_cols(g.a, i0, j0, jend, ca);
        else load_rows(g.a, i0, j0, jend, ca);
        if (KIND == TC_FWD) load_rows(g.b, n0, j0, jend, cb);
        else load_cols(g.b, n0, j0, jend, cb);
        const int b = s & 1;
        if (s >= 2) mbar_wait(&bar[b], ((s - 2) >> 1) & 1);          // the MMAs of slab s - 2 have read this stage
        const uint32_t ta = sbase + (uint32_t)(2 * b) * TC_TILE, tb = ta + TC_TILE;
        if (KIND == TC_DW) store_cols(ta, ca);
        else store_rows(ta, ca);
        if (KIND == TC_FWD) store_rows(tb, cb);
        else store_cols(tb, cb);
        fence_proxy_async();
        fence_before_sync();
        __syncthreads();
        if (threadIdx.x == 0) {
            fence_after_sync();
            const uint64_t ad = desc_sw128(ta), bd = desc_sw128(tb);
#pragma unroll
            for (int k = 0; k < 4; k++) mma_bf16(tmem, ad + 2 * k, bd + 2 * k, idesc, (uint32_t)((s | k) != 0));
            mma_commit(&bar[b]);
        }
    }
    if (ns > 0) mbar_wait(&bar[(ns - 1) & 1], ((ns - 1) >> 1) & 1);   // commits are cumulative: every MMA is done
    fence_after_sync();
    // ---- epilogue: warp w reads accumulator lanes 32 (w % 4) .., columns 64 (w / 4) .., through a 32 x 32 staging tile ----
    float *stage = (float *)smem + warp * 32 * TC_PITCH;
    const Epi &e = g.e;
    float *cout = e.c + (KIND == TC_DW ? (long long)blockIdx.z * g.zstride : 0);
    const int q = warp & 3;
#pragma unroll 1
    for (int half = 0; half < 2; half++) {
        const int col0 = 64 * (warp >> 2) + 32 * half;
        uint32_t v[32];
        const uint32_t taddr = tmem + ((uint32_t)(32 * q) << 16) + (uint32_t)col0;
        tmem_ld16(taddr, v);
        tmem_ld16(taddr + 16, v + 16);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; j++) stage[lane * TC_PITCH + j] = __uint_as_float(v[j]);
        __syncwarp();
        const long long n = n0 + col0 + lane;
        const bool nok = n < e.cols;
        const float bn = (nok && e.bias) ? e.bias[n] : 0.0f;
#pragma unroll 4
        for (int r = 0; r < 32; r++) {
            const long long m = i0 + 32 * q + r;
            if (m >= e.rows || !nok) continue;
            float x = stage[r * TC_PITCH + lane];
            if (e.bias) x += bn;
            if (e.add) x += e.add[m * e.ldadd + n];
            const long long row = e.cidx ? (long long)e.cidx[m] : m;
            if (e.accum) x += cout[row * e.ldc + n];
            if (e.pre) e.pre[m * e.ldc + n] = x;
            if (e.act == 1) x = f32path::gelu_erf(x);
            if (e.gpre) x *= f32grad::gelu_grad(e.gpre[m * e.ldgpre + n]);
            cout[row * e.ldc + n] = x;
        }
        __syncwarp();
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 128);
}

// part[z][n][K] (the bias column of the partials, row stride K + 1) = sum over rows m of chunk z, in row order, of dY[m][n]
__global__ void k_db_part(const float *__restrict__ dy, long long ldy, int N, long long M, long long chunk, int K,
                          float *__restrict__ part) {
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const long long z = blockIdx.y, r0 = z * chunk, r1 = min(M, r0 + chunk);
    float s = 0.0f;
#pragma unroll 8
    for (long long m = r0; m < r1; m++) s += dy[m * ldy + n];     // loads issued ahead, the sum in row order
    part[(z * N + n) * (K + 1) + K] = s;
}

inline bool aligned4(const void *p) { return ((uintptr_t)p & 15) == 0; }
inline Src make_src(const float *p1, const int32_t *idx, long long ld1, int k1, const float *p2, long long ld2, int k2, long long rows) {
    Src s{p1, idx, ld1, k1, p2, ld2, k2, rows, 0};
    s.vec = aligned4(p1) && ld1 % 4 == 0 && k1 % 4 == 0 && (!p2 || (aligned4(p2) && ld2 % 4 == 0 && k2 % 4 == 0));
    return s;
}
inline Epi no_epi() { return Epi{nullptr, nullptr, 0, 0, 0, nullptr, nullptr, 0, 0, nullptr, 0, nullptr, 0}; }

// rows of one weight-gradient chunk (a multiple of 64) and the number of chunks; nch <= f32grad::n_chunks(M), so the
// partials fit the fp32 path's buffer
inline long long dw_chunk(long long M, int *nch) {
    long long c = (M + f32grad::MAX_CHUNKS - 1) / f32grad::MAX_CHUNKS;
    if (c < DW_MIN_CHUNK) c = DW_MIN_CHUNK;
    c = (c + 63) & ~63LL;
    *nch = M > 0 ? (int)((M + c - 1) / c) : 0;
    return c;
}

}  // namespace bf16grad
