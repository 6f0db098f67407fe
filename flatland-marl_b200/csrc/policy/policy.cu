// policy.cu — batched forward pass of the reference policy network on B200 (sm_100a), C ABI of
// include/flatland_policy_b200.h.  Reference semantics: solution/nn/net_tree.py:73-116 (Network),
// solution/nn/TreeLSTM.py:34-154 (TreeLSTM), solution/plfActor.py:27-44 (action choice).
//
// Every matrix product runs on the 5th-generation tensor cores: tcgen05.mma issued by one thread, bf16 operands
// staged in shared memory in the 128-byte-swizzled K-major layout, fp32 accumulators in TMEM, read back with
// tcgen05.ld by the epilogue warps.  Dense operands arrive as TMA tiles (cp.async.bulk.tensor, tensor maps from the
// driver entry point); the Tree-LSTM's rows are tree nodes scattered over the batch, which a tiled TMA box cannot
// address, so they are gathered with 16-byte cp.async copies that arrive on the stage's mbarrier.
//
//   k_lin<MODE,BN> persistent; the CTA's BN (128 / 256) output columns of W stay resident in shared memory, 128-row
//                 tiles of A stream through a ring, two TMEM accumulators so the epilogue of tile i (16 warps) overlaps
//                 the MMAs of tile i+1.  MODE_LINEAR: dense layers (bias, optional GELU).  MODE_TREE_F: forget gates of
//                 one tree level, rows = child nodes, epilogue sigmoid(.) * c_child.
//   k_tree_p      one tree level: i/o/u pre-activations (N = 384) and the W_c reduction (N = 128) of 128 parent
//                 nodes accumulate side by side in all 512 TMEM columns; the epilogue applies the LSTM gates.
//   k_attn_mma    4-head attention over the agents of one environment: S = QK^T and O = PV as tcgen05 MMAs, softmax by
//                 the row's thread straight from TMEM.
//   k_tree_leaf   leaves of the Tree-LSTM (K = 12: one MMA k-step), two 192-column accumulators, 16 epilogue warps.
//   k_prep / k_tree_plan / k_head_final / k_choose: casts, level lists, final 128->5/1 layers, action choice.
//   rollout.cuh: seeded sampling with log-probabilities (k_sample) and GAE (k_gae) for PPO rollouts.
#include <cmath>
#include <cstdlib>
#include <cuda.h>
#include <cuda_runtime.h>
#include <math_constants.h>

#include "../../../include/flatland_policy_b200.h"
#include "rollout.cuh"
#include "umma.cuh"

using namespace umma;
typedef __nv_bfloat16 bf16;

namespace {

constexpr int TILE = 128 * 128;   // bytes of a 128-row x 64-element bf16 tile (one k-block)
constexpr int P_STAGES = 3;       // the ring is what paces k_tree_p: a stage takes ~2.5k cycles to arrive, its MMAs 768
constexpr int P_STAGE_BYTES = 4 * TILE;   // A tile + up to 384 rows of B
constexpr int NODES = 32;         // node slots per tree in the h / c / fc / x scratch (31 used)
constexpr int NULL_COPIES = 1024; // copies of the shared null-node row (one hot row serialises in its L2 slice)

unsigned long long g_launches = 0;

enum { MODE_LINEAR = 0, MODE_TREE_F = 1 };

struct LinArgs {
    const bf16 *a0, *a1, *a2;   // A = [a0 (kb0 k-blocks) | a1 (kb1 k-blocks) | a2 (16 columns, if k16)]
    int lda0, lda1, lda2;
    int kb0, kb1, k16;
    const bf16 *w;              // [n][ldw], the same column order as A
    int ldw;
    const float *bias;
    int rows;
    const int *rows_dev;        // when set: rows = *rows_dev * rows_mul (tree levels are counted on the device)
    int rows_mul;
    int act;
    int stages;                 // A ring depth (<= LIN_MAX_STAGES)
    long long *dbg;             // tuning only: SM-clock timestamps of CTA (0,0), NULL = off
    bf16 *out;                  // MODE_LINEAR: [rows][ldc]
    int ldc;
    const uint32_t *entries;    // MODE_TREE_F: level list (tree | node << 22 | first child << 27)
    const bf16 *cstate;         //              c of every node [tree][32][128]
    bf16 *fc;                   //              f * c_child     [tree][32][128]
    const uint8_t *eflags;      //              per list entry: bit j = child j of the node is a null leaf (shared h / c row)
    uint32_t null_off;          //              element offset of that shared row in h / c
};

// entry of a level list
__device__ __forceinline__ void entry_decode(uint32_t e, uint32_t &tree, uint32_t &node, uint32_t &child0) {
    tree = e & 0x3FFFFFu;
    node = (e >> 22) & 31u;
    child0 = e >> 27;
}

// Warp roles of k_lin: warps 0-15 epilogue (TMEM lane quarter = warp & 3, 32-column group = warp >> 2), warp 16 MMA
// issue, warps 17.. producers.
constexpr int LIN_THREADS = 21 * 32;      // 16 epilogue warps, MMA warp, 4 gather warps
constexpr int LIN_THREADS_TMA = 18 * 32;  // 16 epilogue warps, MMA warp, TMA warp
constexpr int LIN_MAX_STAGES = 8;
constexpr int OUT_PITCH = 272;          // bytes between rows of the staged output tile (256 + 16: conflict-free 16-byte stores)

// MODE_LINEAR: A (one or two dense sources) and W arrive as TMA tiles (tensor maps ta0 / ta1 / tw, one elected
// producer thread); MODE_TREE_F: rows are gathered by 128 producer threads with cp.async (the LDGSTS path tops out
// near 16 B/clk per SM, so it is kept for the gathers only).
// BN = output columns per CTA: 128, or 256 for the dense layers with K <= 256 (one 128x256x16 MMA reads 96 B/clk of
// shared memory instead of 128 and amortises the per-k-block hand-off; A is read half as often).
template <int MODE, int BN>
__global__ void __launch_bounds__(MODE == MODE_LINEAR ? LIN_THREADS_TMA : LIN_THREADS, 1) k_lin(const LinArgs p, const __grid_constant__ CUtensorMap ta0,
                                                        const __grid_constant__ CUtensorMap ta1, const __grid_constant__ CUtensorMap tw) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int nkb = p.kb0 + p.kb1 + p.k16;
    const int S = p.stages;
    const int rows = p.rows_dev ? (*p.rows_dev) * p.rows_mul : p.rows;
    const int mtiles = (rows + 127) >> 7;
    if ((int)blockIdx.x >= mtiles) return;
    uint8_t *sW = smem;
    constexpr int WT = BN / 128;                            // 16 KB tiles per k-block of W
    uint8_t *sA = smem + (size_t)nkb * WT * TILE;
    uint8_t *sC = sA + (size_t)S * TILE;                 // output tile staging: 128 rows, pitch OUT_PITCH
    unsigned long long *rowptr = (unsigned long long *)(sC + 128 * OUT_PITCH);   // MODE_TREE_F: destination of every row
    uint8_t *sCc = (uint8_t *)(rowptr + 128);              // MODE_TREE_F: c of the tile's child rows, pitch OUT_PITCH
    uint32_t *crowoff = (uint32_t *)(sCc + (MODE == MODE_TREE_F ? 128 * OUT_PITCH : 0));
    uint64_t *bars = (uint64_t *)(crowoff + (MODE == MODE_TREE_F ? 128 : 0));
    uint64_t *full = bars, *empty = bars + LIN_MAX_STAGES, *wfull = bars + 2 * LIN_MAX_STAGES;
    uint64_t *tfull = wfull + 1, *tempty = tfull + 2;
    uint32_t *tmem_slot = (uint32_t *)(tempty + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.y * BN;
    if (p.dbg && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) p.dbg[3] = clock64();

    if (warp == 16) {
        if (lane == 0) {
            const uint32_t nprod = MODE == MODE_LINEAR ? 1 : 128;
            for (int s = 0; s < S; s++) { mbar_init(&full[s], nprod); mbar_init(&empty[s], 1); }
            mbar_init(wfull, nprod);
            for (int b = 0; b < 2; b++) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 512); }
            mbar_init_fence();
        }
        __syncwarp();
        tmem_alloc(tmem_slot, 2 * BN);
    }
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    if (MODE == MODE_LINEAR && warp >= 17) {
        // ---------------- producer: one thread issues TMA tile loads ----------------
        if (threadIdx.x == 544) {
            tma_prefetch_desc(&ta0);
            tma_prefetch_desc(&tw);
            mbar_expect_tx(wfull, (uint32_t)nkb * WT * TILE);
            for (int kb = 0; kb < nkb; kb++)
                for (int hh = 0; hh < WT; hh++) tma_load_2d(smem_u32(sW + (size_t)(kb * WT + hh) * TILE), &tw, kb * 64, n0 + hh * 128, wfull);
            uint32_t it = 0;
            for (int mt = blockIdx.x; mt < mtiles; mt += gridDim.x) {
                for (int kb = 0; kb < nkb; kb++, it++) {
                    const int s = it % S;
                    mbar_wait(&empty[s], ((it / S) & 1) ^ 1);
                    if (p.dbg && kb == 0 && blockIdx.x == 0 && blockIdx.y == 0 && it / nkb < 8) p.dbg[80 + it / nkb] = clock64();
                    mbar_expect_tx(&full[s], TILE);
                    if (kb < p.kb0) tma_load_2d(smem_u32(sA + (size_t)s * TILE), &ta0, kb * 64, mt * 128, &full[s]);
                    else tma_load_2d(smem_u32(sA + (size_t)s * TILE), &ta1, (kb - p.kb0) * 64, mt * 128, &full[s]);
                }
            }
        }
    } else if (warp >= 17) {
        // ---------------- producers: 128 threads, thread = (16-byte chunk c, rows r0 + 16 i) ----------------
        const int tp = threadIdx.x - 544;
        const int c = tp & 7, r0 = tp >> 3;
        const uint32_t swz = (uint32_t)((c ^ (r0 & 7)) << 4) + (uint32_t)r0 * 128u;
        for (int kb = 0; kb < nkb; kb++) {
            const bool narrow = p.k16 && kb == nkb - 1;
            const bf16 *src = p.w + (size_t)kb * 64 + c * 8;
            const uint32_t dst = smem_u32(sW + (size_t)kb * TILE) + swz;
            if (!narrow || c < 2) {
#pragma unroll
                for (int i = 0; i < 8; i++) cp_async16(dst + i * 2048, src + (size_t)(n0 + r0 + 16 * i) * p.ldw, 16);
            }
        }
        cp_async_arrive(wfull);

        uint32_t it = 0;
        uint32_t ent[8], efl[8];                           // MODE_TREE_F: list entries / null flags of the tile, fetched one tile ahead
        if (MODE == MODE_TREE_F) {
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int r = (int)blockIdx.x * 128 + r0 + 16 * i;
                ent[i] = efl[i] = 0;
                if (r < rows) { ent[i] = ldg_u32_now(p.entries + r / 3); efl[i] = ldg_u8_now(p.eflags + r / 3); }
            }
        }
        for (int mt = blockIdx.x; mt < mtiles; mt += gridDim.x) {
            uint32_t off0[8], off1[8], off2[8], ok[8];
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int r = mt * 128 + r0 + 16 * i;
                ok[i] = r < rows ? 16u : 0u;
                off0[i] = off1[i] = off2[i] = 0;
                if (ok[i]) {
                    if (MODE == MODE_LINEAR) {
                        off0[i] = (uint32_t)r * (uint32_t)p.lda0;
                        off1[i] = (uint32_t)r * (uint32_t)p.lda1;
                        off2[i] = (uint32_t)r * (uint32_t)p.lda2;
                    } else {
                        uint32_t t, v, ch0;
                        entry_decode(ent[i], t, v, ch0);
                        const uint32_t child = ch0 + (uint32_t)(r % 3);
                        off0[i] = ((efl[i] >> (r % 3)) & 1u) ? p.null_off + (t & (NULL_COPIES - 1)) * (NODES * 128u) : (t * NODES + child) * 128u;
                        off2[i] = (t * NODES + v) * 16u;
                    }
                }
            }
            if (MODE == MODE_TREE_F) {
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    const int r = (mt + (int)gridDim.x) * 128 + r0 + 16 * i;
                    if (r < rows) { ent[i] = ldg_u32_now(p.entries + r / 3); efl[i] = ldg_u8_now(p.eflags + r / 3); }
                }
            }
            for (int kb = 0; kb < nkb; kb++, it++) {
                const int s = it % S;
                mbar_wait(&empty[s], ((it / S) & 1) ^ 1);
                if (p.dbg && tp == 0 && kb == 0 && blockIdx.x == 0 && blockIdx.y == 0 && it / nkb < 8) p.dbg[80 + it / nkb] = clock64();
                const uint32_t dst = smem_u32(sA + (size_t)s * TILE) + swz;
                if (kb < p.kb0) {
                    const bf16 *src = p.a0 + kb * 64 + c * 8;
#pragma unroll
                    for (int i = 0; i < 8; i++) cp_async16(dst + i * 2048, src + off0[i], ok[i]);
                } else if (kb < p.kb0 + p.kb1) {
                    const bf16 *src = p.a1 + (kb - p.kb0) * 64 + c * 8;
#pragma unroll
                    for (int i = 0; i < 8; i++) cp_async16(dst + i * 2048, src + off1[i], ok[i]);
                } else if (c < 2) {
                    const bf16 *src = p.a2 + c * 8;
#pragma unroll
                    for (int i = 0; i < 8; i++) cp_async16(dst + i * 2048, src + off2[i], ok[i]);
                }
                cp_async_arrive(&full[s]);
            }
        }
        cp_async_wait_all();
    } else if (warp == 16) {
        // ---------------- MMA issue: one thread ----------------
        if (lane == 0) {
            const bool dbg = p.dbg && blockIdx.x == 0 && blockIdx.y == 0;
            if (dbg) p.dbg[0] = clock64();
            mbar_wait(wfull, 0);
            fence_after_sync();
            if (dbg) p.dbg[1] = clock64();
            const uint32_t idesc = idesc_bf16(128, BN);
            uint32_t it = 0, tl = 0;
            for (int mt = blockIdx.x; mt < mtiles; mt += gridDim.x, tl++) {
                const uint32_t b = tl & 1;
                mbar_wait(&tempty[b], ((tl >> 1) & 1) ^ 1);
                fence_after_sync();
                if (dbg && tl < 8) p.dbg[8 + tl * 4] = clock64();
                for (int kb = 0; kb < nkb; kb++, it++) {
                    const int s = it % S;
                    mbar_wait(&full[s], (it / S) & 1);
                    fence_after_sync();
                    if (dbg && tl < 8 && kb == 0) p.dbg[8 + tl * 4 + 1] = clock64();
                    if (dbg && tl < 8 && kb == nkb - 1) p.dbg[8 + tl * 4 + 2] = clock64();
                    const uint64_t ad = desc_sw128(smem_u32(sA + (size_t)s * TILE));
                    const uint64_t bd = desc_sw128(smem_u32(sW + (size_t)kb * WT * TILE));
                    const int nk = (p.k16 && kb == nkb - 1) ? 1 : 4;
                    for (int k = 0; k < nk; k++) mma_bf16(tmem + b * BN, ad + 2 * k, bd + 2 * k, idesc, (uint32_t)((kb | k) != 0));
                    mma_commit(&empty[s]);
                }
                mma_commit(&tfull[b]);
            }
        }
        __syncwarp();
    } else {
        // ---------------- epilogue: warp w owns TMEM lanes 32(w&3).. (rows) and columns 32(w>>2).. ----------------
        uint32_t tl = 0;
        const int q = warp & 3, cg = warp >> 2;
        for (int mt = blockIdx.x; mt < mtiles; mt += gridDim.x, tl++) {
            const uint32_t b = tl & 1;
            const int r = mt * 128 + q * 32 + lane;
            const bool valid = r < rows;
            size_t orow = 0, crow = 0;
            if (valid) {
                if (MODE == MODE_LINEAR) {
                    orow = (size_t)r * p.ldc + n0;
                } else {
                    uint32_t t, v, ch0;
                    entry_decode(__ldg(p.entries + r / 3), t, v, ch0);
                    const uint32_t child = ch0 + (uint32_t)(r % 3);
                    orow = ((size_t)t * NODES + child) * 128;
                    crow = ((__ldg(p.eflags + r / 3) >> (r % 3)) & 1u) ? (size_t)p.null_off + (size_t)(t & (NULL_COPIES - 1)) * (NODES * 128) : orow;
                }
            }
            float bias[32];
            if (MODE == MODE_LINEAR && WT == 1) {
#pragma unroll
                for (int j = 0; j < 8; j++) *reinterpret_cast<float4 *>(&bias[4 * j]) = __ldg(reinterpret_cast<const float4 *>(p.bias + n0 + cg * 32) + j);
            }
            uint32_t cw[16];
            if (MODE == MODE_TREE_F) {
                // c of the 128 child rows: fetched row-contiguously (16 lanes per 256-byte row) into shared memory, then
                // every thread picks up its own 64 bytes (a direct read is 32 rows x 16 bytes per instruction)
                if (cg == 0) crowoff[q * 32 + lane] = valid ? (uint32_t)crow : 0xFFFFFFFFu;
                named_bar_sync(3, 512);
                const int te0 = warp * 32 + lane;
                uint4 cv[4];
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const int ci = te0 + 512 * j, row = ci >> 4, cc = ci & 15;
                    const uint32_t off = crowoff[row];
                    cv[j] = off != 0xFFFFFFFFu ? __ldg(reinterpret_cast<const uint4 *>(p.cstate + off) + cc) : make_uint4(0u, 0u, 0u, 0u);
                }
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const int ci = te0 + 512 * j, row = ci >> 4, cc = ci & 15;
                    st_shared_v4(smem_u32(sCc) + (uint32_t)row * OUT_PITCH + cc * 16, cv[j].x, cv[j].y, cv[j].z, cv[j].w);
                }
                named_bar_sync(4, 512);
                const uint32_t crd = smem_u32(sCc) + (uint32_t)(q * 32 + lane) * OUT_PITCH + cg * 64;
#pragma unroll
                for (int j = 0; j < 4; j++) *reinterpret_cast<uint4 *>(&cw[4 * j]) = ld_shared_v4(crd + j * 16);
            }
            mbar_wait(&tfull[b], (tl >> 1) & 1);
            fence_after_sync();
            const bool dbg = p.dbg && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0 && tl < 8;
            if (dbg) p.dbg[48 + tl * 4] = clock64();
#pragma unroll 1
            for (int round = 0; round < WT; round++) {          // 128 output columns per round
            const int nr = n0 + round * 128;
            const uint32_t tbase = tmem + ((uint32_t)(q * 32) << 16) + b * BN + round * 128 + cg * 32;
            uint32_t v[32];
            tmem_ld16(tbase, v);
            tmem_ld16(tbase + 16, v + 16);
            if (WT > 1) {
#pragma unroll
                for (int j = 0; j < 8; j++) *reinterpret_cast<float4 *>(&bias[4 * j]) = __ldg(reinterpret_cast<const float4 *>(p.bias + nr + cg * 32) + j);
            }
            tmem_ld_wait();
            if (round == WT - 1) {
                fence_before_sync();
                mbar_arrive(&tempty[b]);  // the accumulator is in registers: the MMA warp may overwrite the buffer
            }
            if (dbg) p.dbg[48 + tl * 4 + 1] = clock64();
            uint32_t ow[16];
#pragma unroll
            for (int j = 0; j < 16; j++) {
                float f0 = 0.0f, f1 = 0.0f;
                if (MODE == MODE_LINEAR) {
                    f0 = __uint_as_float(v[2 * j]) + bias[2 * j];
                    f1 = __uint_as_float(v[2 * j + 1]) + bias[2 * j + 1];
                    if (p.act & 1) { const float2 g = gelu2_erf(f0, f1); f0 = g.x; f1 = g.y; }
                } else {
                    // forget gate: b_f rides in the MMA and the weights are pre-scaled by 1/2, so f = 0.5 tanh(acc) + 0.5
                    const float2 cc = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&cw[j]));
                    f0 = fmaf(0.5f * cc.x, tanh_fast(__uint_as_float(v[2 * j])), 0.5f * cc.x);
                    f1 = fmaf(0.5f * cc.y, tanh_fast(__uint_as_float(v[2 * j + 1])), 0.5f * cc.y);
                }
                ow[j] = pack_bf16(f0, f1);
            }
            // registers -> padded shared-memory tile -> row-contiguous 16-byte stores (16 lanes cover a 256-byte row).
            // The direct form, 32 lanes writing 16 bytes to 32 different rows, costs 32 store transactions per
            // instruction; one bulk copy per row serialises in the uniform datapath (2.5k cycles per tile).
            if (dbg) p.dbg[96 + tl * 4] = clock64();
            named_bar_sync(1, 512);                       // everybody has finished reading the previous tile
            const uint32_t srow = smem_u32(sC) + (uint32_t)(q * 32 + lane) * OUT_PITCH;
#pragma unroll
            for (int j = 0; j < 4; j++) st_shared_v4(srow + cg * 64 + j * 16, ow[4 * j], ow[4 * j + 1], ow[4 * j + 2], ow[4 * j + 3]);
            if (MODE == MODE_TREE_F && cg == 0) rowptr[q * 32 + lane] = valid ? (unsigned long long)(p.fc + orow) : 0ull;
            if (dbg) p.dbg[96 + tl * 4 + 1] = clock64();
            named_bar_sync(2, 512);
            if (dbg) p.dbg[96 + tl * 4 + 2] = clock64();
            const int te = warp * 32 + lane;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int ci = te + 512 * j, row = ci >> 4, cc = ci & 15;
                const uint4 val = ld_shared_v4(smem_u32(sC) + (uint32_t)row * OUT_PITCH + cc * 16);
                if (MODE == MODE_LINEAR) {
                    const int gr = mt * 128 + row;
                    if (gr < rows) *reinterpret_cast<uint4 *>(p.out + (size_t)gr * p.ldc + nr + cc * 8) = val;
                } else {
                    const unsigned long long dst = rowptr[row];
                    if (dst) *reinterpret_cast<uint4 *>(dst + cc * 16) = val;
                }
            }
            }   // round
            if (dbg) p.dbg[48 + tl * 4 + 2] = clock64();
        }
    }
    fence_before_sync();
    __syncthreads();
    if (p.dbg && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) p.dbg[2] = clock64();
    if (warp == 16) tmem_dealloc(tmem, 2 * BN);
}

// ---------------------------------------------------------------------------------------------------------------
// Leaves of the Tree-LSTM (node_order 0, two thirds of all nodes): iou = W_iou x + b (K = 12, one k16 MMA step),
// c = sig(i) tanh(u), h = sig(o) tanh(c).  W_iou stays resident; the 128-leaf x tiles stream through a ring; each
// tile is processed as two halves of 64 hidden units (i | o | u = 192 TMEM columns per half) so that two
// accumulator buffers fit and the gate epilogue of one half overlaps the MMAs of the next.
struct LeafArgs {
    const uint32_t *entries;
    const int *count_dev;
    const bf16 *x;
    bf16 *h, *c;
    bf16 *emb;
    int emb_ld;
    const bf16 *wiou;
    const float *b_iou;
    long long *dbg;            // tuning only: SM-clock stamps of CTA 0 (fl_policy_debug_clocks)
};
constexpr int LEAF_THREADS = 21 * 32;   // 16 epilogue warps (8 per half of the hidden units), MMA warp, 4 producer warps
constexpr int LEAF_STAGES = 6;
constexpr int LEAF_PITCH = 144;         // 128 bytes (64 hidden units) + 16

__global__ void __launch_bounds__(LEAF_THREADS, 1) k_tree_leaf(const LeafArgs p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int rows = *p.count_dev;
    const int mtiles = (rows + 127) >> 7;
    if ((int)blockIdx.x >= mtiles) return;
    uint8_t *sW = smem;                       // 384 rows x 128 B (first 32 B of every row used)
    uint8_t *sA = smem + 3 * TILE;
    uint8_t *sC = sA + LEAF_STAGES * TILE;    // per half: staged h | c, 2 x 128 rows, pitch LEAF_PITCH
    uint32_t *rowoff = (uint32_t *)(sC + 4 * 128 * LEAF_PITCH);   // per half: element offset of every row's node in h / c
    uint64_t *bars = (uint64_t *)(rowoff + 256);
    uint64_t *full = bars, *empty = bars + LEAF_STAGES, *wfull = bars + 2 * LEAF_STAGES;
    uint64_t *tfull = wfull + 1, *tempty = tfull + 2;
    uint32_t *tmem_slot = (uint32_t *)(tempty + 2);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 16) {
        if (lane == 0) {
            for (int s = 0; s < LEAF_STAGES; s++) { mbar_init(&full[s], 128); mbar_init(&empty[s], 1); }
            mbar_init(wfull, 128);
            for (int b = 0; b < 2; b++) { mbar_init(&tfull[b], 1); mbar_init(&tempty[b], 256); }
            mbar_init_fence();
        }
        __syncwarp();
        tmem_alloc(tmem_slot, 512);
    }
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    if (warp >= 17) {
        // ---------------- producers ----------------
        const int tp = threadIdx.x - 544;
        const int c = tp & 7, r0 = tp >> 3;
        const uint32_t swz = (uint32_t)((c ^ (r0 & 7)) << 4) + (uint32_t)r0 * 128u;
        if (c < 2) {
            const uint32_t dst = smem_u32(sW) + swz;
#pragma unroll 8
            for (int i = 0; i < 24; i++) cp_async16(dst + i * 2048, p.wiou + (size_t)(r0 + 16 * i) * 16 + c * 8, 16);
        }
        cp_async_arrive(wfull);
        uint32_t it = 0;
        uint32_t ent[8];                                   // list entries of the tile, fetched one tile ahead
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int r = (int)blockIdx.x * 128 + r0 + 16 * i;
            ent[i] = (c < 2 && r < rows) ? ldg_u32_now(p.entries + r) : 0u;
        }
        for (int mt = blockIdx.x; mt < mtiles; mt += gridDim.x, it++) {
            const int s = it % LEAF_STAGES;
            uint32_t off[8], ok[8];
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int r = mt * 128 + r0 + 16 * i;
                uint32_t t, v, ch0;
                entry_decode(ent[i], t, v, ch0);
                ok[i] = r < rows ? 16u : 0u;
                off[i] = ok[i] ? (t * NODES + v) * 16u : 0u;
            }
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int r = (mt + (int)gridDim.x) * 128 + r0 + 16 * i;
                if (c < 2 && r < rows) ent[i] = ldg_u32_now(p.entries + r);
            }
            mbar_wait(&empty[s], ((it / LEAF_STAGES) & 1) ^ 1);
            if (c < 2) {
                const uint32_t dst = smem_u32(sA + (size_t)s * TILE) + swz;
#pragma unroll
                for (int i = 0; i < 8; i++) cp_async16(dst + i * 2048, p.x + off[i] + c * 8, ok[i]);
            }
            cp_async_arrive(&full[s]);
        }
        cp_async_wait_all();
    } else if (warp == 16) {
        // ---------------- MMA issue ----------------
        if (lane == 0) {
            mbar_wait(wfull, 0);
            fence_after_sync();
            const uint32_t idesc = idesc_bf16(128, 64);
            const uint32_t w0 = smem_u32(sW);
            uint32_t it = 0;
            for (int mt = blockIdx.x; mt < mtiles; mt += gridDim.x, it++) {
                const int s = it % LEAF_STAGES;
                mbar_wait(&full[s], (it / LEAF_STAGES) & 1);
                fence_after_sync();
                const uint64_t ad = desc_sw128(smem_u32(sA + (size_t)s * TILE));
                for (int half = 0; half < 2; half++) {      // accumulator `half` always holds hidden units 64 half ..
                    mbar_wait(&tempty[half], (it & 1) ^ 1);
                    fence_after_sync();
                    for (int g = 0; g < 3; g++)     // gate g (i, o, u): rows 128 g + 64 half .. of W_iou
                        mma_bf16(tmem + half * 256 + g * 64, ad, desc_sw128(w0 + (uint32_t)(g * 128 + half * 64) * 128u), idesc, 0u);
                    if (half == 1) mma_commit(&empty[s]);
                    mma_commit(&tfull[half]);
                }
            }
        }
        __syncwarp();
    } else {
        // ---------------- epilogue: warps 0-7 own half 0 (hidden units 0..63) of every tile, warps 8-15 half 1, so the
        // gate math of one half overlaps the store drain of the other ----------------
        const int half = warp >> 3, q = warp & 3, sub = (warp >> 2) & 1;   // sub: which 32 of the half's 64 hidden units
        const int n0 = half * 64 + sub * 32;
        uint8_t *sCh = sC + (size_t)half * 2 * 128 * LEAF_PITCH;
        uint32_t *roff = rowoff + half * 128;
        const int te = (warp & 7) * 32 + lane;
        uint32_t tl = 0;
        for (int mt = blockIdx.x; mt < mtiles; mt += gridDim.x, tl++) {
            const bool dbg = p.dbg && blockIdx.x == 0 && threadIdx.x == 0 && tl >= 8 && tl < 12;
            long long *dd = p.dbg + (tl >= 8 ? (tl - 8) * 16 : 0);
            if (dbg) dd[4] = clock64();
            const int r = mt * 128 + q * 32 + lane;
            const bool valid = r < rows;
            uint32_t t = 0, v = 0, ch0 = 0;
            if (valid) entry_decode(__ldg(p.entries + r), t, v, ch0);
            const size_t orow = ((size_t)t * NODES + v) * 128;
            mbar_wait(&tfull[half], tl & 1);
            fence_after_sync();
            if (dbg) dd[5] = clock64();
            const uint32_t tbase = tmem + ((uint32_t)(q * 32) << 16) + half * 256 + sub * 32;
            uint32_t hw[16], cw[16];
#pragma unroll
            for (int u16 = 0; u16 < 2; u16++) {
                uint32_t vi[16], vo[16], vu[16];
                tmem_ld16(tbase + u16 * 16, vi);
                tmem_ld16(tbase + 64 + u16 * 16, vo);
                tmem_ld16(tbase + 128 + u16 * 16, vu);
                tmem_ld_wait();
                if (u16 == 1) {
                    fence_before_sync();
                    mbar_arrive(&tempty[half]);
                }
                // i and o arrive as half their pre-activation (weights pre-scaled): sigmoid(2z) = 0.5 tanh(z) + 0.5
#pragma unroll
                for (int j = 0; j < 16; j += 2) {
                    float cc[2], hh[2];
#pragma unroll
                    for (int k = 0; k < 2; k++) {
                        const float ti = tanh_fast(__uint_as_float(vi[j + k])), to = tanh_fast(__uint_as_float(vo[j + k]));
                        const float tu = tanh_fast(__uint_as_float(vu[j + k]));
                        cc[k] = fmaf(0.5f * tu, ti, 0.5f * tu);
                        const float tc = tanh_fast(cc[k]);
                        hh[k] = fmaf(0.5f * tc, to, 0.5f * tc);
                    }
                    cw[u16 * 8 + (j >> 1)] = pack_bf16(cc[0], cc[1]);
                    hw[u16 * 8 + (j >> 1)] = pack_bf16(hh[0], hh[1]);
                }
            }
            // staged through shared memory so that 8 lanes write one 128-byte row segment (see k_lin)
            if (dbg) dd[6] = clock64();
            named_bar_sync(1 + 2 * half, 256);
            const uint32_t srow = smem_u32(sCh) + (uint32_t)(q * 32 + lane) * LEAF_PITCH;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                st_shared_v4(srow + sub * 64 + j * 16, hw[4 * j], hw[4 * j + 1], hw[4 * j + 2], hw[4 * j + 3]);
                st_shared_v4(srow + 128 * LEAF_PITCH + sub * 64 + j * 16, cw[4 * j], cw[4 * j + 1], cw[4 * j + 2], cw[4 * j + 3]);
            }
            if (sub == 0) roff[q * 32 + lane] = valid ? (uint32_t)orow : 0xFFFFFFFFu;
            named_bar_sync(2 + 2 * half, 256);
            if (dbg) dd[8] = clock64();
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int ci = te + 256 * j, which = ci >> 10, row = (ci >> 3) & 127, cc = ci & 7;
                const uint4 val = ld_shared_v4(smem_u32(sCh) + (uint32_t)(which * 128 + row) * LEAF_PITCH + cc * 16);
                const uint32_t off = roff[row];
                if (off != 0xFFFFFFFFu) *reinterpret_cast<uint4 *>((which ? p.c : p.h) + off + half * 64 + cc * 8) = val;
            }
            if (dbg) dd[9] = clock64();
            if (valid && v == 0) {
                uint4 *oe = reinterpret_cast<uint4 *>(p.emb + (size_t)t * p.emb_ld + n0);
#pragma unroll
                for (int j = 0; j < 4; j++) oe[j] = make_uint4(hw[4 * j], hw[4 * j + 1], hw[4 * j + 2], hw[4 * j + 3]);
            }
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 16) tmem_dealloc(tmem, 512);
}

// ---------------------------------------------------------------------------------------------------------------
struct TreeArgs {
    const uint32_t *entries;   // level list
    const int *count_dev;      // nodes on this level
    int level;
    const bf16 *x;             // [tree][32][16]
    bf16 *h, *c;               // [tree][32][128]
    const bf16 *fc;            // [tree][32][128]
    bf16 *emb;                 // root h goes to emb[tree][emb_ld] (+ column offset folded in)
    int emb_ld;
    const bf16 *uiou, *wiou, *wc;
    const float *b_iou, *b_c;
    const uint8_t *eflags;     // per list entry: bit j = child j of the node is a null leaf: its h is a shared row at null_off
    uint32_t null_off;
};

// The weight k-blocks (U_iou: 384 rows, W_c: 128 rows) come as TMA tiles issued by one producer thread — they are dense and
// would otherwise share the cp.async path (about 16 B/clk per SM) with the gathered node rows.
__global__ void __launch_bounds__(416, 1) k_tree_p(const TreeArgs p, const __grid_constant__ CUtensorMap tu, const __grid_constant__ CUtensorMap tc) {
    // three 64 KB stages + one staging tile fill the 227 KB of the SM to within 500 bytes: no slack for re-aligning the
    // base, which the driver places 1024-aligned when the kernel has no static shared memory (checked, not assumed)
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t *smem = smem_raw;
    if ((smem_u32(smem) & 1023u) != 0) __trap();
    const int rows = *p.count_dev;
    const int mtiles = (rows + 127) >> 7;
    if ((int)blockIdx.x >= mtiles) return;
    uint8_t *sC = smem + P_STAGES * P_STAGE_BYTES;          // staged h, then c, of the tile: 128 rows, pitch OUT_PITCH
    uint32_t *rowoff = (uint32_t *)(sC + 128 * OUT_PITCH);
    uint64_t *bars = (uint64_t *)(rowoff + 128);
    uint64_t *full = bars, *empty = bars + P_STAGES, *tfull = bars + 2 * P_STAGES, *tempty = tfull + 1;
    uint32_t *tmem_slot = (uint32_t *)(tempty + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kfirst = p.level == 0 ? 6 : 0, klast = p.level == 0 ? 6 : 12;   // k-iterations: 0-5 h, 6 x, 7-12 fc

    if (warp == 12) {
        if (lane == 0) {
            for (int s = 0; s < P_STAGES; s++) { mbar_init(&full[s], 129); mbar_init(&empty[s], 1); }   // 128 gather threads + the TMA issuer
            mbar_init(tfull, 1);
            mbar_init(tempty, 256);
            mbar_init_fence();
        }
        __syncwarp();
        tmem_alloc(tmem_slot, 512);
    }
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    if (warp >= 8 && warp < 12) {
        const int tp = threadIdx.x - 256;
        const int c = tp & 7, r0 = tp >> 3;
        const uint32_t swz = (uint32_t)((c ^ (r0 & 7)) << 4) + (uint32_t)r0 * 128u;
        uint32_t it = 0;
        uint32_t ent[8], efl[8];                           // list entries / null flags of the tile, fetched one tile ahead
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const int r = (int)blockIdx.x * 128 + r0 + 16 * i;
            ent[i] = efl[i] = 0;
            if (r < rows) { ent[i] = ldg_u32_now(p.entries + r); efl[i] = ldg_u8_now(p.eflags + r); }
        }
        for (int mt = blockIdx.x; mt < mtiles; mt += gridDim.x) {
            uint32_t offc[8], offx[8], ok[8], nul[8], offn[8];
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int r = mt * 128 + r0 + 16 * i;
                ok[i] = r < rows ? 16u : 0u;
                offc[i] = offx[i] = nul[i] = offn[i] = 0;
                if (ok[i]) {
                    uint32_t t, v, ch0;
                    entry_decode(ent[i], t, v, ch0);
                    offc[i] = (t * NODES + ch0) * 128u;
                    offx[i] = (t * NODES + v) * 16u;
                    nul[i] = efl[i];                                   // which of the three children are null leaves
                    offn[i] = p.null_off + (t & (NULL_COPIES - 1)) * (NODES * 128u);
                }
            }
#pragma unroll
            for (int i = 0; i < 8; i++) {
                const int r = (mt + (int)gridDim.x) * 128 + r0 + 16 * i;
                if (r < rows) { ent[i] = ldg_u32_now(p.entries + r); efl[i] = ldg_u8_now(p.eflags + r); }
            }
            for (int kk = kfirst; kk <= klast; kk++, it++) {
                const int s = it % P_STAGES;
                mbar_wait(&empty[s], ((it / P_STAGES) & 1) ^ 1);
                const uint32_t dstA = smem_u32(smem + (size_t)s * P_STAGE_BYTES) + swz;
                const uint32_t dstB = dstA + TILE;
                if (kk < 6) {
                    // child kk >> 1 of every parent: its own h row, or the shared row of the null nodes
                    const int cj = kk >> 1;
                    const bf16 *src = p.h + kk * 64 + c * 8;
                    const bf16 *nsrc = p.h + (kk & 1) * 64 + c * 8;
#pragma unroll
                    for (int i = 0; i < 8; i++) cp_async16(dstA + i * 2048, ((nul[i] >> cj) & 1u) ? nsrc + offn[i] : src + offc[i], ok[i]);
                    if (tp == 0) {
                        const uint32_t bB = smem_u32(smem + (size_t)s * P_STAGE_BYTES) + TILE;
                        mbar_expect_tx(&full[s], 3 * TILE);
                        for (int hh = 0; hh < 3; hh++) tma_load_2d(bB + hh * TILE, &tu, kk * 64, hh * 128, &full[s]);
                    }
                } else if (kk == 6) {
                    if (c < 2) {
                        const bf16 *src = p.x + c * 8;
#pragma unroll
                        for (int i = 0; i < 8; i++) cp_async16(dstA + i * 2048, src + offx[i], ok[i]);
                        const bf16 *wsrc = p.wiou + c * 8;
#pragma unroll 8
                        for (int i = 0; i < 24; i++) cp_async16(dstB + i * 2048, wsrc + (size_t)(r0 + 16 * i) * 16, 16);
                    }
                    if (tp == 0) mbar_arrive(&full[s]);        // no TMA tile in this stage: the issuer's arrival only
                } else {
                    const bf16 *src = p.fc + (kk - 7) * 64 + c * 8;
#pragma unroll
                    for (int i = 0; i < 8; i++) cp_async16(dstA + i * 2048, src + offc[i], ok[i]);
                    if (tp == 0) {
                        mbar_expect_tx(&full[s], TILE);
                        tma_load_2d(smem_u32(smem + (size_t)s * P_STAGE_BYTES) + TILE, &tc, (kk - 7) * 64, 0, &full[s]);
                    }
                }
                cp_async_arrive(&full[s]);
            }
        }
        cp_async_wait_all();
    } else if (warp == 12) {
        if (lane == 0) {
            const uint32_t id256 = idesc_bf16(128, 256), id128 = idesc_bf16(128, 128);
            uint32_t it = 0, tl = 0;
            for (int mt = blockIdx.x; mt < mtiles; mt += gridDim.x, tl++) {
                mbar_wait(tempty, (tl & 1) ^ 1);
                fence_after_sync();
                for (int kk = kfirst; kk <= klast; kk++, it++) {
                    const int s = it % P_STAGES;
                    mbar_wait(&full[s], (it / P_STAGES) & 1);
                    fence_after_sync();
                    const uint32_t a = smem_u32(smem + (size_t)s * P_STAGE_BYTES);
                    const uint64_t ad = desc_sw128(a), bd = desc_sw128(a + TILE), bd2 = desc_sw128(a + TILE + 256 * 128);
                    if (kk <= 6) {
                        const int nk = kk == 6 ? 1 : 4;
                        for (int k = 0; k < nk; k++) {
                            const uint32_t acc = (uint32_t)(kk > kfirst || k > 0);
                            mma_bf16(tmem, ad + 2 * k, bd + 2 * k, id256, acc);
                            mma_bf16(tmem + 256, ad + 2 * k, bd2 + 2 * k, id128, acc);
                        }
                    } else {
                        for (int k = 0; k < 4; k++) mma_bf16(tmem + 384, ad + 2 * k, bd + 2 * k, id128, (uint32_t)(kk > 7 || k > 0));
                    }
                    mma_commit(&empty[s]);
                }
                mma_commit(tfull);
            }
        }
        __syncwarp();
    } else {
        uint32_t tl = 0;
        const bool inner = p.level > 0;
        for (int mt = blockIdx.x; mt < mtiles; mt += gridDim.x, tl++) {
            const int r = mt * 128 + (warp & 3) * 32 + lane;
            const bool valid = r < rows;
            uint32_t t = 0, v = 0, ch0 = 0;
            if (valid) entry_decode(__ldg(p.entries + r), t, v, ch0);
            const size_t orow = ((size_t)t * NODES + v) * 128;
            mbar_wait(tfull, tl & 1);
            fence_after_sync();
            const uint32_t tbase = tmem + ((uint32_t)((warp & 3) * 32) << 16);
            const uint32_t srow = smem_u32(sC) + (uint32_t)((warp & 3) * 32 + lane) * OUT_PITCH;
            uint32_t cwk[4][8];                            // c of this thread's 64 hidden units waits here while h drains
#pragma unroll
            for (int ch = (warp >> 2) * 4; ch < (warp >> 2) * 4 + 4; ch++) {
                uint32_t vi[16], vo[16], vu[16], vc[16];
                tmem_ld16(tbase + ch * 16, vi);
                tmem_ld16(tbase + 128 + ch * 16, vo);
                tmem_ld16(tbase + 256 + ch * 16, vu);
                if (inner) tmem_ld16(tbase + 384 + ch * 16, vc);
                tmem_ld_wait();
                uint32_t hw[8];
                uint32_t *cw = cwk[ch & 3];
                float bc[16];
#pragma unroll
                for (int j = 0; j < 4; j++) *reinterpret_cast<float4 *>(&bc[4 * j]) = __ldg(reinterpret_cast<const float4 *>(p.b_c + ch * 16) + j);
                // b_iou rides in the MMA (x column 12); i and o arrive as half their pre-activation
#pragma unroll
                for (int j = 0; j < 16; j += 2) {
                    float cc[2], hh[2];
#pragma unroll
                    for (int k = 0; k < 2; k++) {
                        const float ti = tanh_fast(__uint_as_float(vi[j + k])), to = tanh_fast(__uint_as_float(vo[j + k]));
                        const float tu = tanh_fast(__uint_as_float(vu[j + k]));
                        float cn = fmaf(0.5f * tu, ti, 0.5f * tu);
                        if (inner) cn += __uint_as_float(vc[j + k]) + bc[j + k];
                        cc[k] = cn;
                        const float tc = tanh_fast(cn);
                        hh[k] = fmaf(0.5f * tc, to, 0.5f * tc);
                    }
                    cw[j >> 1] = pack_bf16(cc[0], cc[1]);
                    hw[j >> 1] = pack_bf16(hh[0], hh[1]);
                }
                // staged: the rows leave through row-contiguous stores below (see k_lin)
                st_shared_v4(srow + ch * 32, hw[0], hw[1], hw[2], hw[3]);
                st_shared_v4(srow + ch * 32 + 16, hw[4], hw[5], hw[6], hw[7]);
                if (valid && v == 0) {
                    uint4 *oe = reinterpret_cast<uint4 *>(p.emb + (size_t)t * p.emb_ld + ch * 16);
                    oe[0] = make_uint4(hw[0], hw[1], hw[2], hw[3]);
                    oe[1] = make_uint4(hw[4], hw[5], hw[6], hw[7]);
                }
            }
            fence_before_sync();
            mbar_arrive(tempty);                          // every accumulator column of this thread's rows is in shared memory
            if (warp < 4) rowoff[warp * 32 + lane] = valid ? (uint32_t)orow : 0xFFFFFFFFu;
            const int te = warp * 32 + lane;
#pragma unroll 1
            for (int which = 0; which < 2; which++) {      // h, then c, through the one staging tile
                if (which) {
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const int ch = (warp >> 2) * 4 + k;
                        st_shared_v4(srow + ch * 32, cwk[k][0], cwk[k][1], cwk[k][2], cwk[k][3]);
                        st_shared_v4(srow + ch * 32 + 16, cwk[k][4], cwk[k][5], cwk[k][6], cwk[k][7]);
                    }
                }
                named_bar_sync(1, 256);
#pragma unroll 4
                for (int j = 0; j < 8; j++) {
                    const int ci = te + 256 * j, row = ci >> 4, cc = ci & 15;
                    const uint4 val = ld_shared_v4(smem_u32(sC) + (uint32_t)row * OUT_PITCH + cc * 16);
                    const uint32_t off = rowoff[row];
                    if (off != 0xFFFFFFFFu) *reinterpret_cast<uint4 *>((which ? p.c : p.h) + off + cc * 8) = val;
                }
                named_bar_sync(2, 256);                   // the staging tile may be overwritten
            }
        }
    }
    fence_before_sync();
    __syncthreads();
    if (warp == 12) tmem_dealloc(tmem, 512);
}

// ---------------------------------------------------------------------------------------------------------------
// casts: agent_attr f32 [M][83] -> bf16 [M][128] (zero padded); forest f32 [M][31][12] -> bf16 [M][32][16] with
// +inf -> -1 (eval_env.py:76) and zero padding.  One thread writes 16 bytes (attr) or one node's 32 bytes (x).
__global__ void k_prep(const float *__restrict__ attr, const float *__restrict__ forest, bf16 *__restrict__ attr_b,
                       bf16 *__restrict__ x, uint32_t *__restrict__ nullmask, long long M) {
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long n_attr = (M * 16 + 31) & ~31LL, n_x = (M + NULL_COPIES) * NODES;     // x part: one warp per tree (32 node slots)
    if (tid < M * 16) {
        const long long m = tid >> 4;
        const int k0 = (int)(tid & 15) * 8;
        float f[8];
#pragma unroll
        for (int j = 0; j < 8; j++) f[j] = k0 + j < 83 ? attr[m * 83 + k0 + j] : 0.0f;
        reinterpret_cast<uint4 *>(attr_b)[tid] = make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
    } else if (tid >= n_attr && tid < n_attr + n_x) {
        const long long u = tid - n_attr;
        const long long m = u / NODES;
        const int node = (int)(u % NODES);
        float f[12];
#pragma unroll
        for (int j = 0; j < 12; j++) f[j] = 0.0f;
        bool real = node < 31;
        if (m >= M) {
            // trees M.. are not trees: their node 1 carries the null-node features (treeobs.cpp null node: seven inf, five -1),
            // so that the leaf kernel computes the h / c row all null nodes share
            real = node == 1;
#pragma unroll
            for (int j = 0; j < 12; j++) f[j] = real ? -1.0f : 0.0f;
        } else if (real) {
            const float4 *src = reinterpret_cast<const float4 *>(forest + (m * 31 + node) * 12);
#pragma unroll
            for (int j = 0; j < 3; j++) {
                const float4 q = src[j];
                f[4 * j] = q.x; f[4 * j + 1] = q.y; f[4 * j + 2] = q.z; f[4 * j + 3] = q.w;
            }
#pragma unroll
            for (int j = 0; j < 12; j++) f[j] = f[j] == CUDART_INF_F ? -1.0f : f[j];
        }
        bool is_null = real;
#pragma unroll
        for (int j = 0; j < 12; j++) is_null = is_null && f[j] == -1.0f;
        const uint32_t mask = __ballot_sync(0xFFFFFFFFu, is_null && node != 0 && m < M);   // the root is never shared
        if (node == 0 && m < M) nullmask[m] = mask;
        // column 12 is the constant 1 that multiplies the bias column of W_iou / W_f (the biases ride in the MMA)
        uint4 *dst = reinterpret_cast<uint4 *>(x + u * 16);
        dst[0] = make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
        dst[1] = make_uint4(pack_bf16(f[8], f[9]), pack_bf16(f[10], f[11]), pack_bf16(real ? 1.0f : 0.0f, 0.0f), 0u);
    }
}

// Level lists of the Tree-LSTM: every node with node_order == n >= 0 goes to list n as
// tree | node << 22 | first child << 27.  The order inside a list is arbitrary (rows are independent).
__global__ void k_tree_plan(const int32_t *__restrict__ adjacency, const int32_t *__restrict__ node_order,
                            const uint32_t *__restrict__ nullmask, uint32_t *lists, uint8_t *eflags, int *counts, long long M) {
    __shared__ int cnt[FL_POLICY_MAX_LEVELS], base[FL_POLICY_MAX_LEVELS];
    if (threadIdx.x < FL_POLICY_MAX_LEVELS) cnt[threadIdx.x] = 0;
    __syncthreads();
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned char child0[32];
    unsigned short pos[31];
    signed char lvl[31];
    uint32_t shared = 0;   // bit v: node v is a null leaf, whose h / c its parent reads from the shared null row
    if (t < M) {
#pragma unroll 1
        for (int v = 0; v < 32; v++) child0[v] = 0;
#pragma unroll 1
        for (int g = 0; g < 10; g++) {
            const int par = adjacency[(t * 30 + 3 * g) * 3];
            if (par >= 0 && par < 31) child0[par] = (unsigned char)(3 * g + 1);
        }
        const uint32_t nm = nullmask[t];
#pragma unroll 1
        for (int v = 0; v < 31; v++) {
            int o = node_order[t * 31 + v];
            if (o >= FL_POLICY_MAX_LEVELS) o = -1;
            // a null leaf: its h / c is the shared row, nothing to compute.  A null-featured node with children is not
            // shared: its state depends on its subtree, so it is computed in its own row and its parent reads that row.
            if (o == 0 && ((nm >> v) & 1u)) { o = -1; shared |= 1u << v; }
            lvl[v] = (signed char)o;
            if (o >= 0) pos[v] = (unsigned short)atomicAdd(&cnt[o], 1);
        }
    } else if (t < M + NULL_COPIES) {
        // the shared null-node rows: "trees" M.., node 1 (k_prep), one extra leaf each
        for (int v = 0; v < 31; v++) lvl[v] = -1;
        for (int v = 0; v < 32; v++) child0[v] = 0;
        lvl[1] = 0;
        pos[1] = (unsigned short)atomicAdd(&cnt[0], 1);
    }
    __syncthreads();
    if (threadIdx.x < FL_POLICY_MAX_LEVELS) base[threadIdx.x] = cnt[threadIdx.x] ? atomicAdd(&counts[threadIdx.x], cnt[threadIdx.x]) : 0;
    __syncthreads();
    if (t < M + NULL_COPIES) {
#pragma unroll 1
        for (int v = 0; v < 31; v++) {
            const int o = lvl[v];
            if (o < 0) continue;
            const size_t off = o == 0 ? 0 : (size_t)21 * M + NULL_COPIES + (size_t)(o - 1) * 10 * M;
            lists[off + base[o] + pos[v]] = (uint32_t)t | ((uint32_t)v << 22) | ((uint32_t)child0[v] << 27);
            eflags[off + base[o] + pos[v]] = (uint8_t)(o > 0 ? (shared >> child0[v]) & 7u : 0u);
        }
    }
}

// Attention on the tensor cores.  One CTA = one head of one 128-row query tile: R = G*N query rows (G = 128 / N whole
// environments when N <= 128, else 128 agents of one environment) against the key tiles of the same environments.
//   S = Q K^T   tcgen05.mma M=128 N=128 K=64 : Q tile and K tile are 64-column TMA boxes of the qkv buffer
//   softmax     thread = query row (TMEM lane): scale, mask keys of other environments, max / exp / sum in registers;
//               with more than one key tile a first pass over S finds the row maximum, a second pass exponentiates
//   O += P V    P (bf16) written by its row's thread into the swizzled K-major A layout; V is used where the TMA box put
//               it ([key][64 dims] = MN-major B operand), M=128 N=64 K=128
// qkv [M][768] = q | k | v, out [M][256].
struct AttnArgs {
    bf16 *out;
    int N;             // agents per environment
    int E;
    int rows_per_tile; // R
    int tiles_per_env; // query tiles per environment (N > 128), else 0
};
constexpr int ATTN_SMEM = 1024 + 5 * TILE + 256;   // Q, K, V, P (2 k-blocks)

__global__ void __launch_bounds__(128, 2) k_attn_mma(const AttnArgs p, const __grid_constant__ CUtensorMap tq) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint8_t *sQ = smem, *sK = smem + TILE, *sV = smem + 2 * TILE, *sP = smem + 3 * TILE;
    uint64_t *bar_tma = (uint64_t *)(smem + 5 * TILE), *bar_mma = bar_tma + 1;
    uint32_t *tmem_slot = (uint32_t *)(bar_mma + 1);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, hd = blockIdx.y;
    const long long M = (long long)p.E * p.N;
    // rows of this tile and the key range of their environments
    long long qb, key0;
    int nq, nkeys;
    if (p.tiles_per_env) {
        const int e = blockIdx.x / p.tiles_per_env, qt = blockIdx.x % p.tiles_per_env;
        qb = (long long)e * p.N + qt * 128;
        nq = min(128, p.N - qt * 128);
        key0 = (long long)e * p.N;
        nkeys = p.N;
    } else {
        qb = (long long)blockIdx.x * p.rows_per_tile;
        nq = (int)min((long long)p.rows_per_tile, M - qb);
        key0 = qb;
        nkeys = nq;
    }
    const int ktiles = (nkeys + 127) >> 7;
    if (warp == 0) {
        if (lane == 0) { mbar_init(bar_tma, 1); mbar_init(bar_mma, 1); mbar_init_fence(); }
        __syncwarp();
        tmem_alloc(tmem_slot, 256);
    }
    fence_before_sync();
    __syncthreads();
    fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    const uint32_t tS = tmem, tO = tmem + 128;
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    const int r = threadIdx.x;                       // query row of this thread
    const long long m = qb + r;
    // keys this row may attend to: those of its own environment
    const long long env_lo = (m / p.N) * p.N, env_hi = env_lo + p.N;
    uint32_t ph_tma = 0, ph_mma = 0;
    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tq);
        mbar_expect_tx(bar_tma, TILE);
        tma_load_2d(smem_u32(sQ), &tq, hd * 64, (int)qb, bar_tma);
    }
    mbar_wait(bar_tma, ph_tma);
    ph_tma ^= 1;
    float mx = -CUDART_INF_F, den = 0.0f;
    const uint32_t id_s = idesc_bf16(128, 128), id_o = idesc_bf16_bmn(128, 64);
    for (int pass = (ktiles > 1 ? 0 : 1); pass < 2; pass++) {      // pass 0: row maxima only (several key tiles)
        for (int kt = 0; kt < ktiles; kt++) {
            const long long kb = key0 + (long long)kt * 128;
            const int nk = min(128, nkeys - kt * 128);
            if (threadIdx.x == 0) {
                mbar_expect_tx(bar_tma, pass ? 2 * TILE : TILE);
                tma_load_2d(smem_u32(sK), &tq, 256 + hd * 64, (int)kb, bar_tma);
                if (pass) tma_load_2d(smem_u32(sV), &tq, 512 + hd * 64, (int)kb, bar_tma);
            }
            mbar_wait(bar_tma, ph_tma);
            ph_tma ^= 1;
            if (threadIdx.x == 0) {
                fence_after_sync();
                const uint64_t ad = desc_sw128(smem_u32(sQ)), bd = desc_sw128(smem_u32(sK));
                for (int k = 0; k < 4; k++) mma_bf16(tS, ad + 2 * k, bd + 2 * k, id_s, (uint32_t)(k != 0));
                mma_commit(bar_mma);
            }
            mbar_wait(bar_mma, ph_mma);
            ph_mma ^= 1;
            fence_after_sync();
            const int jlo = (int)max(0LL, env_lo - kb), jhi = (int)min((long long)nk, env_hi - kb);
            if (!pass) {
#pragma unroll 1
                for (int c0 = 0; c0 < 128; c0 += 16) {
                    uint32_t v[16];
                    tmem_ld16(tS + lane_base + c0, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; j++)
                        if (c0 + j >= jlo && c0 + j < jhi) mx = fmaxf(mx, __uint_as_float(v[j]) * 0.125f);
                }
                fence_before_sync();
                __syncthreads();          // everybody has read S before the next tile's MMA overwrites it
                continue;
            }
            if (ktiles == 1) {
#pragma unroll 1
                for (int c0 = 0; c0 < 128; c0 += 16) {
                    uint32_t v[16];
                    tmem_ld16(tS + lane_base + c0, v);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; j++)
                        if (c0 + j >= jlo && c0 + j < jhi) mx = fmaxf(mx, __uint_as_float(v[j]) * 0.125f);
                }
            }
            // P = exp(S/8 - max) as bf16 into the A-operand layout: row r, 16-byte chunk c at (c & 7) ^ (r & 7) of k-block c >> 3
            const uint32_t prow = smem_u32(sP) + (uint32_t)r * 128u;
#pragma unroll 1
            for (int c0 = 0; c0 < 128; c0 += 16) {
                uint32_t v[16], w[8];
                tmem_ld16(tS + lane_base + c0, v);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; j += 2) {
                    float p0 = 0.0f, p1 = 0.0f;
                    if (c0 + j >= jlo && c0 + j < jhi) p0 = __expf(__uint_as_float(v[j]) * 0.125f - mx);
                    if (c0 + j + 1 >= jlo && c0 + j + 1 < jhi) p1 = __expf(__uint_as_float(v[j + 1]) * 0.125f - mx);
                    // the denominator sums what the MMA will see: the bf16-rounded probabilities
                    const __nv_bfloat162 pb = __floats2bfloat162_rn(p0, p1);
                    const float2 pf = __bfloat1622float2(pb);
                    den += pf.x + pf.y;
                    w[j >> 1] = *reinterpret_cast<const uint32_t *>(&pb);
                }
                const int ch = c0 >> 3;          // two 16-byte chunks per 16 columns
                st_shared_v4(prow + (uint32_t)(ch >> 3) * TILE + (uint32_t)(((ch & 7) ^ (r & 7)) << 4), w[0], w[1], w[2], w[3]);
                st_shared_v4(prow + (uint32_t)((ch + 1) >> 3) * TILE + (uint32_t)((((ch + 1) & 7) ^ (r & 7)) << 4), w[4], w[5], w[6], w[7]);
            }
            fence_proxy_async();
            fence_before_sync();
            __syncthreads();
            if (threadIdx.x == 0) {
                fence_after_sync();
                const uint32_t pa = smem_u32(sP), vb = smem_u32(sV);
                for (int k = 0; k < 8; k++) {
                    // A: k-block k >> 2 of P, 16 keys at byte 32 (k & 3) of the row; B: key rows 16 k .. of the V tile
                    const uint64_t ad = desc_sw128(pa + (uint32_t)(k >> 2) * TILE) + 2 * (k & 3);
                    const uint64_t bd = desc_sw128(vb + (uint32_t)k * 2048u);
                    mma_bf16(tO, ad, bd, id_o, (uint32_t)(kt != 0 || k != 0));
                }
                mma_commit(bar_mma);
            }
            mbar_wait(bar_mma, ph_mma);       // P, K and V may be overwritten after this
            ph_mma ^= 1;
            fence_after_sync();
        }
    }
    // O / den -> bf16 -> staged in the (now free) P region -> row-contiguous stores
    {
        const float inv = 1.0f / den;
        const uint32_t orow = smem_u32(sP) + (uint32_t)r * 144u;
#pragma unroll 1
        for (int c0 = 0; c0 < 64; c0 += 16) {
            uint32_t v[16];
            tmem_ld16(tO + lane_base + c0, v);
            tmem_ld_wait();
            st_shared_v4(orow + c0 * 2, pack_bf16(__uint_as_float(v[0]) * inv, __uint_as_float(v[1]) * inv),
                         pack_bf16(__uint_as_float(v[2]) * inv, __uint_as_float(v[3]) * inv),
                         pack_bf16(__uint_as_float(v[4]) * inv, __uint_as_float(v[5]) * inv),
                         pack_bf16(__uint_as_float(v[6]) * inv, __uint_as_float(v[7]) * inv));
            st_shared_v4(orow + c0 * 2 + 16, pack_bf16(__uint_as_float(v[8]) * inv, __uint_as_float(v[9]) * inv),
                         pack_bf16(__uint_as_float(v[10]) * inv, __uint_as_float(v[11]) * inv),
                         pack_bf16(__uint_as_float(v[12]) * inv, __uint_as_float(v[13]) * inv),
                         pack_bf16(__uint_as_float(v[14]) * inv, __uint_as_float(v[15]) * inv));
        }
    }
    fence_before_sync();
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 8; j++) {
        const int ci = threadIdx.x + 128 * j, row = ci >> 3, cc = ci & 7;
        if (row < nq) {
            const uint4 val = ld_shared_v4(smem_u32(sP) + (uint32_t)row * 144u + cc * 16);
            *reinterpret_cast<uint4 *>(p.out + (qb + row) * 256 + hd * 64 + cc * 8) = val;
        }
    }
    if (warp == 0) tmem_dealloc(tmem, 256);
}

// Last layers: logits = actor_net.4(y2[:, :128]), value = mean over agents of critic_net.4(y2[:, 128:]).  One CTA per
// environment, one warp per agent at a time: the 512-byte row is read once, 16 bytes per lane (lanes 0-15 hold the actor
// half, 16-31 the critic half), partial dot products reduced with shuffles; the critic mean is a fixed-order sum.
__global__ void __launch_bounds__(256) k_head_final(const bf16 *__restrict__ y2, const float *__restrict__ w3, const float *__restrict__ b3,
                                                    float *__restrict__ logits, float *__restrict__ value, int N) {
    extern __shared__ float vals[];          // per-agent critic outputs
    const int e = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    const int half = lane >> 4, k0 = (lane & 15) * 8;
    // this lane's 8 weights of every output it contributes to: actor rows 0..4 (lanes 0-15) or the critic row (16-31)
    float wreg[5][8];
#pragma unroll
    for (int j = 0; j < 5; j++)
#pragma unroll
        for (int k = 0; k < 8; k++) wreg[j][k] = half == 0 ? w3[j * 128 + k0 + k] : (j == 0 ? w3[5 * 128 + k0 + k] : 0.0f);
    for (int a = warp; a < N; a += nw) {
        const uint4 raw = *reinterpret_cast<const uint4 *>(y2 + ((size_t)e * N + a) * 256 + lane * 8);
        const uint32_t rw[4] = {raw.x, raw.y, raw.z, raw.w};
        float x[8];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162 *>(&rw[k]));
            x[2 * k] = f.x;
            x[2 * k + 1] = f.y;
        }
        float o[5];
#pragma unroll
        for (int j = 0; j < 5; j++) {
            float acc = 0.0f;
#pragma unroll
            for (int k = 0; k < 8; k++) acc = fmaf(x[k], wreg[j][k], acc);
            o[j] = acc;
        }
#pragma unroll
        for (int j = 0; j < 5; j++)
#pragma unroll
            for (int d = 8; d > 0; d >>= 1) o[j] += __shfl_xor_sync(0xFFFFFFFFu, o[j], d);     // within each 16-lane half
        if (lane == 0) {
            float *lo = logits + ((size_t)e * N + a) * 5;
#pragma unroll
            for (int j = 0; j < 5; j++) lo[j] = o[j] + b3[j];
        }
        if (lane == 16) vals[a] = o[0] + b3[5];
    }
    __syncthreads();
    if (warp == 0) {
        float sacc = 0.0f;
        for (int a = lane; a < N; a += 32) sacc += vals[a];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) sacc += __shfl_xor_sync(0xFFFFFFFFu, sacc, d);
        if (lane == 0) value[e] = sacc / (float)N;
    }
}

// plfActor.py:27-44 soft choice: np.random.seed(42); np.random.choice(valid, p=softmax(logits[valid])) draws one
// uniform (0.3745401188473625) and returns the first entry whose normalised cumulative probability exceeds it.
__global__ void k_choose(const float *__restrict__ logits, const uint8_t *__restrict__ valid, uint8_t *__restrict__ actions, long long n) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    actions[i] = rollout::masked_choice(logits + i * 5, valid + i * 5, 0.3745401188473625, nullptr);
}

// ---------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode = nullptr;
int g_num_sms = 0;
long long *g_dbg = nullptr;       // k_lin timeline (fl_policy_linear_debug)
long long *g_leaf_dbg = nullptr;  // k_tree_leaf timeline (fl_policy_debug_clocks)
// the dynamic shared-memory opt-in of a kernel is per DEVICE: one bit per device ordinal, so that a process driving several
// devices opts in on each of them (all B200s of a box have the same SM count)
unsigned long long g_attr_set_mask = 0;

int setup() {
    int dev = 0;
    {
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return (int)e;
    }
    if (!g_num_sms) {
        cudaError_t e = cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
        if (e != cudaSuccess) return (int)e;
    }
    const bool g_attr_set = dev < 64 && ((g_attr_set_mask >> dev) & 1ull);
    if (!g_encode) {
        // the driver's tensor-map encoder, looked up at run time (no link-time dependency on libcuda)
        cudaDriverEntryPointQueryResult qres;
        void *fn = nullptr;
        cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
        if (e != cudaSuccess) return (int)e;
        if (!fn || qres != cudaDriverEntryPointSuccess) return (int)cudaErrorNotSupported;
        g_encode = (EncodeTiledFn)fn;
    }
    if (!g_attr_set) {
        const int lin_max = 1024 + 11 * TILE + 128 * OUT_PITCH + 1024 + 512;
        const int p_bytes = P_STAGES * P_STAGE_BYTES + 128 * OUT_PITCH + 512 + 128;
        const int leaf_bytes = 1024 + (3 + LEAF_STAGES) * TILE + 4 * 128 * LEAF_PITCH + 2048;
        cudaError_t e = cudaFuncSetAttribute(k_lin<MODE_LINEAR, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, lin_max);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_lin<MODE_LINEAR, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, lin_max);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_lin<MODE_TREE_F, 128>, cudaFuncAttributeMaxDynamicSharedMemorySize, 1024 + 9 * TILE + 2 * 128 * OUT_PITCH + 2048 + 512);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_tree_p, cudaFuncAttributeMaxDynamicSharedMemorySize, p_bytes);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_attn_mma, cudaFuncAttributeMaxDynamicSharedMemorySize, ATTN_SMEM);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(k_tree_leaf, cudaFuncAttributeMaxDynamicSharedMemorySize, leaf_bytes);
        if (e != cudaSuccess) return (int)e;
        if (dev < 64) g_attr_set_mask |= 1ull << dev;
    }
    return 0;
}

// nkb = 16 KB tiles of resident W; the A ring takes what is left of 11 tiles beside the staging tile
int lin_stages(int nkb) { return nkb <= 3 ? LIN_MAX_STAGES : 11 - nkb; }
size_t lin_smem(int nkb) { return 1024 + (size_t)(nkb + lin_stages(nkb)) * TILE + 128 * OUT_PITCH + 1024 + 512; }

// 2-D bf16 tensor map: `rows` x `cols` elements, row pitch `ld` elements, box = 64 columns (128 bytes, swizzled) x 128 rows;
// out-of-range rows read as zero.
int make_tmap(CUtensorMap *m, const bf16 *base, unsigned long long rows, unsigned long long cols, unsigned long long ld) {
    cuuint64_t dims[2] = {cols, rows};
    cuuint64_t strides[1] = {ld * 2};
    cuuint32_t box[2] = {64, 128};
    cuuint32_t es[2] = {1, 1};
    CUresult r = g_encode(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void *)base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : 700 + (int)r;
}

int launch_linear(const bf16 *a0, int lda0, int k0, const bf16 *a1, int lda1, int k1, const bf16 *w, const float *bias,
                  bf16 *out, int ldc, long long M, int N, int act, cudaStream_t st) {
    if (k0 % 64 || k1 % 64 || N % 128 || M <= 0 || M > 0x7FFFFF00LL) return -1;
    LinArgs p = {};
    p.a0 = a0; p.a1 = a1; p.a2 = nullptr;
    p.lda0 = lda0; p.lda1 = lda1; p.lda2 = 0;
    p.kb0 = k0 / 64; p.kb1 = k1 / 64; p.k16 = 0;
    p.w = w; p.ldw = k0 + k1; p.bias = bias;
    p.rows = (int)M; p.rows_dev = nullptr; p.rows_mul = 1; p.act = act;
    p.out = out; p.ldc = ldc;
    const bool wide = N % 256 == 0 && p.kb0 + p.kb1 <= 4 && !getenv("FL_POLICY_BN128");   // 256 columns per CTA
    const int wtiles = (p.kb0 + p.kb1) * (wide ? 2 : 1);
    p.stages = lin_stages(wtiles);
    p.dbg = g_dbg;
    const int ny = N / (wide ? 256 : 128);
    const int mtiles = (int)((M + 127) / 128);
    int nx = g_num_sms / ny;
    if (nx < 1) nx = 1;
    if (nx > mtiles) nx = mtiles;
    if (g_dbg && getenv("FL_POLICY_NX")) nx = atoi(getenv("FL_POLICY_NX"));   // tuning only (fl_policy_linear_debug)
    CUtensorMap ta0, ta1, tw;
    int rc = make_tmap(&ta0, a0, (unsigned long long)M, (unsigned long long)k0, (unsigned long long)lda0);
    if (!rc) rc = k1 ? make_tmap(&ta1, a1, (unsigned long long)M, (unsigned long long)k1, (unsigned long long)lda1) : 0;
    if (!rc) rc = make_tmap(&tw, w, (unsigned long long)N, (unsigned long long)(k0 + k1), (unsigned long long)(k0 + k1));
    if (rc) return rc;
    if (!k1) ta1 = ta0;
    if (wide) k_lin<MODE_LINEAR, 256><<<dim3(nx, ny), LIN_THREADS_TMA, lin_smem(wtiles), st>>>(p, ta0, ta1, tw);
    else k_lin<MODE_LINEAR, 128><<<dim3(nx, ny), LIN_THREADS_TMA, lin_smem(wtiles), st>>>(p, ta0, ta1, tw);
    g_launches++;
    return (int)cudaGetLastError();
}

struct Workspace {
    bf16 *x, *h, *c, *fc, *attr, *a1, *a2, *emb, *qkv, *atto, *proj, *ta, *tb, *y1, *y2;
    uint32_t *lists, *nullmask;
    uint8_t *eflags;
    int *counts;
    size_t bytes;
};

Workspace carve(void *base, long long M) {
    Workspace w;
    size_t off = 0;
    auto take = [&](size_t n) { size_t o = off; off += (n + 255) & ~(size_t)255; return (uint8_t *)base + o; };
    const size_t m = (size_t)M;
    w.counts = (int *)take(64 * sizeof(int));
    w.lists = (uint32_t *)take(((21 + 10 * (FL_POLICY_MAX_LEVELS - 1)) * m + NULL_COPIES) * sizeof(uint32_t));
    w.nullmask = (uint32_t *)take((m + 1) * sizeof(uint32_t));
    w.eflags = (uint8_t *)take((21 + 10 * (FL_POLICY_MAX_LEVELS - 1)) * m + NULL_COPIES);
    w.x = (bf16 *)take((m + NULL_COPIES) * NODES * 16 * 2);          // extra "trees": the shared null-node rows
    w.h = (bf16 *)take((m + NULL_COPIES) * NODES * 128 * 2);
    w.c = (bf16 *)take((m + NULL_COPIES) * NODES * 128 * 2);
    w.fc = (bf16 *)take(m * NODES * 128 * 2);
    w.attr = (bf16 *)take(m * 128 * 2);
    w.a1 = (bf16 *)take(m * 256 * 2);
    w.a2 = (bf16 *)take(m * 256 * 2);
    w.emb = (bf16 *)take(m * 256 * 2);
    w.qkv = (bf16 *)take(m * 768 * 2);
    w.atto = (bf16 *)take(m * 256 * 2);
    w.proj = (bf16 *)take(m * 256 * 2);
    w.ta = (bf16 *)take(m * 256 * 2);
    w.tb = (bf16 *)take(m * 256 * 2);
    w.y1 = (bf16 *)take(m * 512 * 2);
    w.y2 = (bf16 *)take(m * 256 * 2);
    w.bytes = off;
    return w;
}

}  // namespace

#include "policy_f32.cuh"
#include "policy_f32_grad.cuh"
#include "policy_bf16_grad.cuh"

// ---- the PPO graph (training forward, loss, backward), shared by the fp32 and the bf16 learner --------------------------
// The two learners differ only in the launchers of the 20 large weight matrices' products (Lin::gemm, Lin::dx, Lin::dw):
// F32Lin runs the fp32 CUDA-core kernels of policy_f32.cuh / policy_f32_grad.cuh, Bf16Lin the tensor-core kernel of
// policy_bf16_grad.cuh.  Everything else (the 12-feature node terms, the heads' last layer, attention, the gates, the loss)
// is launched here with the fp32 kernels in both.
namespace ppograph {
using namespace f32path;
using namespace f32grad;

struct F32Lin {
    cudaStream_t st; float *part;
    // C = act(A W^T + bias) as k_gemm_f32 (GemmArgs)
    void gemm(const float *a1, const int32_t *idx1, long long lda1, int K1, const float *a2, long long lda2, int K2,
              const float *w, const float *bias, float *c, long long ldc, long long M, int Nn, int act, float *pre) {
        if (M <= 0) return;
        GemmArgs g{a1, idx1, lda1, K1, a2, lda2, K2, w, bias, c, ldc, M, nullptr, Nn, act, pre};
        k_gemm_f32<<<dim3((unsigned)((M + 63) / 64), (unsigned)((Nn + 63) / 64)), 256, 0, st>>>(g);
        g_launches++;
    }
    // dX = dY W with the epilogue of k_gemm_dx
    void dx(const float *a, long long lda, int Nn, const float *w, long long ldw, int K, float *c, const int32_t *cidx, long long ldc,
            const float *add, long long ldadd, int accum, const float *pre, long long ldpre, long long M) {
        if (M <= 0) return;
        DxArgs g{a, lda, Nn, w, ldw, K, c, cidx, ldc, add, ldadd, accum, pre, ldpre, M};
        k_gemm_dx<<<dim3((unsigned)((M + 63) / 64), (unsigned)((K + 63) / 64)), 256, 0, st>>>(g);
        g_launches++;
    }
    // dW = dY^T X (and db when db != null) over M rows, fixed chunks, then summed in chunk order
    void dw(const float *dy, long long ldy, int Nn, const float *x1, const int32_t *idx1, long long ldx1, int K1, const float *x2,
            long long ldx2, int K2, long long M, float *dW, float *db) {
        const int bias = db ? 1 : 0, Kp = K1 + K2 + bias;
        int nch = n_chunks(M);
        long long chunk = 0;
        if (nch > 0) {
            chunk = ((M + nch - 1) / nch + 15) & ~15LL;
            nch = (int)((M + chunk - 1) / chunk);
            DwArgs g{dy, ldy, Nn, x1, idx1, ldx1, K1, x2, ldx2, K2, bias, M, chunk, part};
            k_gemm_dw<<<dim3((unsigned)((Nn + 63) / 64), (unsigned)((Kp + 63) / 64), (unsigned)nch), 256, 0, st>>>(g);
            g_launches++;
        }
        k_dw_reduce<<<(unsigned)(((long long)Nn * Kp + 255) / 256), 256, 0, st>>>(part, nch, Nn, K1 + K2, bias, dW, db);
        g_launches++;
    }
};

struct Bf16Lin {
    cudaStream_t st; float *part;
    void gemm(const float *a1, const int32_t *idx1, long long lda1, int K1, const float *a2, long long lda2, int K2,
              const float *w, const float *bias, float *c, long long ldc, long long M, int Nn, int act, float *pre) {
        using namespace bf16grad;
        if (M <= 0) return;
        TcArgs g{};
        g.a = make_src(a1, idx1, lda1, K1, a2, lda2, K2, M);
        g.b = make_src(w, nullptr, K1 + K2, K1 + K2, nullptr, 0, 0, Nn);
        g.red = K1 + K2;
        g.e = no_epi();
        g.e.c = c; g.e.ldc = ldc; g.e.rows = M; g.e.cols = Nn; g.e.bias = bias; g.e.pre = pre; g.e.act = act;
        k_tc_gemm<TC_FWD><<<dim3((unsigned)((M + 127) / 128), (unsigned)((Nn + 127) / 128)), TC_THREADS, TC_SMEM, st>>>(g);
        g_launches++;
    }
    void dx(const float *a, long long lda, int Nn, const float *w, long long ldw, int K, float *c, const int32_t *cidx, long long ldc,
            const float *add, long long ldadd, int accum, const float *pre, long long ldpre, long long M) {
        using namespace bf16grad;
        if (M <= 0) return;
        TcArgs g{};
        g.a = make_src(a, nullptr, lda, Nn, nullptr, 0, 0, M);
        g.b = make_src(w, nullptr, ldw, K, nullptr, 0, 0, Nn);
        g.red = Nn;
        g.e = no_epi();
        g.e.c = c; g.e.cidx = cidx; g.e.ldc = ldc; g.e.rows = M; g.e.cols = K;
        g.e.add = add; g.e.ldadd = ldadd; g.e.accum = accum; g.e.gpre = pre; g.e.ldgpre = ldpre;
        k_tc_gemm<TC_DX><<<dim3((unsigned)((M + 127) / 128), (unsigned)((K + 127) / 128)), TC_THREADS, TC_SMEM, st>>>(g);
        g_launches++;
    }
    void dw(const float *dy, long long ldy, int Nn, const float *x1, const int32_t *idx1, long long ldx1, int K1, const float *x2,
            long long ldx2, int K2, long long M, float *dW, float *db) {
        using namespace bf16grad;
        const int bias = db ? 1 : 0, K = K1 + K2, Kp = K + bias;
        int nch = 0;
        const long long chunk = dw_chunk(M, &nch);
        if (nch > 0) {
            TcArgs g{};
            g.a = make_src(dy, nullptr, ldy, Nn, nullptr, 0, 0, M);
            g.b = make_src(x1, idx1, ldx1, K1, x2, ldx2, K2, M);
            g.red = M; g.chunk = chunk;
            g.e = no_epi();
            g.e.c = part; g.e.ldc = Kp; g.e.rows = Nn; g.e.cols = K;
            g.zstride = (long long)Nn * Kp;
            k_tc_gemm<TC_DW><<<dim3((unsigned)((Nn + 127) / 128), (unsigned)((K + 127) / 128), (unsigned)nch), TC_THREADS, TC_SMEM, st>>>(g);
            g_launches++;
            if (bias) {
                k_db_part<<<dim3((unsigned)((Nn + 127) / 128), (unsigned)nch), 128, 0, st>>>(dy, ldy, Nn, M, chunk, K, part);
                g_launches++;
            }
        }
        k_dw_reduce<<<(unsigned)(((long long)Nn * Kp + 255) / 256), 256, 0, st>>>(part, nch, Nn, K, bias, dW, db);
        g_launches++;
    }
};

// the dynamic shared-memory opt-in of k_tc_gemm, per device (as setup() for the inference kernels)
unsigned long long g_tc_attr_mask = 0;
int bf16_setup() {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return (int)e;
    if (dev < 64 && ((g_tc_attr_mask >> dev) & 1ull)) return 0;
    using namespace bf16grad;
    e = cudaFuncSetAttribute(k_tc_gemm<TC_FWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_tc_gemm<TC_DX>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_tc_gemm<TC_DW>, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM);
    if (e != cudaSuccess) return (int)e;
    if (dev < 64) g_tc_attr_mask |= 1ull << dev;
    return 0;
}

struct PpoIn {
    const float *agent_attr, *forest; const int32_t *adjacency, *node_order;
    const uint8_t *valid, *actions; const float *old_lp, *adv, *ret; const uint8_t *acted;
    float eps, vf, ent;
    float *const *grads; float *logits, *value, *stats;
    const long long *gcnt;   // the loss's denominators [|S|, acted rows] over the whole minibatch; null: these rows' own counts
    // FlPpoOptions (all off by default); gmom: [sum_S A, sum_S A^2] of the whole minibatch, null: these rows' own moments
    const float *old_values = nullptr; const double *gmom = nullptr;
    float vf_clip = 0.0f, adv_eps = 0.0f; int norm_adv = 0;
};

// The forward pass and, when `loss`, the PPO loss and the backward pass.  On F32Lin with the forward-only layout
// (carve(..., false)) this is fl_policy_forward_f32; with the training layout every level and layer keeps its own slice of
// the workspace for the backward.  Both layouts give the same logits and values.  Arguments are checked by the caller.
template <class Lin>
int run(Lin &lin, const float *const *wts, Wg &ws, long long E, long long N, const PpoIn &in, bool loss, cudaStream_t st) {
    F32Lin f32{st, ws.part};
    const long long T = E * N;
    auto copy_cols = [&](const float *src, long long lds, float *dst, long long ldd, long long rows, int cols) {
        k_copy_cols<<<(unsigned)((rows * cols + 255) / 256), 256, 0, st>>>(src, lds, dst, ldd, rows, cols);
        g_launches++;
    };
    auto gelu_bwd = [&](const float *src, long long lds, const float *pre, long long ldp, float *dst, long long ldd, long long rows, int cols) {
        k_gelu_bwd<<<(unsigned)((rows * cols + 255) / 256), 256, 0, st>>>(src, lds, pre, ldp, dst, ldd, rows, cols);
        g_launches++;
    };
    const float *W_iou = wts[0], *b_iou = wts[1], *U_iou = wts[2], *W_c = wts[3], *b_c = wts[4], *W_f = wts[5], *b_f = wts[6], *U_f = wts[7];
    float *const *gr = in.grads;
    const float *d_agent_attr = in.agent_attr, *d_forest = in.forest;

    // ==== forward: Tree-LSTM (TreeLSTM.py:34-154), leaves, then one level at a time ====
    const long long nodes = T * f32path::NODES;
    cudaError_t err = cudaMemsetAsync(ws.h, 0, (size_t)nodes * T_H * 4, st);
    if (err == cudaSuccess) err = cudaMemsetAsync(ws.c, 0, (size_t)nodes * T_H * 4, st);
    if (err == cudaSuccess) err = cudaMemsetAsync(ws.counts, 0, 64 * 4, st);
    if (err != cudaSuccess) return (int)err;
    if (ws.xcl) {   // only the backward reads the cleaned features
        k_clean<<<(unsigned)((nodes * NF + 255) / 256), 256, 0, st>>>(d_forest, ws.xcl, nodes * NF);
        g_launches++;
    }
    k_tl_count<<<(unsigned)((T + 127) / 128), 128, 0, st>>>(in.adjacency, in.node_order, T, ws.child_base, ws.tcnt);
    k_tl_scan<<<dim3((unsigned)ws.nblk, MAX_LEVELS), SCAN, 0, st>>>(ws.tcnt, T, ws.nblk, ws.tpos, ws.btot);
    k_tl_tops<<<1, 32, 0, st>>>(ws.btot, ws.nblk, ws.counts);
    k_tl_fill<<<(unsigned)((T + 127) / 128), 128, 0, st>>>(in.node_order, T, ws.nblk, ws.tpos, ws.btot, ws.counts, ws.lists);
    k_tree_leaves<<<(unsigned)nodes, 128, 0, st>>>(d_forest, in.node_order, nodes, W_iou, b_iou, ws.h, ws.c);
    g_launches += 5;
    int32_t counts[MAX_LEVELS];
    err = cudaMemcpyAsync(counts, ws.counts, sizeof(counts), cudaMemcpyDeviceToHost, st);
    if (err == cudaSuccess) err = cudaStreamSynchronize(st);        // per-level sizes of the launches below; the only host sync
    if (err != cudaSuccess) return (int)err;
    long long loff[MAX_LEVELS + 1];                                  // list offset of every level (leaves first)
    loff[0] = 0;
    for (int lv = 0; lv < MAX_LEVELS; lv++) loff[lv + 1] = loff[lv] + counts[lv];
    const long long n_leaf = counts[0], n_in = loff[MAX_LEVELS] - n_leaf;   // inner index i = list position - n_leaf
    if (n_in > ws.cap) return -1;
    for (int lv = 1; lv < MAX_LEVELS; lv++) {
        const long long M = counts[lv], io = loff[lv] - n_leaf;
        if (M <= 0) continue;
        const int32_t *list = ws.lists + loff[lv], *dM = ws.counts + lv;
        int32_t *mr = ws.merge_row + io, *cr = ws.child_row + 3 * io;
        float *iou = ws.iou + io * 384, *fraw = ws.fraw + io * 384, *fc = ws.fc + io * 384;
        k_level_rows<<<(unsigned)((M + 127) / 128), 128, 0, st>>>(list, dM, ws.child_base, mr, cr);
        g_launches++;
        lin.gemm(ws.h, mr, T_H, 3 * T_H, nullptr, 0, 0, U_iou, nullptr, iou, 3 * T_H, M, 3 * T_H, 0, nullptr);
        lin.gemm(ws.h, cr, T_H, T_H, nullptr, 0, 0, U_f, nullptr, fraw, T_H, 3 * M, T_H, 0, nullptr);
        k_forget<<<(unsigned)M, 384, 0, st>>>(fraw, list, cr, dM, d_forest, W_f, b_f, ws.c, fc);
        lin.gemm(fc, nullptr, 3 * T_H, 3 * T_H, nullptr, 0, 0, W_c, nullptr, ws.craw, T_H, M, T_H, 0, nullptr);
        k_inner<<<(unsigned)M, 128, 0, st>>>(iou, ws.craw, list, dM, d_forest, W_iou, b_iou, b_c, ws.h, ws.c);
        g_launches += 2;
    }
    // attribute MLP (net_tree.py:41-50), emb = cat(attr embedding, h of the root)
    lin.gemm(d_agent_attr, nullptr, 83, 83, nullptr, 0, 0, wts[8], wts[9], ws.aa[0], 256, T, 256, 1, ws.ap[0]);
    lin.gemm(ws.aa[0], nullptr, 256, 256, nullptr, 0, 0, wts[10], wts[11], ws.aa[1], 256, T, 256, 1, ws.ap[1]);
    lin.gemm(ws.aa[1], nullptr, 256, 256, nullptr, 0, 0, wts[12], wts[13], ws.aa[2], 256, T, 256, 1, ws.ap[2]);
    lin.gemm(ws.aa[2], nullptr, 256, 256, nullptr, 0, 0, wts[14], wts[15], ws.emb, 256, T, 128, 1, ws.ap[3]);
    copy_cols(ws.h, (long long)f32path::NODES * T_H, ws.emb + 128, 256, T, 128);
    const float *x = ws.emb;
    for (int l = 0; l < 3; l++) {   // three attention blocks (net_tree.py:20-32)
        const float *const *tw = wts + 16 + 6 * l;
        lin.gemm(x, nullptr, 256, 256, nullptr, 0, 0, tw[0], tw[1], ws.qkv[l], 768, T, 768, 0, nullptr);
        k_attention<<<(unsigned)((T * 4 * 32 + 255) / 256), 256, 0, st>>>(ws.qkv[l], ws.att[l], 256, E, (int)N, ws.lse[l]);
        g_launches++;
        lin.gemm(ws.att[l], nullptr, 256, 256, nullptr, 0, 0, tw[2], tw[3], ws.cat[l] + 256, 512, T, 256, 0, nullptr);
        copy_cols(x, 256, ws.cat[l], 512, T, 256);
        lin.gemm(ws.cat[l], nullptr, 512, 512, nullptr, 0, 0, tw[4], tw[5], ws.xs[l], 256, T, 256, 1, ws.mpre[l]);
        x = ws.xs[l];
    }
    const float *const *aw = wts + 34, *const *cw = wts + 40;
    for (int hd = 0; hd < 2; hd++) {   // heads on cat(emb, att) (net_tree.py:56-71, 100-110)
        const float *const *hw = hd ? cw : aw;
        lin.gemm(ws.emb, nullptr, 256, 256, x, 256, 256, hw[0], hw[1], ws.y1[hd], 256, T, 256, 1, ws.y1p[hd]);
        lin.gemm(ws.y1[hd], nullptr, 256, 256, nullptr, 0, 0, hw[2], hw[3], ws.y2[hd], 128, T, 128, 1, ws.y2p[hd]);
    }
    k_heads_final<<<(unsigned)E, 256, (size_t)N * sizeof(float), st>>>(ws.y2[0], ws.y2[1], aw[4], aw[5], cw[4], cw[5], in.logits, in.value, (int)N);
    g_launches++;
    if (!loss) return (int)cudaGetLastError();

    // ==== PPO loss: d loss / d logits, d loss / d critic output, statistics ====
    // these rows' counts go to words 32..35 of ws.counts (zeroed above), their advantage moments to words 36..39; one shard
    // of a minibatch divides by the minibatch's counts and normalises by its moments
    unsigned long long *cnt = reinterpret_cast<unsigned long long *>(ws.counts + 32);
    double *mom = reinterpret_cast<double *>(ws.counts + 36);
    const long long *gcnt = in.gcnt ? in.gcnt : reinterpret_cast<const long long *>(cnt);
    PpoArgs pa{in.logits, in.value, in.old_lp, in.adv, in.ret, in.valid, in.actions, in.acted, E, (int)N, in.eps, in.vf, in.ent,
               cnt, ws.dlogits, ws.dcrit, ws.rowstats, gcnt, in.old_values, in.gmom ? in.gmom : mom, in.vf_clip, in.adv_eps,
               in.norm_adv};
    k_ppo_count<<<(unsigned)E, 128, 0, st>>>(pa);
    if (in.norm_adv && !in.gmom) {
        k_ppo_moments<<<1, 1024, 0, st>>>(pa, mom);
        g_launches++;
    }
    if (in.norm_adv || in.vf_clip > 0.0f) k_ppo_loss<true><<<(unsigned)E, 128, 0, st>>>(pa);
    else k_ppo_loss<false><<<(unsigned)E, 128, 0, st>>>(pa);
    k_ppo_stats<<<1, 256, 0, st>>>(ws.rowstats, E, cnt, gcnt, in.vf, in.ent, in.stats);
    g_launches += 3;

    // ==== backward: heads (net_tree.py:56-71, 100-110); the last layers (N = 5, 1) stay on F32Lin ====
    f32.dx(ws.dlogits, 5, 5, aw[4], 128, 128, ws.dy2, nullptr, 128, nullptr, 0, 0, ws.y2p[0], 128, T);
    f32.dw(ws.dlogits, 5, 5, ws.y2[0], nullptr, 128, 128, nullptr, 0, 0, T, gr[38], gr[39]);
    lin.dx(ws.dy2, 128, 128, aw[2], 256, 256, ws.dy1, nullptr, 256, nullptr, 0, 0, ws.y1p[0], 256, T);
    lin.dw(ws.dy2, 128, 128, ws.y1[0], nullptr, 256, 256, nullptr, 0, 0, T, gr[36], gr[37]);
    lin.dx(ws.dy1, 256, 256, aw[0], 512, 512, ws.dz, nullptr, 512, nullptr, 0, 0, nullptr, 0, T);
    lin.dw(ws.dy1, 256, 256, ws.emb, nullptr, 256, 256, x, 256, 256, T, gr[34], gr[35]);
    f32.dx(ws.dcrit, 1, 1, cw[4], 128, 128, ws.dy2, nullptr, 128, nullptr, 0, 0, ws.y2p[1], 128, T);
    f32.dw(ws.dcrit, 1, 1, ws.y2[1], nullptr, 128, 128, nullptr, 0, 0, T, gr[44], gr[45]);
    lin.dx(ws.dy2, 128, 128, cw[2], 256, 256, ws.dy1, nullptr, 256, nullptr, 0, 0, ws.y1p[1], 256, T);
    lin.dw(ws.dy2, 128, 128, ws.y1[1], nullptr, 256, 256, nullptr, 0, 0, T, gr[42], gr[43]);
    lin.dx(ws.dy1, 256, 256, cw[0], 512, 512, ws.dz, nullptr, 512, nullptr, 0, 1, nullptr, 0, T);      // dz = d cat(emb, att)
    lin.dw(ws.dy1, 256, 256, ws.emb, nullptr, 256, 256, x, 256, 256, T, gr[40], gr[41]);
    // ==== three attention blocks (net_tree.py:20-32), last to first ====
    int cur = 0;
    gelu_bwd(ws.dz + 256, 512, ws.mpre[2], 256, ws.dx[cur], 256, T, 256);
    for (int l = 2; l >= 0; l--) {
        const float *const *tw = wts + 16 + 6 * l;
        float *const *tg = gr + 16 + 6 * l;
        const float *xin = l ? ws.xs[l - 1] : ws.emb;
        const float *dpm = ws.dx[cur];
        lin.dw(dpm, 256, 256, ws.cat[l], nullptr, 512, 512, nullptr, 0, 0, T, tg[4], tg[5]);                  // att_mlp.0
        lin.dx(dpm, 256, 256, tw[4], 512, 512, ws.dcat, nullptr, 512, nullptr, 0, 0, nullptr, 0, T);
        lin.dw(ws.dcat + 256, 512, 256, ws.att[l], nullptr, 256, 256, nullptr, 0, 0, T, tg[2], tg[3]);         // out_proj
        lin.dx(ws.dcat + 256, 512, 256, tw[2], 256, 256, ws.datt, nullptr, 256, nullptr, 0, 0, nullptr, 0, T);
        k_attn_bwd_q<<<(unsigned)((T * 4 * 32 + 255) / 256), 256, 0, st>>>(ws.qkv[l], ws.att[l], ws.datt, ws.lse[l], ws.dqkv, ws.Dq, E, (int)N);
        k_attn_bwd_kv<<<(unsigned)((T * 4 * 32 + 255) / 256), 256, 0, st>>>(ws.qkv[l], ws.datt, ws.lse[l], ws.Dq, ws.dqkv, E, (int)N);
        g_launches += 2;
        lin.dw(ws.dqkv, 768, 768, xin, nullptr, 256, 256, nullptr, 0, 0, T, tg[0], tg[1]);                      // in_proj
        if (l > 0) {   // d(block input) = d cat[:, :256] + dqkv W_in, through the previous block's GELU
            lin.dx(ws.dqkv, 768, 768, tw[0], 256, 256, ws.dx[cur ^ 1], nullptr, 256, ws.dcat, 512, 0, ws.mpre[l - 1], 256, T);
            cur ^= 1;
        } else {       // d emb = dz[:, :256] (heads) + d cat[:, :256] + dqkv W_in, into dz[:, :256]
            lin.dx(ws.dqkv, 768, 768, tw[0], 256, 256, ws.dz, nullptr, 512, ws.dcat, 512, 1, nullptr, 0, T);
        }
    }
    // ==== attribute MLP (net_tree.py:41-50) on d emb[:, :128] ====
    gelu_bwd(ws.dz, 512, ws.ap[3], 256, ws.dx[0], 256, T, 128);
    lin.dw(ws.dx[0], 256, 128, ws.aa[2], nullptr, 256, 256, nullptr, 0, 0, T, gr[14], gr[15]);
    lin.dx(ws.dx[0], 256, 128, wts[14], 256, 256, ws.dx[1], nullptr, 256, nullptr, 0, 0, ws.ap[2], 256, T);
    lin.dw(ws.dx[1], 256, 256, ws.aa[1], nullptr, 256, 256, nullptr, 0, 0, T, gr[12], gr[13]);
    lin.dx(ws.dx[1], 256, 256, wts[12], 256, 256, ws.dx[0], nullptr, 256, nullptr, 0, 0, ws.ap[1], 256, T);
    lin.dw(ws.dx[0], 256, 256, ws.aa[0], nullptr, 256, 256, nullptr, 0, 0, T, gr[10], gr[11]);
    lin.dx(ws.dx[0], 256, 256, wts[10], 256, 256, ws.dx[1], nullptr, 256, nullptr, 0, 0, ws.ap[0], 256, T);
    lin.dw(ws.dx[1], 256, 256, d_agent_attr, nullptr, 83, 83, nullptr, 0, 0, T, gr[8], gr[9]);
    // ==== Tree-LSTM (TreeLSTM.py:59-154), deepest level first; d h of the roots = d emb[:, 128:] ====
    err = cudaMemsetAsync(ws.dh, 0, (size_t)nodes * T_H * 4, st);
    if (err == cudaSuccess) err = cudaMemsetAsync(ws.dc, 0, (size_t)nodes * T_H * 4, st);
    if (err != cudaSuccess) return (int)err;
    copy_cols(ws.dz + 128, 512, ws.dh, (long long)f32path::NODES * T_H, T, 128);
    for (int lv = MAX_LEVELS - 1; lv >= 1; lv--) {
        const long long M = counts[lv], io = loff[lv] - n_leaf;
        if (M <= 0) continue;
        const int32_t *list = ws.lists + loff[lv], *mr = ws.merge_row + io, *cr = ws.child_row + 3 * io;
        float *dG = ws.dG + loff[lv] * 384, *dC = ws.dC + io * 128, *dFC = ws.dFC + io * 384, *dF = ws.dF + io * 384, *dFs = ws.dFs + io * 128;
        k_inner_bwd<<<(unsigned)M, 128, 0, st>>>(ws.iou + io * 384, list, ws.xcl, W_iou, b_iou, ws.c, ws.dh, ws.dc, dG, dC);
        g_launches++;
        lin.dx(dG, 384, 384, U_iou, 384, 384, ws.dh, mr, T_H, nullptr, 0, 0, nullptr, 0, M);            // children's h via U_iou (first write)
        lin.dx(dC, 128, 128, W_c, 384, 384, dFC, nullptr, 384, nullptr, 0, 0, nullptr, 0, M);           // d(f * c_child)
        k_forget_bwd<<<(unsigned)M, 384, 0, st>>>(ws.fraw + io * 384, list, cr, ws.xcl, W_f, b_f, ws.c, dFC, ws.dc, dF, dFs);
        g_launches++;
        lin.dx(dF, 128, 128, U_f, 128, 128, ws.dh, cr, T_H, nullptr, 0, 1, nullptr, 0, 3 * M);          // children's h via U_f (added)
    }
    if (n_leaf > 0) {
        k_inner_bwd<<<(unsigned)n_leaf, 128, 0, st>>>(nullptr, ws.lists, ws.xcl, W_iou, b_iou, ws.c, ws.dh, ws.dc, ws.dG, nullptr);
        g_launches++;
    }
    f32.dw(ws.dG, 384, 384, ws.xcl, ws.lists, NF, NF, nullptr, 0, 0, n_leaf + n_in, gr[0], gr[1]);                 // W_iou, b_iou
    lin.dw(ws.dG + n_leaf * 384, 384, 384, ws.h, ws.merge_row, T_H, 3 * T_H, nullptr, 0, 0, n_in, gr[2], nullptr); // U_iou
    lin.dw(ws.dC, 128, 128, ws.fc, nullptr, 384, 384, nullptr, 0, 0, n_in, gr[3], gr[4]);                          // W_c, b_c
    f32.dw(ws.dFs, 128, 128, ws.xcl, ws.lists + n_leaf, NF, NF, nullptr, 0, 0, n_in, gr[5], gr[6]);                // W_f, b_f
    lin.dw(ws.dF, 128, 128, ws.h, ws.child_row, T_H, T_H, nullptr, 0, 0, 3 * n_in, gr[7], nullptr);                // U_f
    return (int)cudaGetLastError();
}

// E, N > 0 and E * N * 31 < 2^31: node ids are 32-bit
bool bad_shape(int64_t E, int64_t N) {
    return E <= 0 || N <= 0 || N > (1ll << 31) / f32path::NODES || E > ((1ll << 31) / f32path::NODES) / N;
}

// the observation-side argument checks of every entry point of the fp32 network (FL_ERR_BAD_ARG before any CUDA call);
// carves `ws` out of d_workspace in the training layout when `train`, else in the forward-only one
int check_obs(const float *const *wts, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N, const PpoIn &in,
              Wg &ws, bool train) {
    if (!wts || !d_workspace || !in.agent_attr || !in.forest || !in.adjacency || !in.node_order || !in.logits || !in.value)
        return -1;
    if (bad_shape(E, N)) return -1;
    for (int i = 0; i < FL_POLICY_F32_TENSORS; i++)
        if (!wts[i]) return -1;
    return carve(ws, (unsigned char *)d_workspace, E * N, train) > workspace_bytes ? -1 : 0;
}

// the argument checks of fl_policy_ppo_grad_f32: the observation side and the loss's inputs
int check_args(const float *const *wts, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N, const PpoIn &in,
               const FlPpoParams *params, Wg &ws) {
    if (!in.grads || !params || !in.valid || !in.actions || !in.old_lp || !in.adv || !in.ret || !in.acted || !in.stats) return -1;
    if (!(params->clip_eps > 0.0f)) return -1;
    if (!(in.vf_clip >= 0.0f) || (in.norm_adv != 0 && in.norm_adv != 1) || !(in.adv_eps >= 0.0f) || !std::isfinite(in.adv_eps)) return -1;
    if ((in.vf_clip > 0.0f && !in.old_values) || (in.gmom && !in.gcnt)) return -1;
    for (int i = 0; i < FL_POLICY_F32_TENSORS; i++)
        if (!in.grads[i]) return -1;
    return check_obs(wts, d_workspace, workspace_bytes, E, N, in, ws, true);
}

}  // namespace ppograph

extern "C" {

int fl_policy_abi_version(void) { return FL_POLICY_ABI_VERSION; }

uint64_t fl_policy_launch_count(void) { return g_launches; }

size_t fl_policy_workspace_bytes(int64_t n_agents_total) { return carve(nullptr, n_agents_total).bytes; }

int fl_policy_linear(const uint16_t *d_a, int64_t lda, const uint16_t *d_w, const float *d_bias, uint16_t *d_c, int64_t ldc,
                     int64_t M, int64_t N, int64_t K, int act, void *stream) {
    int rc = setup();
    if (rc) return rc;
    if (K > 512) return -1;
    return launch_linear((const bf16 *)d_a, (int)lda, (int)K, nullptr, 0, 0, (const bf16 *)d_w, d_bias, (bf16 *)d_c, (int)ldc, M, (int)N, act,
                         (cudaStream_t)stream);
}

int fl_policy_linear_debug(const uint16_t *d_a, int64_t lda, const uint16_t *d_w, const float *d_bias, uint16_t *d_c, int64_t ldc,
                           int64_t M, int64_t N, int64_t K, int act, long long *d_clocks, void *stream) {
    int rc = setup();
    if (rc) return rc;
    g_dbg = d_clocks;
    rc = launch_linear((const bf16 *)d_a, (int)lda, (int)K, nullptr, 0, 0, (const bf16 *)d_w, d_bias, (bf16 *)d_c, (int)ldc, M, (int)N, act,
                       (cudaStream_t)stream);
    g_dbg = nullptr;
    return rc;
}

void fl_policy_debug_clocks(long long *d_clocks) { g_leaf_dbg = d_clocks; }

int fl_policy_forward(const FlPolicyWeights *w, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                      const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                      const int32_t *d_node_order, float *d_logits, float *d_value, void *stream) {
    int rc = setup();
    if (rc) return rc;
    const long long M = E * N;
    if (M <= 0 || M > 0x3FFFFF - NULL_COPIES || !w || !d_workspace) return -1;   // 22-bit tree ids in the level lists
    Workspace ws = carve(d_workspace, M);
    if (workspace_bytes < ws.bytes) return -1;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(ws.counts, 0, 64 * sizeof(int), st);
    // a tree without a single edge has node_order -2 everywhere: its root is never evaluated and h stays 0 (TreeLSTM.py:49-50)
    if (e == cudaSuccess) e = cudaMemsetAsync(ws.emb, 0, (size_t)M * 256 * 2, st);
    if (e != cudaSuccess) return (int)e;
    {
        const long long total = ((M * 16 + 31) & ~31LL) + (M + NULL_COPIES) * NODES;
        k_prep<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(d_agent_attr, d_forest, ws.attr, ws.x, ws.nullmask, M);
        k_tree_plan<<<(unsigned)((M + NULL_COPIES + 127) / 128), 128, 0, st>>>(d_adjacency, d_node_order, ws.nullmask, ws.lists, ws.eflags, ws.counts, M);
        g_launches += 2;
    }
    // ---- Tree-LSTM, level by level (TreeLSTM.py:54-56) ----
    for (int lv = 0; lv < FL_POLICY_MAX_LEVELS; lv++) {
        const uint32_t *list = ws.lists + (lv == 0 ? 0 : (size_t)21 * M + NULL_COPIES + (size_t)(lv - 1) * 10 * M);
        const uint32_t null_off = (uint32_t)((M * NODES + 1) * 128);
        if (lv > 0) {
            LinArgs p = {};
            p.a0 = ws.h; p.a2 = ws.x;
            p.kb0 = 2; p.kb1 = 0; p.k16 = 1;
            p.w = (const bf16 *)w->tree_ufwf; p.ldw = 144; p.bias = w->tree_b_f;
            p.rows = 0; p.rows_dev = ws.counts + lv; p.rows_mul = 3;
            p.entries = list; p.cstate = ws.c; p.fc = ws.fc;
            p.eflags = ws.eflags + (list - ws.lists); p.null_off = null_off;
            p.stages = 6;                                   // W 3 tiles + 6 stages + output and c staging tiles
            p.dbg = (lv == 1 && g_leaf_dbg && getenv("FL_POLICY_DBG_F")) ? g_leaf_dbg : nullptr;   // tuning only
            static CUtensorMap dummy;
            k_lin<MODE_TREE_F, 128><<<dim3(g_num_sms, 1), LIN_THREADS, 1024 + 9 * TILE + 2 * 128 * OUT_PITCH + 2048 + 512, st>>>(p, dummy, dummy, dummy);
            g_launches++;
        }
        if (lv == 0) {
            LeafArgs lf = {};
            lf.entries = list; lf.count_dev = ws.counts; lf.x = ws.x; lf.h = ws.h; lf.c = ws.c;
            lf.emb = ws.emb + 128; lf.emb_ld = 256;
            lf.wiou = (const bf16 *)w->tree_wiou; lf.b_iou = w->tree_b_iou; lf.dbg = (g_leaf_dbg && !getenv("FL_POLICY_DBG_F")) ? g_leaf_dbg : nullptr;
            k_tree_leaf<<<g_num_sms, LEAF_THREADS, 1024 + (3 + LEAF_STAGES) * TILE + 4 * 128 * LEAF_PITCH + 2048, st>>>(lf);
            g_launches++;
            continue;
        }
        TreeArgs t = {};
        t.entries = list; t.count_dev = ws.counts + lv; t.level = lv;
        t.x = ws.x; t.h = ws.h; t.c = ws.c; t.fc = ws.fc;
        t.emb = ws.emb + 128; t.emb_ld = 256;
        t.uiou = (const bf16 *)w->tree_uiou; t.wiou = (const bf16 *)w->tree_wiou; t.wc = (const bf16 *)w->tree_wc;
        t.b_iou = w->tree_b_iou; t.b_c = w->tree_b_c;
        t.eflags = ws.eflags + (list - ws.lists); t.null_off = null_off;
        CUtensorMap tu, tc;
        if ((rc = make_tmap(&tu, (const bf16 *)w->tree_uiou, 384, 384, 384))) return rc;
        if ((rc = make_tmap(&tc, (const bf16 *)w->tree_wc, 128, 384, 384))) return rc;
        k_tree_p<<<g_num_sms, 416, P_STAGES * P_STAGE_BYTES + 128 * OUT_PITCH + 512 + 128, st>>>(t, tu, tc);
        g_launches++;
    }
    // ---- attribute MLP (net_tree.py:41-50) ----
    if ((rc = launch_linear(ws.attr, 128, 128, nullptr, 0, 0, (const bf16 *)w->attr_w[0], w->attr_b[0], ws.a1, 256, M, 256, 1, st))) return rc;
    if ((rc = launch_linear(ws.a1, 256, 256, nullptr, 0, 0, (const bf16 *)w->attr_w[1], w->attr_b[1], ws.a2, 256, M, 256, 1, st))) return rc;
    if ((rc = launch_linear(ws.a2, 256, 256, nullptr, 0, 0, (const bf16 *)w->attr_w[2], w->attr_b[2], ws.a1, 256, M, 256, 1, st))) return rc;
    if ((rc = launch_linear(ws.a1, 256, 256, nullptr, 0, 0, (const bf16 *)w->attr_w[3], w->attr_b[3], ws.emb, 256, M, 128, 1, st))) return rc;
    // ---- 3 attention blocks (net_tree.py:10-32, 51-55) ----
    const bf16 *tin = ws.emb;
    bf16 *touts[3] = {ws.ta, ws.tb, ws.ta};
    for (int l = 0; l < FL_POLICY_LAYERS; l++) {
        if ((rc = launch_linear(tin, 256, 256, nullptr, 0, 0, (const bf16 *)w->tf_wqkv[l], w->tf_bqkv[l], ws.qkv, 768, M, 768, 0, st))) return rc;
        {
            AttnArgs at = {};
            at.out = ws.atto; at.N = (int)N; at.E = (int)E;
            unsigned tiles;
            if (N <= 128) {
                const int G = 128 / (int)N;
                at.rows_per_tile = G * (int)N; at.tiles_per_env = 0;
                tiles = (unsigned)((E + G - 1) / G);
            } else {
                at.rows_per_tile = 128; at.tiles_per_env = (int)((N + 127) / 128);
                tiles = (unsigned)(E * at.tiles_per_env);
            }
            CUtensorMap tq;
            if ((rc = make_tmap(&tq, ws.qkv, (unsigned long long)M, 768, 768))) return rc;
            k_attn_mma<<<dim3(tiles, FL_POLICY_HEADS), 128, ATTN_SMEM, st>>>(at, tq);
            g_launches++;
        }
        // out_proj is folded into att_mlp's weights at pack time (policy.py:pack_weights): cat(input, heads) -> GELU
        if ((rc = launch_linear(tin, 256, 256, ws.atto, 256, 256, (const bf16 *)w->tf_wm[l], w->tf_bm[l], touts[l], 256, M, 256, 1, st))) return rc;
        tin = touts[l];
    }
    // ---- actor / critic heads (net_tree.py:56-71, 100-110) ----
    if ((rc = launch_linear(ws.emb, 256, 256, tin, 256, 256, (const bf16 *)w->head_w1, w->head_b1, ws.y1, 512, M, 512, 1, st))) return rc;
    if ((rc = launch_linear(ws.y1, 512, 256, nullptr, 0, 0, (const bf16 *)w->head_w2a, w->head_b2, ws.y2, 256, M, 128, 1, st))) return rc;
    if ((rc = launch_linear(ws.y1 + 256, 512, 256, nullptr, 0, 0, (const bf16 *)w->head_w2c, w->head_b2 + 128, ws.y2 + 128, 256, M, 128, 1, st))) return rc;
    k_head_final<<<(unsigned)E, 256, (size_t)N * sizeof(float), st>>>(ws.y2, w->head_w3, w->head_b3, d_logits, d_value, (int)N);
    g_launches++;
    return (int)cudaGetLastError();
}

// ---- the same forward pass in fp32 on the CUDA cores (policy_f32.cuh): the training graph's forward, forward-only layout
size_t fl_policy_workspace_bytes_f32(int64_t n_agents_total) {
    if (n_agents_total <= 0) return 0;
    f32grad::Wg w;
    return f32grad::carve(w, nullptr, n_agents_total, false);
}

int fl_policy_forward_f32(const float *const *wts, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                          const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                          const int32_t *d_node_order, float *d_logits, float *d_value, void *stream) {
    const ppograph::PpoIn in{d_agent_attr, d_forest, d_adjacency, d_node_order, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                             0.0f, 0.0f, 0.0f, nullptr, d_logits, d_value, nullptr, nullptr};
    f32grad::Wg ws;
    if (ppograph::check_obs(wts, d_workspace, workspace_bytes, E, N, in, ws, false)) return -1;
    ppograph::F32Lin lin{(cudaStream_t)stream, ws.part};
    return ppograph::run(lin, wts, ws, E, N, in, false, (cudaStream_t)stream);
}

// ---- PPO loss and gradients of the fp32 network (policy_f32_grad.cuh) ------------------------------------------------
size_t fl_policy_workspace_bytes_grad_f32(int64_t n_agents_total) {
    if (n_agents_total <= 0) return 0;
    f32grad::Wg w;
    return f32grad::carve(w, nullptr, n_agents_total, true);
}

// The one PPO path: fl_policy_ppo_grad_{f32,bf16} are it with the counts taken from the workspace (gcnt null) and the
// options off, fl_policy_ppo_grad_shard_* with the options off, fl_policy_ppo_grad_ex_* as given
static int ppo_grad(bool bf16, const int64_t *gcnt, const float *const *wts, void *d_workspace, size_t workspace_bytes,
                    int64_t E, int64_t N, const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                    const int32_t *d_node_order, const uint8_t *d_valid_actions, const uint8_t *d_actions,
                    const float *d_old_log_probs, const float *d_advantages, const float *d_returns, const uint8_t *d_acted,
                    const FlPpoParams *params, float *const *d_grads, float *d_logits, float *d_value, float *d_stats,
                    void *stream, const float *d_old_values = nullptr, const double *gmom = nullptr,
                    const FlPpoOptions *opts = nullptr) {
    ppograph::PpoIn in{d_agent_attr, d_forest, d_adjacency, d_node_order, d_valid_actions, d_actions, d_old_log_probs, d_advantages,
                       d_returns, d_acted, params ? params->clip_eps : 0.0f, params ? params->vf_coef : 0.0f,
                       params ? params->ent_coef : 0.0f, d_grads, d_logits, d_value, d_stats,
                       reinterpret_cast<const long long *>(gcnt)};
    in.old_values = d_old_values;
    in.gmom = gmom;
    if (opts) {
        in.vf_clip = opts->vf_clip;
        in.norm_adv = opts->norm_adv;
        in.adv_eps = opts->adv_eps;
    }
    f32grad::Wg ws;
    if (ppograph::check_args(wts, d_workspace, workspace_bytes, E, N, in, params, ws)) return -1;
    if (!bf16) {
        ppograph::F32Lin lin{(cudaStream_t)stream, ws.part};
        return ppograph::run(lin, wts, ws, E, N, in, true, (cudaStream_t)stream);
    }
    const int rc = ppograph::bf16_setup();
    if (rc) return rc;
    ppograph::Bf16Lin lin{(cudaStream_t)stream, ws.part};
    return ppograph::run(lin, wts, ws, E, N, in, true, (cudaStream_t)stream);
}

int fl_policy_ppo_grad_f32(const float *const *wts, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                           const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                           const int32_t *d_node_order, const uint8_t *d_valid_actions, const uint8_t *d_actions,
                           const float *d_old_log_probs, const float *d_advantages, const float *d_returns, const uint8_t *d_acted,
                           const FlPpoParams *params, float *const *d_grads, float *d_logits, float *d_value, float *d_stats,
                           void *stream) {
    return ppo_grad(false, nullptr, wts, d_workspace, workspace_bytes, E, N, d_agent_attr, d_forest, d_adjacency, d_node_order,
                    d_valid_actions, d_actions, d_old_log_probs, d_advantages, d_returns, d_acted, params, d_grads, d_logits, d_value,
                    d_stats, stream);
}

// ---- the same loss and gradients with the dense products on the tensor cores (policy_bf16_grad.cuh) --------------------
size_t fl_policy_workspace_bytes_grad_bf16(int64_t n_agents_total) { return fl_policy_workspace_bytes_grad_f32(n_agents_total); }

int fl_policy_ppo_grad_bf16(const float *const *wts, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                            const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                            const int32_t *d_node_order, const uint8_t *d_valid_actions, const uint8_t *d_actions,
                            const float *d_old_log_probs, const float *d_advantages, const float *d_returns, const uint8_t *d_acted,
                            const FlPpoParams *params, float *const *d_grads, float *d_logits, float *d_value, float *d_stats,
                            void *stream) {
    return ppo_grad(true, nullptr, wts, d_workspace, workspace_bytes, E, N, d_agent_attr, d_forest, d_adjacency, d_node_order,
                    d_valid_actions, d_actions, d_old_log_probs, d_advantages, d_returns, d_acted, params, d_grads, d_logits, d_value,
                    d_stats, stream);
}

// ---- one shard of a data-parallel minibatch: the counts of its rows, and the loss divided by the minibatch's counts ------
int fl_policy_ppo_counts(int64_t E, int64_t N, const uint8_t *d_valid_actions, const uint8_t *d_acted, int64_t *d_counts,
                         void *stream) {
    if (ppograph::bad_shape(E, N) || !d_valid_actions || !d_acted || !d_counts) return -1;      // as fl_policy_ppo_grad_f32
    const cudaStream_t st = (cudaStream_t)stream;
    const cudaError_t err = cudaMemsetAsync(d_counts, 0, 2 * sizeof(int64_t), st);
    if (err != cudaSuccess) return (int)err;
    f32grad::PpoArgs pa{};
    pa.valid = d_valid_actions;
    pa.acted = d_acted;
    pa.E = E;
    pa.N = (int)N;
    pa.cnt = reinterpret_cast<unsigned long long *>(d_counts);
    f32grad::k_ppo_count<<<(unsigned)E, 128, 0, st>>>(pa);
    g_launches++;
    return (int)cudaGetLastError();
}

int fl_policy_ppo_grad_shard_f32(const float *const *wts, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                                 const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                                 const int32_t *d_node_order, const uint8_t *d_valid_actions, const uint8_t *d_actions,
                                 const float *d_old_log_probs, const float *d_advantages, const float *d_returns, const uint8_t *d_acted,
                                 const int64_t *d_global_counts,
                                 const FlPpoParams *params, float *const *d_grads, float *d_logits, float *d_value, float *d_stats,
                                 void *stream) {
    if (!d_global_counts) return -1;
    return ppo_grad(false, d_global_counts, wts, d_workspace, workspace_bytes, E, N, d_agent_attr, d_forest, d_adjacency, d_node_order,
                    d_valid_actions, d_actions, d_old_log_probs, d_advantages, d_returns, d_acted, params, d_grads, d_logits, d_value,
                    d_stats, stream);
}

int fl_policy_ppo_grad_shard_bf16(const float *const *wts, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                                  const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                                  const int32_t *d_node_order, const uint8_t *d_valid_actions, const uint8_t *d_actions,
                                  const float *d_old_log_probs, const float *d_advantages, const float *d_returns, const uint8_t *d_acted,
                                  const int64_t *d_global_counts,
                                  const FlPpoParams *params, float *const *d_grads, float *d_logits, float *d_value, float *d_stats,
                                  void *stream) {
    if (!d_global_counts) return -1;
    return ppo_grad(true, d_global_counts, wts, d_workspace, workspace_bytes, E, N, d_agent_attr, d_forest, d_adjacency, d_node_order,
                    d_valid_actions, d_actions, d_old_log_probs, d_advantages, d_returns, d_acted, params, d_grads, d_logits, d_value,
                    d_stats, stream);
}

// ---- options of the loss: the minibatch's advantage moments, and the PPO path with clipped value loss / normalisation ----
int fl_policy_ppo_moments(int64_t E, int64_t N, const uint8_t *d_valid_actions, const uint8_t *d_acted, const float *d_advantages,
                          double *d_moments, void *stream) {
    if (ppograph::bad_shape(E, N) || !d_valid_actions || !d_acted || !d_advantages || !d_moments) return -1;
    f32grad::PpoArgs pa{};
    pa.valid = d_valid_actions;
    pa.acted = d_acted;
    pa.adv = d_advantages;
    pa.E = E;
    pa.N = (int)N;
    f32grad::k_ppo_moments<<<1, 1024, 0, (cudaStream_t)stream>>>(pa, d_moments);
    g_launches++;
    return (int)cudaGetLastError();
}

int fl_policy_ppo_grad_ex_f32(const float *const *wts, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                              const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                              const int32_t *d_node_order, const uint8_t *d_valid_actions, const uint8_t *d_actions,
                              const float *d_old_log_probs, const float *d_advantages, const float *d_returns, const uint8_t *d_acted,
                              const int64_t *d_global_counts,
                              const FlPpoParams *params, float *const *d_grads, float *d_logits, float *d_value, float *d_stats,
                              void *stream, const float *d_old_values, const double *d_global_moments, const FlPpoOptions *opts) {
    if (!opts) return -1;
    return ppo_grad(false, d_global_counts, wts, d_workspace, workspace_bytes, E, N, d_agent_attr, d_forest, d_adjacency, d_node_order,
                    d_valid_actions, d_actions, d_old_log_probs, d_advantages, d_returns, d_acted, params, d_grads, d_logits, d_value,
                    d_stats, stream, d_old_values, d_global_moments, opts);
}

int fl_policy_ppo_grad_ex_bf16(const float *const *wts, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                               const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                               const int32_t *d_node_order, const uint8_t *d_valid_actions, const uint8_t *d_actions,
                               const float *d_old_log_probs, const float *d_advantages, const float *d_returns, const uint8_t *d_acted,
                               const int64_t *d_global_counts,
                               const FlPpoParams *params, float *const *d_grads, float *d_logits, float *d_value, float *d_stats,
                               void *stream, const float *d_old_values, const double *d_global_moments, const FlPpoOptions *opts) {
    if (!opts) return -1;
    return ppo_grad(true, d_global_counts, wts, d_workspace, workspace_bytes, E, N, d_agent_attr, d_forest, d_adjacency, d_node_order,
                    d_valid_actions, d_actions, d_old_log_probs, d_advantages, d_returns, d_acted, params, d_grads, d_logits, d_value,
                    d_stats, stream, d_old_values, d_global_moments, opts);
}

int fl_policy_forward_train_bf16(const float *const *wts, void *d_workspace, size_t workspace_bytes, int64_t E, int64_t N,
                                 const float *d_agent_attr, const float *d_forest, const int32_t *d_adjacency,
                                 const int32_t *d_node_order, float *d_logits, float *d_value, void *stream) {
    const ppograph::PpoIn in{d_agent_attr, d_forest, d_adjacency, d_node_order, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr,
                             0.0f, 0.0f, 0.0f, nullptr, d_logits, d_value, nullptr, nullptr};
    f32grad::Wg ws;      // the training layout: the header gives this call fl_policy_workspace_bytes_grad_bf16's workspace
    if (ppograph::check_obs(wts, d_workspace, workspace_bytes, E, N, in, ws, true)) return -1;
    const int rc = ppograph::bf16_setup();
    if (rc) return rc;
    ppograph::Bf16Lin lin{(cudaStream_t)stream, ws.part};
    return ppograph::run(lin, wts, ws, E, N, in, false, (cudaStream_t)stream);
}

int fl_policy_tc_product_bf16(const FlTcProduct *p, void *d_workspace, size_t workspace_bytes, void *stream) {
    if (!p || p->M < 0 || p->N <= 0 || p->K <= 0 || !p->c) return -1;
    const bool xok = p->x1 && p->K1 >= 0 && p->K2 >= 0 && p->K1 + p->K2 == p->K && (!p->K2 || p->x2);
    if (p->kind == FL_TC_FORWARD) {
        if (!xok || !p->w) return -1;
    } else if (p->kind == FL_TC_DX) {
        if (!p->dy || !p->w || p->ldw < p->K) return -1;
    } else if (p->kind == FL_TC_DW) {
        if (!p->dy || !xok || !d_workspace) return -1;
        int nch = 0;
        bf16grad::dw_chunk(p->M, &nch);
        if ((size_t)nch * p->N * (p->K + 1) * 4 > workspace_bytes) return -1;
    } else {
        return -1;
    }
    const int rc = ppograph::bf16_setup();
    if (rc) return rc;
    ppograph::Bf16Lin lin{(cudaStream_t)stream, (float *)d_workspace};
    if (p->kind == FL_TC_FORWARD)
        lin.gemm(p->x1, p->idx, p->ldx1, p->K1, p->x2, p->ldx2, p->K2, p->w, p->bias, p->c, p->ldc, p->M, p->N, p->act, p->pre);
    else if (p->kind == FL_TC_DX)
        lin.dx(p->dy, p->lddy, p->N, p->w, p->ldw, p->K, p->c, p->cidx, p->ldc, p->add, p->ldadd, p->accum, p->gpre, p->ldgpre, p->M);
    else
        lin.dw(p->dy, p->lddy, p->N, p->x1, p->idx, p->ldx1, p->K1, p->x2, p->ldx2, p->K2, p->M, p->c, p->db);
    return (int)cudaGetLastError();
}

int fl_policy_choose_actions(const float *d_logits, const uint8_t *d_valid_actions, uint8_t *d_actions, int64_t n, void *stream) {
    if (n <= 0) return -1;
    k_choose<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_logits, d_valid_actions, d_actions, n);
    g_launches++;
    return (int)cudaGetLastError();
}

int fl_policy_sample_actions(const float *d_logits, const uint8_t *d_valid_actions, int64_t E, int64_t N, int64_t env_offset,
                             uint64_t seed, uint64_t step, uint8_t *d_actions, float *d_log_probs, void *stream) {
    if (!d_logits || !d_valid_actions || !d_actions || !d_log_probs || E <= 0 || N <= 0 || env_offset < 0) return -1;
    if (env_offset > (1ll << 32) - E) return -1;                      // the environment id is one 32-bit counter word
    if (N > (1ll << 32) || E > (1ll << 38) / N) return -1;             // agent word; the grid's x extent
    const long long n = E * N;
    rollout::k_sample<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_logits, d_valid_actions, E, N, env_offset, seed,
                                                                                   step, d_actions, d_log_probs);
    g_launches++;
    return (int)cudaGetLastError();
}

int fl_policy_gae(const int32_t *d_rewards, const uint8_t *d_dones, const float *d_values, const uint8_t *d_acted, int64_t T,
                  int64_t E, int64_t N, float gamma, float lam, float *d_advantages, float *d_returns, void *stream) {
    if (!d_rewards || !d_dones || !d_values || !d_acted || !d_advantages || !d_returns || T <= 0 || E <= 0 || N <= 0) return -1;
    if (T >= (1ll << 31) || E >= (1ll << 31) || N >= (1ll << 31) || (T + 1) * E > (1ll << 62) / (N + 1)) return -1;
    rollout::k_gae<<<(unsigned)((E + 3) / 4), 128, 0, (cudaStream_t)stream>>>(d_rewards, d_dones, d_values, d_acted, T, E, N,
                                                                              (double)gamma, (double)lam, d_advantages, d_returns);
    g_launches++;
    return (int)cudaGetLastError();
}

}  // extern "C"
