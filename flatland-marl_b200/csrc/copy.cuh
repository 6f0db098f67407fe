// copy.cuh — k_copy_envs: environment slots of one batch become copies of slots of another (or the same) batch
// (fl_copy_envs): what copy.deepcopy(env) of the reference does, for many environments in one launch.
#pragma once
#include "common.cuh"

// Every per-environment array of struct FlBatch with its extent per environment in elements and the part of
// fl_copy_envs it travels with (0 = per-call scratch of fl_observe, never copied).  fl_batch_slice and fl_copy_envs
// both walk this list.  X(field, elements per environment, part); `b` is a const FlBatch *.  FL_PART_OPTIONAL marks the
// caches, which a batch may leave NULL (fl_observe then recomputes what they hold).
#define FL_PART_SCRATCH 0u
#define FL_PART_OPTIONAL 0x100u
#define FL_BATCH_FIELDS(X, b)                                                                                            \
    X(grid, (b)->grid_stride, FL_COPY_WORLD) X(slot_rc, (b)->n_slots * 2, FL_COPY_WORLD)                               \
    X(dist, (b)->dist_stride, FL_COPY_WORLD) X(max_steps, 1, FL_COPY_WORLD) X(init_rc, (b)->N * 2, FL_COPY_WORLD)      \
    X(tgt_rc, (b)->N * 2, FL_COPY_WORLD) X(init_dir, (b)->N, FL_COPY_WORLD) X(max_count, (b)->N, FL_COPY_WORLD)        \
    X(slot, (b)->N, FL_COPY_WORLD) X(speed, (b)->N, FL_COPY_WORLD) X(earliest, (b)->N, FL_COPY_WORLD)                  \
    X(latest, (b)->N, FL_COPY_WORLD) X(sched, (b)->S * (b)->N, FL_COPY_WORLD)                                          \
    X(ridx, (b)->ridx_stride, FL_COPY_WORLD) X(srec, (b)->state_stride, FL_COPY_WORLD)                                 \
    X(wrec, (b)->state_stride * 4, FL_COPY_WORLD) X(whoff, (b)->state_stride, FL_COPY_WORLD)                           \
    X(wlist, (b)->wlist_stride, FL_COPY_WORLD) X(whits, (b)->whits_stride, FL_COPY_WORLD)                              \
    X(kcls, (b)->state_stride, FL_COPY_WORLD) X(sdist, (b)->n_slots * (b)->state_stride, FL_COPY_WORLD)                \
    X(gtab, (b)->n_slots * (b)->state_stride, FL_COPY_WORLD) X(walk_total, 4, FL_COPY_WORLD)                           \
    X(tree_cache, (b)->N * FL_TREE_CACHE_WORDS, FL_COPY_WORLD | FL_PART_OPTIONAL)                                      \
    X(path_cache, (b)->N * (b)->pc_stride, FL_COPY_WORLD | FL_PART_OPTIONAL)                                           \
    X(rc, (b)->N * 2, FL_COPY_STATE) X(old_rc, (b)->N * 2, FL_COPY_STATE) X(dir, (b)->N, FL_COPY_STATE)                \
    X(old_dir, (b)->N, FL_COPY_STATE) X(state, (b)->N, FL_COPY_STATE) X(ctr, (b)->N, FL_COPY_STATE)                    \
    X(mal, (b)->N, FL_COPY_STATE) X(saved, (b)->N, FL_COPY_STATE) X(sig_mal, (b)->N, FL_COPY_STATE)                    \
    X(deadlocked, (b)->N, FL_COPY_STATE) X(done, (b)->N, FL_COPY_STATE) X(nmal, (b)->N, FL_COPY_STATE)                 \
    X(arrival, (b)->N, FL_COPY_STATE) X(elapsed, 1, FL_COPY_STATE) X(sched_pos, 1, FL_COPY_STATE)                      \
    X(done_all, 1, FL_COPY_STATE) X(status, 1, FL_COPY_STATE) X(stats, 4, FL_COPY_STATE)                              \
    X(entries, (b)->ent_cap, FL_PART_SCRATCH) X(segs, (b)->seg_stride, FL_PART_SCRATCH)                                \
    X(debug_clocks, 32, FL_PART_SCRATCH) X(obs_ws, (b)->ws_stride, FL_PART_SCRATCH)

// The rows of FlObsBuffers, X(field, elements per environment); N = agents per environment.
#define FL_OBS_FIELDS(X, N)                                                                                              \
    X(agent_attr, (N) * FL_ATTR_F) X(forest, (N) * FL_MAX_NODES * FL_NODE_F) X(adjacency, (N) * (FL_MAX_NODES - 1) * 3) \
    X(node_order, (N) * FL_MAX_NODES) X(edge_order, (N) * (FL_MAX_NODES - 1)) X(valid_actions, (N) * 5)                \
    X(dist_target, (N)) X(rewards, (N)) X(dones, (N) + 1)

namespace {

constexpr int COPY_MAX_RANGES = 64;      // FL_BATCH_FIELDS has 47 entries, FL_OBS_FIELDS 9
constexpr int COPY_THREADS = 256;
constexpr int64_t COPY_CHUNK = 32 * 1024; // bytes of one environment pair per CTA: a 12 MB distance map spreads over 384 CTAs

// One field of the work list: environment e of it starts at base + e * bytes.  `voff` is where the field starts in the
// per-pair byte space the CTAs are cut from (a multiple of 16, so that a chunk boundary inside a field keeps the 16-byte
// alignment of the field's blocks).
struct CopyRange {
    const char *src;
    char *dst;
    int64_t bytes;
    int64_t voff;
};

// Passed by value: the list is built on the host for every call (about 1.5 KB of kernel parameters).
struct CopyPlan {
    CopyRange r[COPY_MAX_RANGES];
    int n_ranges;
    int64_t chunks;     // CTAs per environment pair
    int64_t src_E, dst_E;
};

DEVI void copy_bytes(char *__restrict__ d, const char *__restrict__ s, int64_t len, int tid) {
    const uintptr_t mis = reinterpret_cast<uintptr_t>(d) | reinterpret_cast<uintptr_t>(s);
    int64_t done = 0;
    if ((mis & 15) == 0) {
        // the big tables: 16-byte blocks (per-environment strides are multiples of 16 bytes), four loads in flight per thread
        const int64_t nv = len >> 4;
        const uint4 *__restrict__ sv = reinterpret_cast<const uint4 *>(s);
        uint4 *__restrict__ dv = reinterpret_cast<uint4 *>(d);
        int64_t k = tid;
        for (; k + 3 * COPY_THREADS < nv; k += 4 * COPY_THREADS) {
            const uint4 a0 = __ldg(sv + k), a1 = __ldg(sv + k + COPY_THREADS), a2 = __ldg(sv + k + 2 * COPY_THREADS),
                        a3 = __ldg(sv + k + 3 * COPY_THREADS);
            dv[k] = a0; dv[k + COPY_THREADS] = a1; dv[k + 2 * COPY_THREADS] = a2; dv[k + 3 * COPY_THREADS] = a3;
        }
        for (; k < nv; k += COPY_THREADS) dv[k] = __ldg(sv + k);
        done = nv << 4;
    } else if ((mis & 3) == 0) {
        // per-agent arrays of 4-byte elements (rc is N*4 bytes per environment): not 16-byte aligned for every environment
        const int64_t nw = len >> 2;
        const uint32_t *__restrict__ sw = reinterpret_cast<const uint32_t *>(s);
        uint32_t *__restrict__ dw = reinterpret_cast<uint32_t *>(d);
        for (int64_t k = tid; k < nw; k += COPY_THREADS) dw[k] = __ldg(sw + k);
        done = nw << 2;
    }
    for (int64_t k = done + tid; k < len; k += COPY_THREADS) d[k] = s[k];   // byte arrays and tails
}

// grid: pairs * plan.chunks CTAs.  CTA (pair, chunk) copies bytes [chunk, chunk + 1) * COPY_CHUNK of the pair's byte space.
__global__ void __launch_bounds__(COPY_THREADS) k_copy_envs(const CopyPlan plan, const int32_t *__restrict__ src_ids,
                                                           const int32_t *__restrict__ dst_ids) {
    const int64_t pair = blockIdx.x / plan.chunks, chunk = blockIdx.x % plan.chunks;
    const int64_t s = src_ids[pair], d = dst_ids[pair];
    if (s < 0 || s >= plan.src_E || d < 0 || d >= plan.dst_E) return;   // ids are the caller's to check; never write outside
    const int64_t v0 = chunk * COPY_CHUNK, v1 = v0 + COPY_CHUNK;
    for (int f = 0; f < plan.n_ranges; f++) {
        const CopyRange &r = plan.r[f];
        const int64_t a = v0 > r.voff ? v0 : r.voff, e = v1 < r.voff + r.bytes ? v1 : r.voff + r.bytes;
        if (a >= e) continue;
        copy_bytes(r.dst + d * r.bytes + (a - r.voff), r.src + s * r.bytes + (a - r.voff), e - a, threadIdx.x);
    }
}

}  // namespace
