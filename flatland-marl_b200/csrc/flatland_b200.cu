// flatland_b200.cu — hand-written sm_100a kernels + the C ABI declared in include/flatland_b200.h.
//
// Three kernels on the hot path (+ k_reset), all integer / byte work bound by dependent-load latency and HBM/L2,
// no dense contraction anywhere (so no tensor cores):
//   k_step   one CTA per environment, one thread per agent: RailEnv.step up to the observation
//            (rail_env.py:501-632): action preprocessing, MotionCheck as a least fixpoint resolved
//            with shared-memory broadcasts, state machine, counters, end-of-episode rewards.
//   k_observe one CTA per environment with the environment's working set in shared memory (TMA bulk
//            copies of grid + distance maps): loader view + valid actions (loader.cpp:221-327), the
//            serial sticky deadlock checker on a spare lane (deadlock_checker.cpp), greedy shortest-path
//            predictions (predictions.cpp) as a CSR inverse index  cell id -> occupancy intervals, the
//            31-node branch trees (treeobs.cpp:154-610): structure per agent from the static walk tables, then
//            one warp per agent over the flat list of the cells of all its walks, evaluation orders
//            (tool.h:468-524) and the 83-float agent attributes (feature_parser.cpp), written in the policy's
//            input layout (observe.cuh).
//   k_bfs    one CTA per (environment, unique target): DistanceMap (distance_map.py:57-160) as a
//            level-synchronous pull BFS with the whole map in shared memory.  Reset-time only.
// Reference citations are relative to the reference repository root.  No fast-math: every float
// expression mirrors one float expression of the reference (SURVEY.md A.8).
#include "flatland_b200.h"

#include <cuda_runtime.h>

#include <atomic>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <vector>

#include "common.cuh"
#include "step.cuh"
#include "observe.cuh"
#include "bfs.cuh"
#include "wire.cuh"
#include "copy.cuh"
#include "expand_pool.h"

#include <chrono>
#include <condition_variable>
#include <cstdio>
#include <functional>
#include <memory>
#include <thread>

namespace {

std::atomic<uint64_t> g_launches{0};

// Optional per-kernel timing (fl_profile_*): every launch is bracketed by CUDA events recorded on the
// launching stream; fl_profile_collect turns them into per-kernel totals.  Off by default.
enum KernelId : int { K_BFS = 0, K_RESET, K_STEP, K_OBSERVE, K_WALKS, K_OBSERVE_INDEX, K_OBSERVE_TREES, K_PACK, K_COPY, K_COUNT };
const char *const kKernelNames[K_COUNT] = {"k_bfs", "k_reset", "k_step", "k_observe", "k_walks", "k_observe_index", "k_observe_trees", "k_pack", "k_copy_envs"};
struct ProfRec { int id; cudaEvent_t a, b; };
std::mutex g_prof_mu;
bool g_prof_on = false;
std::vector<ProfRec> g_prof_pending;
std::vector<cudaEvent_t> g_prof_free;
double g_prof_ms[K_COUNT];
uint64_t g_prof_n[K_COUNT];

struct LaunchScope {  // RAII: counts the launch and, when profiling, records the event pair around it
    int id; cudaStream_t st; cudaEvent_t a = nullptr, b = nullptr; bool on;
    static cudaEvent_t get() {
        if (!g_prof_free.empty()) { cudaEvent_t e = g_prof_free.back(); g_prof_free.pop_back(); return e; }
        cudaEvent_t e; cudaEventCreate(&e); return e;
    }
    LaunchScope(int id_, cudaStream_t st_) : id(id_), st(st_) {
        g_launches++;
        std::lock_guard<std::mutex> lk(g_prof_mu);
        on = g_prof_on;
        if (on) { a = get(); b = get(); cudaEventRecord(a, st); }
    }
    ~LaunchScope() {
        if (!on) return;
        cudaEventRecord(b, st);
        std::lock_guard<std::mutex> lk(g_prof_mu);
        g_prof_pending.push_back({id, a, b});
    }
};

int round_up(int v, int m) { return (v + m - 1) / m * m; }

int check_batch(const FlBatch *b) {
    if (!b || b->E <= 0 || b->N <= 0 || b->H <= 0 || b->W <= 0 || b->n_slots <= 0 || b->S <= 0) return FL_ERR_BAD_ARG;
    if (b->N >= FL_MAX_AGENTS) return FL_ERR_TOO_MANY_AGENTS;
    if (b->ent_cap < b->N * (int64_t)NPRED) return FL_ERR_BAD_ARG;
    if (b->H >= 1024 || b->W >= 1024) return FL_ERR_BAD_ARG;   // srec packs row and column in 10 bits each
    if (b->ridx_stride < b->H * b->W || b->ridx_stride % 8 || b->state_stride % 32 || b->wlist_stride % 4 || b->whits_stride % 4)
        return FL_ERR_BAD_ARG;
    if (b->state_stride > 0xFFFF) return FL_ERR_BAD_ARG;       // state ids are 16 bit
    // per-environment blocks are 16-byte aligned so that they can be moved with TMA bulk copies
    if (b->grid_stride < b->H * b->W || b->grid_stride % 8 || b->dist_stride < b->n_slots * b->H * b->W * 4 || b->dist_stride % 8)
        return FL_ERR_BAD_ARG;
    return FL_OK;
}

constexpr int SMEM_MAX = 227 * 1024;

int align_up(int v, int a) { return (v + a - 1) / a * a; }

// Plan overrides (fl_observe_override; tuning and tests only).  -1 = default.  Seeded once from FL_OBS_<KEY> environment
// variables when the library is loaded; the launch path reads these atomics, never the environment.
enum ObsKnob : int { KNOB_NT = 0, KNOB_CTAS, KNOB_TABLES, KNOB_SEGCAP, KNOB_ENTCAP, KNOB_SORTSMALL, KNOB_PARTS, KNOB_BMGLOBAL, KNOB_TREENT, KNOB_FLATWALK, KNOB_GROUP, KNOB_TREECACHE, KNOB_PATHCACHE, KNOB_STEPMAP, KNOB_COUNT };
const char *const kKnobNames[KNOB_COUNT] = {"nt", "ctas", "tables", "segcap", "entcap", "sortsmall", "parts", "bmglobal", "treent", "flatwalk", "group", "treecache", "pathcache", "stepmap"};
const char *const kKnobEnv[KNOB_COUNT] = {"FL_OBS_NT", "FL_OBS_CTAS", "FL_OBS_TABLES", "FL_OBS_SEGCAP", "FL_OBS_ENTCAP", "FL_OBS_SORTSMALL", "FL_OBS_PARTS",
                                          "FL_OBS_BMGLOBAL", "FL_OBS_TREENT", "FL_OBS_FLATWALK", "FL_OBS_GROUP", "FL_OBS_TREECACHE", "FL_OBS_PATHCACHE", "FL_STEP_MAP"};
std::atomic<int> g_knob[KNOB_COUNT];
struct KnobInit {
    KnobInit() {
        for (int k = 0; k < KNOB_COUNT; k++) {
            const char *s = getenv(kKnobEnv[k]);
            g_knob[k].store(s && *s ? atoi(s) : -1);
        }
    }
} g_knob_init;
int knob(int k) { return g_knob[k].load(std::memory_order_relaxed); }

// Shared-memory plan of k_observe for one configuration.  Mandatory: barrier + scalars, scan partials, the
// per-agent records, the deadlock scratch, the occupancy word and the bucket offsets per rail cell (and the key
// classes when H > W).  Then, while they fit: rail grid, rail index, the sorted predicted-occupancy entries at their
// typical size ("core").  The budget per CTA is the largest that lets `ctas` CTAs share an SM, ctas being the largest
// count for which the core fits (more resident warps hide the latency of the table lookups, which then go to L2).
// What is left of the budget takes the static walk tables in the order of their use per visited cell.
// fl_observe_override("ctas" / "tables" / "nt", ...) override (tuning only).
// group > 1: the plan of ONE environment of a group-mode CTA (k_observe<..., G>): `group` copies of it, each a multiple of
// 128 bytes, share the CTA's shared memory.
ObsLayout make_obs_layout(const FlBatch *b, int nt, int mode, int parts, int *ctas_out = nullptr, int group = 1) {
    const int N = (int)b->N, Rmax = (int)(b->state_stride / 4), Np = (N + 3) & ~3;
    ObsLayout L;
    int off = 0;
    // regions are 16-byte aligned (what the bulk copies need); every byte counts towards one more resident CTA per SM
    auto take = [&](long long bytes) { const int o = off; off = align_up(off + (int)bytes, 16); return o; };
    L.parts = mode == OBS_FUSED ? 0 : parts;
    // FlBatch.obs_ws of the split launch: [header 16 B | six agent arrays] [occupancy words | bucket offsets | filter]
    L.ws_ag = 0; L.ws_ag_bytes = (4 + 6 * Np) * 4;
    L.ws_idx = L.ws_ag_bytes; L.ws_idx_bytes = Rmax * 4 + (Rmax + 4) * 4 + Rmax * 32;
    L.bar = take(16 + 4 * OBS_MISC_WORDS);                     // mbarrier, then the scalars of the environment
    L.part = take(128);                                         // one scan partial per warp
    L.ag = take(mode == OBS_TREES ? (long long)L.ws_ag_bytes : (long long)(4 + 6 * Np + 5 * N) * 4);
    L.dl = mode == OBS_TREES ? 0 : take(26 * N + 8);
    L.ci = take((long long)Rmax * 4);
    L.ks = take((long long)(Rmax + 4) * 4);
    // time-slot filter of the prediction index: one / two entries per slot; it may stay in the workspace (global memory)
    // ("bmglobal" knob; in every mode it stays in the workspace when the mandatory regions would not fit beside it: it is
    // written with plain stores once its bucket is sorted, so it can live anywhere)
    const long long sq_bytes = (long long)(mode == OBS_TREES ? (nt / 32) * 64 : (10 * N > (nt / 32) * 64 ? 10 * N : (nt / 32) * 64)) * 8;
    L.cmp = take((nt / 32) * 32);                               // per warp: "r-th lane of a ballot" table
    const bool bm_fits = (long long)off + (long long)Rmax * 32 + sq_bytes + (b->H > b->W ? Rmax * 2 : 0) + 4096 <= SMEM_MAX;
    const bool bm_global = b->obs_ws && b->ws_stride > 0 && (knob(KNOB_BMGLOBAL) >= 0 ? knob(KNOB_BMGLOBAL) != 0 : !bm_fits);
    L.bm = bm_global ? -1 : take((long long)Rmax * 32);
    L.seg_cap = mode == OBS_TREES ? 0 : 10 * N;                 // path segments of phase 3 share the room of the phase-4 queues
    if (L.seg_cap < (nt / 32) * 64) L.seg_cap = (nt / 32) * 64;
    L.sq_words = L.seg_cap * 2;
    L.flat_walk = knob(KNOB_FLATWALK) >= 0 ? knob(KNOB_FLATWALK) : 3;
    L.tree_cache = b->tree_cache && knob(KNOB_TREECACHE) != 0;
    L.path_cache = b->path_cache && b->pc_stride >= 2 && knob(KNOB_PATHCACHE) != 0;   // "pathcache" 0: every predicted path walked every step  // "treecache" 0: recompute every tree's structure every step
    int seg_cap_use = L.seg_cap;                                // "segcap" / "entcap" overrides (tests): smaller capacities in
    if (knob(KNOB_SEGCAP) >= 0 && knob(KNOB_SEGCAP) < seg_cap_use) seg_cap_use = knob(KNOB_SEGCAP);                            // the same room,
    L.sq = take((long long)L.seg_cap * 8);                      // per-warp queues of the full conflict checks / segment pool
    L.kcls = b->H > b->W ? take((long long)Rmax * 2) : -1;      // key classes of the reference's c*W + r (walks.cuh)
    const long long ent_typ = (long long)N * 56 * 4;
    const long long grid_b = b->grid_stride * 2, ridx_b = b->ridx_stride * 2;
    const long long st_b = b->state_stride * 4, wl_b = b->wlist_stride * 4, wh_b = b->whits_stride * 4;
    const long long sd_b = b->n_slots * b->state_stride * 2;
    const long long core = off + ridx_b + ent_typ + 3 * 16;
    int want_tables = 0x77;                                     // bit k: wlist, wrec, sdist, (srec: unused by k_observe), whoff, whits
    if (knob(KNOB_TABLES) >= 0) want_tables = knob(KNOB_TABLES);
    if (mode == OBS_TREES) want_tables &= ~0x40;                // the tree kernel never reads the grid
    const int max_ctas = nt >= 1024 ? 1 : nt == 512 ? 2 : nt == 256 ? 4 : nt == 192 || nt == 160 ? 7 : nt == 128 ? 8 : 12;
    int ctas = 0;
    if (knob(KNOB_CTAS) >= 0) ctas = knob(KNOB_CTAS) > 0 ? knob(KNOB_CTAS) : 1;
    if (!ctas)
        for (int c = max_ctas; c >= 1; c--)
            if (core <= SMEM_MAX / c - 1024 || c == 1) { ctas = c; break; }
    if (group > 1) ctas = group;
    if (ctas_out) *ctas_out = ctas;
    const int budget = group > 1 ? (((SMEM_MAX - 1024) / group) & ~127) : SMEM_MAX / ctas - 1024;
    auto opt = [&](long long bytes) { if ((long long)off + bytes + 16 > budget) return -1; return take(bytes); };
    L.ridx = opt(ridx_b);
    long long reserve = ent_typ + 16;                            // keep room for the entries while placing the tables
    auto table = [&](int bit, long long bytes) {
        if (!((want_tables >> bit) & 1) || (long long)off + bytes + 16 + reserve > budget) return -1;
        return take(bytes);
    };
    L.wlist = table(0, wl_b);
    L.wrec = table(1, 4 * st_b);
    L.sdist = table(2, sd_b);
    L.srec = table(3, st_b);
    L.whoff = table(4, st_b);
    L.whits = table(5, wh_b);
    L.grid = table(6, grid_b);                                  // only phase 1 reads the grid
    // entries: at least the typical size, at most twice that (more is never needed; larger counts spill to global memory)
    long long ent_b = ((long long)budget - off - 16) & ~15ll;
    if (ent_b > 2 * ent_typ) ent_b = 2 * ent_typ;
    if (ent_b > (long long)N * NPRED * 4) ent_b = (long long)N * NPRED * 4;
    if (ent_b < 0) ent_b = 0;
    L.ent = take(ent_b);
    L.ent_cap = (int)(ent_b / 4);
    L.sort_small = 16;                                          // buckets up to this size are sorted by one thread (40: +2..4 % time, profiles/r02_l_experiments.txt)
    if (knob(KNOB_SORTSMALL) >= 1) L.sort_small = knob(KNOB_SORTSMALL);
    L.seg_cap = seg_cap_use;                                    // to force the per-agent path walk and the global spill of the entries
    if (knob(KNOB_ENTCAP) >= 0 && knob(KNOB_ENTCAP) < L.ent_cap) L.ent_cap = knob(KNOB_ENTCAP);
    L.total = group > 1 ? align_up(off, 128) : off;
    return L;
}

// Threads per CTA: one CTA per environment, so small batches of large environments get more warps per CTA to keep the
// SM's warp slots filled (about 32 resident warps per SM); only tiny environments (up to 8 agents) get 64-thread CTAs
// (Test_02's 20 agents: 115.7 M agent-steps/s with 128 threads against 92 M with 64).
int obs_threads(const FlBatch *b) {
    {
        const int v = knob(KNOB_NT);
        if (v == 64 || v == 128 || v == 160 || v == 192 || v == 256 || v == 512 || v == 1024) return v;
    }
    if (b->N <= 8) return 64;
    const long long per_sm = (b->E + 147) / 148;                // environments per SM (B200: 148 SMs)
    if (per_sm >= 5) return 128;
    if (per_sm >= 3) return 256;
    if (per_sm >= 2) return 512;
    return b->N > 128 ? 1024 : 512;
}

// CTAs per environment of the tree kernel (0 = fused kernel).  Measured on B200 (profiles/r02_launch_shapes.txt): the fused
// kernel wins when one-CTA-per-environment fills the chip's CTA slots in whole waves and an environment has enough agents
// to keep its CTA's warps busy (Test_03: 1024 environments on 148 x 7 slots); otherwise the split launch does — few large
// environments spread their trees over more SMs (Test_14), a ragged last wave is cut into smaller units (Test_08), and
// small environments no longer hold 128-thread CTAs through their serial phases (Test_02).
int obs_parts(const FlBatch *b) {
    if (!b->obs_ws || b->ws_stride <= 0) return 0;
    const int v = knob(KNOB_PARTS);
    if (v >= 0) return v > 32 ? 32 : v;
    if (b->N < 16) return 0;
    const int by_agents = (int)(b->N / 16);
    if (b->E < 148) {                                            // one wave of tree CTAs over the SMs
        int p = (int)(148 / b->E);
        if (p > by_agents) p = by_agents;
        if (p > 32) p = 32;
        return p <= 1 ? 0 : p;
    }
    int ctas = 1;
    make_obs_layout(b, obs_threads(b), OBS_FUSED, 0, &ctas);
    const double waves = (double)b->E / (148.0 * ctas), frac = waves - (double)(long long)waves;
    const bool whole_waves = waves >= 0.95 && (frac <= 0.03 || frac >= 0.95);
    if (whole_waves && b->N >= 32) return 0;
    // Test_02 (8192 x 20 agents): split 140 M agent-steps/s against 102-117 M fused (profiles/r02_g_sweep.txt, r02_h_sweep.txt)
    return b->N >= 20 ? 2 : 0;
}

// Environments per CTA of the fused kernel (group mode, observe.cuh; 1 = one CTA per environment).  As many as the
// one-CTA-per-environment plan would put on an SM, so that the launch shape on the chip is the same and only the tree
// phase is shared; needs the fused plan (no split launch) and at least one full group per SM.
int obs_group(const FlBatch *b, int nt) {
    const int v = knob(KNOB_GROUP);
    if (v == 0 || v == 1) return 1;
    int ctas = 1;
    make_obs_layout(b, nt, OBS_FUSED, 0, &ctas);
    int g = v > 1 ? v : ctas;
    if (g > 7) g = 7;
    while (g > 1 && g * nt > 1024) g--;
    // the instantiated shapes: 128 threads x 4..7, 256 x 2..3, 64 x 7 environments
    if (nt == 128) { if (g < 4) return 1; }
    else if (nt == 256) { if (g < 2) return 1; if (g > 3) g = 3; }
    else if (nt == 64) { if (g < 7) return 1; }
    else return 1;
    {   // the mandatory regions + typical entries must fit the group's per-environment budget
        const ObsLayout L = make_obs_layout(b, nt, OBS_FUSED, 0, nullptr, g);
        if (L.total * g > SMEM_MAX - 1024 || L.ent_cap < (int)b->N * 8) return 1;
    }
    if (v > 1) return g;
    return 1;                                                   // default: off until measured (profiles/)
}

// threads per CTA of the tree kernel: one warp per agent at a time; enough warps to cover its share of the agents
int tree_threads(const FlBatch *b, int parts) {
    for (int v : {knob(KNOB_TREENT), knob(KNOB_NT)})
        if (v == 64 || v == 128 || v == 256 || v == 512 || v == 1024) return v;
    const long long per = (b->N + parts - 1) / parts;           // agents per CTA
    if (per >= 192) return 1024;
    if (per >= 96) return 512;
    if (per >= 32) return 256;
    return 128;
}

// Threads per environment of the launch that obs_parts chose.  The fused kernel at the headline shape (128 threads, seven
// environments per SM, all environments resident in one wave) runs with FIVE warps per environment: 35 instead of 28 warps
// per SM hide more of the latency the kernel is bound by (ncu: issue slots 62.7 % instead of 59.4 % busy, -4 % time,
// profiles/r02_m_sweep.txt); the register budget is then 56 per thread.  160 / 192 threads exist for the fused kernel only.
int obs_threads_for(const FlBatch *b, int parts) {
    int nt = obs_threads(b);
    if (parts) return nt == 160 || nt == 192 ? 128 : nt;
    if (knob(KNOB_NT) >= 0 || nt != 128 || b->N < 32) return nt;
    int ctas = 1, ctas160 = 1;
    make_obs_layout(b, 128, OBS_FUSED, 0, &ctas);
    make_obs_layout(b, 160, OBS_FUSED, 0, &ctas160);
    return ctas == 7 && ctas160 == 7 && knob(KNOB_CTAS) < 0 ? 160 : nt;
}

int finish(cudaError_t launch_err) { return launch_err == cudaSuccess ? FL_OK : (int)launch_err; }

}  // namespace

extern "C" {

int fl_abi_version(void) { return FL_ABI_VERSION; }
size_t fl_batch_sizeof(void) { return sizeof(FlBatch); }
uint64_t fl_launch_count(void) { return g_launches.load(); }

int fl_observe_override(const char *key, int value) {
    if (!key) return FL_ERR_BAD_ARG;
    for (int k = 0; k < KNOB_COUNT; k++)
        if (!strcmp(key, kKnobNames[k])) { g_knob[k].store(value < 0 ? -1 : value); return FL_OK; }
    return FL_ERR_BAD_ARG;
}

int fl_profile_num_kernels(void) { return K_COUNT; }
const char *fl_profile_kernel_name(int k) { return k >= 0 && k < K_COUNT ? kKernelNames[k] : ""; }

void fl_profile_enable(int on) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    g_prof_on = on != 0;
}

int fl_profile_collect(double *ms_out, uint64_t *launches_out, int reset) {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (const ProfRec &r : g_prof_pending) {
        cudaError_t err = cudaEventSynchronize(r.b);
        if (err != cudaSuccess) return (int)err;
        float ms = 0.0f;
        err = cudaEventElapsedTime(&ms, r.a, r.b);
        if (err != cudaSuccess) return (int)err;
        g_prof_ms[r.id] += ms; g_prof_n[r.id] += 1;
        g_prof_free.push_back(r.a); g_prof_free.push_back(r.b);
    }
    g_prof_pending.clear();
    for (int k = 0; k < K_COUNT; k++) {
        if (ms_out) ms_out[k] = g_prof_ms[k];
        if (launches_out) launches_out[k] = g_prof_n[k];
        if (reset) { g_prof_ms[k] = 0.0; g_prof_n[k] = 0; }
    }
    return FL_OK;
}

const char *fl_error_string(int code) {
    switch (code) {
    case FL_OK: return "ok";
    case FL_ERR_BAD_ARG: return "flatland_b200: bad argument (null batch, non-positive dimension, ent_cap too small)";
    case FL_ERR_TOO_MANY_AGENTS: return "flatland_b200: more than FL_MAX_AGENTS-1 agents per environment";
    case FL_ERR_SMEM: return "flatland_b200: configuration needs more shared memory than one SM has";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "flatland_b200: unknown error";
    }
}

int fl_distance_map_ids(const FlBatch *b, const int32_t *d_env_ids, int64_t n_ids, void *stream) {
    if (int rc = check_batch(b)) return rc;
    if (d_env_ids && (n_ids <= 0 || n_ids > b->E)) return FL_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const int HW = (int)(b->H * b->W);
    const size_t smem = (size_t)HW * 4 * sizeof(uint16_t);
    const int nt = HW >= 4096 ? 1024 : 256;
    const unsigned grid = (unsigned)((d_env_ids ? n_ids : b->E) * b->n_slots);
    if (smem <= 227 * 1024) {
        if (smem > 48 * 1024) {
            cudaError_t err = cudaFuncSetAttribute(k_bfs<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (err != cudaSuccess) return (int)err;
        }
        LaunchScope ls(K_BFS, st);
        k_bfs<true><<<grid, nt, smem, st>>>(*b, d_env_ids);
    } else {
        LaunchScope ls(K_BFS, st);
        k_bfs<false><<<grid, nt, 0, st>>>(*b, d_env_ids);
    }
    return finish(cudaGetLastError());
}

int fl_distance_map(const FlBatch *b, void *stream) { return fl_distance_map_ids(b, nullptr, 0, stream); }

int fl_walk_tables_ids(const FlBatch *b, int fill, const int32_t *d_env_ids, int64_t n_ids, void *stream) {
    if (int rc = check_batch(b)) return rc;
    if (!b->ridx || !b->walk_total) return FL_ERR_BAD_ARG;
    if (d_env_ids && (n_ids <= 0 || n_ids > b->E)) return FL_ERR_BAD_ARG;
    if (fill && (!b->srec || !b->wrec || !b->whoff || !b->wlist || !b->whits || !b->kcls || !b->sdist || !b->gtab || !b->dist || b->state_stride <= 0 || b->wlist_stride <= 0 ||
                 b->whits_stride <= 0))
        return FL_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem = (size_t)((b->H * b->W + 31) / 32) * 4;   // one bit per cell: a slot's target stands here
    if (smem > 200 * 1024) return FL_ERR_SMEM;
    if (smem > 40 * 1024) {
        cudaError_t err = cudaFuncSetAttribute(k_walks<true, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err == cudaSuccess) err = cudaFuncSetAttribute(k_walks<false, 256>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err != cudaSuccess) return (int)err;
    }
    const unsigned grid = (unsigned)(d_env_ids ? n_ids : b->E);
    LaunchScope ls(K_WALKS, st);
    if (fill) k_walks<true, 256><<<grid, 256, smem, st>>>(*b, d_env_ids);
    else k_walks<false, 256><<<grid, 256, smem, st>>>(*b, d_env_ids);
    return finish(cudaGetLastError());
}

int fl_walk_tables(const FlBatch *b, int fill, void *stream) { return fl_walk_tables_ids(b, fill, nullptr, 0, stream); }

int fl_reset_ex(const FlBatch *b, const uint8_t *d_env_mask, uint32_t flags, void *stream) {
    if (int rc = check_batch(b)) return rc;
    {
        LaunchScope ls(K_RESET, (cudaStream_t)stream);
        k_reset<<<(unsigned)b->E, 128, 0, (cudaStream_t)stream>>>(*b, d_env_mask, flags);
    }
    return finish(cudaGetLastError());
}

int fl_reset(const FlBatch *b, const uint8_t *d_env_mask, void *stream) { return fl_reset_ex(b, d_env_mask, 0u, stream); }

int fl_step(const FlBatch *b, const uint8_t *d_actions, int32_t *d_rewards, uint8_t *d_dones, uint32_t flags,
            void *stream) {
    if (int rc = check_batch(b)) return rc;
    if (!d_actions || !d_rewards || !d_dones) return FL_ERR_BAD_ARG;
    const int nt = round_up((int)b->N, 32);
    // MotionCheck through per-rail-cell tables from 32 agents on ("stepmap" knob: 0 never, 1 always); they need the rail index
    // of fl_walk_tables and three words per rail cell of shared memory.  k_step at 425 agents: 44 -> 17 us; at 50 agents
    // 17.2 -> 16.6 us (profiles/r02_aa_stepmap.txt)
    int map_cells = 0;
    const int want_map = knob(KNOB_STEPMAP);
    if (want_map != 0 && (want_map > 0 || b->N >= 32) && b->ridx && b->walk_total && b->state_stride > 0) map_cells = (int)(b->state_stride / 4);
    size_t smem = (4 * (size_t)b->N + 3 * (size_t)map_cells) * sizeof(int);
    if (smem > (size_t)SMEM_MAX) { map_cells = 0; smem = 4 * (size_t)b->N * sizeof(int); }
    if (smem > 48 * 1024) {
        cudaError_t err = cudaFuncSetAttribute(k_step, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (err != cudaSuccess) return (int)err;
    }
    {
        LaunchScope ls(K_STEP, (cudaStream_t)stream);
        k_step<<<(unsigned)b->E, nt, smem, (cudaStream_t)stream>>>(*b, d_actions, d_rewards, d_dones, flags, map_cells);
    }
    return finish(cudaGetLastError());
}

int fl_observe(const FlBatch *b, float *d_agent_attr, float *d_forest, int32_t *d_adjacency, int32_t *d_node_order,
               int32_t *d_edge_order, uint8_t *d_valid_actions, float *d_dist_target, void *stream) {
    if (int rc = check_batch(b)) return rc;
    if (!d_agent_attr || !d_forest || !d_adjacency || !d_node_order || !d_edge_order || !d_valid_actions || !d_dist_target)
        return FL_ERR_BAD_ARG;
    if (!b->srec || !b->wrec || !b->whoff || !b->wlist || !b->whits || !b->kcls || !b->sdist || !b->gtab || !b->ridx || !b->walk_total) return FL_ERR_BAD_ARG;   // fl_walk_tables first
    cudaStream_t st = (cudaStream_t)stream;
    using Kern = void (*)(FlBatch, ObsLayout, float *, float *, int32_t *, int32_t *, int32_t *, uint8_t *, float *);
    auto pick = [](int nt, int ctas, int mode) -> Kern {
        // the register budget follows the number of CTAs the shared-memory plan lets share an SM
#define FL_K(NT_, RES_) (mode == OBS_FUSED ? (Kern)k_observe<NT_, RES_, OBS_FUSED> : mode == OBS_INDEX ? (Kern)k_observe<NT_, RES_, OBS_INDEX> : (Kern)k_observe<NT_, RES_, OBS_TREES>)
        if (nt == 64) return ctas > 8 ? FL_K(64, 12) : FL_K(64, 8);
        // five / six warps per environment, seven environments per SM: fused kernel only (the "nt" knob; tuning)
        if (nt == 160) return mode == OBS_FUSED ? (Kern)k_observe<160, 7, OBS_FUSED> : nullptr;
        if (nt == 192) return mode == OBS_FUSED ? (Kern)k_observe<192, 7, OBS_FUSED> : nullptr;
        if (nt == 128) return ctas > 7 ? FL_K(128, 8) : ctas > 6 ? FL_K(128, 7) : ctas > 4 ? FL_K(128, 6) : FL_K(128, 4);
        if (nt == 256) return ctas > 3 ? FL_K(256, 4) : ctas > 2 ? FL_K(256, 3) : FL_K(256, 2);
        if (nt == 512) return ctas > 1 ? FL_K(512, 2) : FL_K(512, 1);
        return FL_K(1024, 1);
#undef FL_K
    };
    auto pick_group = [](int nt, int g) -> Kern {
        if (nt == 128) return g == 7 ? (Kern)k_observe<128, 1, OBS_FUSED, 7> : g == 6 ? (Kern)k_observe<128, 1, OBS_FUSED, 6>
                            : g == 5 ? (Kern)k_observe<128, 1, OBS_FUSED, 5> : (Kern)k_observe<128, 1, OBS_FUSED, 4>;
        if (nt == 256) return g == 3 ? (Kern)k_observe<256, 1, OBS_FUSED, 3> : (Kern)k_observe<256, 1, OBS_FUSED, 2>;
        return (Kern)k_observe<64, 1, OBS_FUSED, 7>;
    };
    auto launch = [&](int mode, int nt, int parts, int kid, int group = 1) -> int {
        int ctas = 1;
        const ObsLayout lay = make_obs_layout(b, nt, mode, parts, &ctas, group);
        const int smem = lay.total * group;
        if (smem > SMEM_MAX) return FL_ERR_SMEM;
        Kern kern = group > 1 ? pick_group(nt, group) : pick(nt, ctas, mode);
        if (!kern) return FL_ERR_BAD_ARG;
        if (smem > 48 * 1024) {
            cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            if (err != cudaSuccess) return (int)err;
        }
        LaunchScope ls(kid, st);
        const unsigned grid = group > 1 ? (unsigned)((b->E + group - 1) / group) : (unsigned)(b->E * (mode == OBS_TREES ? parts : 1));
        kern<<<grid, nt * group, smem, st>>>(*b, lay, d_agent_attr, d_forest, d_adjacency, d_node_order, d_edge_order, d_valid_actions,
                                             d_dist_target);
        return finish(cudaGetLastError());
    };
    const int parts = obs_parts(b);
    if (parts == 0) {
        const int nt = obs_threads_for(b, 0);
        return launch(OBS_FUSED, nt, 0, K_OBSERVE, obs_group(b, nt));
    }
    if (b->ws_stride < fl_observe_ws_words(b)) return FL_ERR_BAD_ARG;
    if (int rc = launch(OBS_INDEX, obs_threads_for(b, parts), parts, K_OBSERVE_INDEX)) return rc;
    return launch(OBS_TREES, tree_threads(b, parts), parts, K_OBSERVE_TREES);
}

int64_t fl_observe_ws_words(const FlBatch *b) {
    if (!b || b->N <= 0 || b->state_stride <= 0) return 0;
    const int64_t Np = (b->N + 3) & ~(int64_t)3, Rmax = b->state_stride / 4;
    return 4 + 6 * Np + Rmax + (Rmax + 4) + 8 * Rmax;
}

int fl_batch_slice(const FlBatch *b, int64_t e0, int64_t n, FlBatch *out) {
    if (!b || !out || e0 < 0 || n <= 0 || e0 + n > b->E) return FL_ERR_BAD_ARG;
    *out = *b;
    out->E = n;
#define FL_ADV(field, per_env, part) out->field = b->field ? b->field + (size_t)e0 * (size_t)(per_env) : b->field;
    FL_BATCH_FIELDS(FL_ADV, b)
#undef FL_ADV
    return FL_OK;
}

int fl_copy_envs(const FlBatch *src, const FlBatch *dst, const int32_t *d_src_ids, const int32_t *d_dst_ids, int64_t n,
                 uint32_t parts, const FlObsBuffers *d_src_out, const FlObsBuffers *d_dst_out, void *stream) {
    if (!src || !dst || !d_src_ids || !d_dst_ids || (parts & ~(FL_COPY_WORLD | FL_COPY_STATE))) return FL_ERR_BAD_ARG;
    const bool outs = d_src_out && d_dst_out;
    if (!parts && !outs) return FL_ERR_BAD_ARG;
    if ((d_src_out != nullptr) != (d_dst_out != nullptr)) return FL_ERR_BAD_ARG;
    if (src->E <= 0 || dst->E <= 0 || src->N <= 0 || src->N != dst->N || n <= 0 || n > dst->E) return FL_ERR_BAD_ARG;
    if (parts & FL_COPY_WORLD) {
        // the world part depends on every shape and table stride; the tables must be built (state_stride > 0)
        if (src->H != dst->H || src->W != dst->W || src->n_slots != dst->n_slots || src->S != dst->S ||
            src->grid_stride != dst->grid_stride || src->dist_stride != dst->dist_stride || src->ridx_stride != dst->ridx_stride ||
            src->state_stride != dst->state_stride || src->wlist_stride != dst->wlist_stride ||
            src->whits_stride != dst->whits_stride || src->pc_stride != dst->pc_stride || src->state_stride <= 0)
            return FL_ERR_BAD_ARG;
        // a cache present in the destination only would keep entries of the world it held before
        if (!src->tree_cache != !dst->tree_cache || !src->path_cache != !dst->path_cache) return FL_ERR_BAD_ARG;
    }
    CopyPlan plan;
    plan.n_ranges = 0;
    int64_t voff = 0;
    bool missing = false;
    auto add = [&](const void *s, void *d, int64_t bytes) {
        if (!s || !d) { missing = true; return; }
        plan.r[plan.n_ranges++] = {static_cast<const char *>(s), static_cast<char *>(d), bytes, voff};
        voff += (bytes + 15) / 16 * 16;
    };
#define FL_RANGE(field, per_env, part)                                                                                   \
    if ((part) & parts) {                                                                                                  \
        if (((part) & FL_PART_OPTIONAL) && !src->field) {}                                                                 \
        else add(src->field, (void *)dst->field, (int64_t)(per_env) * (int64_t)sizeof(*src->field));                   \
    }
    FL_BATCH_FIELDS(FL_RANGE, src)
#undef FL_RANGE
    if (outs) {
#define FL_RANGE(field, per_env) add(d_src_out->field, d_dst_out->field, (int64_t)(per_env) * (int64_t)sizeof(*d_src_out->field));
        FL_OBS_FIELDS(FL_RANGE, src->N)
#undef FL_RANGE
    }
    if (missing) return FL_ERR_BAD_ARG;
    plan.chunks = (voff + COPY_CHUNK - 1) / COPY_CHUNK;
    plan.src_E = src->E;
    plan.dst_E = dst->E;
    if (n * plan.chunks > 0x7fffffffll) return FL_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    {
        LaunchScope ls(K_COPY, st);
        k_copy_envs<<<(unsigned)(n * plan.chunks), COPY_THREADS, 0, st>>>(plan, d_src_ids, d_dst_ids);
    }
    return finish(cudaGetLastError());
}

namespace {
// events that order the copy stream behind the compute stream, one per chunk and device, created on first use
cudaEvent_t chunk_event(int k) {
    static std::mutex mu;
    static std::vector<std::vector<cudaEvent_t>> pool;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(mu);
    if ((int)pool.size() <= dev) pool.resize(dev + 1);
    while ((int)pool[dev].size() <= k) {
        cudaEvent_t e;
        cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
        pool[dev].push_back(e);
    }
    return pool[dev][k];
}
// extra compute streams of the host-buffer step (one set per device): the kernels of successive environment ranges run on
// alternating streams, so that a range's latency-bound kernels overlap the next range's instead of queueing behind them
cudaStream_t lane_stream(int k) {
    static std::mutex mu;
    static std::vector<std::vector<cudaStream_t>> pool;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(mu);
    if ((int)pool.size() <= dev) pool.resize(dev + 1);
    while ((int)pool[dev].size() <= k) {
        cudaStream_t s;
        cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking);
        pool[dev].push_back(s);
    }
    return pool[dev][k];
}
}  // namespace

namespace {
ExpandPool g_pool;
}  // namespace

int fl_host_threads(int n) {
    if (n > 0) g_pool.set_threads(n);
    return g_pool.threads();
}

size_t fl_wire_bytes(const FlBatch *b, int n_chunks) {
    if (!b || b->E <= 0 || b->N <= 0) return 0;
    (void)n_chunks;
    return ((size_t)b->E * (size_t)b->N * WIRE_MAX_WORDS + (size_t)b->E + 64 * 16 + 64) * 4;   // worst case: every node of every tree is real
}

int fl_step_observe_host_compact(const FlBatch *b, const uint8_t *h_actions, uint8_t *d_actions, const FlObsBuffers *d_out,
                                 const FlObsBuffers *h_out, void *h_wire, uint32_t *d_cursor, uint64_t *wire_bytes_out,
                                 uint32_t flags, int n_chunks, void *stream, void *copy_stream) {
    if (int rc = check_batch(b)) return rc;
    if (!h_actions || !d_actions || !d_out || !h_out || !h_wire || !d_cursor) return FL_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream, cs = copy_stream ? (cudaStream_t)copy_stream : st;
    if (n_chunks < 1) n_chunks = 1;
    if (n_chunks > 64) n_chunks = 64;
    if (n_chunks > b->E) n_chunks = (int)b->E;
    uint32_t *wire_dev = nullptr;
    cudaError_t err = cudaHostGetDevicePointer((void **)&wire_dev, h_wire, 0);      // pinned + mapped host memory (UVA)
    if (err != cudaSuccess) return (int)err;
    const size_t N = (size_t)b->N;
    const int smem = (int)((2 * ((N + 3) & ~(size_t)3) + 4 + (PACK_THREADS / 32) * WIRE_MAX_WORDS) * 4);
    // expansion: 3 = AVX2 + non-temporal stores for every tensor, 2 = AVX2 + non-temporal forest stores (default), 1 = AVX2,
    // 0 = portable; FL_WIRE_TIMING=1 prints where a call's time goes
    static const int expand_mode = getenv("FL_WIRE_EXPAND") ? atoi(getenv("FL_WIRE_EXPAND")) : 2;
    static const bool timing = getenv("FL_WIRE_TIMING") != nullptr;
    const auto t_start = std::chrono::steady_clock::now();
    double t_wait = 0.0, t_expand = 0.0;
    if ((err = cudaMemcpyAsync(d_actions, h_actions, (size_t)b->E * N, cudaMemcpyHostToDevice, st)) != cudaSuccess) return (int)err;
    if ((err = cudaMemsetAsync(d_cursor, 0, sizeof(uint32_t) * (size_t)n_chunks, st)) != cudaSuccess) return (int)err;
    // compute lanes: range c runs on lane c % n_lanes (lane 0 = the caller's stream).  A range of 128 environments is one
    // latency-bound wave of CTAs (0.2 ms whatever its size); two lanes keep the device ahead of the host's expansion
    static const int lanes_env = getenv("FL_WIRE_LANES") ? atoi(getenv("FL_WIRE_LANES")) : 2;
    const int n_lanes = copy_stream && n_chunks >= 2 ? (lanes_env < 1 ? 1 : lanes_env > 4 ? 4 : lanes_env) : 1;
    if (n_lanes > 1) {
        cudaEvent_t ev0 = chunk_event(160);
        if ((err = cudaEventRecord(ev0, st)) != cudaSuccess) return (int)err;
        for (int l = 1; l < n_lanes; l++)
            if ((err = cudaStreamWaitEvent(lane_stream(l - 1), ev0, 0)) != cudaSuccess) return (int)err;
    }
    std::vector<size_t> chunk_word0((size_t)n_chunks);
    for (int c = 0; c < n_chunks; c++) {
        const int64_t e0 = b->E * c / n_chunks, e1 = b->E * (c + 1) / n_chunks, n = e1 - e0;
        const size_t a0 = (size_t)e0 * N;
        chunk_word0[c] = ((a0 * WIRE_MAX_WORDS + (size_t)e0 + 7) & ~(size_t)7) + 16 * (size_t)c;   // worst-case prefix, 32-byte aligned: regions never overlap
        FlBatch sub;
        if (int rc = fl_batch_slice(b, e0, n, &sub)) return rc;
        cudaStream_t ls = c % n_lanes == 0 ? st : lane_stream(c % n_lanes - 1);
        if (int rc = fl_step(&sub, d_actions + a0, d_out->rewards + a0, d_out->dones + (size_t)e0 * (N + 1), flags, (void *)ls)) return rc;
        if (int rc = fl_observe(&sub, d_out->agent_attr + a0 * FL_ATTR_F, d_out->forest + a0 * FL_MAX_NODES * FL_NODE_F,
                                d_out->adjacency + a0 * (FL_MAX_NODES - 1) * 3, d_out->node_order + a0 * FL_MAX_NODES,
                                d_out->edge_order + a0 * (FL_MAX_NODES - 1), d_out->valid_actions + a0 * 5,
                                d_out->dist_target + a0, (void *)ls))
            return rc;
        if (cs != ls) {
            cudaEvent_t ev = chunk_event(c);
            if ((err = cudaEventRecord(ev, ls)) != cudaSuccess) return (int)err;
            if ((err = cudaStreamWaitEvent(cs, ev, 0)) != cudaSuccess) return (int)err;
        }
        WireSrc src{d_out->agent_attr + a0 * FL_ATTR_F, d_out->forest + a0 * FL_MAX_NODES * FL_NODE_F, d_out->dist_target + a0,
                    d_out->adjacency + a0 * (FL_MAX_NODES - 1) * 3, d_out->node_order + a0 * FL_MAX_NODES,
                    d_out->edge_order + a0 * (FL_MAX_NODES - 1), d_out->rewards + a0, d_out->dones + (size_t)e0 * (N + 1)};
        {
            LaunchScope ls(K_PACK, cs);
            k_pack<<<(unsigned)n, PACK_THREADS, smem, cs>>>(src, (int)N, (int)n, wire_dev + chunk_word0[c], d_cursor + c);
        }
        if ((err = cudaGetLastError()) != cudaSuccess) return (int)err;
        if ((err = cudaEventRecord(chunk_event(64 + c), cs)) != cudaSuccess) return (int)err;
    }
    // expansion on the host while the device works on the later chunks
    const WireDst dst{h_out->agent_attr, h_out->forest, h_out->dist_target, h_out->adjacency, h_out->node_order, h_out->edge_order,
                      h_out->rewards, h_out->valid_actions, h_out->dones};
    std::atomic<uint64_t> words{0};
    const auto t_launched = std::chrono::steady_clock::now();
    for (int c = 0; c < n_chunks; c++) {
        const auto t0 = std::chrono::steady_clock::now();
        if ((err = cudaEventSynchronize(chunk_event(64 + c))) != cudaSuccess) return (int)err;
        const auto t1 = std::chrono::steady_clock::now();
        const int64_t e0 = b->E * c / n_chunks, e1 = b->E * (c + 1) / n_chunks;
        const uint32_t *wire = reinterpret_cast<const uint32_t *>(h_wire) + chunk_word0[c];
        const int Ni = (int)N;
        const std::function<void(int)> job = [&](int el) { words.fetch_add(expand_env(wire, el, e0 + el, Ni, dst, expand_mode) + 1); };
        g_pool.parallel_for((int)(e1 - e0), job);
        t_wait += std::chrono::duration<double>(t1 - t0).count();
        t_expand += std::chrono::duration<double>(std::chrono::steady_clock::now() - t1).count();
    }
    if (timing)
        fprintf(stderr, "fl_step_observe_host_compact: launch %.3f ms, waiting for the device %.3f ms, expanding %.3f ms (%d chunks, %d threads, %.1f MB wire)\n",
                1e3 * std::chrono::duration<double>(t_launched - t_start).count(), 1e3 * t_wait, 1e3 * t_expand, n_chunks, g_pool.threads(),
                words.load() * 4 / 1e6);
    if (wire_bytes_out) *wire_bytes_out = words.load() * 4;
    if (cs != st) {
        if ((err = cudaStreamWaitEvent(st, chunk_event(64 + n_chunks - 1), 0)) != cudaSuccess) return (int)err;
    }
    return FL_OK;
}

int fl_observe_plan(const FlBatch *b, int32_t *out, int n_out) {
    if (int rc = check_batch(b)) return rc;
    if (!out || n_out < 20) return FL_ERR_BAD_ARG;
    const int parts = obs_parts(b), nt = obs_threads_for(b, parts);
    const int group = parts ? 1 : obs_group(b, nt);
    int ctas = 1;
    const ObsLayout L = make_obs_layout(b, nt, parts ? OBS_INDEX : OBS_FUSED, parts, &ctas, group);
    const int v[20] = {nt, L.total, ctas, L.ent_cap, L.kcls, L.grid, L.ci, L.ks, L.ent, L.sdist,
                       L.ridx, L.srec, L.wrec, L.whoff, L.wlist, L.ag, L.dl, L.part, SMEM_MAX / (L.total + 1024), L.whits};
    for (int k = 0; k < 20; k++) out[k] = v[k];
    if (n_out >= 24) {                                          // the split launch: parts, and the tree kernel's threads / bytes / CTAs per SM
        int tctas = 0;
        const int tnt = parts ? tree_threads(b, parts) : 0;
        const ObsLayout T = parts ? make_obs_layout(b, tnt, OBS_TREES, parts, &tctas) : L;
        out[20] = parts; out[21] = tnt; out[22] = parts ? T.total : 0; out[23] = tctas;
    }
    if (n_out >= 25) out[24] = group;                           // environments per CTA of the fused kernel
    return FL_OK;
}

int fl_step_observe_host(const FlBatch *b, const uint8_t *h_actions, uint8_t *d_actions, const FlObsBuffers *d_out,
                         const FlObsBuffers *h_out, uint32_t flags, int n_chunks, void *stream, void *copy_stream) {
    if (int rc = check_batch(b)) return rc;
    if (!h_actions || !d_actions || !d_out || !h_out) return FL_ERR_BAD_ARG;
    cudaStream_t st = (cudaStream_t)stream, cs = copy_stream ? (cudaStream_t)copy_stream : st;
    if (n_chunks < 1 || !copy_stream) n_chunks = 1;
    if (n_chunks > b->E) n_chunks = (int)b->E;
    const size_t N = (size_t)b->N;
    cudaError_t err = cudaMemcpyAsync(d_actions, h_actions, (size_t)b->E * N, cudaMemcpyHostToDevice, st);
    if (err != cudaSuccess) return (int)err;
    for (int c = 0; c < n_chunks; c++) {
        const int64_t e0 = b->E * c / n_chunks, e1 = b->E * (c + 1) / n_chunks, n = e1 - e0;
        const size_t a0 = (size_t)e0 * N, an = (size_t)n * N;       // first agent / agents of the chunk
        FlBatch sub;
        if (int rc = fl_batch_slice(b, e0, n, &sub)) return rc;
        if (int rc = fl_step(&sub, d_actions + a0, d_out->rewards + a0, d_out->dones + (size_t)e0 * (N + 1), flags, stream)) return rc;
        if (int rc = fl_observe(&sub, d_out->agent_attr + a0 * FL_ATTR_F, d_out->forest + a0 * FL_MAX_NODES * FL_NODE_F,
                                d_out->adjacency + a0 * (FL_MAX_NODES - 1) * 3, d_out->node_order + a0 * FL_MAX_NODES,
                                d_out->edge_order + a0 * (FL_MAX_NODES - 1), d_out->valid_actions + a0 * 5,
                                d_out->dist_target + a0, stream))
            return rc;
        if (cs != st) {                                             // the chunk's copies wait for its kernels only
            cudaEvent_t ev = chunk_event(c);
            if ((err = cudaEventRecord(ev, st)) != cudaSuccess) return (int)err;
            if ((err = cudaStreamWaitEvent(cs, ev, 0)) != cudaSuccess) return (int)err;
        }
#define FL_D2H(field, first, count, elem)                                                                              \
    if (h_out->field) {                                                                                                \
        err = cudaMemcpyAsync(h_out->field + (first), d_out->field + (first), (size_t)(count) * (elem), cudaMemcpyDeviceToHost, cs); \
        if (err != cudaSuccess) return (int)err;                                                                       \
    }
        FL_D2H(rewards, a0, an, 4)
        FL_D2H(dones, (size_t)e0 * (N + 1), (size_t)n * (N + 1), 1)
        FL_D2H(agent_attr, a0 * FL_ATTR_F, an * FL_ATTR_F, 4)
        FL_D2H(forest, a0 * FL_MAX_NODES * FL_NODE_F, an * FL_MAX_NODES * FL_NODE_F, 4)
        FL_D2H(adjacency, a0 * (FL_MAX_NODES - 1) * 3, an * (FL_MAX_NODES - 1) * 3, 4)
        FL_D2H(node_order, a0 * FL_MAX_NODES, an * FL_MAX_NODES, 4)
        FL_D2H(edge_order, a0 * (FL_MAX_NODES - 1), an * (FL_MAX_NODES - 1), 4)
        FL_D2H(valid_actions, a0 * 5, an * 5, 1)
        FL_D2H(dist_target, a0, an, 4)
#undef FL_D2H
    }
    if (cs != st) {                                                 // `stream` completes when the last copy has landed
        cudaEvent_t ev = chunk_event(n_chunks);
        if ((err = cudaEventRecord(ev, cs)) != cudaSuccess) return (int)err;
        if ((err = cudaStreamWaitEvent(st, ev, 0)) != cudaSuccess) return (int)err;
    }
    return FL_OK;
}

}  // extern "C"

