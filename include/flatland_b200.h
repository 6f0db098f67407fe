/* flatland_b200.h — C ABI of the B200-native batched Flatland-3 hot path.
 *
 * Drop-in boundary.  The reference (RoboEden/flatland-marl) exposes this path through two
 * duck-typed Python interfaces, `RailEnv.reset/step` (pure Python) and the pybind11 class
 * `flatland_cutils.TreeObsForRailEnv` (flatland_cutils/src/main.cpp:17-22); neither is a C ABI, so
 * this header defines the C ABI that sits UNDER Python classes keeping those signatures
 * (flatland-marl_b200/rail_env.py, tree_obs.py).  Every entry point cites the reference interface
 * it replaces; citations are relative to the reference repository root.
 *
 * Conventions: plain pointers and sizes only (no torch / pybind types); every pointer inside
 * `FlBatch` and every `d_` argument is a DEVICE pointer owned by the caller; `h_` arguments are
 * HOST pointers (pinned for async copies); `stream` is a `cudaStream_t` passed as `void*`; the
 * library never allocates or frees device memory and keeps no global state except a launch counter
 * and the optional fl_profile_* event log; return value is 0 or
 * an `FlStatus` / CUDA error code (see fl_error_string); no exceptions cross the boundary.
 * Calls on one FlBatch must be serialised by the caller (one stream); different batches are
 * independent.
 */
#ifndef FLATLAND_B200_H
#define FLATLAND_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FL_ABI_VERSION 5

/* fixed by the reference (solution/impl_config.py:4-21, flatland_cutils/src/tool.h:67-93) */
#define FL_MAX_NODES 31     /* num_tree_obs_nodes = 1 + 3*10 */
#define FL_NODE_F 12        /* floats per tree node (treeobs.cpp:562-573) */
#define FL_ATTR_F 83        /* floats per agent attribute vector (feature_parser.cpp:19-94) */
#define FL_PRED_DEPTH 500   /* tree_pred_path_depth */
#define FL_ACTION_ABSENT 255 /* agent key not present in action_dict (rail_env.py:527) */
#define FL_NO_AGENT 0xFFFFu
#define FL_DIST_INF 0xFFFFu /* unreachable in the uint16 distance map (np.inf in distance_map.py:66) */
#define FL_MAX_AGENTS 1024

enum FlStatus {
    FL_OK = 0,
    FL_ERR_BAD_ARG = -1,
    FL_ERR_TOO_MANY_AGENTS = -2,
    FL_ERR_SMEM = -3
};

/* per-environment status bits written by fl_step into FlBatch.status */
#define FL_ST_STEP_AFTER_DONE 1u /* step() on a finished episode: reference raises (rail_env.py:508-509) */
#define FL_ST_AUTO_RESET 2u      /* the env was reset in place by this call (FL_FLAG_AUTO_RESET) */
#define FL_ST_BAD_CELL 4u        /* tree walk met a cell with 0 transitions (treeobs.cpp:527-535 throws) */

/* fl_step flags */
#define FL_FLAG_AUTO_RESET 1u   /* a finished env is reset in place instead of stepped: env.reset(False, False) of the
                                   reference (rail_env.py:260-357 with nothing regenerated) — no schedule rows are consumed by
                                   the call, and, as in the reference, EnvAgent.reset (agent_utils.py:90-105) keeps arrival_time:
                                   a train that arrived in the previous episode carries its old arrival_time, so when it
                                   reaches its target again handle_done_state (rail_env.py:493-499) leaves it standing there */
#define FL_FLAG_FRESH_AGENTS 2u /* with FL_FLAG_AUTO_RESET: arrival_time is cleared too (fresh agent objects, what a reset that
                                   regenerates the schedule gives: EnvAgent.from_line, rail_env.py:315-317) */

/* fl_reset_ex flags */
#define FL_RESET_KEEP_SCHEDULE 1u /* do not rewind the malfunction schedule (the reference's generator carries on) */
#define FL_RESET_KEEP_ARRIVAL 2u  /* keep arrival_time (EnvAgent.reset semantics, see FL_FLAG_AUTO_RESET) */

/* Device-resident state of E lock-step environments of one configuration (same N, H, W).
 * Struct of arrays; E is the slowest index everywhere.  "rc" arrays hold (row, col) int16 pairs.
 * Layout rationale: DESIGN.md §3. */
typedef struct FlBatch {
    int64_t E, N, H, W;
    int64_t n_slots;   /* unique-target slots allocated per env (max over envs) */
    int64_t S;         /* malfunction-schedule rows per env */
    int64_t ent_cap;   /* capacity of `entries` per env, >= N * (FL_PRED_DEPTH + 1) */
    int64_t grid_stride; /* uint16 elements between the grids of consecutive envs, >= H*W, multiple of 8 */
    int64_t dist_stride; /* uint16 elements between the distance maps of consecutive envs,
                            >= n_slots*H*W*4, multiple of 8 (16-byte aligned blocks: moved by TMA bulk copies) */
    int64_t *debug_clocks; /* tuning only: [E][32] SM-clock timestamps of k_observe's phases, NULL = off */
    int64_t ridx_stride;   /* uint16 elements per env of ridx, >= H*W, multiple of 8 */
    int64_t state_stride;  /* elements per env of srec / wrec / whoff / kcls, >= 4 * rail cells, multiple of 32 */
    int64_t wlist_stride;  /* uint32 elements per env of wlist, multiple of 4, with 8 elements of slack at the end */
    int64_t whits_stride;  /* uint32 elements per env of whits, multiple of 4 */
    int64_t seg_stride;    /* uint64 elements per env of segs (0 = none) */
    int64_t pc_stride;     /* uint2 elements per AGENT of path_cache: 1 header + the longest predicted path it can hold (0 = none) */
    int64_t ws_stride;     /* uint32 elements per env of obs_ws: >= fl_observe_ws_words(b), multiple of 4 (0 = none: fused kernel only) */

    /* ---- world, static after upload (RailEnv.reset generators stay reference Python) ---- */
    const uint16_t *grid;      /* [E][grid_stride] transition bitmask per cell (core/transition_map.py:144) */
    const int16_t *slot_rc;    /* [E][n_slots][2] target cell of each unique-target slot, (-1,-1) unused */
    uint16_t *dist;            /* [E][dist_stride] = per env [n_slots][H*W][4] distance map, written by fl_distance_map */
    const int32_t *max_steps;  /* [E] _max_episode_steps */
    const int16_t *init_rc;    /* [E][N][2] */
    const int16_t *tgt_rc;     /* [E][N][2] */
    const uint8_t *init_dir;   /* [E][N] */
    const uint8_t *max_count;  /* [E][N] int(1/speed)-1 (speed_counter.py:40-42) */
    const uint16_t *slot;      /* [E][N] index into the env's distance-map slots */
    const double *speed;       /* [E][N] */
    const int32_t *earliest;   /* [E][N] earliest_departure */
    const int32_t *latest;     /* [E][N] latest_arrival */
    const uint8_t *sched;      /* [E][S][N] pre-drawn malfunction durations (0 = none); row sched_pos % S */
    /* static branch-walk tables written by fl_walk_tables (csrc/walks.cuh): which states the tree observation's
     * walk from a (cell, direction) state visits (treeobs.cpp:258-610 _explore_branch, rail-only part) */
    uint16_t *ridx;            /* [E][ridx_stride] rail index per cell, 0xFFFF = no rail; state id = 4*ridx + dir */
    uint32_t *srec;            /* [E][state_stride] row | col<<10 | dir<<20 | transitions nibble<<22 | unusable switch<<26 */
    uint32_t *wrec;            /* [E][state_stride][4] per walk: offset in wlist; steps | kind<<16 | target hits<<20
                                  (kind 1 switch, 2 dead end, 3 cycle, 0 bad cell); child0 | child1<<16;
                                  child2 | first unusable-switch step<<16 (0xFFFF = null / none).  16-byte aligned. */
    uint32_t *whoff;           /* [E][state_stride] offset of the walk's target hits in whits */
    uint32_t *wlist;           /* [E][wlist_stride] visited states, walk after walk: state id | transitions nibble<<16 */
    uint32_t *whits;           /* [E][whits_stride] step | slot<<16 of every walk state standing on a slot's target */
    uint16_t *kcls;            /* [E][state_stride] per rail cell: lowest rail index among the cells sharing the reference's
                                  prediction key c*W + r (only cells of grids with H > W have partners) */
    uint16_t *sdist;           /* [E][n_slots][state_stride] the distance map indexed by state id (copy of `dist` on the rail
                                  cells only; fl_walk_tables(fill) runs after fl_distance_map) */
    uint32_t *gtab;            /* [E][n_slots][state_stride] where the shortest path to the slot's target continues after the
                                  walk from a state: next state (0xFFFF = the path ends with this walk) | last step of the walk
                                  on the path<<16 (14 bits) | direction of the state at that step<<30 */
    int32_t *walk_total;       /* [E][4] written by fl_walk_tables: states, wlist elements, whits elements, 1 if a walk is
                                  longer than 16383 steps (unsupported) */

    /* ---- agent state (agent_utils.py:58-105 and step_utils/*) ---- */
    int16_t *rc;          /* [E][N][2] position, (-1,-1) = None */
    int16_t *old_rc;      /* [E][N][2] */
    uint8_t *dir;         /* [E][N] */
    uint8_t *old_dir;     /* [E][N] 255 = None */
    uint8_t *state;       /* [E][N] TrainState */
    uint8_t *ctr;         /* [E][N] speed counter */
    uint8_t *mal;         /* [E][N] malfunction_down_counter */
    uint8_t *saved;       /* [E][N] saved action, 0 = None */
    uint8_t *sig_mal;     /* [E][N] st_signals.in_malfunction of the last step */
    uint8_t *deadlocked;  /* [E][N] sticky deadlock flag (deadlock_checker.cpp) */
    uint8_t *done;        /* [E][N] dones[i] */
    uint16_t *nmal;       /* [E][N] num_malfunctions */
    int32_t *arrival;     /* [E][N] arrival_time, -1 = None */

    /* ---- environment state ---- */
    int32_t *elapsed;     /* [E] _elapsed_steps */
    int32_t *sched_pos;   /* [E] schedule rows consumed so far */
    uint8_t *done_all;    /* [E] dones["__all__"] */
    uint32_t *status;     /* [E] FL_ST_* bits, sticky until cleared by the caller */
    int64_t *stats;       /* [E][4] running totals since upload: episodes finished, "arrived" agents at episode end with
                                    the predicate of eval_env.py:81-94 final_metric (position is None and state !=
                                    READY_TO_DEPART: includes trains that never left), sum of end-of-episode rewards,
                                    agent-steps */

    /* ---- per-step observation workspace (rebuilt by every fl_observe) ---- */
    uint32_t *entries;    /* [E][ent_cap] predicted-occupancy entries grouped by rail cell (spill space: used only
                                       when an environment's entries do not fit in shared memory; its free tail is
                                       the scratch of the sort of large buckets) */
    uint64_t *segs;       /* [E][seg_stride] path segments that do not fit in the shared-memory pool (spill space) */
    uint32_t *obs_ws;     /* [E][ws_stride] split launch of fl_observe (k_observe as two kernels, see csrc/observe.cuh): the
                                       prediction index of an environment between the index kernel and the tree kernel.
                                       NULL = fl_observe always runs the fused kernel */
    uint32_t *tree_cache; /* [E][N][FL_TREE_CACHE_WORDS] the structure of every agent's branch tree (which walk each of the 31
                                       nodes stands for, where it ends, parents, evaluation orders) as fl_observe left it,
                                       keyed by the agent's rail state: the structure is a function of the static walk
                                       tables and the agent's (cell, direction) alone, and most agents stand where they stood
                                       a step ago.  Invalidated by fl_walk_tables / fl_reset.  NULL = recomputed every step */
    uint64_t *path_cache; /* [E][N][pc_stride] (key class of the rail cell, index entry) of every element of an agent's predicted
                                       path as fl_observe last computed it, behind a header (key, elements): the predicted
                                       path and its timing relative to "now" are a function of the static tables and the
                                       agent's (cell, direction, speed, done) alone.  Invalidated like tree_cache.  NULL = the
                                       paths are walked every step */
} FlBatch;
#define FL_TREE_CACHE_WORDS 160 /* 5 words per lane of the agent's warp; lane 31 (no node) holds the key */

int fl_abi_version(void);
size_t fl_batch_sizeof(void);
const char *fl_error_string(int code);

/* Replaces DistanceMap._compute/_distance_map_walker (flatland/envs/distance_map.py:57-160): one BFS
 * over (cell, orientation) per unique target slot, writing FlBatch.dist.  Reset-time only. */
int fl_distance_map(const FlBatch *b, void *stream);

/* Builds the static branch-walk tables of every environment (reset time, after the grid upload).  Two
 * passes: fill == 0 only writes walk_total (ridx and walk_total must be allocated) so that the caller can
 * size srec / wrec / whoff / wlist / whits; fill != 0 writes all tables, and needs the distance maps (fl_distance_map
 * earlier on the same stream) for sdist.  No reference counterpart: the reference
 * re-walks the rail cell by cell in every _explore_branch call (treeobs.cpp:258-610). */
int fl_walk_tables(const FlBatch *b, int fill, void *stream);

/* The same two for a list of environments of the batch only (d_env_ids: device int32[n_ids], distinct indices), one launch
 * each: what RailEnv.reset(regenerate_rail=True, ...) costs for SOME environments of a running batch (rail_env.py:260-357;
 * distance_map.py:57-160 is 16.9 s of Python per reset at Test_14).  Used by the reset pipeline (BatchedRailEnv.replace_worlds). */
int fl_distance_map_ids(const FlBatch *b, const int32_t *d_env_ids, int64_t n_ids, void *stream);
int fl_walk_tables_ids(const FlBatch *b, int fill, const int32_t *d_env_ids, int64_t n_ids, void *stream);

/* Replaces the tail of RailEnv.reset (flatland/envs/rail_env.py:335-347: reset_agents, elapsed=0,
 * dones cleared) and TreeObsForRailEnv::reset (flatland_cutils/src/treeobs.cpp:22-28: a fresh
 * DeadlockChecker).  d_env_mask: [E] bytes, non-zero = reset this env; NULL = all. */
int fl_reset(const FlBatch *b, const uint8_t *d_env_mask, void *stream);
/* The same with flags: FL_RESET_KEEP_SCHEDULE | FL_RESET_KEEP_ARRIVAL is env.reset(False, False) on the reference (the
 * agent objects and the malfunction generator live on); 0 is fl_reset (fresh agents, schedule rewound: a new upload). */
int fl_reset_ex(const FlBatch *b, const uint8_t *d_env_mask, uint32_t flags, void *stream);

/* Replaces RailEnv.step(action_dict) up to but excluding the observation
 * (flatland/envs/rail_env.py:501-632, step_utils/*, agent_chains.py MotionCheck).
 * d_actions [E][N] uint8 (FL_ACTION_ABSENT = key missing); d_rewards [E][N] int32;
 * d_dones [E][N+1] uint8, last column = "__all__".  From 32 agents on MotionCheck uses the rail index of fl_walk_tables
 * (FlBatch.ridx, walk_total) when it is built; without it every pair of agents is compared, with the same result. */
int fl_step(const FlBatch *b, const uint8_t *d_actions, int32_t *d_rewards, uint8_t *d_dones,
            uint32_t flags, void *stream);

/* Replaces TreeObsForRailEnv::get_many + get_properties (flatland_cutils/src/treeobs.cpp:30-108,
 * 612-640; loader.cpp:221-327; predictions.cpp; deadlock_checker.cpp; feature_parser.cpp), output in
 * the policy's input layout (solution/plfActor.py:48-74):
 *   d_agent_attr [E][N][83] f32, d_forest [E][N][31][12] f32, d_adjacency [E][N][30][3] i32,
 *   d_node_order [E][N][31] i32, d_edge_order [E][N][30] i32, d_valid_actions [E][N][5] u8,
 *   d_dist_target [E][N] f32 (inf = unreachable).  `deadlocked` is read from FlBatch.deadlocked. */
int fl_observe(const FlBatch *b, float *d_agent_attr, float *d_forest, int32_t *d_adjacency,
               int32_t *d_node_order, int32_t *d_edge_order, uint8_t *d_valid_actions,
               float *d_dist_target, void *stream);

/* uint32 words per environment fl_observe's split launch needs in FlBatch.obs_ws (depends on N and state_stride: call it after
 * fl_walk_tables sized the static tables). */
int64_t fl_observe_ws_words(const FlBatch *b);

/* Tuning and test hook (no reference counterpart): overrides one knob of the shared-memory / launch plan fl_observe derives
 * from the batch shape, process-wide, value < 0 = back to the default.  Keys: "nt" (threads per CTA: 64..1024), "ctas"
 * (CTAs per SM the plan is cut for), "tables" (bit mask of the static tables staged in shared memory), "segcap", "entcap"
 * (capacities of the shared-memory segment pool / entry array, to force the global spill paths), "sortsmall" (largest bucket
 * sorted by one thread), "parts" (CTAs per environment of the tree kernel; 0 = fused kernel), "treent" (threads per CTA of the
 * tree kernel), "bmglobal" (1: the tree kernel reads the time-slot filter from the workspace instead of shared memory),
 * "flatwalk" (bit 0 / 1: path segments walked by warps as flat lists in the counting / scatter pass), "group" (environments
 * per CTA of the fused kernel, 1 = one CTA per environment), "treecache" / "pathcache" (0: FlBatch.tree_cache / path_cache
 * are not used), and one knob of fl_step: "stepmap" (MotionCheck through per-rail-cell tables: 0 never, 1 always; default from
 * 32 agents on).  The same knobs are read ONCE from the environment variables FL_OBS_<KEY> (FL_STEP_MAP for "stepmap") when the
 * library is loaded; fl_observe itself never calls getenv.
 * Returns 0, or FL_ERR_BAD_ARG for an unknown key. */
int fl_observe_override(const char *key, int value);

/* Diagnostics: the shared-memory plan fl_observe uses for this batch.  out[0..19] = threads per CTA, dynamic
 * shared bytes, CTAs per SM planned for, entry capacity, byte offsets of key classes, grid, occupancy,
 * bucket offsets, entries, sdist, ridx, srec, wrec, whoff, wlist (-1 = stays in global memory / unused),
 * agents, deadlock scratch, scan partials, CTAs per SM that fit, whits. */
int fl_observe_plan(const FlBatch *b, int32_t *out, int n_out);

/* A view of environments [e0, e0+n) of a batch: every pointer advanced by e0 environments, E = n.  The view
 * aliases the parent's memory; stepping disjoint views on different streams is allowed. */
int fl_batch_slice(const FlBatch *b, int64_t e0, int64_t n, FlBatch *out);

/* One env.step as the reference's caller sees it (solution/eval_env.py:108-114) with HOST buffers:
 * copies h_actions to d_actions, runs fl_step + fl_observe, copies rewards, dones and every
 * observation tensor back to the h_ buffers (any h_ output may be NULL to leave it on the device).
 * With n_chunks > 1 and a copy_stream the batch is cut into n_chunks environment ranges and the
 * device-to-host copies of one range (on copy_stream) overlap the kernels of the next (on stream).
 * All work is ordered before the end of `stream`; the caller synchronises `stream`. */
typedef struct FlObsBuffers {
    float *agent_attr;
    float *forest;
    int32_t *adjacency;
    int32_t *node_order;
    int32_t *edge_order;
    uint8_t *valid_actions;
    float *dist_target;
    int32_t *rewards;
    uint8_t *dones;
} FlObsBuffers;

int fl_step_observe_host(const FlBatch *b, const uint8_t *h_actions, uint8_t *d_actions,
                         const FlObsBuffers *d_out, const FlObsBuffers *h_out, uint32_t flags,
                         int n_chunks, void *stream, void *copy_stream);

/* fl_copy_envs parts */
#define FL_COPY_WORLD 1u   /* world, schedule, reset-time tables, tree/path caches */
#define FL_COPY_STATE 2u   /* agent and environment state, status and stats included */

/* copy.deepcopy(env) of the reference (rail_env.py RailEnv is a plain Python object) for many environments in one launch:
 * slot d_dst_ids[i] of `dst` becomes slot d_src_ids[i] of `src` (device int32[n] each) for the requested parts; the output
 * rows (observation tensors, rewards, dones) are copied too when d_src_out and d_dst_out are both non-NULL (host structs of
 * device pointers, [E][...] as in fl_step_observe_host).  Given the same actions, a copied slot then produces the same bytes
 * as its source, across episode ends too (the schedule rows and sched_pos travel with it).  The per-call scratch of
 * fl_observe (entries, segs, obs_ws, debug_clocks) is never copied.  `src` may equal `dst`; one source may feed several
 * destinations; the destination ids must be distinct, and within one batch no id may be both a source and a destination
 * (the caller's to guarantee, as with fl_distance_map_ids).  A snapshot store is a batch with only the state pointers set:
 * the shapes and pointers are checked per requested part.  FL_ERR_BAD_ARG before any CUDA call when n is out of range, a
 * pointer a requested part needs is NULL in either batch, the two batches differ in a shape or stride the requested parts
 * depend on, or the tree / path caches are present in one batch only (FL_COPY_WORLD).  One launch (k_copy_envs). */
int fl_copy_envs(const FlBatch *src, const FlBatch *dst, const int32_t *d_src_ids, const int32_t *d_dst_ids, int64_t n,
                 uint32_t parts, const FlObsBuffers *d_src_out, const FlObsBuffers *d_dst_out, void *stream);

/* The same step with a compact device-to-host format (csrc/wire.cuh): instead of copying 2,438 bytes per agent, a pack
 * kernel rewrites each environment range into ~1.1 KB per agent — tree nodes that are the all -1 "no branch" vector as one
 * bit, adjacency / orders as int8, the 70 flag entries of the attribute vector as bits, every other float as its own 32
 * bits — straight into `h_wire` (pinned, device-mapped host memory of at least fl_wire_bytes(b) bytes, e.g. cudaHostAlloc /
 * torch pin_memory), and host threads of this library (fl_host_threads) expand it into the same h_out tensors, bit for bit
 * what fl_step_observe_host delivers, while the device works on the next range.  d_cursor: device uint32[64] scratch.
 * SYNCHRONOUS: every h_out tensor is complete when the call returns.  wire_bytes_out (may be NULL): bytes that crossed PCIe. */
int fl_step_observe_host_compact(const FlBatch *b, const uint8_t *h_actions, uint8_t *d_actions,
                                 const FlObsBuffers *d_out, const FlObsBuffers *h_out, void *h_wire, uint32_t *d_cursor,
                                 uint64_t *wire_bytes_out, uint32_t flags, int n_chunks, void *stream, void *copy_stream);
size_t fl_wire_bytes(const FlBatch *b, int n_chunks);
/* Host threads of the expansion: n > 0 sets the count (before the first compact step; default: hardware threads divided by
 * LOCAL_WORLD_SIZE, at most 32); returns the count in use. */
int fl_host_threads(int n);

/* Number of kernel launches issued by this library since load (bench.py reports it as gpu_launches). */
uint64_t fl_launch_count(void);

/* Measurement hooks (no reference counterpart; BASELINE.json asks for per-kernel numbers).  While
 * enabled, every kernel launch of this library is bracketed by two CUDA events recorded on the
 * launching stream.  fl_profile_collect waits for the pending events and writes the accumulated
 * device time in ms and the launch count per kernel into ms_out / launches_out
 * (fl_profile_num_kernels() entries each; either may be NULL); reset != 0 zeroes the totals. */
int fl_profile_num_kernels(void);
const char *fl_profile_kernel_name(int k);
void fl_profile_enable(int on);
int fl_profile_collect(double *ms_out, uint64_t *launches_out, int reset);

#ifdef __cplusplus
}
#endif
#endif
