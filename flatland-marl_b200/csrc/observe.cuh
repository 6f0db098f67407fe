// observe.cuh — k_observe: TreeObsForRailEnv::get_many + get_properties (treeobs.cpp:30-108, 612-640) for
// one environment per CTA, the per-environment working set staged in shared memory.
//
// Phases of one CTA (= one environment):
//   0  stage the rail grid, the rail index and (as far as they fit) the static walk tables into shared memory
//      with 1-D TMA bulk copies (cp.async.bulk + mbarrier) while phase 1 reads the agents.
//   1  loader view per agent (loader.cpp:8-179, 221-327): virtual position, valid actions, distance to
//      target, the occupancy word per RAIL CELL (treeobs.cpp:67-92) built with shared-memory atomics, and the
//      one-hot part of the attribute vector as three bit masks.
//   2  the serial, sticky DeadlockChecker (deadlock_checker.cpp:11-110) on lane 0 of the last warp, running
//      concurrently with phases 3 and 4 (its result is only needed by the attribute vector).
//   3  shortest-path predictions (predictions.cpp:13-235) as occupancy intervals, one lane per agent hopping
//      from static walk to static walk (walks.cuh): a counting pass, a scan and a scatter pass build a CSR inverse
//      index  rail cell -> intervals, every bucket ordered by start time so that the tree walk only scans the
//      entries of a three-step time window.  (The reference keys positions by c * W + r, which makes distinct
//      cells of a grid with H > W share predictions; kcls of walks.cuh maps a rail cell to its key class so
//      that these false conflicts are reproduced.)
//   4  the 31-node branch trees (treeobs.cpp:154-610), one warp per agent taken from a shared counter:
//      STRUCTURE: node n of the tree lives in lane n.  Which walk a node stands for, where it ends and what its
//        children are follows from the static walk records alone (steps, kind, children, the steps at which the walk
//        crosses the target of a slot), so the reference's FIFO becomes one ballot + shuffle round per tree level.
//      FEATURES: the cells of all walks of the agent form one flat list (about 130 cells); the warp takes it 32
//        cells at a time, one cell per lane — no idle lanes, no queue, no atomics.  The owner node of a cell follows
//        from a ballot + a bit mask of segment starts; what the lanes find (trains, predicted conflicts) returns
//        to the lane that owns the node as ballots masked by the node's segment.  Lane n then writes node n of the
//        forest (three 16-byte stores), its adjacency row and its evaluation orders (tool.h:468-524).
//   5  the 83-float attribute vector (feature_parser.cpp:3-98), written with coalesced stores.
// Arrays that do not fit in shared memory for a configuration (large grids) stay in global memory behind
// the same generic pointers (ObsLayout offsets < 0).
#pragma once
#include "common.cuh"
#include "walks.cuh"

namespace {

constexpr int I_INF = 0x7fffffff;

struct ObsLayout {   // byte offsets into dynamic shared memory (host: make_obs_layout); < 0 = lives in global memory
    int bar, part, cmp, ag, dl, ci, ks, bm, sq, seg_cap, sort_small, kcls, grid, ridx, ent, ent_cap, total;
    int srec, wrec, whoff, whits, wlist, sdist;   // static walk tables (walks.cuh)
    int sq_words;                                 // uint32 words of the sq region (seg_cap may be lowered by a test override)
    int path_cache;                               // FlBatch.path_cache is in use (the "pathcache" knob turns it off)
    int tree_cache;                               // FlBatch.tree_cache is in use (the "treecache" knob turns it off)
    int flat_walk;                                // path segments walked by warps as flat lists: bit 0 counting pass, bit 1 scatter pass
    int parts;                                    // split launch: CTAs per environment of the tree kernel (0 = fused kernel)
    int ws_ag, ws_idx, ws_ag_bytes, ws_idx_bytes; // split launch: byte offsets / sizes of the two blocks of FlBatch.obs_ws
};

// k_observe comes in three shapes.  OBS_FUSED: one CTA per environment does everything (the headline shape: all of the
// working set stays in shared memory).  OBS_INDEX + OBS_TREES: the same code cut after phase 3 — the first kernel (one CTA
// per environment) builds the loader view, the deadlock flags, the prediction index and the attribute vectors and leaves
// the index in FlBatch.obs_ws; the second (`parts` CTAs per environment) stages it back into shared memory with bulk
// copies and walks the trees of every parts-th agent.  Few large environments (Test_14: 64 x 425 agents) then fill the
// chip, and many small ones are cut into more, smaller units of work than there are CTA slots.
enum : int { OBS_FUSED = 0, OBS_INDEX = 1, OBS_TREES = 2 };
// The fused kernel also runs as a GROUP (template parameter G > 1): one CTA of G x NT threads holds G environments side by
// side — G copies of the shared-memory plan, the index phases of each behind its own pair of named barriers — and the tree
// phase takes (environment, agent) pairs from all of them: a warp whose own environment has no agent left walks the trees
// of its neighbours.  With one CTA per environment the warps of an environment that finishes early leave the SM while the
// slowest environment of the SM (the launch is one wave) runs on at a quarter of the SM's issue rate; as a group the SM's
// warps stay busy until all of its environments are done.
constexpr int OBS_MISC_WORDS = 8;   // [0] path segments, then entries  [1] next agent of phase 4  [2] max rows per cell  [3] bad cell met
                                    // [4] group mode: the index is complete, trees may be taken by any warp of the CTA

// ---- mbarrier + 1-D TMA bulk copy (global -> shared), sm_90+ ------------------------------------
DEVI uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
DEVI void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
DEVI void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
DEVI void tma_load_1d(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
DEVI void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!ok);
}
DEVI void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

DEVI uint32_t ld_vol_u32(const uint32_t *p) { return *reinterpret_cast<const volatile uint32_t *>(p); }
DEVI int ld_vol_i32(const int *p) { return *reinterpret_cast<const volatile int *>(p); }
DEVI unsigned ld_vol_u16(const uint16_t *p) { return *reinterpret_cast<const volatile uint16_t *>(p); }

DEVI uint32_t pack_entry(int agent, int t0, int t1, int dh, int dp, int dn, uint32_t extra);
DEVI uint32_t entry_extra(int tpc, bool done);
// Predicted occupancy of one agent (predictions.cpp:13-235 + the transpose in treeobs.cpp:50-65) from the static walk
// tables.  The greedy descent of the distance map is forced inside a walk (one successor per state) and, because the
// distance of a state is one more than the lowest distance among its successors, always continues at the end of a
// walk into the child with the lowest distance, the first of equals in the order left, forward, right
// (predictions.cpp:13-76) — unless the start state cannot reach the target at all, in which case the path is its first
// element.  The path ends on the agent's target cell (a target hit of the walk) or after 500 moves.  Path element idx >= 1
// is occupied for prediction rows [1 + (idx-1)*tpc, idx*tpc], the last element until row 500, element 0 for row 0 only
// (or all rows when the path has a single element).  Emit(rail cell, t0, t1, entry) is called once per occupied element.
template <class Emit>
DEVI void predict_path(const uint4 *wrec, const uint32_t *whoff, const uint32_t *whits, const uint32_t *wlist,
                       const uint16_t *sd, unsigned sid, unsigned slot, int tpc, int agent, uint32_t extra, Emit emit) {
    int dp = (int)(sid & 3u);                        // direction of the previous element (element 0: its own)
    if (sd[sid] == FL_DIST_INF) {                    // no move lowers the distance: the path is its first element
        // (a start state on the target has distance 0 and ends through the target hit below)
        emit(sid >> 2, 0, NPRED - 1, pack_entry(agent, 0, NPRED - 1, dp, dp, dp, extra));
        return;
    }
    int kk = 0;                                      // path element index of the walk's first state
    while (true) {
        const uint4 w = wrec[sid];
        const int L = (int)(w.y & 0xFFFFu), kind = (int)((w.y >> 16) & 15u), nh = (int)((w.y >> 20) & 255u);
        int kend = L;
        bool hit = false;
        if (nh) {
            const uint32_t ho = whoff[sid];
            for (int q = 0; q < nh; q++) {
                const uint32_t hv = whits[ho + q];
                if ((hv >> 16) == slot) { kend = (int)(hv & 0xFFFFu); hit = true; break; }
            }
        }
        unsigned nxt = 0xFFFFu;                      // where the path continues after this walk
        if (!hit && (kind == WK_SWITCH || kind == WK_DEADEND)) {
            const unsigned ch[3] = {w.z & 0xFFFFu, w.z >> 16, w.w & 0xFFFFu};
            unsigned best = FL_DIST_INF;
#pragma unroll
            for (int j = 0; j < 3; j++)
                if (ch[j] != 0xFFFFu) { const unsigned v = sd[ch[j]]; if (v < best) { best = v; nxt = ch[j]; } }
        }
        // four elements per round: their states are loaded together (one memory latency per round, not per element;
        // the list has 8 elements of slack at its end, so reading past the walk is harmless)
        for (int k0 = 0; k0 <= kend; k0 += 4) {
            unsigned sv[5];
#pragma unroll
            for (int u = 0; u < 5; u++) sv[u] = wlist[w.x + k0 + u] & 0xFFFFu;
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int k = k0 + u;
                if (k > kend) break;
                const int idx = kk + k;
                const int t0 = idx ? 1 + (idx - 1) * tpc : 0;
                if (t0 >= NPRED) return;
                const bool last = (k == kend && (hit || nxt == 0xFFFFu)) || idx >= FL_PRED_DEPTH;
                const unsigned s = sv[u], sn = k < kend ? sv[u + 1] : nxt;
                const int d = (int)(s & 3u), dn = last ? d : (int)(sn & 3u);
                const int t1 = last ? NPRED - 1 : min(idx ? idx * tpc : 0, NPRED - 1);
                emit(s >> 2, t0, t1, pack_entry(agent, t0, t1, d, dp, dn, extra));
                if (last) return;
                dp = d;
            }
        }
        sid = nxt; kk += kend + 1;
    }
}

// Predicted-occupancy entry, 4 bytes, laid out so that entries order like their sort key (long-lived entries first, then by
// start row): regular << 31 | t0 << 22 | (bit 21 free) | rows per cell > 8 (read it from the agent record instead) << 20 |
// agent is DONE << 19 | (rows per cell - 1) << 16 | dir_next << 14 | dir_prev << 12 | dir_here << 10 | agent.
// "regular" is 0 for the last element of a path, which stays occupied until row 500 (long-lived).  The interval end is
// implied: 500 for a long-lived entry, 0 for element 0, t0 + tpc - 1 otherwise.
DEVI uint32_t pack_entry(int agent, int t0, int t1, int dh, int dp, int dn, uint32_t extra) {
    return (uint32_t)agent | ((uint32_t)dh << 10) | ((uint32_t)dp << 12) | ((uint32_t)dn << 14) | ((uint32_t)t0 << 22) |
           ((uint32_t)(t1 != NPRED - 1) << 31) | extra;
}
DEVI uint32_t entry_extra(int tpc, bool done) {
    return (tpc <= 8 ? (uint32_t)(tpc - 1) << 16 : 1u << 20) | ((uint32_t)done << 19);
}
// acc |= x when cond != 0, as one predicated OR (the compiler's select + OR is one more instruction per index entry)
DEVI void or_if(unsigned &acc, unsigned x, unsigned cond) {
    asm("{\n.reg .pred p;\nsetp.ne.u32 p, %2, 0;\n@p or.b32 %0, %0, %1;\n}" : "+r"(acc) : "r"(x), "r"(cond));
}
// rows an entry's agent spends per cell (info: the agents' records, only read for speeds below 1/8)
DEVI int entry_tpc(uint32_t en, const uint32_t *info) { return ((en >> 20) & 1u) ? (int)(info[en & 1023u] >> 24) : (int)((en >> 16) & 7u) + 1; }
DEVI uint32_t entry_sort_key(uint32_t en) { return en >> 22; }          // 10 bits: long-lived first, then by t0
DEVI bool entry_long_lived(uint32_t en) { return !(en >> 31); }
DEVI int entry_t0(uint32_t en) { return (int)((en >> 22) & 511u); }

// loader.cpp:273-312: valid-action mask, bit a = action a allowed
DEVI int valid_actions_of(const uint16_t *g, int W, int st, int ctr, int r, int c, int d) {
    int va = 0;
    if (st == MOVING || st == STOPPED) {
        if (ctr == 0) {
            const unsigned cell = g[r * W + c];
            const int nb = nibble(cell, d);
            int cnt = 0;
            bool branch_next = false;
            for (int a = A_LEFT; a <= A_RIGHT; a++) {
                const int nd = (d + a - 2) & 3;
                if (tbit(nb, nd)) {
                    va |= 1 << a;
                    cnt++;
                    if (__popc(g[(r + d_row(nd)) * W + c + d_col(nd)]) > 2) branch_next = true;
                }
            }
            if (__popc(cell) > 2 || (cnt == 1 && branch_next)) va |= 1 << A_STOP;
        } else va = 1 << A_NOTHING;
    } else if (st == READY) va = (1 << A_FORWARD) | (1 << A_STOP);
    else va = 1 << A_NOTHING;
    return va;
}

// Serial, order-dependent and sticky: an exact restatement of DeadlockChecker::update_deadlocks /
// _check_blocked / _fix_deps (deadlock_checker.cpp:11-110) with the recursion turned into an explicit
// stack.  Runs on one lane per environment while the other warps walk predictions and trees.
struct DeadlockScratch {
    uint8_t *checked, *ndep, *dl, *ct, *stk_d, *stk_phase;   // ct: transitions nibble of the agent's (cell, direction) | 16 if the agent is ACTIVE (on the map)
    uint16_t *dep, *stk_h, *stk_opp;
    int16_t *opp;      // [N][4] the ACTIVE agent standing on the neighbour cell in direction dd (highest handle), -1 = none:
                       // filled by all threads before the serial lane starts (deadlock_checker.cpp:15-20 agent_positions)
};

DEVI void update_deadlocks(const DeadlockScratch &x, int N) {
    for (int a0 = 0; a0 < N; a0++) {
        if (!(x.ct[a0] & 16) || x.dl[a0] || x.checked[a0]) continue;
        int sp = 0;
        x.stk_h[0] = a0; x.stk_d[0] = 0; x.stk_phase[0] = 0; x.checked[a0] = 1; sp = 1;
        while (sp > 0) {
            const int f = sp - 1, h = x.stk_h[f];
            bool popped = false, pushed = false;
            while (x.stk_d[f] < 4) {
                const int dd = x.stk_d[f];
                int opp;
                if (x.stk_phase[f] == 1) { opp = x.stk_opp[f]; x.stk_phase[f] = 0; }
                else {
                    if (!tbit(x.ct[h] & 15, dd)) { x.stk_d[f]++; continue; }
                    opp = x.opp[h * 4 + dd];
                    if (opp < 0) { x.checked[h] = 2; popped = true; break; }           // road is free
                    if (x.dl[opp]) { x.stk_d[f]++; continue; }                          // road is blocked
                    if (x.checked[opp] == 0) {                                          // recurse
                        x.stk_phase[f] = 1; x.stk_opp[f] = (uint16_t)opp;
                        x.stk_h[sp] = (uint16_t)opp; x.stk_d[sp] = 0; x.stk_phase[sp] = 0; x.checked[opp] = 1; sp++;
                        pushed = true;
                        break;
                    }
                }
                if (x.checked[opp] == 2 && !x.dl[opp]) { x.checked[h] = 2; popped = true; break; }  // may become free
                x.dep[h * 4 + x.ndep[h]] = (uint16_t)opp; x.ndep[h]++;
                x.stk_d[f]++;
            }
            if (pushed) continue;
            if (!popped && x.ndep[h] == 0) {
                x.checked[h] = 2;
                if ((x.ct[h] & 15) != 0) x.dl[h] = 1;
            }
            sp--;
        }
    }
    bool any = true;                                                                    // _fix_deps
    while (any) {
        any = false;
        for (int h = 0; h < N; h++) {
            if (x.checked[h] != 1) continue;
            int cnt = 0;
            for (int k = 0; k < x.ndep[h]; k++) {
                const int o = x.dep[h * 4 + k];
                if (x.checked[o] == 2) {
                    if (x.dl[o]) cnt++;
                    else { x.checked[h] = 2; any = true; }
                }
            }
            if (cnt == x.ndep[h]) { x.checked[h] = 2; x.dl[h] = 1; any = true; }
        }
    }
    for (int h = 0; h < N; h++) if (x.checked[h] == 1) { x.dl[h] = 1; x.checked[h] = 2; }
}

// rotate_transition (tool.h:300-335): rotate the 4 bits inside every orientation block right by k,
// then rotate the four blocks right by k
DEVI int rotate_transition(int t, int k) {
    int v = 0;
#pragma unroll
    for (int o = 0; o < 4; o++) {
        int bl = (t >> ((3 - o) * 4)) & 0xF;
        bl = ((bl >> k) | (bl << (4 - k))) & 0xF;
        v |= bl << ((3 - o) * 4);
    }
    return (((v & ((1 << (k * 4)) - 1)) << ((4 - k) * 4)) | (v >> (k * 4))) & 0xFFFF;
}

__constant__ int c_road_types[11] = {0x0000, 0x8020, 0x9220, 0x8421, 0x9621, 0xCC33,
                                     0x5202, 0x2000, 0x4002, 0x1200, 0xC022};  // loader.cpp:123-134

DEVI int road_type_of(int trans) {  // loader.cpp:122-161: first rotation that is in the table
    for (int q = 0; q < 4; q++) {
        const int rot = q == 0 ? trans : rotate_transition(trans, q);
        for (int k = 0; k < 11; k++) if (c_road_types[k] == rot) return k;
    }
    return 0;
}

// a / b correctly rounded (identical to IEEE division for the integer-valued operands of this kernel) from the
// correctly rounded reciprocal rb = __frcp_rn(b): q0 = RN(a*rb), r = a - b*q0 (exact in an FMA), q = RN(q0 + r*rb).
// The only inputs for which this sequence can misround have an all-ones significand in b; b is a step or agent
// count here.  Replaces the ~20-instruction division sequence on the per-node path.
DEVI float div_rn(float a, float b, float rb) {
    const float q0 = a * rb;
    const float r = fmaf(-q0, b, a);
    return fmaf(r, rb, q0);
}
struct Scale { float T, rT, N, rN; };
DEVI float scale_i(int v, const Scale &sc) { return v != I_INF ? div_rn((float)v, sc.T, sc.rT) : -1.0f; }  // treeobs.cpp:111-152
DEVI float scale_n(int v, const Scale &sc) { return div_rn((float)v, sc.N, sc.rN); }

// state id of the cell entered from (r, c) in direction cd; 0xFFFFFFFF when the rail leads nowhere (invalid grid)
DEVI uint32_t child_state(const uint16_t *ridx, int H, int W, int r, int c, int cd) {
    const int rr = r + d_row(cd), cc = c + d_col(cd);
    if (rr < 0 || cc < 0 || rr >= H || cc >= W) return 0xFFFFFFFFu;
    const unsigned ri = ridx[rr * W + cc];
    return ri == 0xFFFFu ? 0xFFFFFFFFu : ri * 4u + (uint32_t)cd;
}

DEVI void store_node(float *forest_node, float4 a, float4 b, float4 c) {
    float4 *p = reinterpret_cast<float4 *>(forest_node);
    p[0] = a; p[1] = b; p[2] = c;
}
DEVI void store_null_node(float *forest_node) {
    const float4 m = make_float4(-1.0f, -1.0f, -1.0f, -1.0f);
    store_node(forest_node, m, m, m);
}

// per-agent shared-memory record (struct of arrays, N entries each)
constexpr int OBS_AGENT_WORDS = 11;
struct ObsAgents {
    uint32_t *vrc;      // virtual position r | c << 16 (loader.cpp:87-101)
    uint32_t *sid0;     // state id of the virtual position and direction (walks.cuh), 0xFFFF = not on a rail cell
    uint32_t *info;     // dir | st << 2 | done << 5 | slot << 8 | tpc << 24
    float *speed;       // (float)speed
    float *dt;          // dist_target, INFINITY = unreachable
    int *cellid;        // on-map cell index, -1 otherwise
    int *initcell;      // initial cell index while off map, -1 otherwise
    uint32_t *rec_a;    // st | road << 3 | idir << 7 | od << 9 | ctr << 11 | maxc << 19 | va << 27
    uint32_t *rec_b;    // trans | nmal01 << 16 | mal01 << 17 | sig_mal << 18 | transitions nibble of the virtual position << 20
    uint32_t *m0, *m1;  // attribute entries 0..63 as bits (feature_parser.cpp:19-77), entry 41 (deadlocked) left out
};

DEVI ObsAgents obs_agents_at(uint32_t *ws_hdr, int N) {
    const int Np = (N + 3) & ~3;
    ObsAgents A;
    uint32_t *p = ws_hdr + 4;
    A.vrc = p; p += Np; A.sid0 = p; p += Np; A.info = p; p += Np;
    A.speed = reinterpret_cast<float *>(p); p += Np; A.dt = reinterpret_cast<float *>(p); p += Np;
    A.rec_b = p; p += Np;
    A.cellid = reinterpret_cast<int *>(p); p += N; A.initcell = reinterpret_cast<int *>(p); p += N;
    A.rec_a = p; p += N; A.m0 = p; p += N; A.m1 = p; p += N;
    return A;
}

// What the tree phase reads of one environment: static tables (shared-memory copy when the layout has room, else global
// memory), the prediction index and the agent block.  Group mode builds it for whichever environment of the CTA an agent
// belongs to.
struct ObsEnv {
    const uint16_t *ridx, *sdist, *kcls;
    const uint4 *wrec;
    const uint32_t *whoff, *whits, *wlist, *gtab;
    uint32_t *ci, *ks, *ent_s, *ent_g;
    uint2 *bm, *bm_s;
    int *misc;
    ObsAgents A;
};
DEVI ObsEnv obs_env_of(const FlBatch &b, const ObsLayout &lay, unsigned char *sm, int e) {
    const int SS = (int)b.state_stride;
    ObsEnv V;
    V.ridx = lay.ridx >= 0 ? reinterpret_cast<const uint16_t *>(sm + lay.ridx) : b.ridx + (size_t)e * b.ridx_stride;
    V.wrec = lay.wrec >= 0 ? reinterpret_cast<const uint4 *>(sm + lay.wrec) : reinterpret_cast<const uint4 *>(b.wrec) + (size_t)e * SS;
    V.whoff = lay.whoff >= 0 ? reinterpret_cast<const uint32_t *>(sm + lay.whoff) : b.whoff + (size_t)e * SS;
    V.whits = lay.whits >= 0 ? reinterpret_cast<const uint32_t *>(sm + lay.whits) : b.whits + (size_t)e * b.whits_stride;
    V.wlist = lay.wlist >= 0 ? reinterpret_cast<const uint32_t *>(sm + lay.wlist) : b.wlist + (size_t)e * b.wlist_stride;
    V.sdist = lay.sdist >= 0 ? reinterpret_cast<const uint16_t *>(sm + lay.sdist) : b.sdist + (size_t)e * b.n_slots * SS;
    V.kcls = lay.kcls >= 0 ? reinterpret_cast<const uint16_t *>(sm + lay.kcls) : nullptr;   // only when H > W
    V.gtab = b.gtab + (size_t)e * b.n_slots * SS;
    V.ci = reinterpret_cast<uint32_t *>(sm + lay.ci);
    V.ks = reinterpret_cast<uint32_t *>(sm + lay.ks) + 1;
    V.bm_s = reinterpret_cast<uint2 *>(sm + (lay.bm >= 0 ? lay.bm : 0));
    V.bm = lay.bm >= 0 ? V.bm_s : reinterpret_cast<uint2 *>(b.obs_ws + (size_t)e * b.ws_stride + lay.ws_idx / 4 + 2 * (SS / 4) + 4);
    V.ent_s = reinterpret_cast<uint32_t *>(sm + lay.ent);
    V.ent_g = b.entries + (size_t)e * b.ent_cap;
    V.misc = reinterpret_cast<int *>(sm + lay.bar + 16);
    V.A = obs_agents_at(reinterpret_cast<uint32_t *>(sm + lay.ag), (int)b.N);
    return V;
}

DEVI unsigned warp_excl_scan(unsigned v, int lane, unsigned &total) {
    unsigned x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned y = __shfl_up_sync(0xFFFFFFFFu, x, o);
        if (lane >= o) x += y;
    }
    total = __shfl_sync(0xFFFFFFFFu, x, 31);
    return x - v;
}

// NT threads per environment, RES CTAs per SM the register budget is cut for, MODE: OBS_FUSED / OBS_INDEX / OBS_TREES,
// G environments per CTA (group mode, fused kernel only; the CTA has G * NT threads)
template <int NT, int RES, int MODE, int G = 1>
__global__ void __launch_bounds__(NT * G, RES)
k_observe(FlBatch b, ObsLayout lay, float *__restrict__ out_attr, float *__restrict__ out_forest,
          int32_t *__restrict__ out_adj, int32_t *__restrict__ out_norder, int32_t *__restrict__ out_eorder,
          uint8_t *__restrict__ out_valid, float *__restrict__ out_dist_target) {
    static_assert(G == 1 || (MODE == OBS_FUSED && G <= 7 && NT * G <= 1024), "group mode: fused kernel, two named barriers per environment");
    const int sub = G > 1 ? (int)threadIdx.x / NT : 0;                 // which environment of the group this thread belongs to
    const int e_raw = MODE == OBS_TREES ? (int)blockIdx.x / lay.parts : (int)blockIdx.x * G + sub;
    const bool live = G == 1 || e_raw < (int)b.E;                       // the last group may be ragged: its spare threads only walk trees
    const int e = live ? e_raw : (int)b.E - 1;                          // (addresses only; a spare thread never dereferences them)
    const int part = MODE == OBS_TREES ? (int)blockIdx.x - e * lay.parts : 0, n_parts = MODE == OBS_TREES ? lay.parts : 1;
    const int N = (int)b.N, H = (int)b.H, W = (int)b.W;
    const int tid = (int)threadIdx.x - sub * NT, lane = tid & 31, warp = tid >> 5;
    extern __shared__ __align__(128) unsigned char obs_smem[];
    unsigned char *const smraw = obs_smem + (G > 1 ? (size_t)sub * lay.total : 0);
    // barriers of one environment: A = all of its NT threads, B = the NT - 32 threads that build the prediction index, C = the
    // hand-over index -> deadlock warp (arrive / sync over NT).  Group mode has 16 hardware barriers for G environments: C
    // reuses A (between phase 1 and the hand-over nobody waits on A), 0 stays the CTA-wide barrier.
    const int BAR_A = G > 1 ? 1 + 2 * sub : 0, BAR_B = G > 1 ? 2 + 2 * sub : 1, BAR_C = G > 1 ? BAR_A : 2;
    auto env_sync = [&]() { if (G > 1) named_bar_sync(BAR_A, NT); else __syncthreads(); };
    const int R = b.walk_total[(size_t)e * 4] >> 2;         // rail cells of this environment
    const int SS = (int)b.state_stride;

    // ---- pointers: shared-memory copy when the layout has room, global memory otherwise ---------
    const uint16_t *g_grid = b.grid + (size_t)e * b.grid_stride;
    const uint16_t *g_ridx = b.ridx + (size_t)e * b.ridx_stride;
    const uint32_t *g_srec = b.srec + (size_t)e * SS, *g_whoff = b.whoff + (size_t)e * SS;
    const uint4 *g_wrec = reinterpret_cast<const uint4 *>(b.wrec) + (size_t)e * SS;
    const uint32_t *g_wlist = b.wlist + (size_t)e * b.wlist_stride;
    const uint32_t *g_whits = b.whits + (size_t)e * b.whits_stride;
    const uint16_t *g_sdist = b.sdist + (size_t)e * b.n_slots * SS;
    const uint32_t *gtab = b.gtab + (size_t)e * b.n_slots * SS;
    (void)g_srec; (void)g_sdist;
    const uint16_t *grid = lay.grid >= 0 ? reinterpret_cast<const uint16_t *>(smraw + lay.grid) : g_grid;
    const ObsEnv X = obs_env_of(b, lay, smraw, e);
    const uint16_t *ridx = X.ridx, *sdist = X.sdist, *kcls = X.kcls;
    const uint4 *wrec = X.wrec;
    const uint32_t *whoff = X.whoff, *whits = X.whits, *wlist = X.wlist;
    uint32_t *ci = X.ci;                            // [R] occupancy word per rail cell
    uint32_t *ks = X.ks;                            // ks[-1..R]: bucket r = [ks[r-1], ks[r])
    // [R][4] bit s of .x / .y: at least one / two prediction entries of the key overlap rows 4s..4s+3.  In shared memory, or —
    // when its 32 bytes per rail cell do not fit beside the mandatory regions (lay.bm < 0: large worlds) — in its place in
    // the workspace: it is written with plain stores and read twice per visited cell with independent loads
    uint2 *bm = X.bm;
    const bool bm_smem = lay.bm >= 0;               // reads and atomics go through typed shared-memory accesses when they can
    uint2 *const bm_s = X.bm_s;
    uint2 *sq = reinterpret_cast<uint2 *>(smraw + lay.sq) + warp * 64;       // this warp's queue of cells that need the full conflict check
    // per warp: a 32-byte table "r-th set lane of a ballot" (five popc steps per look-up otherwise: 9 % of the kernel's instructions)
    uint8_t *const cmp_s = smraw + lay.cmp + warp * 32;
    uint32_t *s_part = reinterpret_cast<uint32_t *>(smraw + lay.part);
    uint64_t *bar = reinterpret_cast<uint64_t *>(smraw + lay.bar);
    int *s_misc = reinterpret_cast<int *>(smraw + lay.bar + 16);

    // the first six arrays (+ a 16-byte header in front of them: entries, longest time per cell) are what the tree phase
    // reads; the split launch hands exactly this block from the index kernel to the tree kernel
    const int Np = (N + 3) & ~3;
    uint32_t *ws_hdr = reinterpret_cast<uint32_t *>(smraw + lay.ag);
    const ObsAgents A = X.A;
    uint32_t *g_ws = b.obs_ws ? b.obs_ws + (size_t)e * b.ws_stride : nullptr;
    DeadlockScratch D;
    {
        uint16_t *p = reinterpret_cast<uint16_t *>(smraw + lay.dl);
        D.dep = p; p += 4 * N; D.stk_h = p; p += N; D.stk_opp = p; p += N;
        uint8_t *q = reinterpret_cast<uint8_t *>(p);
        D.checked = q; q += N; D.ndep = q; q += N; D.dl = q; q += N; D.ct = q; q += N; D.stk_d = q; q += N; D.stk_phase = q; q += N;
        D.opp = reinterpret_cast<int16_t *>(q);      // byte offset 18 N from a 128-byte aligned base: even
    }

    // optional phase timestamps (tuning only): FlBatch.debug_clocks [E][16] int64, NULL = off
    // [E][32]: slots 0..15 of the fused / index kernel, 16.. of the tree kernel of a split launch (its CTA 0 of the environment)
    int64_t *dbg = b.debug_clocks && part == 0 && live ? b.debug_clocks + (size_t)e * 32 : nullptr;
#define OBS_TICK(k) do { if (dbg && tid == 0) dbg[(MODE == OBS_TREES ? 16 : 0) + (k)] = clock64(); } while (0)
    if (dbg && tid == 0) {
        dbg[MODE == OBS_TREES ? 31 : 15] = clock64();
        if (MODE != OBS_TREES || n_parts == 1) { dbg[12] = 0; dbg[13] = 0; dbg[14] = 0; for (int k = 26; k <= 30; k++) dbg[k] = 0; }
    }
    // ---- phase 0: TMA bulk copies of the static world ---------------------------------------------
    const bool use_tma = MODE == OBS_TREES || lay.grid >= 0 || lay.ridx >= 0 || lay.srec >= 0 || lay.wrec >= 0 || lay.whoff >= 0 ||
                         lay.whits >= 0 || lay.wlist >= 0 || lay.kcls >= 0 || lay.sdist >= 0;
    uint32_t *ent = reinterpret_cast<uint32_t *>(smraw + lay.ent);
    uint32_t *const ent_s = ent;                   // the shared-memory copy (typed loads are cheaper than generic ones)
    if (use_tma && tid == 0 && live) {
        mbar_init(bar, 1);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        const uint32_t gb = lay.grid >= 0 ? (uint32_t)(b.grid_stride * 2) : 0u;
        const uint32_t rb = lay.ridx >= 0 ? (uint32_t)(b.ridx_stride * 2) : 0u;
        const uint32_t sb = (uint32_t)(SS * 4);
        const uint32_t lb = lay.wlist >= 0 ? (uint32_t)(b.wlist_stride * 4) : 0u;
        const uint32_t hb = lay.whits >= 0 ? (uint32_t)(b.whits_stride * 4) : 0u;
        const uint32_t kb = lay.kcls >= 0 ? (uint32_t)(SS / 2) : 0u;     // one uint16 per rail cell
        const uint32_t db = lay.sdist >= 0 ? (uint32_t)(b.n_slots * SS * 2) : 0u;
        // split launch, tree kernel: the index the first kernel left in FlBatch.obs_ws comes back with four bulk copies
        // (agent block, occupancy words, bucket offsets, time-slot filter) and the entries with a fifth when they fit
        uint32_t wsb = 0, eb = 0;
        if (MODE == OBS_TREES) {
            const int n_ent_g = (int)g_ws[0];
            wsb = (uint32_t)(lay.ws_ag_bytes + lay.ws_idx_bytes) - (lay.bm >= 0 ? 0u : 8u * (uint32_t)(SS / 4) * 4u);
            eb = (n_ent_g <= lay.ent_cap && !(b.ent_cap & 3)) ? (uint32_t)((n_ent_g * 4 + 15) & ~15) : 0u;   // 16-byte aligned blocks only
        }
        mbar_expect_tx(bar, wsb + eb + gb + rb + lb + hb + kb + db + (lay.srec >= 0 ? sb : 0u) + (lay.wrec >= 0 ? 4 * sb : 0u) + (lay.whoff >= 0 ? sb : 0u));
        if (MODE == OBS_TREES) {
            const unsigned char *gw = reinterpret_cast<const unsigned char *>(g_ws);
            const uint32_t Rb = (uint32_t)(SS / 4) * 4u;                     // bytes of one uint32 per rail cell (capacity)
            tma_load_1d(smraw + lay.ag, gw, (uint32_t)lay.ws_ag_bytes, bar);
            tma_load_1d(smraw + lay.ci, gw + lay.ws_idx, Rb, bar);
            tma_load_1d(smraw + lay.ks, gw + lay.ws_idx + Rb, Rb + 16u, bar);
            if (lay.bm >= 0) tma_load_1d(smraw + lay.bm, gw + lay.ws_idx + 2u * Rb + 16u, 8u * Rb, bar);
            if (eb) tma_load_1d(smraw + lay.ent, b.entries + (size_t)e * b.ent_cap, eb, bar);
        }
        if (gb) tma_load_1d(smraw + lay.grid, g_grid, gb, bar);
        if (rb) tma_load_1d(smraw + lay.ridx, g_ridx, rb, bar);
        if (kb) tma_load_1d(smraw + lay.kcls, b.kcls + (size_t)e * SS, kb, bar);
        if (db) tma_load_1d(smraw + lay.sdist, g_sdist, db, bar);
        if (lay.wrec >= 0) tma_load_1d(smraw + lay.wrec, g_wrec, 4 * sb, bar);
        if (lay.srec >= 0) tma_load_1d(smraw + lay.srec, g_srec, sb, bar);
        if (lay.whoff >= 0) tma_load_1d(smraw + lay.whoff, g_whoff, sb, bar);
        if (hb) tma_load_1d(smraw + lay.whits, g_whits, hb, bar);
        if (lb) tma_load_1d(smraw + lay.wlist, g_wlist, lb, bar);
    }
    // zero the bucket counters and the occupancy words
    if (MODE != OBS_TREES && live) {
        for (int k = tid; k <= R + 1; k += NT) ks[k - 1] = 0;
        for (int k = tid; k < R; k += NT) ci[k] = 0;
        for (int k = tid; k < R * 4; k += NT) bm[k] = make_uint2(0u, 0u);
    }
    const float T_ = (float)b.max_steps[e], Nf = (float)N;
    const Scale sc{T_, __frcp_rn(T_), Nf, __frcp_rn(Nf)};
    const int elapsed = b.elapsed[e];
    // OBS_MISC_WORDS scalars; a spare environment slot of a ragged group reads "ready, no agent left"
    if (tid < OBS_MISC_WORDS) s_misc[tid] = live ? 0 : (tid == 1 ? N : tid == 4 ? 1 : 0);
    __syncthreads();                               // (the whole CTA) mbarrier initialised, counters zeroed
    OBS_TICK(0);
    if (use_tma && live) mbar_wait(bar, 0);
    int tpc_max = 0;
    if (MODE != OBS_TREES && live) {

    // ---- phase 1: loader view (loader.cpp:8-179, 221-327) -----------------------------------------
    for (int i = tid; i < N; i += NT) {
        const size_t ea = (size_t)e * N + i;
        const short2 p = reinterpret_cast<const short2 *>(b.rc)[ea];
        const short2 ip = reinterpret_cast<const short2 *>(b.init_rc)[ea];
        const short2 tp = reinterpret_cast<const short2 *>(b.tgt_rc)[ea];
        const int r = p.x, c = p.y, d = b.dir[ea], st = b.state[ea], idir = b.init_dir[ea];
        const int slot = b.slot[ea], ctr = b.ctr[ea], maxc = b.max_count[ea];
        const double speed_d = b.speed[ea];
        const float speed = (float)speed_d;
        int vr, vc;
        if (off_map(st)) { vr = ip.x; vc = ip.y; } else if (on_map(st)) { vr = r; vc = c; } else { vr = tp.x; vc = tp.y; }
        const int tpc = (int)(1.0f / speed);                             // predictions.cpp:184
        const uint16_t *sd = sdist + (size_t)slot * SS;
        const unsigned vri = ridx[vr * W + vc], iri = ridx[ip.x * W + ip.y];
        A.vrc[i] = (uint32_t)(vr & 0xFFFF) | ((uint32_t)vc << 16);
        A.sid0[i] = vri != 0xFFFFu ? vri * 4u + (uint32_t)d : 0xFFFFu;
        A.info[i] = (uint32_t)d | ((uint32_t)st << 2) | ((uint32_t)(st == DONE) << 5) | ((uint32_t)slot << 8) |
                    ((uint32_t)min(tpc, 255) << 24);
        A.speed[i] = speed;
        atomicMax(&s_misc[2], min(tpc, 255));
        // the tree's occupancy maps take every agent that is not off the map and has a position (treeobs.cpp:74-80): the trains
        // on the map and — a case only the second episode after an in-place reset produces — a train standing on its target
        // in state DONE (see reset_env in step.cuh); the deadlock checker looks at ACTIVE agents only (D.ct bit 4)
        A.cellid[i] = (!off_map(st) && r >= 0) ? r * W + c : -1;
        A.initcell[i] = off_map(st) ? ip.x * W + ip.y : -1;
        const int trans = on_map(st) ? (int)grid[r * W + c] : 0;
        D.ct[i] = on_map(st) ? (uint8_t)(nibble(trans, d) | 16) : 0;
        D.dl[i] = b.deadlocked[ea]; D.checked[i] = 0; D.ndep[i] = 0;
        const int va = valid_actions_of(grid, W, st, ctr, r, c, d);
        for (int k = 0; k < 5; k++) out_valid[ea * 5 + k] = (va >> k) & 1;
        const unsigned idv = iri != 0xFFFFu ? sd[iri * 4u + idir] : FL_DIST_INF;
        float dt;                                                        // loader.cpp:163-179
        if (st == DONE) dt = 0.0f;
        else {
            const unsigned dv = off_map(st) ? idv : (vri != 0xFFFFu ? (unsigned)sd[vri * 4u + d] : FL_DIST_INF);
            dt = dv == FL_DIST_INF ? INFINITY : (float)dv;
        }
        out_dist_target[ea] = dt;
        A.dt[i] = dt;
        // attribute record (feature_parser.cpp:19-94)
        const int od_raw = b.old_dir[ea], od = od_raw == 255 ? d : od_raw;
        const int trans_attr = r >= 0 ? (int)grid[r * W + c] : 0;
        const int road = r >= 0 ? road_type_of(trans_attr) : 0;
        const int nmal01 = b.nmal[ea] != 0, mal01 = b.mal[ea] != 0, sig_mal = b.sig_mal[ea] != 0;
        A.rec_a[i] = (uint32_t)st | ((uint32_t)road << 3) | ((uint32_t)idir << 7) | ((uint32_t)od << 9) |
                     ((uint32_t)ctr << 11) | ((uint32_t)maxc << 19) | ((uint32_t)va << 27);
        A.rec_b[i] = (uint32_t)trans_attr | ((uint32_t)nmal01 << 16) | ((uint32_t)mal01 << 17) | ((uint32_t)sig_mal << 18) |
                     ((uint32_t)nibble(grid[vr * W + vc], d) << 20);
        // entries 0..63 of the attribute vector are one-hot codes and flags: bit k of (m0, m1) = entry k
        A.m0[i] = (1u << st) | (1u << (7 + road)) | (1u << (18 + nmal01)) | (1u << (28 + idir));
        A.m1[i] = (1u << d) | (1u << (4 + od)) | ((uint32_t)(st == MOVING) << 8) | ((uint32_t)sig_mal << 10) | ((uint32_t)!mal01 << 11) |
                  ((uint32_t)(ctr == 0) << 12) | ((uint32_t)(ctr == maxc) << 13) | ((uint32_t)(st == MALFUNCTION || st == MAL_OFF) << 14) |
                  ((uint32_t)off_map(st) << 15) | ((uint32_t)on_map(st) << 16) | (__brev((unsigned)trans_attr) << 1);
        // entries 70..82 are floats (feature_parser.cpp:78-94): written here by the agent's own lane, every lane in the
        // same expression at the same time (phase 5 writes the flag entries 0..69)
        {
            const float max_dist = (float)((H + W) * 8);
            const float curr_step = (float)elapsed / T_;
            const float latest = (float)b.latest[ea] / T_, before_late = __fsub_rn(latest, curr_step);
            const float dist_f = dt == INFINITY ? 8.0f : dt / max_dist;
            float *fa = out_attr + ea * FL_ATTR_F + 70;
            fa[0] = (float)i / Nf;
            fa[1] = curr_step;
            fa[2] = (float)b.earliest[ea] / T_;
            fa[3] = latest;
            fa[4] = (float)b.arrival[ea] / T_;
            fa[5] = before_late;
            fa[6] = dist_f;
            fa[7] = before_late < dist_f ? before_late : dist_f;
            fa[8] = (float)maxc / 10.0f;
            fa[9] = speed / 1.0f;
            fa[10] = (float)ctr / 10.0f;
            fa[11] = (float)mal01 / 10.0f;
            fa[12] = idv == FL_DIST_INF ? 8.0f : (float)idv / max_dist;
        }
    }
    env_sync();
    // occupancy word per rail cell (treeobs.cpp:67-92, deadlock_checker.cpp:15-20): the HIGHEST handle standing on the
    // cell (std::map assignment in handle order = last writer) in the top bits so atomicMax picks it, its
    // direction and malfunction flag; then the number of off-map trains whose initial cell it is.
    for (int i = tid; i < N; i += NT) {
        const int cellid = A.cellid[i];
        if (cellid >= 0) {
            const unsigned ri = ridx[cellid];
            if (ri != 0xFFFFu)
                atomicMax(&ci[ri], ((uint32_t)(i + 1) << 21) | ((A.info[i] & 3u) << 9) | (((A.rec_b[i] >> 17) & 1u) << 8));
        }
    }
    env_sync();
    for (int i = tid; i < N; i += NT) {
        const int ic = A.initcell[i];
        if (ic >= 0) {
            const unsigned ri = ridx[ic];
            if (ri != 0xFFFFu && ld_vol_u32(&ci[ri]) != 0) atomicAdd(&ci[ri], 1u << 11);
        }
    }
    env_sync();
    // deadlock_checker.cpp:15-20 agent_positions, hoisted out of the serial lane: the highest ACTIVE handle per rail cell (in
    // the still unused bucket counters), then for every active agent the occupant of each neighbour cell its transitions lead to
    {
        uint32_t *ca = ks;                            // ks[0..R) is zero until the counting pass of phase 3
        for (int i = tid; i < N; i += NT)
            if (D.ct[i] & 16) { const unsigned ri = ridx[A.cellid[i]]; if (ri != 0xFFFFu) atomicMax(&ca[ri], (uint32_t)(i + 1)); }
        env_sync();
        for (int k = tid; k < N * 4; k += NT) {
            const int i = k >> 2, dd = k & 3;
            int opp = -1;
            if ((D.ct[i] & 16) && tbit(D.ct[i] & 15, dd)) {
                const int cid = A.cellid[i], rr = cid / W + d_row(dd), cc = cid % W + d_col(dd);
                if (rr >= 0 && cc >= 0 && rr < H && cc < W) {
                    const unsigned ri = ridx[rr * W + cc];
                    if (ri != 0xFFFFu) opp = (int)ld_vol_u32(&ca[ri]) - 1;
                }
            }
            D.opp[k] = (int16_t)opp;
        }
        env_sync();
        for (int k = tid; k < R; k += NT) ca[k] = 0;
        env_sync();
    }
    OBS_TICK(1);

    // ---- phase 2 (lane 0 of the last warp): deadlocks; phase 3 (the other warps, named barrier B): predictions ----
    // The last warp runs the serial deadlock lane WHILE the other warps build the prediction index and joins the tree phase
    // afterwards.  (Building the index with all warps and running the lane beside the tree phase instead was measured: 9 % more
    // instructions, 7 % more time — profiles/r02_n_ab.txt.)
    const bool dl_warp = warp == NT / 32 - 1;
    constexpr int NW = NT - 32;                    // threads walking predictions
    auto run_deadlocks = [&]() {
        if (lane == 0) { update_deadlocks(D, N); if (dbg) dbg[8] = clock64(); }
        __syncwarp();
        if (G > 1) {
            // group mode has no common end of the tree phase: the sticky flags go back to the agent records and the flag
            // entries of the attribute vectors (phase 5 below) are written here, by the warp that computed the flags
            for (int i = lane; i < N; i += 32) b.deadlocked[(size_t)e * N + i] = D.dl[i];
            float *dst = out_attr + (size_t)e * N * FL_ATTR_F;
            for (int idx = lane; idx < N * 70; idx += 32) {
                const int i = idx / 70, k = idx - i * 70;
                float v;
                if (k < 64) {
                    const uint32_t m = k < 32 ? A.m0[i] : A.m1[i];
                    v = (float)((m >> (k & 31)) & 1u);
                    if (k == 41) v = D.dl[i] != 0;
                } else {
                    const uint32_t ra = A.rec_a[i], rb = A.rec_b[i];
                    v = k == 64 ? (float)(rb & 1u) : (float)((ra >> (27 + k - 65)) & 1u);
                }
                dst[i * FL_ATTR_F + k] = v;
            }
        }
    };
    if (dl_warp) {
        run_deadlocks();
        asm volatile("bar.sync %0, %1;" ::"r"(BAR_C), "r"(NT) : "memory");    // the prediction index is complete (the other warps only arrive)
        if (s_misc[0] > lay.ent_cap) ent = b.entries + (size_t)e * b.ent_cap;
    } else {
        // Predicted paths as segments (predictions.cpp:13-235): a path is a chain of static walks, gtab tells where it
        // continues after each of them.  One lane per agent follows the chain (one dependent load per walk) and writes
        // a segment record per walk into a pool; the occupancy intervals of a segment are then emitted by any thread.
        uint2 *pool = reinterpret_cast<uint2 *>(smraw + lay.sq);      // state | last step << 16 | direction before << 30,
                                                                      // agent | first path index << 10 | direction after << 19 | last << 21
        uint2 *pool_g = reinterpret_cast<uint2 *>(b.segs) + (size_t)e * b.seg_stride;   // segments beyond the shared-memory pool
        const int seg_gcap = b.segs ? (int)b.seg_stride : 0;
        // Path cache (FlBatch.path_cache): the elements of an agent's predicted path — rail key and index entry, rows counted
        // from "now" — depend on the static tables and the agent's (cell, direction, rows per cell, done) alone.  An agent
        // whose key matches what the cache holds takes its elements from there (two streaming passes, no walk); the others
        // are walked as before and leave their elements behind for the next step.  pc_n[i]: elements of agent i, | 0x10000
        // when they come from the cache (the room of A.initcell, which only the occupancy pass of phase 1 reads).
        uint2 *const pcache = lay.path_cache ? reinterpret_cast<uint2 *>(b.path_cache) + (size_t)e * N * b.pc_stride : nullptr;
        const int PC = (int)b.pc_stride;
        int *const pc_n = A.initcell;
        auto path_key = [&](int i) { const uint32_t inf = A.info[i]; return 0x80000000u | (((inf >> 5) & 1u) << 24) | ((inf >> 24) << 16) | (A.sid0[i] & 0xFFFFu); };
        for (int i = tid; i < N; i += NW) {
            const uint32_t info = A.info[i];
            const unsigned slot = (info >> 8) & 0xFFFFu;
            unsigned sid = A.sid0[i];
            pc_n[i] = 0;
            if (sid == 0xFFFFu) continue;
            if (pcache) {
                const uint2 hdr = pcache[(size_t)i * PC];
                if (hdr.x == path_key(i)) { pc_n[i] = (int)(hdr.y | 0x10000u); continue; }
            }
            const int tpc = (int)(info >> 24);
            const uint32_t *gt = gtab + (size_t)slot * SS;
            unsigned dp = sid & 3u;
            int kk = 0;
            const bool stuck = sdist[(size_t)slot * SS + sid] == FL_DIST_INF;   // no move lowers the distance: a single element
            while (true) {
                const uint32_t g = stuck ? 0xFFFFu : gt[sid];
                const unsigned nxt = g & 0xFFFFu, kend = (g >> 16) & 0x3FFFu;
                const int pos = atomicAdd(&s_misc[0], 1);
                const uint2 rec = make_uint2(sid | (kend << 16) | (dp << 30),
                                             (unsigned)i | ((unsigned)kk << 10) | ((nxt & 3u) << 19) | ((nxt == 0xFFFFu ? 1u : 0u) << 21));
                if (pos < lay.seg_cap) pool[pos] = rec;
                else if (pos - lay.seg_cap < seg_gcap) pool_g[pos - lay.seg_cap] = rec;
                kk += (int)kend + 1;
                if (nxt == 0xFFFFu || kk > FL_PRED_DEPTH || 1 + (kk - 1) * tpc >= NPRED) break;
                dp = g >> 30; sid = nxt;
            }
        }
        named_bar_sync(BAR_B, NW);
        const int n_seg = s_misc[0];
        if (dbg && tid == 0) dbg[11] = n_seg;
        const bool pooled = n_seg <= lay.seg_cap + seg_gcap;  // else: every lane walks its agent's path itself (predict_path), twice
        // Emit(rail cell, t0, t1, entry) for every occupied element of pool segment j (one thread per segment)
        auto emit_segment = [&](int j, auto emit) {
            const uint2 sg = j < lay.seg_cap ? pool[j] : pool_g[j - lay.seg_cap];
            const unsigned sid = sg.x & 0xFFFFu;
            const int kend = (int)((sg.x >> 16) & 0x3FFFu), agent = (int)(sg.y & 1023u), kk = (int)((sg.y >> 10) & 511u);
            const bool seg_last = (sg.y >> 21) & 1u;
            const uint32_t ainf = A.info[agent];
            const int tpc = (int)(ainf >> 24);
            const uint32_t extra = entry_extra(tpc, (ainf >> 5) & 1u);
            int dp = (int)(sg.x >> 30);
            const uint32_t wx = wrec[sid].x;
            for (int k0 = 0; k0 <= kend; k0 += 4) {  // four states per round: one memory latency per round (8 elements of slack in wlist)
                unsigned sv[5];
#pragma unroll
                for (int u = 0; u < 5; u++) sv[u] = wlist[wx + k0 + u];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int k = k0 + u;
                    if (k > kend) return;
                    const int idx = kk + k;
                    const int t0 = idx ? 1 + (idx - 1) * tpc : 0;
                    if (t0 >= NPRED) return;
                    const bool last = (k == kend && seg_last) || idx >= FL_PRED_DEPTH;
                    const int d = (int)(sv[u] & 3u), dn = last ? d : (k < kend ? (int)(sv[u + 1] & 3u) : (int)((sg.y >> 19) & 3u));
                    const int t1 = last ? NPRED - 1 : min(idx ? idx * tpc : 0, NPRED - 1);
                    emit((sv[u] & 0xFFFFu) >> 2, t0, t1, pack_entry(agent, t0, t1, d, dp, dn, extra));
                    if (last) return;
                    dp = d;
                }
            }
        };
        // The same for every pool segment, a warp at a time (lay.flat_walk bit 0: counting pass, bit 1: scatter pass): 32 segments per batch, their occupied elements as one flat list, one
        // element per lane and round — every load of a round is independent, so a batch costs about three memory round trips
        // (segment record -> walk offset -> states) instead of three per segment and thread.  dirs: the entry's directions are
        // needed (scatter pass) or only its rail cell (counting pass).
        auto emit_pool_flat = [&](bool dirs, auto emit) {
            constexpr int NWP = NW / 32;
            for (int j0 = warp * 32; j0 < n_seg; j0 += NWP * 32) {
                const int j = j0 + lane;
                const bool has = j < n_seg;
                uint2 sg = make_uint2(0u, 0u);
                if (has) sg = j < lay.seg_cap ? pool[j] : pool_g[j - lay.seg_cap];
                const unsigned sid = sg.x & 0xFFFFu;
                const int kend = (int)((sg.x >> 16) & 0x3FFFu), agent = (int)(sg.y & 1023u), kk = (int)((sg.y >> 10) & 511u);
                const uint32_t ainf = has ? A.info[agent] : (1u << 24);
                const int tpc = max((int)(ainf >> 24), 1);
                const uint32_t wx = has ? wrec[sid].x : 0u;
                // elements kk .. last_idx of the path are emitted: up to the end of the segment, path element 500, and row 500
                const int last_idx = min(min(kk + kend, FL_PRED_DEPTH), (NPRED - 2) / tpc + 1);
                const unsigned cnt = has ? (unsigned)max(last_idx - kk + 1, 0) : 0u;
                unsigned total;
                const unsigned off = warp_excl_scan(cnt, lane, total);
                const unsigned nonempty = __ballot_sync(0xFFFFFFFFu, cnt > 0);
                __syncwarp();
                if (cnt > 0) cmp_s[__popc(nonempty & ((1u << lane) - 1u))] = (uint8_t)lane;   // r-th segment with elements
                __syncwarp();
                // what an element needs of its segment, fetched from the owner lane: a = walk offset, b = first step's offset in the
                // flat list, c = kk | kend << 9 | tpc << 23, d = the segment record's second word (agent, next direction, last),
                // e = direction before the segment
                const uint32_t rc_ = (uint32_t)kk | ((uint32_t)kend << 9) | ((uint32_t)min(tpc, 255) << 23);
                // four rounds of 32 elements at a time: owners and addresses first, then all loads, then the emits — the loads
                // of a batch of rounds are in flight together
                for (unsigned base0 = 0; base0 < total; base0 += 128) {
                    uint32_t o_off[4], o_c[4], o_y[4], o_dp[4], o_wx[4];
                    unsigned sv[4], sn[4], sp[4];
#pragma unroll
                    for (int r = 0; r < 4; r++) {
                        const unsigned base = base0 + 32u * r, f = base + lane;
                        if (base >= total) { o_off[r] = 0; o_c[r] = 0; o_y[r] = 0; o_dp[r] = 0; o_wx[r] = 0; continue; }   // warp-uniform
                        const int cnt0 = __popc(__ballot_sync(0xFFFFFFFFu, cnt > 0 && off <= base));
                        const unsigned starts = __reduce_or_sync(0xFFFFFFFFu, (cnt > 0 && off > base && off < base + 32) ? 1u << (off - base) : 0u);
                        const int rank = cnt0 - 1 + __popc(starts & (0xFFFFFFFFu >> (31 - lane)));
                        const int owner = f < total ? (int)cmp_s[rank] : 0;
                        o_wx[r] = __shfl_sync(0xFFFFFFFFu, wx, owner); o_off[r] = __shfl_sync(0xFFFFFFFFu, off, owner);
                        o_c[r] = __shfl_sync(0xFFFFFFFFu, rc_, owner); o_y[r] = __shfl_sync(0xFFFFFFFFu, sg.y, owner);
                        o_dp[r] = __shfl_sync(0xFFFFFFFFu, sg.x >> 30, owner);
                    }
#pragma unroll
                    for (int r = 0; r < 4; r++) {
                        const unsigned f = base0 + 32u * r + lane;
                        sv[r] = 0; sn[r] = 0; sp[r] = 0;
                        if (f < total) {
                            const int k = (int)(f - o_off[r]), o_kend = (int)((o_c[r] >> 9) & 0x3FFFu);
                            sv[r] = wlist[o_wx[r] + k];
                            if (dirs) {
                                if (k < o_kend) sn[r] = wlist[o_wx[r] + k + 1];
                                if (k > 0) sp[r] = wlist[o_wx[r] + k - 1];
                            }
                        }
                    }
#pragma unroll
                    for (int r = 0; r < 4; r++) {
                        const unsigned f = base0 + 32u * r + lane;
                        if (f < total) {
                            const int k = (int)(f - o_off[r]), o_kk = (int)(o_c[r] & 511u), o_kend = (int)((o_c[r] >> 9) & 0x3FFFu), o_tpc = (int)(o_c[r] >> 23);
                            const int idx = o_kk + k;
                            const int t0 = idx ? 1 + (idx - 1) * o_tpc : 0;
                            const bool last = (k == o_kend && ((o_y[r] >> 21) & 1u)) || idx >= FL_PRED_DEPTH;
                            const int d = (int)(sv[r] & 3u), dn = last ? d : (k < o_kend ? (int)(sn[r] & 3u) : (int)((o_y[r] >> 19) & 3u));
                            const int dp = k > 0 ? (int)(sp[r] & 3u) : (int)o_dp[r];
                            const int t1 = last ? NPRED - 1 : min(idx ? idx * o_tpc : 0, NPRED - 1);
                            const int ag = (int)(o_y[r] & 1023u);
                            emit((sv[r] & 0xFFFFu) >> 2, t0, t1, dirs ? pack_entry(ag, t0, t1, d, dp, dn, entry_extra((int)(A.info[ag] >> 24), (A.info[ag] >> 5) & 1u)) : 0u);
                        }
                    }
                }
            }
        };
        auto count_emit = [&](unsigned rail, int, int, uint32_t) { atomicAdd(&ks[kcls ? (unsigned)kcls[rail] : rail], 1u); };
        // the cached paths: a warp per agent, a lane per element
        auto for_cached = [&](auto fn) {
            if (!pcache) return;
            for (int i = warp; i < N; i += NW / 32) {
                const int pn = pc_n[i];
                if (!(pn & 0x10000)) continue;
                const uint2 *lst = pcache + (size_t)i * PC + 1;
                const int n_el = pn & 0xFFFF;
                for (int j0 = lane; j0 < n_el; j0 += 128) {                  // four loads in flight per lane: the lists are in L2 / HBM
                    uint2 el[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) if (j0 + 32 * u < n_el) el[u] = lst[j0 + 32 * u];
#pragma unroll
                    for (int u = 0; u < 4; u++) if (j0 + 32 * u < n_el) fn(el[u]);
                }
            }
        };
        // counting pass: entries per rail cell (or key class)
        if (pooled) { if (lay.flat_walk & 1) emit_pool_flat(false, count_emit); else for (int j = tid; j < n_seg; j += NW) emit_segment(j, count_emit); }
        else
            for (int i = tid; i < N; i += NW) {
                const uint32_t info = A.info[i];
                const unsigned slot = (info >> 8) & 0xFFFFu, s0 = A.sid0[i];
                if (s0 != 0xFFFFu && !(pc_n[i] & 0x10000)) predict_path(wrec, whoff, whits, wlist, sdist + (size_t)slot * SS, s0, slot, (int)(info >> 24), i, entry_extra((int)(info >> 24), (info >> 5) & 1u), count_emit);
            }
        for_cached([&](uint2 el) { atomicAdd(&ks[el.x], 1u); });
        named_bar_sync(BAR_B, NW);
        OBS_TICK(2);
        // exclusive scan of ks[0..R] (R+1 values; the last becomes the total)
        const int per = (R + 1 + NW - 1) / NW, lo = min(tid * per, R + 1), hi = min(lo + per, R + 1);
        uint32_t sum = 0;
        for (int k = lo; k < hi; k++) sum += ks[k];
        uint32_t incl = sum;                        // inclusive scan of the partial sums: shuffles inside the warp, warp totals through shared memory
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, incl, o);
            if (lane >= o) incl += y;
        }
        if (lane == 31) s_part[warp] = incl;
        named_bar_sync(BAR_B, NW);
        uint32_t run = incl - sum, n_total = 0;
#pragma unroll
        for (int w2 = 0; w2 < NW / 32; w2++) {
            const uint32_t wt = s_part[w2];
            if (w2 < warp) run += wt;
            n_total += wt;
        }
        for (int k = lo; k < hi; k++) { const uint32_t v = ks[k]; ks[k] = run; run += v; }
        named_bar_sync(BAR_B, NW);
        const int n_ent = (int)n_total;
        if (tid == 0) s_misc[0] = n_ent;
        if (n_ent > lay.ent_cap) ent = b.entries + (size_t)e * b.ent_cap;   // does not fit in shared memory: global spill space
        // scatter pass.  ks[key] is advanced to the END of its bucket; bucket r is [ks[r-1], ks[r]) afterwards (ks[-1] = 0).
        auto scatter_key = [&](unsigned key, int t0, int t1, uint32_t en) {
            ent[atomicAdd(&ks[key], 1u)] = en;
            const int sa = t0 >> 2, sb = t1 >> 2;             // time slots of 4 rows the entry overlaps
            for (int wd = sa >> 5; wd <= sb >> 5; wd++) {
                const int lo_b = max(sa - 32 * wd, 0), hi_b = min(sb - 32 * wd, 31);
                const uint32_t m = (0xFFFFFFFFu >> (31 - hi_b)) & (0xFFFFFFFFu << lo_b);
                uint2 *w2 = (bm_smem ? bm_s : bm) + key * 4 + wd;
                const uint32_t twice = (bm_smem ? atomicOr(&bm_s[key * 4 + wd].x, m) : atomicOr(&w2->x, m)) & m;     // slots that already had an entry
                if (twice) { if (bm_smem) atomicOr(&bm_s[key * 4 + wd].y, twice); else atomicOr(&w2->y, twice); }
            }
        };
        auto scatter_emit = [&](unsigned rail, int t0, int t1, uint32_t en) {
            const unsigned key = kcls ? (unsigned)kcls[rail] : rail;
            scatter_key(key, t0, t1, en);
            if (pcache) {                              // a walked path leaves its elements in the cache: element idx at slot 1 + idx
                const int ag = (int)(en & 1023u), tpc = entry_tpc(en, A.info);
                const int idx = t0 ? (t0 - 1) / tpc + 1 : 0;
                if (idx + 1 < PC) pcache[(size_t)ag * PC + 1 + idx] = make_uint2(key, en);
                atomicMax(&pc_n[ag], idx + 1);
            }
        };
        if (pooled) { if (lay.flat_walk & 2) emit_pool_flat(true, scatter_emit); else for (int j = tid; j < n_seg; j += NW) emit_segment(j, scatter_emit); }
        else
            for (int i = tid; i < N; i += NW) {
                const uint32_t info = A.info[i];
                const unsigned slot = (info >> 8) & 0xFFFFu, s0 = A.sid0[i];
                if (s0 != 0xFFFFu && !(pc_n[i] & 0x10000)) predict_path(wrec, whoff, whits, wlist, sdist + (size_t)slot * SS, s0, slot, (int)(info >> 24), i, entry_extra((int)(info >> 24), (info >> 5) & 1u), scatter_emit);
            }
        for_cached([&](uint2 el) {
            const uint32_t en = el.y;
            const int t0 = entry_t0(en);
            scatter_key(el.x, t0, entry_long_lived(en) ? NPRED - 1 : (t0 ? t0 + entry_tpc(en, A.info) - 1 : 0), en);
        });
        named_bar_sync(BAR_B, NW);
        if (pcache)                                    // headers of the paths walked in this step (too long for the cache: no key)
            for (int i = tid; i < N; i += NW) {
                const int pn = pc_n[i];
                if (pn > 0 && !(pn & 0x10000)) pcache[(size_t)i * PC] = pn < PC ? make_uint2(path_key(i), (uint32_t)pn) : make_uint2(0u, 0u);
            }
        OBS_TICK(4);
        // order every bucket: long-lived entries first, then by t0, so that the tree walk scans a time window only.
        // Entries in shared memory: buckets up to sort_small by one thread each (insertion sort: 32 buckets per warp at a
        // time), larger ones queued and sorted by a warp.  Entries spilled to global memory (large environments), where a
        // dependent chain of loads per compare would cost an L2 round trip each: every bucket by a warp — up to 32 entries as
        // one load, a bitonic network of register shuffles and one store; longer ones by a two-pass radix sort (5 + 5 bits
        // of the 10-bit key) that streams the bucket through a scratch copy with coalesced loads.
        const int SORT_SMALL = lay.sort_small;
        const bool in_smem = ent == ent_s;
        uint32_t *bigq = reinterpret_cast<uint32_t *>(smraw + lay.sq);          // the segment pool is no longer needed
        const int bigq_cap = lay.sq_words - 32 * (NT / 32);                     // its tail: 32 digit counters per warp
        uint32_t *hist = bigq + bigq_cap + 32 * warp;
        // scratch copy of a bucket at the same offsets: the free tail of the shared-memory entries, else the environment's
        // global spill space (all of it while the entries are in shared memory, its tail otherwise)
        uint32_t *g_ent = b.entries + (size_t)e * b.ent_cap;
        uint32_t *scratch = in_smem ? (2 * n_ent <= lay.ent_cap ? ent_s + n_ent : g_ent)
                                    : (2ll * n_ent <= (long long)b.ent_cap ? g_ent + n_ent : nullptr);
        auto insertion_sort = [&](int s0, int s1) {
            for (int x = s0 + 1; x < s1; x++) {
                const uint32_t v = ent[x];                   // entries order like their keys (ties: by their low bits, any order will do)
                int y = x - 1;
                while (y >= s0 && ent[y] > v) { ent[y + 1] = ent[y]; y--; }
                ent[y + 1] = v;
            }
        };
        // up to 32 entries, one per lane (v0: the lane's entry, already loaded): bitonic network of register shuffles
        auto warp_sort_regs = [&](int key, int s0, int n, uint32_t v0) {
            uint32_t kv = lane < n ? v0 : 0xFFFFFFFFu;                   // entries order like their keys; no entry is all ones (t0 <= 500)
#pragma unroll
            for (int k2 = 2; k2 <= 32; k2 <<= 1)
#pragma unroll
                for (int j2 = k2 >> 1; j2 > 0; j2 >>= 1) {
                    const uint32_t o = __shfl_xor_sync(0xFFFFFFFFu, kv, j2);
                    const bool up = (lane & k2) == 0, low = (lane & j2) == 0;
                    kv = (low == up) ? min(kv, o) : max(kv, o);
                }
            if (lane < n) ent[s0 + lane] = kv;
        };
        // more than 32 entries: two stable radix passes (5 + 5 bits of the 10-bit key) through the scratch copy, the bucket
        // taken 256 entries at a time so that eight loads per lane are in flight (one memory round trip per 256 entries and
        // loop instead of one per 32)
        auto warp_sort_radix = [&](int key, int s0, int n) {
            if (!scratch) { if (lane == 0) insertion_sort(s0, s0 + n); __syncwarp(); return; }
            uint32_t *bufa = ent + s0, *bufb = scratch + s0;
#pragma unroll 1
            for (int pass = 0; pass < 2; pass++) {
                const uint32_t *src = pass ? bufb : bufa;
                uint32_t *dst = pass ? bufa : bufb;
                const int sh = 5 * pass;
                hist[lane] = 0;
                __syncwarp();
                for (int x0 = 0; x0 < n; x0 += 256) {
                    uint32_t v[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) { const int x = x0 + u * 32 + lane; v[u] = x < n ? src[x] : 0u; }
#pragma unroll
                    for (int u = 0; u < 8; u++)
                        if (x0 + u * 32 + lane < n) atomicAdd(&hist[(entry_sort_key(v[u]) >> sh) & 31u], 1u);
                }
                __syncwarp();
                unsigned tot;
                const unsigned c = hist[lane], base = warp_excl_scan(c, lane, tot);
                __syncwarp();
                hist[lane] = base;
                __syncwarp();
                for (int x0 = 0; x0 < n; x0 += 256) {
                    uint32_t v[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) { const int x = x0 + u * 32 + lane; v[u] = x < n ? src[x] : 0u; }
#pragma unroll
                    for (int u = 0; u < 8; u++) {                               // in order: the passes must be stable
                        if (x0 + u * 32 >= n) break;                            // warp-uniform
                        const bool valid = x0 + u * 32 + lane < n;
                        const unsigned dg = valid ? ((entry_sort_key(v[u]) >> sh) & 31u) : 32u + (unsigned)lane;
                        const unsigned m = __match_any_sync(0xFFFFFFFFu, dg);
                        const int rank = __popc(m & ((1u << lane) - 1u));
                        if (valid) dst[hist[dg] + rank] = v[u];
                        __syncwarp();
                        if (valid && rank == 0) hist[dg] += (unsigned)__popc(m);
                        __syncwarp();
                    }
                }
            }
        };
        constexpr int NWARPS = NW / 32;
        if (in_smem) {
            for (int key = tid; key < R; key += NW) {
                const int s0 = (int)ks[key - 1], s1 = (int)ks[key];
                if (s1 - s0 <= SORT_SMALL) { insertion_sort(s0, s1); continue; }
                const int pos = atomicAdd(&s_misc[1], 1);
                if (pos < bigq_cap) bigq[pos] = (uint32_t)key; else insertion_sort(s0, s1);
            }
            named_bar_sync(BAR_B, NW);
            OBS_TICK(9);
            const int n_big = min(ld_vol_i32(&s_misc[1]), bigq_cap);
            for (int q = warp; q < n_big; q += NWARPS) {
                const int key = (int)bigq[q], s0 = (int)ks[key - 1], n = (int)ks[key] - s0;
                if (n <= 32) warp_sort_regs(key, s0, n, lane < n ? ent[s0 + lane] : 0u);
                else warp_sort_radix(key, s0, n);
            }
        } else {
            OBS_TICK(9);
            // (Packing consecutive small buckets into one 32-entry network per pass, a contiguous bucket range per warp, was
            // measured: nothing at Test_08, the index kernel of Test_14 0.31 -> 0.42 ms — profiles/r02_w_packed_sort.txt.)
            // every non-empty bucket by a warp; the entries of the warp's next two buckets are in flight while the current
            // one is sorted (a bucket costs one L2 / DRAM round trip that nothing else hides at 32 warps per SM)
            auto fetch = [&](int key, int &s0, int &n, uint32_t &v) {
                n = 0; v = 0u; s0 = 0;
                if (key < R) { s0 = (int)ks[key - 1]; n = (int)ks[key] - s0; if (n >= 2 && n <= 32 && lane < n) v = ent[s0 + lane]; }
            };
            constexpr int PF = 2;                       // buckets in flight per warp (four measured: no change — profiles/r02_y_prefetch4.txt)
            int s0q[PF], nq[PF];
            uint32_t vq[PF];
#pragma unroll
            for (int u = 0; u < PF; u++) fetch(warp + u * NWARPS, s0q[u], nq[u], vq[u]);
            for (int key = warp; key < R; key += NWARPS) {
                const int s0a = s0q[0], na = nq[0];
                const uint32_t va = vq[0];
#pragma unroll
                for (int u = 0; u + 1 < PF; u++) { s0q[u] = s0q[u + 1]; nq[u] = nq[u + 1]; vq[u] = vq[u + 1]; }
                fetch(key + PF * NWARPS, s0q[PF - 1], nq[PF - 1], vq[PF - 1]);
                if (na > 32) warp_sort_radix(key, s0a, na);
                else if (na >= 2) warp_sort_regs(key, s0a, na, va);
            }
        }
        named_bar_sync(BAR_B, NW);
        if (tid == 0) s_misc[1] = 0;                // phase 4 takes its agents from this counter
        named_bar_sync(BAR_B, NW);
        if (G > 1 && tid == 0) {                    // publish: every write of the index phases happened before the barrier above
            __threadfence_block();
            *reinterpret_cast<volatile int *>(&s_misc[4]) = 1;
        }
        if (MODE == OBS_INDEX) {
            // split launch: the index goes to FlBatch.obs_ws in the layout the tree kernel's bulk copies expect
            // (header + agent block | occupancy words | bucket offsets from ks[-1] | time-slot filter), the entries to
            // FlBatch.entries unless they already spilled there
            const int Rcap = SS / 4;
            if (tid == 0) { g_ws[0] = (uint32_t)n_ent; g_ws[1] = (uint32_t)ld_vol_i32(&s_misc[2]); g_ws[2] = 0u; g_ws[3] = 0u; }
            for (int k = 4 + tid; k < 4 + 6 * Np; k += NW) g_ws[k] = ws_hdr[k];
            uint32_t *gi = g_ws + lay.ws_idx / 4;
            for (int k = tid; k < R; k += NW) gi[k] = ci[k];
            for (int k = tid; k <= R + 1; k += NW) gi[Rcap + k] = ks[k - 1];
            uint2 *gb = reinterpret_cast<uint2 *>(gi + 2 * Rcap + 4);
            if (lay.bm >= 0) for (int k = tid; k < 4 * R; k += NW) gb[k] = bm[k];     // else it was built there
            if (ent == ent_s) {
                uint32_t *ge = b.entries + (size_t)e * b.ent_cap;
                for (int k = tid; k < n_ent; k += NW) ge[k] = ent_s[k];
            }
        }
        asm volatile("bar.arrive %0, %1;" ::"r"(BAR_C), "r"(NT) : "memory");  // lets the deadlock warp go on when it is done
    }
    OBS_TICK(3);
    if (dbg && tid == 0) dbg[10] = s_misc[0];
    tpc_max = ld_vol_i32(&s_misc[2]);
    } else if (MODE == OBS_TREES) {
        // tree kernel of the split launch: everything above arrived through the bulk copies
        const int n_ent_g = (int)ws_hdr[0];
        tpc_max = (int)ws_hdr[1];
        if (n_ent_g > lay.ent_cap || (b.ent_cap & 3)) ent = b.entries + (size_t)e * b.ent_cap;
    }

    // ---- phase 4: branch trees, one warp per agent, agents taken from a shared counter --------------------
    const bool spill_home = ent != ent_s;
    uint32_t *const ent_home = ent;
    const int tpc_max_home = tpc_max;
    uint2 *const sq_home = sq;
    const float T_home = T_;
    const Scale sc_home = sc;
    while (MODE != OBS_INDEX) {
        int h = 0, s_sel = sub;
        if (G == 1) {
            if (lane == 0) h = part + n_parts * atomicAdd(&s_misc[1], 1);     // the tree kernel's CTA `part` takes every n_parts-th agent
            h = __shfl_sync(0xFFFFFFFFu, h, 0);
            if (h >= N) break;
        } else {
            // group mode: the next agent of the warp's own environment, else of the first neighbour that has one left; an
            // environment whose index is still being built is waited for (its own warps are on it)
            int found = -1;
            if (lane == 0) {
                while (true) {
                    bool pending = false;
                    for (int k = 0; k < G; k++) {
                        const int s2 = sub + k < G ? sub + k : sub + k - G;
                        int *m = reinterpret_cast<int *>(obs_smem + (size_t)s2 * lay.total + lay.bar + 16);
                        if (!ld_vol_i32(&m[4])) { pending = true; continue; }
                        if (ld_vol_i32(&m[1]) >= N) continue;
                        const int hh = atomicAdd(&m[1], 1);
                        if (hh < N) { found = s2 | (hh << 4); break; }
                    }
                    if (found >= 0 || !pending) break;
                    __nanosleep(200);
                }
            }
            found = __shfl_sync(0xFFFFFFFFu, found, 0);
            if (found < 0) break;
            s_sel = found & 15; h = found >> 4;
            __threadfence_block();                  // acquire: the index was published before its ready flag
        }
        // ---- the environment the agent belongs to (group mode: possibly a neighbour's) shadows the home environment's names ----
        const int e_home = e;
        const ObsEnv V = G > 1 ? obs_env_of(b, lay, obs_smem + (size_t)s_sel * lay.total, (int)blockIdx.x * G + s_sel) : X;
        const int e = G > 1 ? (int)blockIdx.x * G + s_sel : e_home;
        const uint16_t *const ridx = V.ridx, *const sdist = V.sdist, *const kcls = V.kcls;
        const uint4 *const wrec = V.wrec;
        const uint32_t *const whoff = V.whoff, *const whits = V.whits, *const wlist = V.wlist, *const gtab = V.gtab;
        uint32_t *const ci = V.ci, *const ks = V.ks;
        uint2 *const bm = V.bm;
        const ObsAgents A = V.A;
        const bool spill = G > 1 ? ld_vol_i32(&V.misc[0]) > lay.ent_cap : spill_home;
        uint32_t *const ent = G > 1 ? (spill ? V.ent_g : V.ent_s) : ent_home;
        const int tpc_max = G > 1 ? ld_vol_i32(&V.misc[2]) : tpc_max_home;
        uint2 *const sq = sq_home;                  // the queue stays the warp's own
        const float T_ = G > 1 ? (float)b.max_steps[e] : T_home;
        const Scale sc = G > 1 ? Scale{T_, __frcp_rn(T_), Nf, __frcp_rn(Nf)} : sc_home;   // (two correctly rounded reciprocals: not per agent)
        // one generic load (address + LD) wherever the entries live; selecting between a typed shared-memory load and a global
        // one per access compiles to a branch with a reconvergence point around every load: 8 instructions instead of 2
        // (-4.7 % of the kernel's instructions, profiles/r02_o_ab.txt)
        auto ent_at = [&](uint32_t i) { return ent[i]; };
        const size_t ea = (size_t)e * N + h;
        const uint32_t ainfo = A.info[h];
        const unsigned slot = (ainfo >> 8) & 0xFFFFu;
        const uint16_t *sd = sdist + (size_t)slot * SS;
        const int n = lane;
        // ---- structure: node n in lane n (treeobs.cpp:171-256 FIFO, 583-608 children) ----
        // Which walk each node stands for, where it ends, parents and evaluation orders follow from the static walk tables and
        // the agent's rail state (cell, direction) alone, and most agents stand where they stood a step ago (95 % of the
        // agent-steps of the benchmark's random-action episodes, fewer under a policy that keeps trains moving): the structure
        // is kept per agent in FlBatch.tree_cache under that state as key — five coalesced loads instead of three
        // ballot/shuffle rounds over the walk records.  Everything that depends on other trains (stages 1 and 2) is computed
        // every step.
        unsigned sid = 0xFFFFu, wx = 0, kunus = 0xFFFFu, dv_end = 0;
        int tot0 = 0, kend = 0, kind = 0, parent = 0, ad = 0, count = 4, order = -2, porder = -2;
        bool onp = false, exists = false, real = false;
        uint32_t *tc = lay.tree_cache ? b.tree_cache + ((size_t)e * N + h) * FL_TREE_CACHE_WORDS : nullptr;
        const uint32_t tkey = 0x80000000u | A.sid0[h];
        bool cached = false;
        uint32_t cw0 = 0;
        if (tc) { cw0 = tc[lane]; cached = __shfl_sync(0xFFFFFFFFu, cw0, 31) == tkey; }
        float tpc_f;                                                                      // rows per cell as treeobs.cpp:304 has it
        if (cached) {                                                                     // warp-uniform
            const uint32_t cw1 = tc[32 + lane], cw2 = tc[64 + lane], cw3 = tc[96 + lane], cw4 = tc[128 + lane];
            tpc_f = __uint_as_float(__shfl_sync(0xFFFFFFFFu, cw1, 31));                   // lane 31 holds no node: its second word keeps the quotient
            sid = cw0 & 0xFFFFu; kend = (int)(cw0 >> 16); wx = cw1; tot0 = (int)cw2;
            kunus = cw3 & 0xFFFFu; dv_end = cw3 >> 16;
            kind = (int)(cw4 & 7u); parent = (int)((cw4 >> 3) & 31u); ad = (int)((cw4 >> 8) & 3u) - 1; onp = (cw4 >> 10) & 1u;
            exists = (cw4 >> 11) & 1u; order = (int)((cw4 >> 12) & 63u) - 2; porder = (int)((cw4 >> 18) & 63u) - 2;
            count = (int)((cw4 >> 24) & 63u);
            if (n == 31) { sid = 0xFFFFu; exists = false; }
            real = n >= 1 && exists && sid != 0xFFFFu;
        } else {
            tpc_f = (float)(1.0 / (double)A.speed[h]);                                    // (a double-precision division: ~60 instructions)
            unsigned c01 = 0xFFFFFFFFu, c2 = 0xFFFFu;
            int level = 0, cb = 1;                                                            // cb: index of the node's first child
            // onp: the node's walk is part of the observer's own predicted path (its cell at distance tot is path element tot),
            // gnx: the state the own path continues in after the node's walk (0xFFFF: it does not)
            unsigned gnx = 0xFFFFu;
            const uint32_t *gt = gtab + (size_t)slot * SS;
            if (n >= 1 && n <= 3) {                                                           // roots (treeobs.cpp:171-221)
                const int vr = (int)(short)(A.vrc[h] & 0xFFFF), vc = (int)(A.vrc[h] >> 16), dir = (int)(ainfo & 3);
                const int nb = (int)((A.rec_b[h] >> 20) & 15u);
                int orientation = dir;
                if (__popc(nb) == 1) orientation = first_dir(nb);
                ad = n - 2;
                const int bd = (orientation + ad) & 3;
                sid = (tbit(nb, bd) ? child_state(ridx, H, W, vr, vc, bd) : 0xFFFFFFFFu) & 0xFFFFu;
                tot0 = 1; level = 1; cb = FL_MAX_NODES;
                const unsigned s0 = A.sid0[h];
                if (sid != 0xFFFFu && s0 != 0xFFFFu && sd[s0] != FL_DIST_INF) {
                    const uint32_t g0 = gt[s0];                                               // how the own path leaves the root cell
                    onp = ((g0 >> 16) & 0x3FFFu) ? true : sid == (g0 & 0xFFFFu);             // along the walk (one child) or into the greedy child
                }
            }
            int ls = 1, le = 4, cur = 1;
            count = 4;
            bool bad = false;
            while (true) {
                const bool real_l = n >= ls && n < le && sid != 0xFFFFu;
                const unsigned lmask = __ballot_sync(0xFFFFFFFFu, real_l);
                if (!lmask) break;
                if (real_l) {
                    const uint4 w = wrec[sid];
                    const int L = (int)(w.y & 0xFFFFu), skind = (int)((w.y >> 16) & 15u), nh = (int)((w.y >> 20) & 255u);
                    kend = L;
                    bool hit = false;
                    if (nh) {                                                    // the observer's own target ends the walk early
                        const uint32_t ho = whoff[sid];
                        for (int q = 0; q < nh; q++) {
                            const uint32_t hv = whits[ho + q];
                            if ((hv >> 16) == slot) { kend = (int)(hv & 0xFFFFu); hit = true; break; }
                        }
                    }
                    kind = hit ? 4 : (skind == WK_BAD ? 3 : skind);
                    if (!hit && skind == WK_BAD) bad = true;                     // treeobs.cpp:527-535 throws
                    wx = w.x; kunus = w.w >> 16; c01 = w.z; c2 = w.w & 0xFFFFu;
                    cb = le + 3 * __popc(lmask & ((1u << n) - 1u));
                    if (onp && !hit) gnx = gt[sid] & 0xFFFFu;
                }
                if (le >= FL_MAX_NODES) break;
                const int nle = min(FL_MAX_NODES, le + 3 * __popc(lmask));
                const bool pull = n >= le && n < nle;
                const int rt = pull ? (n - le) / 3 : 0, j = pull ? (n - le) - 3 * rt : 0;
                if (real_l) cmp_s[__popc(lmask & ((1u << n) - 1u))] = (uint8_t)n;     // r-th real node of the level
                __syncwarp();
                const int p = pull ? (int)cmp_s[rt] : 0;
                __syncwarp();
                const unsigned pz = __shfl_sync(0xFFFFFFFFu, c01, p), pw = __shfl_sync(0xFFFFFFFFu, c2, p);
                const int pk = __shfl_sync(0xFFFFFFFFu, kind, p), ptot = __shfl_sync(0xFFFFFFFFu, tot0 + kend + 1, p);
                const unsigned pg = __shfl_sync(0xFFFFFFFFu, gnx, p);
                if (pull) {
                    unsigned cs = j == 0 ? (pz & 0xFFFFu) : j == 1 ? (pz >> 16) : pw;
                    if (pk > 2) cs = 0xFFFFu;
                    sid = cs; tot0 = ptot; parent = p; ad = j - 1; level = cur + 1; cb = FL_MAX_NODES;
                    onp = cs != 0xFFFFu && cs == pg; gnx = 0xFFFFu;
                }
                ls = le; le = nle; count = nle; cur++;
            }
            if (bad) { if (G > 1) atomicOr(&b.status[e], FL_ST_BAD_CELL); else s_misc[3] = 1; }
            exists = n < count;
            real = n >= 1 && exists && sid != 0xFFFFu;
            // evaluation orders (tool.h:468-524): node_order = height above the leaves, bottom level first
            order = exists ? 0 : -2;
            for (int lev = cur; lev >= 0; lev--) {
                const int c0 = min(cb, 31);
                const int o0 = __shfl_sync(0xFFFFFFFFu, order, c0), o1 = __shfl_sync(0xFFFFFFFFu, order, min(cb + 1, 31)),
                          o2 = __shfl_sync(0xFFFFFFFFu, order, min(cb + 2, 31));
                if (level == lev && (n == 0 || real) && cb < count) {
                    int m = o0;
                    if (cb + 1 < count) m = max(m, o1);
                    if (cb + 2 < count) m = max(m, o2);
                    order = m + 1;
                }
            }
            porder = __shfl_sync(0xFFFFFFFFu, order, parent);
            if (real && kind != 4) dv_end = sd[wlist[wx + kend] & 0xFFFFu];
            if (tc && !bad) {                                                             // (a bad cell keeps raising its status bit)
                tc[lane] = n == 31 ? tkey : (sid & 0xFFFFu) | ((uint32_t)kend << 16);
                tc[32 + lane] = n == 31 ? __float_as_uint(tpc_f) : wx; tc[64 + lane] = (uint32_t)tot0;
                tc[96 + lane] = (kunus & 0xFFFFu) | (dv_end << 16);
                tc[128 + lane] = (uint32_t)kind | ((uint32_t)parent << 3) | ((uint32_t)(ad + 1) << 8) | ((uint32_t)onp << 10) |
                                 ((uint32_t)exists << 11) | ((uint32_t)(order + 2) << 12) | ((uint32_t)(porder + 2) << 18) |
                                 ((uint32_t)count << 24);
            }
        }
        // ---- features: the flat list of the cells of all walks of the agent, 32 cells at a time ----
        const unsigned len = real ? (unsigned)kend + 1u : 0u;
        unsigned total;
        const unsigned off = warp_excl_scan(len, lane, total);
        const unsigned real_mask = __ballot_sync(0xFFFFFFFFu, real);
        const int nreal = __popc(real_mask);
        // lane q holds the q-th real node's (offset, list base, tot0): the owner of a cell is found by rank
        if (real) cmp_s[__popc(real_mask & ((1u << lane) - 1u))] = (uint8_t)lane;
        __syncwarp();
        const unsigned src = lane < nreal ? (unsigned)cmp_s[lane] : 31u;
        __syncwarp();
        const unsigned c_off = __shfl_sync(0xFFFFFFFFu, off, src), c_wb = __shfl_sync(0xFFFFFFFFu, wx, src);
        const unsigned c_t0 = __shfl_sync(0xFFFFFFFFu, (unsigned)tot0 | ((onp ? 1u : 0u) << 31), src);   // bit 31: node on the own path
        const bool c_valid = lane < nreal;
        int k_other = I_INF, k_conf = I_INF, same = 0, opp = 0, malf = 0, rtdn = 0, spd_bits = 0x3F800000;  // min speed starts at 1.0f
        const int my_rank = __popc(real_mask & ((1u << lane) - 1u));
        int qn = 0;                                    // cells waiting in the warp's queue for the full conflict check
        unsigned base = 0;
        while (true) {
            const bool more = base < total;            // warp-uniform
            if (more) {
                // ---- stage 1: one cell per lane: trains on the cell, and the time-slot filter of the prediction index ----
                const unsigned j = base + lane;
                const int cnt0 = __popc(__ballot_sync(0xFFFFFFFFu, c_valid && c_off <= base));
                const unsigned starts = __reduce_or_sync(0xFFFFFFFFu, (c_valid && c_off > base && c_off < base + 32) ? 1u << (c_off - base) : 0u);
                const int rank = cnt0 - 1 + __popc(starts & (0xFFFFFFFFu >> (31 - lane)));
                const unsigned o_off = __shfl_sync(0xFFFFFFFFu, c_off, rank), o_wb = __shfl_sync(0xFFFFFFFFu, c_wb, rank);
                const unsigned o_t0 = __shfl_sync(0xFFFFFFFFu, c_t0, rank);
                bool f_agent = false, f_same = false, f_malf = false, surv = false;
                int my_rtd = 0, my_spd = 0x3F800000, k = 0, pt = 0;
                unsigned sidc = 0;                                                  // state id | transitions nibble << 16
                if (j < total) {
                    k = (int)(j - o_off);
                    sidc = wlist[o_wb + k];
                    const unsigned rail = (sidc & 0xFFFFu) >> 2;
                    const int tot = (int)(o_t0 & 0x7FFFFFFFu) + k;
                    const uint32_t cinfo = ci[rail];
                    if (cinfo) {                   // treeobs.cpp:322-360 (the observer itself counts too)
                        f_agent = true;
                        f_malf = (cinfo >> 8) & 1u;
                        const int cnt = (int)((cinfo >> 11) & 1023u);
                        my_rtd = cnt ? cnt - 1 : 0;
                        f_same = ((cinfo >> 9) & 3u) == (sidc & 3u);
                        if (f_same) my_spd = __float_as_int(A.speed[(cinfo >> 21) - 1]);
                    }
                    pt = (int)__fmul_rn((float)tot, tpc_f);                         // treeobs.cpp:378
                    if (pt < NPRED && tot < NPRED) {                                 // treeobs.cpp:379-465
                        const unsigned bk = kcls ? (unsigned)kcls[rail] : rail;    // the reference's position key c*W + r
                        const int sa = max(0, pt - 1) >> 2, sb = min(NPRED - 1, pt + 1) >> 2;
                        const uint2 wa = bm[bk * 4 + (sa >> 5)], wb = bm[bk * 4 + (sb >> 5)];
                        // On the own path the observer's own entry (path element tot, rows t0o..t1o) is in the index too: a slot it
                        // covers needs a second entry to matter.  (t1o is a lower bound for the last element: errs towards checking.)
                        bool own_a = false, own_b = false;
                        if ((o_t0 >> 31) && tot <= FL_PRED_DEPTH) {
                            const int tpc_i = (int)(ainfo >> 24), t0o = 1 + (tot - 1) * tpc_i, t1o = min(tot * tpc_i, NPRED - 1);
                            if (t0o < NPRED) { own_a = sa >= (t0o >> 2) && sa <= (t1o >> 2); own_b = sb >= (t0o >> 2) && sb <= (t1o >> 2); }
                        }
                        surv = (((own_a ? wa.y : wa.x) >> (sa & 31)) | ((own_b ? wb.y : wb.x) >> (sb & 31))) & 1u;
                    }
                }
                // what the lanes found returns to the lane owning the node: ballots masked by the node's segment of this window
                const unsigned b_agent = __ballot_sync(0xFFFFFFFFu, f_agent);
                if (b_agent) {                                                       // warp-uniform
                    const int lo_ = max((int)off - (int)base, 0), hi_ = min((int)(off + len) - (int)base, 32);
                    const unsigned seg = (real && lo_ < hi_) ? ((hi_ == 32 ? 0xFFFFFFFFu : ((1u << hi_) - 1u)) & ~((1u << lo_) - 1u)) : 0u;
                    const unsigned b_same = __ballot_sync(0xFFFFFFFFu, f_same), b_malf = __ballot_sync(0xFFFFFFFFu, f_malf);
                    const unsigned m = b_agent & seg;
                    if (m) {
                        k_other = min(k_other, (int)base + __ffs(m) - 1 - (int)off);
                        same += __popc(b_same & seg); opp += __popc(m & ~b_same);
                        malf |= (b_malf & seg) != 0u;
                    }
                    // ready-to-depart counts and speeds below 1.0 are rare: to the owner by shuffle
                    for (unsigned mm = __ballot_sync(0xFFFFFFFFu, my_rtd != 0 || my_spd != 0x3F800000); mm; mm &= mm - 1) {
                        const int s = __ffs(mm) - 1;
                        const int r_ = __shfl_sync(0xFFFFFFFFu, my_rtd, s), sp = __shfl_sync(0xFFFFFFFFu, my_spd, s);
                        if ((seg >> s) & 1u) { rtdn += r_; spd_bits = min(spd_bits, sp); }   // positive floats order like their bits
                    }
                }
                // cells that passed the filter go to the queue: state | owner rank << 16 | row << 21, walk step | transitions nibble << 16
                const unsigned b_surv = __ballot_sync(0xFFFFFFFFu, surv);
                if (surv) sq[qn + __popc(b_surv & ((1u << lane) - 1u))] = make_uint2((sidc & 0xFFFFu) | ((unsigned)rank << 16) | ((unsigned)pt << 21), (unsigned)k | (sidc & 0xF0000u));
                qn += __popc(b_surv);
                if (dbg && lane == 0) { atomicAdd(reinterpret_cast<unsigned long long *>(&dbg[12]), (unsigned long long)__popc(b_surv)); atomicAdd(reinterpret_cast<unsigned long long *>(&dbg[13]), 1ull); }
                base += 32;
            }
            if (qn >= 32 || (!more && qn > 0)) {
                // ---- stage 2: the full conflict check (treeobs.cpp:379-465) of up to 32 queued cells, one per lane ----
                // (a flat list of (cell, candidate) pairs over the lanes was measured too: 22.7 instead of 19 active lanes per
                // instruction, but 3 % MORE instructions and the same time — profiles/r02_l_experiments.txt)
                __syncwarp();
                const int nq = min(qn, 32);
                if (dbg && lane == 0) atomicAdd(reinterpret_cast<unsigned long long *>(&dbg[14]), 1ull);
                bool f_conf = false;
                unsigned cases = 0;                                                 // (debug counters, see below)
                uint2 q = make_uint2(0u, 0u);
                if (lane < nq) {
                    q = sq[lane];
                    const unsigned sidc = q.x & 0xFFFFu, rail = sidc >> 2;
                    const int d = (int)(sidc & 3u), pt = (int)(q.x >> 21);
                    const unsigned bk = kcls ? (unsigned)kcls[rail] : rail;
                    const uint32_t s0 = ks[(int)bk - 1], s1 = ks[bk];
                    const int pre = max(0, pt - 1), post = min(NPRED - 1, pt + 1);
                    // Everything that depends on the cell alone is settled before the first entry, so that an entry costs a few
                    // shifts.  m4 below is the entry's rows of the window, shifted left by 2 (bit 2: pt, 3: pre, 4: post).
                    // * Rows: byte k of GE holds the rows at or after t0 = pt - 1 + k, byte k of LE the rows at or before
                    //   t1 = pt + 1 - k; a clamping shift by 8 k with k >= 0 selects the byte (k >= 4 reads 0).  Where the window
                    //   is cut (pt = 0: pre = pt, pt = 500: post = pt) the coinciding rows are set together, as the three separate
                    //   interval tests set them.
                    // * The entry's direction at row pt is dh when the entry covers pt, dpv when its interval starts after pt (it
                    //   then covers post alone, m4 = 16) and dn when it ends before pt (pre alone, m4 = 8): nibble m4 / 4 of PD is
                    //   the bit position of that direction in the entry.  (Its odd neighbour nibbles never reach the low five bits
                    //   that a wrapping shift uses: all entries of PD are even.)
                    // * It crosses the observer when it moves in a direction p != d whose reverse leaves the cell
                    //   (tbit(nb, (p + 2) & 3) is bit p ^ 1 of nb); Xrep repeats that 4-bit mask over the word, so that a
                    //   rotation by any amount whose low two bits are p brings bit p to bit 0.
                    const unsigned nb = (q.y >> 16) & 15u;
                    const unsigned Xrep = (((nb & 5u) << 1 | (nb >> 1 & 5u)) & ~(1u << d)) * 0x11111111u;
                    const uint32_t GE = 0x0010141Cu | (pt == 0 ? 0x0800u : 0u), LE = 0x00080C1Cu | (pt == NPRED - 1 ? 0x1000u : 0u);
                    constexpr uint32_t PD = 0xAAACAEAAu;
                    const int cge = 8 - 8 * pt, cle = 8 * pt + 8;                // GE shift = 8 t0 + cge, LE shift = cle - 8 t1
                    unsigned acc_o = 0, acc_c = 0;                               // m4 of the entries of other agents / of crossing ones
                    auto visit = [&](uint32_t en, uint32_t m4) {
                        const uint32_t pdir = __funnelshift_r(en, 0u, PD >> m4);                    // low two bits: direction
                        or_if(acc_o, m4, (en ^ (uint32_t)h) & 1023u);
                        or_if(acc_c, m4, (__funnelshift_r(Xrep, Xrep, pdir) | en >> 19) & 1u);     // crosses, or its agent is DONE
                    };
                    uint32_t idx = s0;
                    for (; idx < s1; idx++) {                                    // long-lived entries come first: t1 = 500
                        const uint32_t en = ent_at(idx);
                        const int t0 = (int)entry_sort_key(en);
                        if (t0 > post) break;                                    // a regular entry, or none of the rest has started yet
                        visit(en, __funnelshift_rc(GE, 0u, (unsigned)max(8 * t0 + cge, 0)) & 0x1Cu);
                    }
                    if (dbg && idx > s0) cases |= 8u;
                    // regular entries follow, ordered by t0: only those with pre - tpc_max < t0 <= post can matter.  The search runs
                    // on the bucket's sort key (long-lived entries first), so long-lived entries still ahead of idx are skipped too
                    const int t_lo = pre - tpc_max + 1;
                    const uint32_t key_lo = (uint32_t)(512 + max(t_lo, 0));
                    uint32_t lo = idx, hi = s1;
                    while (lo < hi) {
                        const uint32_t mid = (lo + hi) >> 1;
                        if (ent_at(mid) < (key_lo << 22)) lo = mid + 1; else hi = mid;
                    }
                    // Two entries per round, loaded together.  The entries that matter are a prefix (sorted by t0, up to the first t0
                    // past post, which covers no row); the round's second entry is the later one, so it alone decides the break.
                    // Past the bucket's end reads a sentinel entry whose t0 is past every window.
                    constexpr uint32_t PAST = 0xFFC00000u;
                    for (idx = lo;; idx += 2) {
                        uint32_t en2[2];
                        int tpc1[2];                                             // rows per cell - 1
#pragma unroll
                        for (int u = 0; u < 2; u++) {
                            en2[u] = idx + u < s1 ? ent_at(idx + u) : PAST;
                            tpc1[u] = (int)((en2[u] >> 16) & 7u);
                        }
                        if ((en2[0] | en2[1]) & (1u << 20)) {                    // slower than 1/8: rare, kept off the common path
#pragma unroll
                            for (int u = 0; u < 2; u++) tpc1[u] = entry_tpc(en2[u], A.info) - 1;
                            if (dbg) cases |= 16u;
                        }
#pragma unroll
                        for (int u = 0; u < 2; u++) {
                            const uint32_t en = en2[u];
                            const int t0 = (int)entry_sort_key(en) - 512;
                            const int t1 = min(t0 + tpc1[u], t0 << 9);           // element 0 (t0 = 0) is row 0 only
                            visit(en, __funnelshift_rc(GE, 0u, (unsigned)max(8 * t0 + cge, 0)) &
                                      __funnelshift_rc(LE, 0u, (unsigned)max(cle - 8 * t1, 0)) & 0x1Cu);
                        }
                        if ((int)entry_sort_key(en2[1]) > 512 + post) break;
                    }
                    const unsigned acc = acc_o >> 2 | acc_c << 1;            // bits 0-2: rows with another agent, 3-5: crossing
                    if (dbg) cases |= (pt <= 1 ? 1u : 0u) | (pt == NPRED - 1 ? 2u : 0u) | (s1 - s0 > 16 ? 4u : 0u);
                    // treeobs.cpp:379-465: the first of the rows cur, pre, post that holds another agent decides, and it decides
                    // "conflict" when an entry of that row crosses the observer's direction (or belongs to a DONE agent):
                    // (acc & 1) ? (acc & 8) : (acc & 2) ? (acc & 16) : (acc & 4) ? (acc & 32) : false, as a 64-entry bit table
                    f_conf = (bool)((0xfe54ba10ee44aa00ull >> acc) & 1ull);
                }
                if (dbg) {
                    // checks whose window starts at row 0 / ends at row 500, of buckets above 16 entries, that visited long-lived
                    // entries, that met an entry of a train slower than 1/8 (the cases the tests of the conflict check must reach)
                    for (int k = 0; k < 5; k++) {
                        const unsigned m = __ballot_sync(0xFFFFFFFFu, (cases >> k) & 1u);
                        if (lane == 0 && m) atomicAdd(reinterpret_cast<unsigned long long *>(&dbg[26 + k]), (unsigned long long)__popc(m));
                    }
                }
                {
                    // A node keeps the FIRST conflict of its walk.  The queue holds cells in flat-list order (node after node,
                    // walk step after walk step), so the lowest conflicting lane of a node has it: those lanes leave the step in
                    // a 32-word table indexed by node rank (the room of the queue slots just read), the owners pick it up.
                    const unsigned cm = __ballot_sync(0xFFFFFFFFu, f_conf);
                    if (cm) {                                                        // warp-uniform
                        const unsigned myr = (q.x >> 16) & 31u;
                        const unsigned peers = __match_any_sync(0xFFFFFFFFu, f_conf ? myr : 32u + (unsigned)lane);
                        const unsigned rmask = __reduce_or_sync(0xFFFFFFFFu, f_conf ? 1u << myr : 0u);
                        uint32_t *kc = reinterpret_cast<uint32_t *>(sq);
                        if (f_conf && __ffs(peers) - 1 == lane) kc[myr] = q.y & 0xFFFFu;
                        __syncwarp();
                        if (real && ((rmask >> my_rank) & 1u)) k_conf = min(k_conf, (int)kc[my_rank]);
                        __syncwarp();
                    }
                }
                // the rest of the queue moves to the front
                uint2 mv = make_uint2(0u, 0u);
                if (lane + 32 < qn) mv = sq[lane + 32];
                __syncwarp();
                if (lane + 32 < qn) sq[lane] = mv;
                qn -= nq;
                __syncwarp();
            } else if (!more) break;
        }
        // ---- lane n writes node n (scale_node, treeobs.cpp:111-152), its adjacency row and its orders ----
        if (n < FL_MAX_NODES) {
            float4 v0, v1, v2;
            if (n == 0) {
                const float dtv = A.dt[h];
                v0 = make_float4(0.f, 0.f, 0.f, 0.f);
                // (integer-valued operands: div_rn is the IEEE quotient, like every other node feature)
                v1 = make_float4(0.f, 0.f, dtv != INFINITY ? div_rn(dtv, sc.T, sc.rT) : -1.0f, 0.f);
                v2 = make_float4(0.f, div_rn((float)((A.rec_b[h] >> 16) & 1u), sc.N, sc.rN), A.speed[h], 0.f);
            } else if (real) {
                const int tot = tot0 + kend;
                const bool tb = kind == 4;
                int dnb, dmin;
                if (tb) { dnb = tot; dmin = 0; }
                else {
                    dmin = dv_end == FL_DIST_INF ? I_INF : (int)dv_end;
                    dnb = kind == 3 ? I_INF : tot;
                }
                const bool unus = kunus != 0xFFFFu && (int)kunus < kend;
                v0 = make_float4(tb ? scale_i(tot, sc) : -1.0f, -1.0f, k_other != I_INF ? scale_i(tot0 + k_other, sc) : -1.0f,
                                 k_conf != I_INF ? scale_i(tot0 + k_conf, sc) : -1.0f);
                v1 = make_float4(unus ? scale_i(tot0 + (int)kunus, sc) : -1.0f, scale_i(dnb, sc), scale_i(dmin, sc), scale_n(same, sc));
                v2 = make_float4(scale_n(opp, sc), scale_n(malf, sc), __int_as_float(spd_bits), scale_n(rtdn, sc));
            } else {
                v0 = v1 = v2 = make_float4(-1.0f, -1.0f, -1.0f, -1.0f);
            }
            store_node(out_forest + ea * (FL_MAX_NODES * FL_NODE_F) + n * FL_NODE_F, v0, v1, v2);
            out_norder[ea * FL_MAX_NODES + n] = order;
            if (n >= 1) {
                int32_t *adj = out_adj + ea * ((FL_MAX_NODES - 1) * 3) + (n - 1) * 3;
                adj[0] = exists ? parent : -2; adj[1] = exists ? n : -2; adj[2] = exists ? ad : -2;
                out_eorder[ea * (FL_MAX_NODES - 1) + n - 1] = exists ? porder : -2;
            }
        }
    }
    if (G > 1) {                                    // group mode: a warp leaves when no environment of the CTA has an agent left
        if (dbg && lane == 0) for (int k = 5; k <= 7; k++) atomicMax(reinterpret_cast<unsigned long long *>(&dbg[k]), (unsigned long long)clock64());
        return;
    }
    __syncthreads();
    OBS_TICK(5);
    if (tid == 0 && s_misc[3]) atomicOr(&b.status[e], FL_ST_BAD_CELL);
    if (MODE == OBS_TREES) return;
    for (int i = tid; i < N; i += NT) b.deadlocked[(size_t)e * N + i] = D.dl[i];
    OBS_TICK(6);

    // ---- phase 5: the flag entries 0..69 of the agent attributes (feature_parser.cpp:19-77) from the bit masks ---------
    {
        float *dst = out_attr + (size_t)e * N * FL_ATTR_F;
        for (int idx = tid; idx < N * 70; idx += NT) {
            const int i = idx / 70, k = idx - i * 70;
            float v;
            if (k < 64) {
                const uint32_t m = k < 32 ? A.m0[i] : A.m1[i];
                v = (float)((m >> (k & 31)) & 1u);
                if (k == 41) v = D.dl[i] != 0;
            } else {
                const uint32_t ra = A.rec_a[i], rb = A.rec_b[i];
                v = k == 64 ? (float)(rb & 1u) : (float)((ra >> (27 + k - 65)) & 1u);
            }
            dst[i * FL_ATTR_F + k] = v;
        }
    }
    __syncthreads();
    OBS_TICK(7);
#undef OBS_TICK
}

}  // namespace
