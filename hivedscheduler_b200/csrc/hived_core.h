// The scheduling program of the B200-native HiveD hot path (device code; see hived_prims.h for
// the execution model).  It implements, over the flat HBM-resident arrays of hived_dev.h, the
// behaviour of the reference's pkg/algorithm (HivedAlgorithm.Schedule -> intra-VC topology-aware
// search -> buddy-cell virtual->physical mapping -> commit) — each function cites the reference
// lines whose observable behaviour it reproduces.  This is a re-design, not a translation:
//   * cells are ids into SoA arrays; children / leaves of a cell are contiguous id ranges and every
//     cell carries its ancestor per level, so a leaf-to-root walk is ONE warp-wide gather
//     (lane = level) instead of a chain of dependent loads;
//   * per-priority used-leaf maps are not stored: used[q](cell) == #leaves below it with priority q,
//     so a cluster-view node's sort key is recomputed from its leaf priorities with coalesced loads;
//   * free / bad-free / doomed lists keep the reference's order semantics (append, swap-remove) but
//     carry a position index per cell, so contains/remove are O(1) instead of linear scans;
//   * findPhysicalLeafCell's scan over all leaves is a (node, chain) -> leaves table lookup;
//   * the cluster-view pass (key computation, stable counting sort, greedy first-fit) is
//     data-parallel over the whole CTA; the rest runs on the leader warp as SIMT code: uniform
//     control flow, with lanes spread over tree levels, over the children of a cell, over the
//     candidates of a free list and over the leaf cells of a gang;
//   * commit, release and virtual->physical mapping handle a whole gang at once (commitGroupBatched,
//     deleteGroupBatched, mapPlacementBatched): lanes over the gang's leaves, one step per tree level, a
//     rank/select per level replacing the reference's leaf-by-leaf walks; the leaf-by-leaf code remains as the
//     fallback for everything outside their preconditions (preemption, bad cells, pinned cells, recovery);
//   * virtual clusters run on different CTAs and meet only in ordered shared sections (sharedEnter).
// Everything on the leader's per-event path is inlined into the kernel (an out-of-line call costs a spill and
// refill of the live registers); cold generic paths stay out of line behind inlined fast checks.
#pragma once
#include <cstddef>

#include "../../include/hived.h"
#include "hived_dev.h"
#include "hived_prims.h"

namespace hived {

#ifndef HIVED_TOPO_CONSTS
constexpr int MAXL = 16;
constexpr int MAX_NODE_LEAVES = 64;
constexpr int MAX_FANOUT = 64;
#endif

constexpr int MAX_BINS = 4 * (MAX_NODE_LEAVES + 1);
constexpr int MAX_WARPS = 16;  // warps per CTA (hived_cuda.cu launches 512 threads)
constexpr int FREE_PRIO = HIVED_FREE_PRIORITY;
constexpr int OPP_PRIO = HIVED_OPPORTUNISTIC_PRIORITY;
constexpr int PF_AT_OR_ABOVE_NODE_BIT = 1, PF_NODE_LEVEL_BIT = 2, PF_PINNED_BIT = 4;

// shared-memory block of the CTA
// resident mode (Core::serve): slot geometry in 32-bit words
constexpr int SERVE_MAX_EVENTS = 8, SERVE_POOL_WINDOW = 16384, SERVE_EV_OFF = 32, SERVE_SUGG_MAX = 8 * 512, SERVE_AUX_MAX = 8192;
constexpr int SERVE_RES_OFF = SERVE_EV_OFF + SERVE_MAX_EVENTS * 32 + SERVE_SUGG_MAX + SERVE_AUX_MAX;
constexpr int SERVE_DONE_OFF = SERVE_RES_OFF + SERVE_MAX_EVENTS * 32 + SERVE_POOL_WINDOW;
constexpr int SERVE_SLOT_WORDS = SERVE_DONE_OFF + 32;

struct Sm {
  int cmd;  // CMD_*
  // ---- view-pass arguments
  int a_sched, a_prio, a_ignore, a_npods;
  const uint32_t* a_sugg;
  // ---- view-pass results
  int r_ok, r_reason, r_cell;
  // ---- scratch
  int best;
  int cnt[MAX_BINS * MAX_WARPS];
  int part[MAX_WARPS + 32];
  // ---- the current event, fetched with one coalesced 128-byte load
  alignas(16) int32_t ev_words[2][sizeof(hived_event_t) / 4];  // double buffer: the next event arrives while this one runs
  // ---- lean-lane workspace of the leader warp: values per tree level (lane = level) and per bucket
  int lw_va[MAXL], lw_pa[MAXL], lw_vold[MAXL], lw_vpc[MAXL], lw_vc0[MAXL], lw_vn[MAXL], lw_pold[MAXL], lw_pst[MAXL], lw_pvc[MAXL],
      lw_pc0[MAXL], lw_pn[MAXL], lw_pin[MAXL];
  int lw_omaxv[MAXL], lw_omaxp[MAXL], lw_oflagv[MAXL], lw_oflagp[MAXL];
  int un_p[32], un_c[32], un_ls[32];   // planned units: physical cell, commit-time virtual cell, first bound level above
  int un_pl0[32], un_vl0[32], un_node[32];  // ... their first physical / virtual leaf and the view node they will sit in
  int pl_anc[8][32], pl_bnd[8][32];    // planLeanMulti: path and bindings per (level, unit)
  int bkc_sched;              // the view whose bucket heads are cached below (-1: none)
  int bkc_head[BK_STRIDE];
  int own_win[64];            // window of the CTA's event-index list
  // the small scratch arrays of a decision that are read back right after they are written (a global store does not
  // allocate in L1: reading it back is a round trip to L2) live here when the group sizes allow (LS <= 64, PS <= 16)
  int32_t sc_pl_v[64], sc_pl_p[64], sc_pl_v2[64], sc_pl_p2[64], sc_pod_need[16], sc_pod_pos[16], sc_pod_cell[16], sc_pod_unit[16];
  int stop_k;                 // multi-GPU partition: index (in the CTA's list) of the event the CTA stopped before; nOwn when done
  int lead_k;                 // index (in the CTA's list) of the event the leader works on; 0x7fffffff when it is done
  // ---- written back at kernel exit
  int panic;
  long long pool_off;
};
#if defined(__CUDACC__) && !defined(HIVED_SIMT_EMU) && !defined(HIVED_EMU)
__shared__ Sm g_hived_sm;  // one per CTA (both kernels of hived_cuda.cu use it)
// The device's view of the scheduler state (array pointers and sizes, hived_dev.h) lives in the CONSTANT bank: `d.p_prio[i]`
// is one load whose base address is an instruction operand (c[3][offset]).  Through a `const Dev&` member the
// compiler fetched the pointer with a generic load (LD.E.64) before nearly every data load — a dependent L1 round trip
// on the leader warp's critical path and a third of its memory instructions (profiles/r2_sass_summary.md).  One
// context's Dev is loaded per device at a time; launchProgram / the per-call path reload it when the owner changes
// (hived_cuda.cu: ensureDevLoaded).
__constant__ Dev g_hived_dev;
#define HIVED_DEV_IN_CONSTANT 1
#endif

enum { CMD_IDLE = 0, CMD_VIEW = 1, CMD_EXIT = 2 };

// uniform store: every lane of the (converged) leader warp writes the same value
#ifdef HIVED_SIMT_EMU
// the functional emulator runs the lanes of a warp one after the other between two collectives: a uniform
// read-modify-write is made phase-correct by finishing every lane's reads (value evaluated, barrier) before the write
#define ST(lvalue, val) do { auto st_v_ = (val); hv_phase(); (lvalue) = st_v_; } while (0)
#else
#define ST(lvalue, val) ((lvalue) = (val))
#endif

struct Core {
#ifdef HIVED_DEV_IN_CONSTANT
#define d g_hived_dev  /* (until the end of this header) */
#else
  const Dev& d;
#endif
#if defined(__CUDACC__) && !defined(HIVED_SIMT_EMU) && !defined(HIVED_EMU)
  // the CTA's shared block is ONE file-scope __shared__ object: every access compiles to LDS / STS / ATOMS (through a
  // generic Sm* the compiler loses the address space as soon as `this` goes through memory: LD.E / ATOM.E)
  HIVED_DEV static Sm* smp() { return &g_hived_sm; }
#else
  Sm* sm_;
  Sm* smp() const { return sm_; }
#endif
  const uint32_t* sugg;  // suggested-node bitmap of the current event (nullptr = every node)
  int32_t* pool;
  long long pool_cap;
  long long poolOff;
  int panicCode;  // sticky platform-error code of the current event
  const int lane;
  const int AS;
  Scratch s;                // this CTA's private scratch arrays
  // ---- VC-parallel execution (several CTAs, one per group of VCs; see run())
  const int cta, nCta;
  bool multi;
  // multi-GPU partition (hived_multigpu.h): 0 off; 1 this CTA runs its VCs' events up to the first one that may touch
  // the cluster-wide state and stops BEFORE it (nothing of that event is written); 2 one such event, alone on the
  // cluster (every other CTA of every rank is parked), the cluster-wide state being this rank's to write
  int mgMode = 0, mgStart = 0;
  bool mgStop = false;
  int curEvent;      // index (in the batch) of the event being processed
  bool sharedHeld;   // this event already holds the right to touch the cluster-wide free-list state

  HIVED_DEV Core(const Dev& dev, Sm* s_, int32_t* pool_, long long cap, int nCta_)
      :
#ifndef HIVED_DEV_IN_CONSTANT
        d(dev),
#endif
#if !(defined(__CUDACC__) && !defined(HIVED_SIMT_EMU) && !defined(HIVED_EMU))
        sm_(s_),
#endif
        sugg(nullptr), pool(pool_), pool_cap(cap), poolOff(0), panicCode(0), lane(hv_lane()), AS(dev.S.AS),
        s(dev.scratch[hv_cta()]), cta(hv_cta()), nCta(nCta_), multi(nCta_ > 1), curEvent(0), sharedHeld(false), prioMask(0) {
    for (int i = 0; i < N_WORK; i++) work[i] = 0;
    for (int i = 0; i < PC_COUNT; i++) pathCnt[i] = 0;
    if (dev.S.LS <= 64 && dev.S.PS <= 16) {
      s.pl_v = smp()->sc_pl_v; s.pl_p = smp()->sc_pl_p; s.pl_v2 = smp()->sc_pl_v2; s.pl_p2 = smp()->sc_pl_p2;
      s.pod_need = smp()->sc_pod_need; s.pod_pos = smp()->sc_pod_pos; s.pod_cell = smp()->sc_pod_cell; s.pod_unit = smp()->sc_pod_unit;
    }
  }

  // Multi-CTA ordering.  VCs are partitioned over the CTAs; an event only touches its VC's virtual
  // tree and the physical cells bound into it, EXCEPT for the chain-wide free lists / counters used
  // when a preassigned cell is bound or released.  Those sections run in batch order: a CTA enters
  // one only when every other CTA is already working on a later event (so all earlier events are
  // complete), and later events that need the shared state wait for this one the same way.
  HIVED_DEV void sharedEnter() {
    if (!multi || sharedHeld) return;
    if (mgMode == 2) { sharedHeld = true; stat_add(ST_SHARED_SECTIONS, 1); return; }
    if (mgMode == 1) { panic(HIVED_ERR_PLATFORM); return; }  // (unreachable: such an event stops before it starts)
    sharedEnterSlow();
  }
  HIVED_DEV void setMultiGpu(int mode, int start) { mgMode = mode; mgStart = start; if (mode) multi = true; }
  HIVED_DEV_NOINLINE void sharedEnterSlow() {
    long long tw0 = pclock();
    while (true) {
      int mn = 0x7fffffff;
      for (int b = 0; b < nCta; b += HIVED_WARPSZ) {
        int i = b + lane;
        if (i < nCta && i != cta) { int v = hv_ld_volatile(d.progress + i); if (v < mn) mn = v; }
      }
      mn = hv_reduce_min(mn);
      if (mn > curEvent) break;
    }
    hv_fence();  // acquire: drop stale L1 lines of state written by the other CTAs
    stat_add(ST_CYC_WAIT, pclock() - tw0);
    stat_add(ST_SHARED_SECTIONS, 1);
    sharedHeld = true;
  }
  // highest physical level an event of this VC may write: in multi-CTA mode the cells above the
  // physical cell bound to the virtual leaf's preassigned cell are shared between VCs; their
  // priority/state (never read by a decision) are re-derived after the batch (repairSharedAncestors)
  HIVED_DEV int ceilOf(int vLeaf) const { return (multi && vLeaf >= 0) ? d.v_prelevel[vLeaf] : AS; }

  // ======================================================================================
  // warp-level building blocks (leader warp; with HIVED_WARPSZ == 1 they degenerate to loops)
  // ======================================================================================
  // bit l (lo <= l < hi <= 32) set iff pred(l)
  template <typename F>
  HIVED_DEV unsigned levelMask(int lo, int hi, F pred) const {
    unsigned m = 0;
    for (int b = 0; b < hi; b += HIVED_WARPSZ) {
      int l = b + lane;
      bool p = l >= lo && l < hi && pred(l);
      m |= hv_ballot(p) << b;
    }
    return m;
  }
  // smallest i in [0,n) with pred(i), else -1
  template <typename F>
  HIVED_DEV int firstIdx(int n, F pred) const {
    for (int b = 0; b < n; b += HIVED_WARPSZ) {
      int i = b + lane;
      unsigned m = hv_ballot(i < n && pred(i));
      if (m) return b + hv_ffs(m) - 1;
    }
    return -1;
  }
  template <typename F>
  HIVED_DEV int maxOver(int n, F val, int init) const {
    int v = init;
    for (int b = 0; b < n; b += HIVED_WARPSZ) {
      int i = b + lane;
      if (i < n) { int x = val(i); if (x > v) v = x; }
    }
    v = hv_reduce_max(v);
    return v;
  }

  // ---- scans over the children of one cell per lane (whole-gang steps).  All lanes call; `act` lanes hold a cell,
  // lanes that share a cell get the same answer.  Two strategies, chosen per call by a cost estimate: every lane
  // walks its own cell's children (one dependent round trip, n serial iterations of a single warp), or one
  // warp-wide pass (lane = child) per DISTINCT cell (D round trips, no serial loop).
  HIVED_DEV bool preferCooperative(bool act, int cell, int n, unsigned& heads) const {
    // cooperative passes pay one round trip per distinct cell, the per-lane walk n serial iterations: wide cells
    // (racks, pods: few distinct ones per gang) go cooperative, narrow ones (nodes: up to one per lane) per lane
    (void)cell;
    heads = hv_ballot(act);
    return hv_reduce_max(act ? n : 0) > 8;
  }
  // V: max v_prio and "some child is bound";  !V: max p_prio and "some child is not Free"
  template <bool V>
  HIVED_DEV void childrenSummary(bool act, int cell, int& mx, bool& flag) const {
    const int32_t* prio = V ? d.v_prio : d.p_prio;
    const int32_t* other = V ? d.v_pcell : d.p_state;
    const int c0 = act ? (V ? d.v_child0[cell] : d.p_child0[cell]) : 0;
    const int n = act ? (V ? d.v_nchild[cell] : d.p_nchild[cell]) : 0;
    mx = FREE_PRIO; flag = false;
    unsigned heads;
    if (preferCooperative(act, cell, n, heads)) {
      for (unsigned todo = heads; todo;) {  // one pass per distinct cell: the first pending lane names it
        const int src = hv_ffs(todo) - 1;
        const int gc0 = hv_shfl(c0, src), gn = hv_shfl(n, src), gcell = hv_shfl(cell, src);
        todo &= ~hv_ballot(act && cell == gcell);
        int m = FREE_PRIO; bool f = false;
        for (int b = 0; b < gn; b += HIVED_WARPSZ) {
          int j = b + lane;
          if (j < gn) {
            int q = prio[gc0 + j]; if (q > m) m = q;
            int o = other[gc0 + j]; if (V ? o >= 0 : o != HIVED_CELL_FREE) f = true;
          }
        }
        m = hv_reduce_max(m);
        f = hv_ballot(f) != 0;
        if (act && cell == gcell) { mx = m; flag = f; }
      }
    } else if (act) {
#pragma unroll 4
      for (int j = 0; j < n; j++) {
        int q = prio[c0 + j]; if (q > mx) mx = q;
        int o = other[c0 + j]; if (V ? o >= 0 : o != HIVED_CELL_FREE) flag = true;
      }
    }
  }
  // the (want)-th child of virtual cell pv that is free and unbound (cell_allocation.go:348-372, first branch), or -1
  HIVED_DEV int selectFreeUnboundChild(bool act, int pv, int want) const {
    const int c0 = act ? d.v_child0[pv] : 0, n = act ? d.v_nchild[pv] : 0;
    int sel = -1;
    unsigned heads;
    if (preferCooperative(act, pv, n, heads)) {
      for (unsigned todo = heads; todo;) {
        const int src = hv_ffs(todo) - 1;
        const int gc0 = hv_shfl(c0, src), gn = hv_shfl(n, src), gpv = hv_shfl(pv, src);
        todo &= ~hv_ballot(act && pv == gpv);
        int before = 0;
        for (int b = 0; b < gn; b += HIVED_WARPSZ) {
          int j = b + lane;
          unsigned fm = hv_ballot(j < gn && d.v_prio[gc0 + j] == FREE_PRIO && d.v_pcell[gc0 + j] < 0);
          int cnt = hv_popc(fm);
          if (act && pv == gpv && want >= before && want < before + cnt) sel = gc0 + b + hv_fns(fm, want - before);
          before += cnt;
        }
      }
    } else if (act) {
      int cnt = 0;
#pragma unroll 4
      for (int j = 0; j < n; j++) {
        bool fr = d.v_prio[c0 + j] == FREE_PRIO && d.v_pcell[c0 + j] < 0;
        if (fr && cnt == want) sel = c0 + j;
        cnt += fr ? 1 : 0;
      }
    }
    return sel;
  }
  // the (want)-th unbound child of physical cell pp, or -1; unusable: some unbound child is bad or opportunistically used
  HIVED_DEV int selectUnboundPhysChild(bool act, int pp, int want, bool& unusable) const {
    const int c0 = act ? d.p_child0[pp] : 0, n = act ? d.p_nchild[pp] : 0;
    int sel = -1;
    bool bad = false;
    unsigned heads;
    if (preferCooperative(act, pp, n, heads)) {
      for (unsigned todo = heads; todo;) {
        const int src = hv_ffs(todo) - 1;
        const int gc0 = hv_shfl(c0, src), gn = hv_shfl(n, src), gpp = hv_shfl(pp, src);
        todo &= ~hv_ballot(act && pp == gpp);
        int before = 0;
        for (int b = 0; b < gn; b += HIVED_WARPSZ) {
          int j = b + lane;
          bool unbound = j < gn && d.p_vcell[gc0 + j] < 0;
          if (unbound && (!d.p_healthy[gc0 + j] || d.p_usedopp[gc0 + j] != 0)) bad = true;
          unsigned um = hv_ballot(unbound);
          int cnt = hv_popc(um);
          if (act && pp == gpp && want >= before && want < before + cnt) sel = gc0 + b + hv_fns(um, want - before);
          before += cnt;
        }
      }
    } else if (act) {
      int cnt = 0;
#pragma unroll 4
      for (int j = 0; j < n; j++) {
        bool unbound = d.p_vcell[c0 + j] < 0;
        if (unbound && (!d.p_healthy[c0 + j] || d.p_usedopp[c0 + j] != 0)) bad = true;
        if (unbound && cnt == want) sel = c0 + j;
        cnt += unbound ? 1 : 0;
      }
    }
    unusable = hv_ballot(bad) != 0;
    return sel;
  }

  // ======================================================================================
  // small helpers
  // ======================================================================================
  HIVED_DEV void panic(int code) { if (panicCode == 0) panicCode = code; }
  HIVED_DEV bool node_suggested(int node) const {
    if (sugg == nullptr) return true;
    if (node < 0) return false;
    return (sugg[node >> 5] >> (node & 31)) & 1u;
  }
  // Work counters (ST_VIEW_NODES .. ST_PRIO_MASK): accumulated per CTA in 32-bit slots and added to d.stats when the
  // batch ends (a batch is far below 2^31 of anything).  The SM-cycle counters (ST_CYC_* and the scratch ST_DBG*)
  // exist only in profiling builds (-DHIVED_PROFILE): in the product neither the clock reads nor the updates are
  // compiled in — they were 6 % of the leader warp's time.
  static constexpr int N_WORK = ST_PRIO_MASK;  // counters [0, N_WORK) are the work counters
  int work[N_WORK];
  int pathCnt[PC_COUNT];  // which path the events took (ST_PATH0 + PC_*)
  unsigned long long prioMask;
  HIVED_DEV void path_add(int which, int v = 1) { pathCnt[which] += v; }
#ifdef HIVED_PROFILE
  HIVED_DEV long long pclock() const { return hv_clock(); }
  HIVED_DEV void stat_add(int which, long long v) {
    if (which < N_WORK) work[which] += (int)v;
    else if (lane == 0) hv_atomic_add64(&d.stats[which], v);
  }
  HIVED_DEV void dbg(int k, long long& t) { long long n = pclock(); stat_add(ST_DBG0 + k, n - t); t = n; }
#else
  HIVED_DEV long long pclock() const { return 0; }
  HIVED_DEV void stat_add(int which, long long v) { if (which < N_WORK) work[which] += (int)v; }
  HIVED_DEV void dbg(int, long long&) {}
#endif
  HIVED_DEV void flushWork() {
    if (lane == 0) {
      for (int i = 0; i < N_WORK; i++) if (work[i]) hv_atomic_add64(&d.stats[i], work[i]);
      for (int i = 0; i < PC_COUNT; i++) if (pathCnt[i]) hv_atomic_add64(&d.stats[ST_PATH0 + i], pathCnt[i]);
      if (prioMask) hv_atomic_or64(&d.stats[ST_PRIO_MASK], (long long)prioMask);
    }
    for (int i = 0; i < N_WORK; i++) work[i] = 0;
    for (int i = 0; i < PC_COUNT; i++) pathCnt[i] = 0;
    prioMask = 0;
    hv_warp_sync();
  }
  HIVED_DEV int cl(int chain, int level) const { return chain * MAXL + level; }
  HIVED_DEV int vcl(int vc, int chain, int level) const { return (vc * d.S.nChains + chain) * MAXL + level; }

  // ---- free list of the physical cluster: order semantics of types.go:78-95 (swap-remove) and append.
  // (read everything, re-converge, then write: a lane must not see another lane's update of the length)
  // The reference's list is a slice and nothing stops it from holding a cell twice (a preassigned cell released again
  // while it is already free): p_flpos is the position of a cell's FIRST occurrence (what CellList.remove finds), fl_dup
  // counts the later occurrences of a segment; while a segment has none the position table is exact and O(1).
  HIVED_DEV void fl_append(int chain, int level, int cell) {
    int k = cl(chain, level);
    int n = d.fl_len[k];
    if (n >= d.fl_cap[k]) { panic(HIVED_ERR_CAPACITY); return; }  // more duplicates than FL_DUP_SLACK (hived_topo.hpp)
    const int first = d.p_flpos[cell];
    const int dups = d.fl_dup[k];
    hv_warp_sync();
    ST(d.fl_data[d.fl_base[k] + n], cell);
    if (first < 0) ST(d.p_flpos[cell], n); else ST(d.fl_dup[k], dups + 1);
    ST(d.fl_len[k], n + 1);
  }
  HIVED_DEV void fl_remove(int chain, int level, int cell) {
    int k = cl(chain, level);
    int pos = d.p_flpos[cell];
    if (pos < 0) { panic(HIVED_ERR_PLATFORM); return; }  // "Cell not not found in list when removing"
    int n = d.fl_len[k];
    int last = d.fl_data[d.fl_base[k] + n - 1];
    const int dups = d.fl_dup[k];
    hv_warp_sync();
    ST(d.fl_data[d.fl_base[k] + pos], last);
    ST(d.fl_len[k], n - 1);
    if (dups == 0) {
      ST(d.p_flpos[last], pos);
      ST(d.p_flpos[cell], -1);
      return;
    }
    // the segment holds duplicates: first occurrences and their number again, in list order (uniform, short lists)
    int32_t* a = d.fl_data + d.fl_base[k];
    ST(d.p_flpos[cell], -1);
    for (int i = 0; i < n - 1; i++) ST(d.p_flpos[a[i]], -1);
    int nd = 0;
    for (int i = 0; i < n - 1; i++) {
      const int c = a[i];
      if (d.p_flpos[c] < 0) ST(d.p_flpos[c], i); else nd++;
    }
    ST(d.fl_dup[k], nd);
  }
  HIVED_DEV bool fl_contains(int cell) const { return d.p_flpos[cell] >= 0; }
  // ---- bad free cells (badFreeCells, hived_algorithm.go:78)
  // Its segment has the free list's capacity (fl_cap).  A cell can be listed only once here (p_bfpos is its position):
  // a second append — the reference's slice would take it — and an append to a full segment report HIVED_ERR_CAPACITY
  // instead of writing into the neighbouring segment.
  HIVED_DEV void bf_append(int chain, int level, int cell) {
    int k = cl(chain, level);
    int n = d.bf_len[k];
    if (n >= d.fl_cap[k] || d.p_bfpos[cell] >= 0) { panic(HIVED_ERR_CAPACITY); return; }
    hv_warp_sync();
    ST(d.bf_data[d.fl_base[k] + n], cell);
    ST(d.p_bfpos[cell], n);
    ST(d.bf_len[k], n + 1);
  }
  HIVED_DEV void bf_remove(int chain, int level, int cell) {
    int k = cl(chain, level);
    int pos = d.p_bfpos[cell];
    if (pos < 0) { panic(HIVED_ERR_PLATFORM); return; }
    int n = d.bf_len[k];
    int last = d.bf_data[d.fl_base[k] + n - 1];
    hv_warp_sync();
    ST(d.bf_data[d.fl_base[k] + pos], last);
    ST(d.p_bfpos[last], pos);
    ST(d.p_bfpos[cell], -1);
    ST(d.bf_len[k], n - 1);
  }
  // ---- doomed bad cells of a VC (vcDoomedBadCells, hived_algorithm.go:80)
  // The reference's list keeps STALE entries: a doomed bad cell that a pod used is unbound when the pod leaves
  // (releaseLeafCell unbinds it but skips releasePreassignedCell because the cell is still listed), its virtual cell can
  // be bound to another bad cell, and the list outgrows the VC's preassigned cells (synthetic fuzz seed 2098).  The
  // segment has room for DM_STALE_SLACK such entries (hived_topo.hpp); beyond that, or for a cell that is already on a
  // doomed bad list (p_dmpos / p_dmvc hold one position per cell), the call reports HIVED_ERR_CAPACITY.
  HIVED_DEV void dm_append(int vc, int chain, int level, int cell) {
    int k = vcl(vc, chain, level);
    int n = d.dm_len[k];
    if (n >= d.dm_cap[k] || d.p_dmpos[cell] >= 0) { panic(HIVED_ERR_CAPACITY); return; }
    hv_warp_sync();
    ST(d.dm_data[d.dm_base[k] + n], cell);
    ST(d.p_dmpos[cell], n);
    ST(d.p_dmvc[cell], vc);
    ST(d.dm_len[k], n + 1);
  }
  HIVED_DEV void dm_remove(int vc, int chain, int level, int cell) {
    int k = vcl(vc, chain, level);
    int pos = d.p_dmpos[cell];
    if (pos < 0 || d.p_dmvc[cell] != vc) { panic(HIVED_ERR_PLATFORM); return; }
    int n = d.dm_len[k];
    int last = d.dm_data[d.dm_base[k] + n - 1];
    hv_warp_sync();
    ST(d.dm_data[d.dm_base[k] + pos], last);
    ST(d.p_dmpos[last], pos);
    ST(d.p_dmpos[cell], -1);
    ST(d.p_dmvc[cell], -1);
    ST(d.dm_len[k], n - 1);
  }
  HIVED_DEV bool dm_contains(int vc, int cell) const { return d.p_dmpos[cell] >= 0 && d.p_dmvc[cell] == vc; }

  // ======================================================================================
  // cell primitives
  // ======================================================================================
  // utils.go:381-391
  HIVED_DEV bool inFreeCellList(int c) const {
    while (true) {
      if (d.p_vcell[c] >= 0 || d.p_split[c]) return false;
      int par = d.p_parent[c];
      if (par < 0 || d.p_split[par]) return true;
      c = par;
    }
  }
  // cell.go:195-204 + utils.go:397-415.  Used propagates unconditionally: one gather over the levels.
  HIVED_DEV_NOINLINE void setCellState(int c, int s, int ceil = 1 << 20) {
    hv_phase();
    if (s == HIVED_CELL_USED) {
      for (int b = 0; b < AS; b += HIVED_WARPSZ) {
        int l = b + lane;
        if (l < AS && l <= ceil) {
          int a = d.p_anc[c * AS + l];
          if (a >= 0) {
            d.p_state[a] = HIVED_CELL_USED;
            int v = d.p_vcell[a];
            if (v >= 0) d.v_state[v] = HIVED_CELL_USED;
          }
        }
      }
      hv_warp_sync();
      return;
    }
    while (true) {
      ST(d.p_state[c], s);
      int vc = d.p_vcell[c];
      if (vc >= 0) ST(d.v_state[vc], s);
      int par = d.p_parent[c];
      if (par < 0 || d.p_level[c] >= ceil) return;
      int c0 = d.p_child0[par], n = d.p_nchild[par];
      if (firstIdx(n, [&](int i) { return d.p_state[c0 + i] != s; }) >= 0) return;
      c = par;
    }
  }
  // cell_allocation.go:422-441.  A raise (p above the cell's priority) is max(old, p) on every
  // ancestor independently, because a parent's priority is the max of its children's.
  template <bool V>
  HIVED_DEV_NOINLINE void setPriority(int c, int p, int ceil = 1 << 20) {
    if (V) bkMarkLeaf(c);  // the key of the view node above this virtual leaf changes
    int32_t* prio = V ? d.v_prio : d.p_prio;
    const int32_t* anc = V ? d.v_anc : d.p_anc;
    const int32_t* parent = V ? d.v_parent : d.p_parent;
    const int32_t* child0 = V ? d.v_child0 : d.p_child0;
    const int32_t* nchild = V ? d.v_nchild : d.p_nchild;
    const bool raise = p > prio[c];
    hv_phase();
    if (raise) {
      for (int b = 0; b < AS; b += HIVED_WARPSZ) {
        int l = b + lane;
        if (l < AS && l <= ceil) {
          int a = anc[c * AS + l];
          if (a >= 0 && prio[a] < p) prio[a] = p;
        }
      }
      hv_warp_sync();
      return;
    }
    while (true) {
      int orig = prio[c];
      ST(prio[c], p);
      int par = parent[c];
      if (par < 0 || (V ? d.v_level[c] : d.p_level[c]) >= ceil) return;
      int pp = prio[par];
      if (p > pp) { c = par; continue; }
      if (orig == pp && p < orig) {
        int c0 = child0[par];
        int mx = maxOver(nchild[par], [&](int i) { return prio[c0 + i]; }, FREE_PRIO);
        c = par;
        p = mx;
        continue;
      }
      return;
    }
  }
  // cell_allocation.go:443-454 — only the opportunistic count of physical cells is ever read back
  // (getUsablePhysicalCells :238-241); every other used[] value is recomputed from leaf priorities.
  HIVED_DEV_NOINLINE void updateUsedOpp(int c, int delta) {
    sharedEnter();  // the counts of the upper cells are read by every VC's buddy allocation
    hv_phase();
    for (int b = 0; b < AS; b += HIVED_WARPSZ) {
      int l = b + lane;
      if (l < AS) {
        int a = d.p_anc[c * AS + l];
        if (a >= 0) d.p_usedopp[a] += delta;
      }
    }
    hv_warp_sync();
  }
  // cell.go:264-277, 401-419
  HIVED_DEV void bindPair(int pc, int vc) {
    ST(d.p_vcell[pc], vc);
    ST(d.v_pcell[vc], pc);
    ST(d.v_healthy[vc], d.p_healthy[pc]);
  }
  HIVED_DEV void unbindPair(int pc, int vc) {
    ST(d.p_vcell[pc], -1);
    ST(d.v_pcell[vc], -1);
    ST(d.v_state[vc], HIVED_CELL_FREE);
    ST(d.v_healthy[vc], 1);
  }
  // cell_allocation.go:384-397: binds the unbound run of ancestors starting at (pc, vc)
  HIVED_DEV_NOINLINE void bindCell(int pc, int vc) {
    int lv = d.v_level[vc];
    unsigned stopMask = levelMask(lv, AS, [&](int l) {
      int va = d.v_anc[vc * AS + l];
      return va < 0 || d.v_pcell[va] >= 0;
    });
    int stop = stopMask ? hv_ffs(stopMask) - 1 : AS;
    for (int b = 0; b < stop; b += HIVED_WARPSZ) {
      int l = b + lane;
      if (l >= lv && l < stop) {
        int va = d.v_anc[vc * AS + l], pa = d.p_anc[pc * AS + l];
        d.p_vcell[pa] = va;
        d.v_pcell[va] = pa;
        d.v_healthy[va] = d.p_healthy[pa];
      }
    }
    hv_warp_sync();
  }
  // cell_allocation.go:399-420
  HIVED_DEV_NOINLINE void unbindCell(int c) {
    int bv = d.p_vcell[c];
    while (!(d.p_flags[d.v_pcell[bv]] & PF_PINNED_BIT)) {
      int bp = d.v_pcell[bv];
      unbindPair(bp, bv);
      int par = d.v_parent[bv];
      if (par < 0) return;
      int c0 = d.v_child0[par];
      if (firstIdx(d.v_nchild[par], [&](int i) { return d.v_pcell[c0 + i] >= 0; }) >= 0) return;
      bv = par;
    }
  }
  // cell_allocation.go:374-382 over a contiguous child range
  HIVED_DEV int unboundChild(int vparent) const {
    int c0 = d.v_child0[vparent];
    int i = firstIdx(d.v_nchild[vparent], [&](int j) { return d.v_pcell[c0 + j] < 0; });
    return i < 0 ? -1 : c0 + i;
  }

  // ======================================================================================
  // bad cells, doomed bad cells, preassigned cell (de)allocation  (hived_algorithm.go:466-653, 1354-1565)
  // ======================================================================================
  // hived_algorithm.go:1502-1527
  HIVED_DEV_NOINLINE int removeCellFromFreeList(int c) {
    int chain = d.p_chain[c];
    while (true) {
      int l = d.p_level[c];
      int par = d.p_parent[c];
      bool terminate = false;
      if (par >= 0) {
        if (d.p_split[par]) {
          terminate = true;
        } else {
          int c0 = d.p_child0[par], n = d.p_nchild[par];
          for (int i = 0; i < n; i++) fl_append(chain, l, c0 + i);
          ST(d.p_split[par], 1);
        }
      } else {
        terminate = true;
      }
      fl_remove(chain, l, c);
      if (terminate) return l;
      c = par;
    }
  }
  // hived_algorithm.go:1529-1565
  HIVED_DEV_NOINLINE int addCellToFreeList(int c) {
    int chain = d.p_chain[c];
    while (true) {
      int l = d.p_level[c];
      int par = d.p_parent[c];
      bool terminate = false;
      if (par >= 0) {
        int c0 = d.p_child0[par], n = d.p_nchild[par];
        bool allBuddyFree = firstIdx(n, [&](int i) { return c0 + i != c && d.p_flpos[c0 + i] < 0; }) < 0;
        if (!allBuddyFree) {
          terminate = true;
        } else {
          for (int i = 0; i < n; i++)
            if (c0 + i != c) fl_remove(chain, l, c0 + i);
          ST(d.p_split[par], 0);
        }
      } else {
        terminate = true;
      }
      if (terminate) { fl_append(chain, l, c); return l; }
      c = par;
    }
  }

  // ---- allocate/releasePreassignedCell and tryBind/tryUnbindDoomedBadCell call each other in the reference
  // (hived_algorithm.go:602-653, 1354-1485): binding a doomed bad cell allocates it as a preassigned cell, which may
  // leave another level short of healthy cells, and so on.  Every nested call is a doomed-bad one and only looks at
  // levels ABOVE its own, so the nesting is bounded by the height of the chain; the four functions are templates on
  // the nesting depth D (the call graph is a finite DAG, the device stack stays statically sized) and a cascade deeper
  // than DOOM_DEPTH reports HIVED_ERR_CAPACITY.  D > 0 implies doomedBad.
  static constexpr int DOOM_DEPTH = 6;  // nested calls go strictly up the chain: enough for chains of 7 levels (C3 has 5, the design config 7)
  HIVED_DEV void tryBindDoomedBadCell(int chain, int l) { tryBindDoomedBadCellT<0>(chain, l); }
  HIVED_DEV void tryUnbindDoomedBadCell(int chain, int l) { tryUnbindDoomedBadCellT<0>(chain, l); }
  HIVED_DEV bool allocatePreassignedCell(int c, int vc, bool doomedBad) { return allocatePreassignedCellT<0>(c, vc, doomedBad); }
  HIVED_DEV void releasePreassignedCell(int c, int vc, bool doomedBad) { releasePreassignedCellT<0>(c, vc, doomedBad); }
  // hived_algorithm.go:602-628 (VCs in ascending id order)
  template <int D>
  HIVED_DEV_NOINLINE void tryBindDoomedBadCellT(int chain, int l) {
    int k = cl(chain, l);
    // no VC is short of healthy cells (lane = VC: the largest vcFree decides; the sum allVCFree is no bound once a
    // safety violation has driven some VC's count negative)
    {
      const int room = d.totalLeft[k] - d.bf_len[k];
      int mx = -0x7fffffff;
      for (int b = 0; b < d.S.nVCs; b += HIVED_WARPSZ) {
        const int vc = b + lane;
        if (vc < d.S.nVCs && d.vc_chain_counter[vc * d.S.nChains + chain]) { const int f = d.vcFree[vcl(vc, chain, l)]; if (f > mx) mx = f; }
      }
      if (hv_reduce_max(mx) <= room) return;
    }
    for (int vc = 0; vc < d.S.nVCs; vc++) {
      if (!d.vc_chain_counter[vc * d.S.nChains + chain]) continue;
      int kv = vcl(vc, chain, l);
      int guard = 0;
      while (d.vcFree[kv] > d.totalLeft[k] - d.bf_len[k]) {
        if (d.bf_len[k] <= 0) { panic(HIVED_ERR_PLATFORM); return; }  // badFreeCells[c][l][0] of an empty slice in the reference
        // a device limit, not the reference's: it would go on binding (one bad free cell per round, each leaves the list)
        if (++guard > d.S.NP) { panic(HIVED_ERR_CAPACITY); return; }
        int pc = d.bf_data[d.fl_base[k] + 0];
        const int32_t* pre = d.pre_list + d.pre_off[kv];
        int idx = firstIdx(d.pre_cnt[kv], [&](int i) { return d.v_pcell[pre[i]] < 0; });
        if (idx < 0) { panic(HIVED_ERR_PLATFORM); return; }
        int vcell = pre[idx];
        bindPair(pc, vcell);
        dm_append(vc, chain, l, pc);
        ST(d.allVCDoomed[k], d.allVCDoomed[k] + 1);
        if constexpr (D < DOOM_DEPTH) allocatePreassignedCellT<D + 1>(pc, vc, true);
        else panic(HIVED_ERR_CAPACITY);
        if (panicCode) return;
      }
    }
  }
  // hived_algorithm.go:630-653
  template <int D>
  HIVED_DEV_NOINLINE void tryUnbindDoomedBadCellT(int chain, int l) {
    int k = cl(chain, l);
    if (d.allVCDoomed[k] == 0) return;  // no doomed bad cell of any VC at this level
    for (int vc = 0; vc < d.S.nVCs; vc++) {
      if (!d.vc_chain_counter[vc * d.S.nChains + chain]) continue;
      int kv = vcl(vc, chain, l);
      int guard = 0;
      while (d.dm_len[kv] != 0 && d.vcFree[kv] < d.totalLeft[k] - d.bf_len[k]) {
        if (++guard > d.S.NP) { panic(HIVED_ERR_CAPACITY); return; }  // a device limit: every round takes one entry off the list
        int pc = d.dm_data[d.dm_base[kv] + 0];
        if (d.p_vcell[pc] < 0) { panic(HIVED_ERR_PLATFORM); return; }  // nil virtual cell dereferenced in the reference (:643-646)
        unbindPair(pc, d.p_vcell[pc]);
        dm_remove(vc, chain, l, pc);
        ST(d.allVCDoomed[k], d.allVCDoomed[k] - 1);
        if constexpr (D < DOOM_DEPTH) releasePreassignedCellT<D + 1>(pc, vc, true);
        else panic(HIVED_ERR_CAPACITY);
        if (panicCode) return;
      }
    }
  }
  // The reference walks the bad cells below a cell recursively, parent before children, children in order
  // (hived_algorithm.go:1429-1447, 1487-1500).  Here: the same pre-order walk with an explicit stack of (cell, next
  // child) — the device program does not recurse, so its stack is sized by the compiler (no cudaLimitStackSize).
  template <typename Body>
  HIVED_DEV void forEachBadCellBelow(int c, Body body) {
    int cell[MAXL], next[MAXL];
    if (!body(c)) return;
    int sp = 0;
    cell[0] = c; next[0] = 0;
    while (sp >= 0) {
      const int x = cell[sp], i = next[sp];
      if (i >= d.p_nchild[x]) { sp--; continue; }
      next[sp] = i + 1;
      const int ch = d.p_child0[x] + i;
      if (!d.p_healthy[ch] && body(ch) && sp + 1 < MAXL) { sp++; cell[sp] = ch; next[sp] = 0; }
    }
  }
  // hived_algorithm.go:1429-1447
  HIVED_DEV_NOINLINE void allocateBadCell(int c0_) {
    forEachBadCellBelow(c0_, [&](int c) {
      if (d.p_bfpos[c] >= 0) bf_remove(d.p_chain[c], d.p_level[c], c);
      if (d.p_vcell[c] < 0) {
        int par = d.p_parent[c];
        int pv = par >= 0 ? d.p_vcell[par] : -1;
        int vc = pv >= 0 ? unboundChild(pv) : -1;
        if (vc < 0) { panic(HIVED_ERR_PLATFORM); return false; }
        bindPair(c, vc);
      }
      return true;
    });
  }
  // hived_algorithm.go:1487-1500
  HIVED_DEV_NOINLINE void releaseBadCell(int c0_) {
    forEachBadCellBelow(c0_, [&](int c) {
      bf_append(d.p_chain[c], d.p_level[c], c);
      int vc = d.p_vcell[c];
      if (vc >= 0) unbindPair(c, vc);
      return true;
    });
  }
  // hived_algorithm.go:1354-1427
  template <int D>
  HIVED_DEV_NOINLINE bool allocatePreassignedCellT(int c, int vc, bool doomedBad) {
    if (c < 0) { panic(HIVED_ERR_PLATFORM); return false; }  // nil *PhysicalCell dereferenced in the reference (:1358): see allocateLeafCell
    sharedEnter();
    bool safetyOk = true;
    int chain = d.p_chain[c], level = d.p_level[c];
    int kv = vcl(vc, chain, level), k = cl(chain, level);
    if (!d.vc_chain_counter[vc * d.S.nChains + chain]) { panic(HIVED_ERR_PLATFORM); return false; }  // write to a nil map in the reference (:1364)
    ST(d.vcFree[kv], d.vcFree[kv] - 1);
    ST(d.allVCFree[k], d.allVCFree[k] - 1);
    ST(d.totalLeft[k], d.totalLeft[k] - 1);
    int splitLevelUpTo = removeCellFromFreeList(c);
    int parent = d.p_parent[c];
    for (int l = level + 1; l <= splitLevelUpTo; l++) {
      int kl = cl(chain, l);
      ST(d.totalLeft[kl], d.totalLeft[kl] - 1);
      if (d.totalLeft[kl] < d.allVCFree[kl]) safetyOk = false;
      if (!d.p_healthy[parent]) {
        bf_remove(chain, l, parent);
      } else {
        tryBindDoomedBadCellT<D>(chain, l);
      }
      parent = d.p_parent[parent];
    }
    if (!d.p_healthy[c]) {
      allocateBadCell(c);
      if constexpr (D == 0) { if (!doomedBad) tryUnbindDoomedBadCellT<D>(chain, level); }
    } else {
      tryBindDoomedBadCellT<D>(chain, level);
    }
    int numToReduce = d.p_nchild[c];
    for (int l = level - 1; l >= 1; l--) {
      int kl = cl(chain, l);
      ST(d.totalLeft[kl], d.totalLeft[kl] - numToReduce);
      if (d.totalLeft[kl] < d.allVCFree[kl]) safetyOk = false;
      if constexpr (D == 0) { if (!doomedBad) tryBindDoomedBadCellT<D>(chain, l); }
      numToReduce *= d.chain_lvl_nchild[kl];
    }
    return safetyOk;
  }
  // hived_algorithm.go:1449-1485
  template <int D>
  HIVED_DEV_NOINLINE void releasePreassignedCellT(int c, int vc, bool doomedBad) {
    sharedEnter();
    int chain = d.p_chain[c], level = d.p_level[c];
    int kv = vcl(vc, chain, level), k = cl(chain, level);
    if (!d.vc_chain_counter[vc * d.S.nChains + chain]) { panic(HIVED_ERR_PLATFORM); return; }  // write to a nil map in the reference (:1454)
    ST(d.vcFree[kv], d.vcFree[kv] + 1);
    ST(d.allVCFree[k], d.allVCFree[k] + 1);
    ST(d.totalLeft[k], d.totalLeft[k] + 1);
    int mergeLevelUpTo = addCellToFreeList(c);
    int parent = d.p_parent[c];
    for (int l = level + 1; l <= mergeLevelUpTo; l++) {
      int kl = cl(chain, l);
      ST(d.totalLeft[kl], d.totalLeft[kl] + 1);
      if (!d.p_healthy[parent]) {
        bf_append(chain, l, parent);
      } else {
        tryUnbindDoomedBadCellT<D>(chain, l);
      }
      parent = d.p_parent[parent];
    }
    if (!d.p_healthy[c]) {
      releaseBadCell(c);
      if constexpr (D == 0) { if (!doomedBad) tryBindDoomedBadCellT<D>(chain, level); }
    } else {
      tryUnbindDoomedBadCellT<D>(chain, level);
    }
    int numToAdd = d.p_nchild[c];
    for (int l = level - 1; l >= 1; l--) {
      int kl = cl(chain, l);
      ST(d.totalLeft[kl], d.totalLeft[kl] + numToAdd);
      if constexpr (D == 0) { if (!doomedBad) tryUnbindDoomedBadCellT<D>(chain, l); }
      numToAdd *= d.chain_lvl_nchild[kl];
    }
  }
  // cell.go:302-312
  HIVED_DEV void setHealthiness(int c, int healthy) {
    ST(d.p_healthy[c], healthy);
    int vc = d.p_vcell[c];
    if (vc >= 0) ST(d.v_healthy[vc], healthy);
  }
  // hived_algorithm.go:562-581
  HIVED_DEV_NOINLINE void addBadFreeCell(int c) {
    int chain = d.p_chain[c], level = d.p_level[c];
    if (!d.chain_in_vc[chain]) { panic(HIVED_ERR_PLATFORM); return; }  // nil-map write in the reference
    bf_append(chain, level, c);
    int k = cl(chain, level);
    if (d.allVCFree[k] > d.totalLeft[k] - d.bf_len[k]) tryBindDoomedBadCell(chain, level);
  }
  // hived_algorithm.go:500-522.  The reference marks the cell, recurses into the parent and only then handles the cell
  // itself: the healthy path is marked bottom-up first, then its cells are handled top-down (no recursion here).
  HIVED_DEV_NOINLINE void setBadCell(int c) {
    int path[MAXL];
    int n = 0;
    for (int x = c; x >= 0 && n < MAXL && d.p_healthy[x]; x = d.p_parent[x]) { setHealthiness(x, 0); path[n++] = x; }
    for (int k = n - 1; k >= 0; k--) {
      const int x = path[k];
      if (inFreeCellList(x)) {
        addBadFreeCell(x);
      } else if (d.p_vcell[x] < 0 && !d.p_split[x]) {
        int par = d.p_parent[x];
        int pv = par >= 0 ? d.p_vcell[par] : -1;
        int vc = pv >= 0 ? unboundChild(pv) : -1;
        if (vc < 0) { panic(HIVED_ERR_PLATFORM); continue; }
        bindPair(x, vc);
      }
    }
  }
  // hived_algorithm.go:524-560
  HIVED_DEV_NOINLINE void setHealthyCell(int c) {
    while (true) {
      if (d.p_healthy[c]) return;
      setHealthiness(c, 1);
      if (inFreeCellList(c)) {
        // removeBadFreeCell :583-600
        bf_remove(d.p_chain[c], d.p_level[c], c);
        tryUnbindDoomedBadCell(d.p_chain[c], d.p_level[c]);
      } else {
        int vc = d.p_vcell[c];
        if (vc >= 0 && !(d.p_flags[c] & PF_PINNED_BIT) && d.p_prio[c] < 0) {
          int vcid = d.v_vc[vc];
          bool preassigned = d.v_parent[vc] < 0;
          unbindPair(c, vc);
          if (preassigned) {
            dm_remove(vcid, d.p_chain[c], d.p_level[c], c);
            int k = cl(d.p_chain[c], d.p_level[c]);
            ST(d.allVCDoomed[k], d.allVCDoomed[k] - 1);
            releasePreassignedCell(c, vcid, true);
          }
        }
      }
      int par = d.p_parent[c];
      if (par < 0) return;
      int c0 = d.p_child0[par];
      if (firstIdx(d.p_nchild[par], [&](int i) { return !d.p_healthy[c0 + i]; }) >= 0) return;
      c = par;
    }
  }
  // hived_algorithm.go:466-498: the leaves of a node, chain by chain, in level-1 list order
  HIVED_DEV_NOINLINE void setNodeHealth(int node, bool healthy) {
    if (multi) { panic(HIVED_ERR_PLATFORM); return; }  // the host never runs health events VC-parallel
    if (node < 0 || node >= d.S.nNodes) return;
    if (healthy) {
      if (!d.node_bad[node]) return;
      ST(d.node_bad[node], 0);
      ST(d.nbad[0], d.nbad[0] - 1);  // bad nodes in the cluster (0: the bucketed cluster views apply)
    } else {
      if (d.node_bad[node]) return;
      ST(d.node_bad[node], 1);
      ST(d.nbad[0], d.nbad[0] + 1);
    }
    for (int chain = 0; chain < d.S.nChains; chain++) {
      int k = node * d.S.nChains + chain;
      for (int i = 0; i < d.ncl_cnt[k]; i++) {
        int leaf = d.ncl_list[d.ncl_off[k] + i];
        if (healthy) setHealthyCell(leaf); else setBadCell(leaf);
        if (panicCode) return;
      }
    }
  }

  // ======================================================================================
  // leaf cell allocation / release (hived_algorithm.go:1292-1352)
  // ======================================================================================
  // The reference keeps a map priority -> number of used leaf cells on every cell and updates it incrementally
  // (cell_allocation.go:443-454): +1 at p in allocateLeafCell, -1 at the leaf's CURRENT priority in releaseLeafCell
  // (hived_algorithm.go:1302-1317, 1329, 1350).  Here the counts are derived from the leaf priorities, which is the
  // same thing as long as every allocation meets a free leaf and every release a used one.  The reference's own call
  // sequences break that in two ways, and its counters then drift for good (nothing ever repairs them):
  //   * allocateLeafCell on a leaf that still has a priority o (a bind that lands on Reserved cells while their
  //     preemptor is alive; cells re-allocated around lazy preemption): the entry at o is never decremented;
  //   * releaseLeafCell on a leaf whose priority is already FREE (a gang lazy-preempted on a bad node keeps its
  //     bindings, :1332-1335, and is released again when deleted): the entry at freePriority goes negative.
  // The cluster views sort and fit on those counters (topology_aware_scheduler.go:138-154), so the differences are
  // kept — (priority, difference) pairs on the leaf and all its ancestors — and added to the derived counts of a
  // view whose s_anom is non-zero (viewNodeInfo); such a view leaves the bucketed form for good.
  template <bool V>
  HIVED_DEV_NOINLINE void noteDelta(int leaf, int prio, int delta) {
    int32_t* dprio = V ? d.v_dprio : d.p_dprio;
    int32_t* dcnt = V ? d.v_dcnt : d.p_dcnt;
    const int32_t* anc = V ? d.v_anc : d.p_anc;
    hv_phase();
    bool full = false;
    for (int b = 0; b < AS; b += HIVED_WARPSZ) {
      int l = b + lane;
      if (l < AS) {
        int a = anc[leaf * AS + l];
        if (a >= 0) {
          int slot = -1;
          for (int i = 0; i < DELTA_SLOTS; i++) if (dprio[a * DELTA_SLOTS + i] == prio) slot = i;
          if (slot < 0) for (int i = DELTA_SLOTS - 1; i >= 0; i--) if (dprio[a * DELTA_SLOTS + i] == DELTA_EMPTY) slot = i;
          if (slot < 0) full = true;
          else { dprio[a * DELTA_SLOTS + slot] = prio; dcnt[a * DELTA_SLOTS + slot] += delta; }
        }
      }
    }
    if (hv_ballot(full)) { panic(HIVED_ERR_CAPACITY); return; }
    hv_warp_sync();
    int sched = -1;
    if (V) sched = schedOfVirtual(leaf);
    else { const int chain = d.p_chain[leaf]; sched = chain >= 0 ? d.opp_sched[chain] : -1; }
    if (sched >= 0) ST(d.s_anom[sched], d.s_anom[sched] + 1);
    if (V) bkMarkLeaf(leaf);
  }
  HIVED_DEV_NOINLINE bool allocateLeafCell(int pLeaf, int vLeaf, int p, int vc) {
    bool safetyOk = true;
    stat_add(ST_LEAVES, 1);
    if (vLeaf >= 0) {
      if (d.v_prio[vLeaf] != FREE_PRIO) noteDelta<true>(vLeaf, d.v_prio[vLeaf], 1);   // the old entry stays in the reference's map
      if (d.p_prio[pLeaf] != FREE_PRIO) noteDelta<false>(pLeaf, d.p_prio[pLeaf], 1);
      setPriority<true>(vLeaf, p);
      setPriority<false>(pLeaf, p, ceilOf(vLeaf));
      if (p == OPP_PRIO) updateUsedOpp(pLeaf, 1);
      int pac = d.v_pre[vLeaf];
      bool newlyBound = d.v_pcell[pac] < 0;
      if (d.p_vcell[pLeaf] < 0) bindCell(pLeaf, vLeaf);
      if (newlyBound) safetyOk = allocatePreassignedCell(d.v_pcell[pac], vc, false);
    } else {
      if (d.p_prio[pLeaf] != FREE_PRIO) noteDelta<false>(pLeaf, d.p_prio[pLeaf], 1);
      setPriority<false>(pLeaf, OPP_PRIO);
      updateUsedOpp(pLeaf, 1);
    }
    return safetyOk;
  }
  HIVED_DEV_NOINLINE void releaseLeafCell(int pLeaf, int vc) {
    stat_add(ST_LEAVES, 1);
    int vLeaf = d.p_vcell[pLeaf];
    const int ceil = ceilOf(vLeaf);
    if (vLeaf >= 0) {
      if (d.v_prio[vLeaf] == FREE_PRIO) noteDelta<true>(vLeaf, FREE_PRIO, -1);  // decremented at the free priority in the reference
      setPriority<true>(vLeaf, FREE_PRIO);
      int pre = d.v_pre[vLeaf];
      int preassignedPhysical = d.v_pcell[pre];
      if (preassignedPhysical < 0) { panic(HIVED_ERR_PLATFORM); return; }  // nil dereference in the reference (hived_algorithm.go:1343)
      if (d.p_healthy[pLeaf]) unbindCell(pLeaf);
      if (!(d.p_flags[preassignedPhysical] & PF_PINNED_BIT) && d.v_prio[pre] < 0 && !dm_contains(vc, preassignedPhysical))
        releasePreassignedCell(preassignedPhysical, vc, false);
    }
    if (d.p_prio[pLeaf] == OPP_PRIO) updateUsedOpp(pLeaf, -1);
    if (d.p_prio[pLeaf] == FREE_PRIO) noteDelta<false>(pLeaf, FREE_PRIO, -1);
    setPriority<false>(pLeaf, FREE_PRIO, ceil);
  }

  // ---- fused fast paths of the two per-leaf sequences that dominate commit and delete.  Each is the
  // exact composition of the generic functions above for the common case (guarded by the preconditions);
  // anything else falls back to the generic sequence.

  // == allocateLeafCell(pLeaf, vLeaf, p, vc); p_using = g; setCellState(pLeaf, Used, ceil)
  //    for a guaranteed allocation that raises both leaves' priorities and whose preassigned cell is bound:
  //    one gather over the levels (lane = level) instead of five dependent walks.
  HIVED_DEV_NOINLINE bool commitLeaf(int pLeaf, int vLeaf, int p, int vc, int g) {
    const int ceil = ceilOf(vLeaf);
    bool fast = vLeaf >= 0 && p > OPP_PRIO && d.v_prio[vLeaf] == FREE_PRIO && d.p_prio[pLeaf] == FREE_PRIO && d.v_pcell[d.v_pre[vLeaf]] >= 0;
    if (!fast) {
      bool safetyOk = allocateLeafCell(pLeaf, vLeaf, p, vc);
      ST(d.p_using[pLeaf], g);
      setCellState(pLeaf, HIVED_CELL_USED, ceil);
      return safetyOk;
    }
    stat_add(ST_LEAVES, 1);
    bkMarkLeaf(vLeaf);
    const bool leafUnbound = d.p_vcell[pLeaf] < 0;
    // bindCell: the run of unbound virtual ancestors starting at the leaf
    unsigned stopMask = leafUnbound ? levelMask(1, AS, [&](int l) { int va = d.v_anc[vLeaf * AS + l]; return va < 0 || d.v_pcell[va] >= 0; }) : 2u;
    const int stop = stopMask ? hv_ffs(stopMask) - 1 : AS;
    hv_phase();
    for (int b = 0; b < AS; b += HIVED_WARPSZ) {
      int l = b + lane;
      if (l >= 1 && l < AS) {
        int pa = d.p_anc[pLeaf * AS + l], va = d.v_anc[vLeaf * AS + l];
        if (va >= 0 && d.v_prio[va] < p) d.v_prio[va] = p;                 // setPriority<true>: raise
        if (pa >= 0) {
          if (l <= ceil && d.p_prio[pa] < p) d.p_prio[pa] = p;             // setPriority<false>: raise up to the ceiling
          int bound = d.p_vcell[pa];
          if (leafUnbound && l < stop) {                                   // bindCell
            d.p_vcell[pa] = va; d.v_pcell[va] = pa; d.v_healthy[va] = d.p_healthy[pa];
            bound = va;
          }
          if (l <= ceil) { d.p_state[pa] = HIVED_CELL_USED; if (bound >= 0) d.v_state[bound] = HIVED_CELL_USED; }  // setCellState(Used)
        }
      }
    }
    hv_warp_sync();
    ST(d.p_using[pLeaf], g);
    return true;
  }

  // == releaseLeafCell(pLeaf, vc); setCellState(pLeaf, Free, ceil)  for a healthy, bound, non-opportunistic leaf.
  // The four upward walks of the generic code (virtual priority, unbinding, physical priority, state) advance
  // together, one level per iteration, sharing one warp-wide scan of the siblings (lane = child).
  HIVED_DEV_NOINLINE void releaseLeafAndFree(int pLeaf, int vc) {
    int vLeaf = d.p_vcell[pLeaf];
    const int ceil = ceilOf(vLeaf);
    if (vLeaf < 0 || !d.p_healthy[pLeaf] || d.p_prio[pLeaf] < 0 || d.v_prio[vLeaf] == FREE_PRIO) {
      releaseLeafCell(pLeaf, vc);
      setCellState(pLeaf, HIVED_CELL_FREE, ceil);
      return;
    }
    stat_add(ST_LEAVES, 1);
    bkMarkLeaf(vLeaf);
    const int pre = d.v_pre[vLeaf];
    const int preP = d.v_pcell[pre];
    if (preP < 0) { panic(HIVED_ERR_PLATFORM); return; }  // nil dereference in the reference (hived_algorithm.go:1343)
    int vOrig = d.v_prio[vLeaf], vNew = FREE_PRIO;
    int pOrig = d.p_prio[pLeaf], pNew = FREE_PRIO;
    bool wU = !(d.p_flags[pLeaf] & PF_PINNED_BIT);
    hv_warp_sync();
    ST(d.v_prio[vLeaf], FREE_PRIO);
    ST(d.p_prio[pLeaf], FREE_PRIO);
    if (wU) unbindPair(pLeaf, vLeaf);
    ST(d.p_state[pLeaf], HIVED_CELL_FREE);
    if (!wU) ST(d.v_state[vLeaf], HIVED_CELL_FREE);
    bool wV = true, wP = true, wS = true;
    int cv = vLeaf, cp = pLeaf;
    for (int l = 2; l < AS + 1 && (wV || wU || wP || wS); l++) {
      int pv = wV || wU ? d.v_parent[cv] : -1;
      int pp = wP || wS ? d.p_parent[cp] : -1;
      if (pv < 0) { wV = false; wU = false; }
      if (pp < 0 || l - 1 >= ceil) { wP = false; wS = false; }
      if (wV || wU) {
        int vpp = d.v_prio[pv];
        bool contV = wV && vOrig == vpp && vNew < vOrig;
        int c0 = d.v_child0[pv], n = d.v_nchild[pv];
        int mx = FREE_PRIO; bool anyBound = false;
        for (int b = 0; b < n; b += HIVED_WARPSZ) {
          int i = b + lane;
          if (i < n && c0 + i != cv) {
            int q = d.v_prio[c0 + i]; if (q > mx) mx = q;
            if (d.v_pcell[c0 + i] >= 0) anyBound = true;
          }
        }
        mx = hv_reduce_max(mx);
        anyBound = hv_ballot(anyBound) != 0;
        if (wU) {
          if (anyBound) {
            wU = false;
          } else {
            int pvP = d.v_pcell[pv];
            if (d.p_flags[pvP] & PF_PINNED_BIT) wU = false; else unbindPair(pvP, pv);
          }
        }
        if (contV) { int np = mx > vNew ? mx : vNew; vOrig = vpp; vNew = np; ST(d.v_prio[pv], np); } else wV = false;
        cv = pv;
      }
      if (wP || wS) {
        int ppp = d.p_prio[pp];
        bool contP = wP && pOrig == ppp && pNew < pOrig;
        int c0 = d.p_child0[pp], n = d.p_nchild[pp];
        int mx = FREE_PRIO; bool anyNotFree = false;
        for (int b = 0; b < n; b += HIVED_WARPSZ) {
          int i = b + lane;
          if (i < n && c0 + i != cp) {
            int q = d.p_prio[c0 + i]; if (q > mx) mx = q;
            if (d.p_state[c0 + i] != HIVED_CELL_FREE) anyNotFree = true;
          }
        }
        mx = hv_reduce_max(mx);
        anyNotFree = hv_ballot(anyNotFree) != 0;
        if (wS) {
          if (anyNotFree) {
            wS = false;
          } else {
            ST(d.p_state[pp], HIVED_CELL_FREE);
            int v = d.p_vcell[pp];
            if (v >= 0) ST(d.v_state[v], HIVED_CELL_FREE);
          }
        }
        if (contP) { int np = mx > pNew ? mx : pNew; pOrig = ppp; pNew = np; ST(d.p_prio[pp], np); } else wP = false;
        cp = pp;
      }
    }
    // hived_algorithm.go:1343-1347: the preassigned cell is released once nothing in it is in real use
    if (!(d.p_flags[preP] & PF_PINNED_BIT) && d.v_prio[pre] < 0 && !dm_contains(vc, preP)) releasePreassignedCell(preP, vc, false);
  }

  // ======================================================================================
  // the lean lane: incremental (bucketed) cluster view, gangs as units, plan / apply / release
  // ======================================================================================
#include "hived_lean.inc"
#include "hived_runahead.inc"

  // ======================================================================================
  // cluster-view pass: data-parallel over the CTA
  //   updateClusterView + sort.Stable + findNodesForPods (topology_aware_scheduler.go:231-306)
  // ======================================================================================
  // info word of a view node: free(8b) | usedSame(8b)<<8 | usedHigher(8b)<<16 | healthy<<24 | suggested<<25
  HIVED_DEV int viewNodeInfo(int cell, bool isVirtual, bool cross, int p, bool ignoreSuggested, bool anomalous) const {
    int leaf0, nleaf, healthy = 1, suggested = 1;
    const int32_t* prio;
    if (isVirtual) {
      leaf0 = d.v_leaf0[cell]; nleaf = d.v_nleaf[cell]; prio = d.v_prio;
      int pc = d.v_pcell[cell];
      if (pc >= 0) { healthy = d.p_healthy[pc]; suggested = ignoreSuggested || node_suggested(d.p_node[pc]); }
    } else {
      leaf0 = d.p_leaf0[cell]; nleaf = d.p_nleaf[cell]; prio = d.p_prio;
      healthy = d.p_healthy[cell]; suggested = ignoreSuggested || node_suggested(d.p_node[cell]);
    }
    int same = 0, higher = 0, ge = 0;
    for (int i = 0; i < nleaf; i++) {
      int q = prio[leaf0 + i];
      if (q < OPP_PRIO) continue;  // free leaf
      if (q == p) same++;
      else if (cross) same++;
      else if (q > p) higher++;
      if (q >= p) ge++;
    }
    int free = nleaf - ge;
    if (anomalous) {  // add what the reference's counters hold beyond the leaf priorities (noteDelta)
      const int32_t* dprio = isVirtual ? d.v_dprio : d.p_dprio;
      const int32_t* dcnt = isVirtual ? d.v_dcnt : d.p_dcnt;
      for (int i = 0; i < DELTA_SLOTS; i++) {
        const int q = dprio[cell * DELTA_SLOTS + i], c = dcnt[cell * DELTA_SLOTS + i];
        if (q == DELTA_EMPTY || c == 0) continue;
        if (q == p) same += c;
        else if (cross) same += c;
        else if (q > p) higher += c;
        if (q >= p) free -= c;
      }
    }
    // free, same, higher: 9 bits each, biased by 128 (the reference's counters may be negative or exceed the leaf count)
    return ((free + 128) & 511) | (((same + 128) & 511) << 9) | (((higher + 128) & 511) << 18) | (healthy << 27) | (suggested << 28);
  }
  HIVED_DEV static int infoFree(int w) { return (w & 511) - 128; }
  HIVED_DEV static int infoSame(int w) { return ((w >> 9) & 511) - 128; }
  HIVED_DEV static int infoHigher(int w) { return ((w >> 18) & 511) - 128; }
  HIVED_DEV static int infoHealthy(int w) { return (w >> 27) & 1; }
  HIVED_DEV static int infoSuggested(int w) { return (w >> 28) & 1; }

  // CTA-wide exclusive prefix sum of smp()->cnt[0..n) (row-major: bin-major, warp-minor)
  HIVED_DEV void ctaExclusiveScan(int n) {
    int nth = hv_nth(), tid = hv_tid(), w = hv_warp(), W = hv_nwarps();
    if (n <= 32 * HIVED_WARPSZ) {  // few counters (the usual 36 bins x 16 warps): one warp scans them, one barrier
      if (w == 0) {
        int per = (n + HIVED_WARPSZ - 1) / HIVED_WARPSZ;
        int lo = lane * per, hi = lo + per < n ? lo + per : n;
        int sum = 0;
        for (int i = lo; i < hi; i++) sum += smp()->cnt[i];
        int incl = sum;
        for (int o = 1; o < HIVED_WARPSZ; o <<= 1) { int t = hv_shfl_up(incl, o); if (lane >= o) incl += t; }
        int run = incl - sum;
        for (int i = lo; i < hi; i++) { int v = smp()->cnt[i]; smp()->cnt[i] = run; run += v; }
      }
      hv_cta_sync();
      return;
    }
    int per = (n + nth - 1) / nth;
    int lo = tid * per, hi = lo + per < n ? lo + per : n;
    int s = 0;
    for (int i = lo; i < hi; i++) s += smp()->cnt[i];
    int incl = s;
    for (int o = 1; o < HIVED_WARPSZ; o <<= 1) { int t = hv_shfl_up(incl, o); if (lane >= o) incl += t; }
    if (lane == HIVED_WARPSZ - 1) smp()->part[w] = incl;
    hv_cta_sync();
    if (w == 0) {
      int v = lane < W ? smp()->part[lane] : 0;
      int inc = v;
      for (int o = 1; o < HIVED_WARPSZ; o <<= 1) { int t = hv_shfl_up(inc, o); if (lane >= o) inc += t; }
      if (lane < W) smp()->part[lane] = inc - v;
    }
    hv_cta_sync();
    int run = smp()->part[w] + incl - s;
    for (int i = lo; i < hi; i++) { int v = smp()->cnt[i]; smp()->cnt[i] = run; run += v; }
    hv_cta_sync();
  }

  // one stable counting pass: out[rank] = in[i] ordered by bin(info[in[i]]), ties by position
  // prezeroed: the caller cleared the counters before its last barrier.  cvOut != nullptr (the last pass): the
  // scatter also persists the order (cvOut[rank] = cell) and lays the infos out in order (s.vw_sinfo[rank]).
  template <typename BinFn>
  HIVED_DEV void stablePass(const int32_t* in, int32_t* out, int n, int nbins, BinFn binOf, bool prezeroed, int32_t* cvOut) {
    int W = hv_nwarps(), w = hv_warp();
    if (!prezeroed) {
      for (int i = hv_tid(); i < nbins * W; i += hv_nth()) smp()->cnt[i] = 0;
      hv_cta_sync();
    }
    int chunk = (n + W - 1) / W;
    chunk = (chunk + HIVED_WARPSZ - 1) / HIVED_WARPSZ * HIVED_WARPSZ;
    int lo = w * chunk, hi = lo + chunk < n ? lo + chunk : n;
    for (int base = lo; base < hi; base += HIVED_WARPSZ) {
      int i = base + lane;
      int b = i < hi ? binOf(s.vw_info[in[i]]) : -1 - lane;  // inactive lanes get unique dummies
      unsigned peers = hv_match(b);
      if (i < hi && (peers & hv_lanemask_lt()) == 0) smp()->cnt[b * W + w] += hv_popc(peers);
      hv_warp_sync();
    }
    hv_cta_sync();
    ctaExclusiveScan(nbins * W);
    for (int base = lo; base < hi; base += HIVED_WARPSZ) {
      int i = base + lane;
      int b = i < hi ? binOf(s.vw_info[in[i]]) : -1 - lane;
      unsigned peers = hv_match(b);
      if (i < hi) {
        int rank = smp()->cnt[b * W + w] + hv_popc(peers & hv_lanemask_lt());
        int src = in[i];
        out[rank] = src;
        if (cvOut) { cvOut[rank] = s.vw_cell[src]; s.vw_sinfo[rank] = s.vw_info[src]; }
      }
      hv_warp_sync();
      if (i < hi && (peers & hv_lanemask_lt()) == 0) smp()->cnt[b * W + w] += hv_popc(peers);
      hv_warp_sync();
    }
    hv_cta_sync();
  }

  // all threads of the CTA
  HIVED_DEV void viewOp() {
    const int sched = smp()->a_sched, p = smp()->a_prio, npods = smp()->a_npods;
    const bool ignoreSuggested = smp()->a_ignore != 0;
    const int off = d.s_off[sched], n = d.s_n[sched];
    const bool cross = d.s_cross[sched] != 0, isVirtual = d.s_virtual[sched] != 0;
    const int L = d.s_maxleaf[sched];
    const int tid = hv_tid(), nth = hv_nth();
    // 1. per-node keys from leaf priorities (coalesced int32 loads of contiguous leaf ranges); the counters of the
    //    first sorting pass are cleared under the same barrier
    const int W = hv_nwarps();
    const bool anomalous = d.s_anom[sched] != 0;
    const int firstBins = cross ? 4 * (L + 1) : L + 1;
    for (int i = tid; i < firstBins * W; i += nth) smp()->cnt[i] = 0;
    for (int i = tid; i < n; i += nth) {
      int cell = d.cv[off + i];
      s.vw_cell[i] = cell;
      s.vw_info[i] = viewNodeInfo(cell, isVirtual, cross, p, ignoreSuggested, anomalous);
      s.vw_ordA[i] = i;
    }
    hv_cta_sync();
    // 2. stable sort by (healthy desc, suggested desc, usedSame desc, usedHigher asc): LSD passes.  The last pass also
    // 3. persists the new order (the reference sorts its slice in place) and lays the infos out in order.
    if (anomalous) {
      // keys outside [0, L] (noteDelta): a stable insertion sort on the full keys by one thread — the order is the
      // persisted one from the last pass, so it is nearly sorted already
      if (tid == 0) {
        auto key = [&](int w) {
          return ((long long)((1 - infoHealthy(w)) * 2 + (1 - infoSuggested(w))) << 40) | ((long long)(512 - infoSame(w)) << 20) |
                 (long long)(infoHigher(w) + 128);
        };
        for (int i = 1; i < n; i++) {
          const int idx = s.vw_ordA[i];
          const long long k = key(s.vw_info[idx]);
          int j = i - 1;
          while (j >= 0 && key(s.vw_info[s.vw_ordA[j]]) > k) { s.vw_ordA[j + 1] = s.vw_ordA[j]; j--; }
          s.vw_ordA[j + 1] = idx;
        }
        for (int i = 0; i < n; i++) { const int src = s.vw_ordA[i]; d.cv[off + i] = s.vw_cell[src]; s.vw_sinfo[i] = s.vw_info[src]; }
      }
      hv_cta_sync();
    } else {
      int32_t* cur = s.vw_ordA;
      int32_t* nxt = s.vw_ordB;
      if (!cross) {
        stablePass(cur, nxt, n, L + 1, [](int w) { return infoHigher(w); }, true, nullptr);
        int32_t* t = cur; cur = nxt; nxt = t;
      }
      stablePass(cur, nxt, n, 4 * (L + 1), [L](int w) {
        return ((1 - infoHealthy(w)) * 2 + (1 - infoSuggested(w))) * (L + 1) + (L - infoSame(w));
      }, cross, d.cv + off);
    }
    const int32_t* sinfo = s.vw_sinfo;
    // 4. greedy first-fit (findNodesForPods :278-305); every thread tracks the same scalar state
    int nodeIndex = 0, picked = 0, ok = 1, reason = 0, rcell = -1;
    for (int k = 0; k < npods && ok; k++) {
      int need = s.pod_need[k];
      int found = -1;
      if (nodeIndex < n && infoFree(sinfo[nodeIndex]) - picked >= need) {
        found = nodeIndex;
      } else {
        if (tid == 0) smp()->best = n;
        hv_cta_sync();
        int mine = n;
        for (int j = nodeIndex + 1 + tid; j < n; j += nth)
          if (infoFree(sinfo[j]) >= need) { mine = j; break; }
        mine = hv_reduce_min(mine);
        if (lane == 0 && mine < n) hv_atomic_min(&smp()->best, mine);
        hv_cta_sync();
        int b = smp()->best;
        hv_cta_sync();
        if (b < n) { found = b; picked = 0; }
      }
      if (found < 0) { ok = 0; reason = HIVED_WAIT_INSUFFICIENT; rcell = -1; break; }
      int w = sinfo[found];
      if (!infoHealthy(w) || !infoSuggested(w)) {
        ok = 0;
        reason = !infoHealthy(w) ? HIVED_WAIT_BAD_NODE : HIVED_WAIT_NON_SUGGESTED_NODE;
        int cell = d.cv[off + found];
        rcell = isVirtual ? d.v_pcell[cell] : cell;
        break;
      }
      nodeIndex = found;
      picked += need;
      if (tid == 0) { s.pod_pos[k] = found; s.pod_cell[k] = d.cv[off + found]; }
    }
    if (tid == 0) { smp()->r_ok = ok; smp()->r_reason = reason; smp()->r_cell = rcell; }
    hv_cta_sync();
  }

  // leader: post the view pass to the CTA and take part in it
  HIVED_DEV bool runViewPass(int sched, int p, bool ignoreSuggested, int npods, int& reason, int& rcell) {
    if (d.bk_valid[sched]) bkMaterialise(sched);  // the general pass sorts the order array
    path_add(PC_GENERAL_VIEW);
    ST(smp()->a_sched, sched);
    ST(smp()->a_prio, p);
    ST(smp()->a_ignore, ignoreSuggested ? 1 : 0);
    ST(smp()->a_npods, npods);
    ST(smp()->a_sugg, sugg);
    ST(smp()->cmd, CMD_VIEW);
    hv_cta_sync();
    viewOp();
    stat_add(ST_VIEW_NODES, d.s_n[sched]);
    reason = smp()->r_reason;
    rcell = smp()->r_cell;
    return smp()->r_ok != 0;
  }

  // ======================================================================================
  // intra-node leaf search (topology_aware_scheduler.go:308-476)
  // ======================================================================================
  // :443-462 with the ancestor tables: lowest level >= level(higher) where both have the same ancestor
  template <bool V>
  HIVED_DEV int findLCA(int lower, int higher) const {
    const int32_t* anc = V ? d.v_anc : d.p_anc;
    int lh = V ? d.v_level[higher] : d.p_level[higher];
    unsigned m = levelMask(lh, AS, [&](int l) {
      int x = anc[lower * AS + l];
      return x >= 0 && x == anc[higher * AS + l];
    });
    if (!m) return -1;
    return anc[lower * AS + hv_ffs(m) - 1];
  }
  // :389-399
  HIVED_DEV int optimalAffinity(int chain, int leafNum) const {
    for (int l = 1; l <= d.chain_top[chain]; l++)
      if (d.chain_lvl_leafnum[cl(chain, l)] >= leafNum) return l;
    return -1;
  }
  // :308-387.  slot = index of this node's candidate list (nodeAvailableLeafCells); out = leaf ids
  template <bool V>
  HIVED_DEV void findLeafCellsInNode(int node, int k, int p, int slot, bool fresh, int chain, int32_t* out) {
    int32_t* avail = s.cand + slot * MAX_NODE_LEAVES;
    int navail;
    if (fresh) {
      // getLeafCellsFromNode :464-476: free leaves in DFS order, then preemptible ones (ballot compaction)
      int leaf0 = V ? d.v_leaf0[node] : d.p_leaf0[node];
      int nleaf = V ? d.v_nleaf[node] : d.p_nleaf[node];
      const int32_t* prio = V ? d.v_prio : d.p_prio;
      int n = 0;
      for (int b = 0; b < nleaf; b += HIVED_WARPSZ) {
        int i = b + lane;
        bool f = i < nleaf && prio[leaf0 + i] == FREE_PRIO;
        unsigned m = hv_ballot(f);
        if (f) avail[n + hv_popc(m & hv_lanemask_lt())] = leaf0 + i;
        n += hv_popc(m);
      }
      if (p > OPP_PRIO) {
        for (int b = 0; b < nleaf; b += HIVED_WARPSZ) {
          int i = b + lane;
          int q = i < nleaf ? prio[leaf0 + i] : FREE_PRIO;
          bool f = q != FREE_PRIO && q < p;
          unsigned m = hv_ballot(f);
          if (f) avail[n + hv_popc(m & hv_lanemask_lt())] = leaf0 + i;
          n += hv_popc(m);
        }
      }
      hv_warp_sync();
      navail = n;
    } else {
      navail = s.cand_len[slot];
    }
    if (k == navail && k <= MAX_NODE_LEAVES && optimalAffinity(chain, k) >= 0) {
      // every available leaf is needed: the search below has exactly one combination to find (the leaves of one
      // view node always share that node as an ancestor) — take them in list order and empty the list
      for (int i = lane; i < k; i += HIVED_WARPSZ) out[i] = avail[i];
      hv_warp_sync();
      ST(s.cand_len[slot], 0);
      return;
    }
    int curIdx[MAX_NODE_LEAVES], curAff[MAX_NODE_LEAVES], bestIdx[MAX_NODE_LEAVES];
    const int HIGHEST = 0x7fffffff;
    int bestAffinity = HIGHEST;
    int optimal = optimalAffinity(chain, k);
    if (k > MAX_NODE_LEAVES) { panic(HIVED_ERR_CAPACITY); return; }  // the search's arrays (a device limit)
    if (optimal < 0) { panic(HIVED_ERR_PLATFORM); return; }
    int ai = 0, si = 0;
    bool done = false;
    while (!done) {
      while (ai < navail) {
        int leaf = avail[ai];
        curIdx[si] = ai;
        if (si == 0) {
          curAff[si] = leaf;
        } else {
          curAff[si] = findLCA<V>(leaf, curAff[si - 1]);
          int lv = curAff[si] >= 0 ? (V ? d.v_level[curAff[si]] : d.p_level[curAff[si]]) : 0;
          if ((curAff[si] < 0 && bestAffinity < HIGHEST) || (curAff[si] >= 0 && lv > bestAffinity)) {
            ai++;
            continue;
          }
        }
        if (si == k - 1) {
          if (curAff[k - 1] < 0) { panic(HIVED_ERR_PLATFORM); return; }
          int affinity = V ? d.v_level[curAff[k - 1]] : d.p_level[curAff[k - 1]];
          bool foundOptimal = false;
          if (affinity < bestAffinity) {
            for (int i = 0; i < k; i++) bestIdx[i] = curIdx[i];
            bestAffinity = affinity;
            foundOptimal = affinity == optimal;
          }
          if (foundOptimal) { done = true; break; }
        } else {
          si++;
        }
        ai++;
      }
      if (done) break;
      si--;
      if (si < 0) {
        if (bestAffinity == HIGHEST) { panic(HIVED_ERR_PLATFORM); return; }  // "Assert Failure"
        break;
      }
      ai = curIdx[si] + 1;
    }
    for (int i = 0; i < k; i++) ST(out[i], avail[bestIdx[i]]);
    // removePickedLeafCells :425-441 (order preserving)
    int w = 0, b = 0;
    for (int i = 0; i < navail; i++) {
      if (b < k && bestIdx[b] == i) { b++; continue; }
      int v = avail[i];
      hv_warp_sync();
      ST(avail[w], v);
      w++;
    }
    ST(s.cand_len[slot], w);
  }

  // ======================================================================================
  // topologyAwareScheduler.Schedule (topology_aware_scheduler.go:65-116)
  //   members: ascending leaf numbers (merged); placement written to `outLeaves` in
  //   (member, pod, leaf) order.  Returns false + reason on failure.
  // ======================================================================================
  HIVED_DEV bool tasSchedule(int sched, int nmem, const int* memLeaf, const int* memPods, int p,
                                      bool ignoreSuggested, int32_t* outLeaves, int& reason, int& rcell) {
    int npods = 0;
    for (int m = 0; m < nmem; m++)
      for (int i = 0; i < memPods[m]; i++) { ST(s.pod_need[npods], memLeaf[m]); npods++; }
    int priority = OPP_PRIO;
    long long tc0 = pclock();
    if (fastEligible(sched, nmem, ignoreSuggested)) {
      const int fp = fastPlace(sched, memLeaf[0], memPods[0], outLeaves);
      if (panicCode) return false;
      if (fp == 1) {
        fastPlaced = true; fastK = memLeaf[0]; fastM = memPods[0]; fastSched = sched;
        path_add(PC_FAST_VIEW);
        stat_add(ST_VIEW_NODES, d.s_n[sched]);
        stat_add(ST_PODS, npods);
        stat_add(ST_CYC_VIEW, pclock() - tc0);
        reason = 0; rcell = -1;
        return true;
      }
    }
    if (mgMode == 1) { mgStop = true; return false; }  // not a lean placement: the event runs alone, later
    bool ok = runViewPass(sched, priority, ignoreSuggested, npods, reason, rcell);
    if (!ok && p > OPP_PRIO) {
      priority = p;
      ok = runViewPass(sched, priority, ignoreSuggested, npods, reason, rcell);
    }
    long long tc1 = pclock();
    stat_add(ST_CYC_VIEW, tc1 - tc0);
    if (!ok) return false;
    stat_add(ST_PODS, npods);
    const bool isVirtual = d.s_virtual[sched] != 0;
    const int chain = d.s_chain[sched];
    int nslots = 0, outOff = 0;
    for (int k = 0; k < npods; k++) {
      int node = s.pod_cell[k];
      int slot = -1;
      for (int j = 0; j < nslots; j++)
        if (s.cand_node[j] == node) { slot = j; break; }
      bool fresh = slot < 0;
      if (fresh) { slot = nslots++; ST(s.cand_node[slot], node); }
      int need = s.pod_need[k];
      if (isVirtual) findLeafCellsInNode<true>(node, need, priority, slot, fresh, chain, outLeaves + outOff);
      else findLeafCellsInNode<false>(node, need, priority, slot, fresh, chain, outLeaves + outOff);
      if (panicCode) return false;
      outOff += need;
    }
    stat_add(ST_CYC_LEAF, pclock() - tc1);
    reason = 0;
    rcell = -1;
    return true;
  }

  // ======================================================================================
  // virtual -> physical mapping (types.go:282-340, cell_allocation.go:34-315)
  // ======================================================================================
  int vxCount;   // vertices in use
  int paCount;   // preassigned roots
  int npCount;   // non-preassigned buddy groups
  int epochNow;
  HIVED_DEV int newVertex(int vcell) {
    int v = vxCount++;
    if (v >= d.S.VX) { panic(HIVED_ERR_CAPACITY); return 0; }
    ST(s.vx_cell[v], vcell);
    ST(s.vx_child[v], -1);
    ST(s.vx_last[v], -1);
    ST(s.vx_next[v], -1);
    ST(s.vx_nch[v], 0);
    ST(d.vx_of[vcell], v);
    ST(d.vx_stamp[vcell], epochNow);
    return v;
  }
  HIVED_DEV int vertexOf(int vcell) const { return d.vx_stamp[vcell] == epochNow ? d.vx_of[vcell] : -1; }
  HIVED_DEV void addChildVertex(int parentV, int childV) {
    int last = s.vx_last[parentV];
    int nch = s.vx_nch[parentV];
    hv_warp_sync();
    if (last < 0) ST(s.vx_child[parentV], childV); else ST(s.vx_next[last], childV);
    ST(s.vx_last[parentV], childV);
    ST(s.vx_nch[parentV], nch + 1);
  }
  // types.go:282-340
  HIVED_DEV_NOINLINE void toBindingPaths(const int32_t* vleaves, int nleaves) {
    epochNow = d.epoch[cta] + 1;
    hv_warp_sync();
    ST(d.epoch[cta], epochNow);
    vxCount = 0; paCount = 0; npCount = 0;
    for (int i = 0; i < nleaves; i++) {
      int leaf = vleaves[i];
      int pl = d.v_pcell[leaf];
      if (pl >= 0) { ST(d.binding[leaf], pl); continue; }
      // the unbound run of ancestors that are not yet vertices: levels [1, stop)
      unsigned stopMask = levelMask(1, AS, [&](int l) {
        int a = d.v_anc[leaf * AS + l];
        return a < 0 || d.v_pcell[a] >= 0 || vertexOf(a) >= 0;
      });
      int stop = stopMask ? hv_ffs(stopMask) - 1 : AS;
      if (stop <= 1) { panic(HIVED_ERR_PLATFORM); return; }
      int root = d.v_anc[leaf * AS + stop - 1];
      int n = newVertex(root);
      int par = d.v_parent[root];
      if (par < 0) {
        ST(s.pa_list[paCount], n); paCount++;
      } else if (d.v_pcell[par] >= 0) {
        bool buddy = false;
        for (int g = 0; g < npCount; g++) {
          if (d.v_parent[s.vx_cell[s.np_head[g]]] == par) {
            // append to the group's chain (roots are linked through vx_next)
            int t = s.np_head[g];
            while (s.vx_next[t] >= 0) t = s.vx_next[t];
            int cnt = s.np_cnt[g];
            hv_warp_sync();
            ST(s.vx_next[t], n);
            ST(s.np_cnt[g], cnt + 1);
            buddy = true;
            break;
          }
        }
        if (!buddy) { ST(s.np_head[npCount], n); ST(s.np_cnt[npCount], 1); npCount++; }
      } else {
        addChildVertex(vertexOf(par), n);
      }
      for (int l = stop - 2; l >= 1; l--) {
        int c = d.v_anc[leaf * AS + l];
        int nn = newVertex(c);
        addChildVertex(vertexOf(d.v_parent[c]), nn);
      }
      if (panicCode) return;
    }
  }

  // cell_allocation.go:199-243.  candidates: in[i] or (in == nullptr) the id range base+i.
  // out: usable ones, stably sorted ascending by used[opportunistic].  returns -1 for nil.
  HIVED_DEV bool cellUsable(int c, bool ignoreSuggested) const {
    if (d.p_vcell[c] >= 0) return false;
    int nn = d.p_nodes_cnt[c];
    if (nn == 1 && !d.p_healthy[c]) return false;
    if (!ignoreSuggested) {
      int o = d.p_nodes_off[c];
      for (int j = 0; j < nn; j++)
        if (node_suggested(d.nodes_flat[o + j])) return true;
      return false;
    }
    return true;
  }
  HIVED_DEV_NOINLINE int getUsablePhysicalCells(const int32_t* in, int base, int nin, int numNeeded, bool ignoreSuggested, int32_t* out) {
    stat_add(ST_FREE_CELLS, nin);
    // order-preserving filter, one warp-wide ballot per 32 candidates
    int n = 0;
    for (int b0 = 0; b0 < nin; b0 += HIVED_WARPSZ) {
      int i = b0 + lane;
      int c = i < nin ? (in ? in[i] : base + i) : -1;
      bool ok = c >= 0 && cellUsable(c, ignoreSuggested);
      unsigned m = hv_ballot(ok);
      if (ok) out[n + hv_popc(m & hv_lanemask_lt())] = c;
      n += hv_popc(m);
    }
    hv_warp_sync();
    if (n < numNeeded) return -1;
    // sort.SliceStable by used[opportunistic]: only when some neighbour pair is out of order
    if (firstIdx(n - 1, [&](int i) { return d.p_usedopp[out[i]] > d.p_usedopp[out[i + 1]]; }) >= 0) {
      for (int i = 1; i < n; i++) {
        int c = out[i], key = d.p_usedopp[c];
        int j = i - 1;
        if (d.p_usedopp[out[j]] <= key) continue;
        while (j >= 0 && d.p_usedopp[out[j]] > key) { int v = out[j]; hv_warp_sync(); ST(out[j + 1], v); j--; }
        ST(out[j + 1], c);
      }
    }
    return n;
  }

  // cell_allocation.go:245-315.  cells: ncells vertices linked through vx_next from firstV.
  // The reference recurses into the children of every candidate it tries (one call per tree level) and backtracks over
  // the candidates of a level.  Here the same search runs as one loop over explicit frames, one per level: the frame's
  // candidate list / picked indices / cell list already live in per-depth scratch rows (mc0 / mcbuf, mcpick, mccells),
  // the frame's scalars (usable candidates, cells, current cell, candidate being tried) in four small arrays.  The
  // order of everything observable — candidates tried, bindings written, where a level resumes after a failed
  // subtree, the picked indices a revisited cell starts from — is the reference's.
  HIVED_DEV_NOINLINE bool mapVirtualCellsToPhysical(int firstV, int ncells0, const int32_t* candIn, int candBase, int ncand0,
                                                    bool ignoreSuggested, int /*depth0*/, int32_t* pickedOut) {
    int fN[MAXL], fNc[MAXL], fCi[MAXL], fCand[MAXL];
    int depth = 0;
    int aFirst = firstV, aNc = ncells0, aBase = candBase, aNcand = ncand0;  // arguments of the frame being entered
    const int32_t* aIn = candIn;
    bool ret = false;  // what the frame that just ended returned
    enum { ENTER = 0, NEWCELL = 1, RESUME = 2, POP = 3 };
    int st = ENTER;
    while (true) {
      if (st == ENTER) {
        if (depth >= MAXL || aNc > MAX_FANOUT || (depth > 0 && aNcand > MAX_FANOUT)) { panic(HIVED_ERR_CAPACITY); return false; }
        int32_t* cands = depth == 0 ? s.mc0 : s.mcbuf + depth * MAX_FANOUT;
        const int n = getUsablePhysicalCells(aIn, aBase, aNcand, aNc, ignoreSuggested, cands);
        if (n < 0) { ret = false; st = POP; continue; }
        int32_t* pickedIdx = s.mcpick + depth * MAX_FANOUT;
        int32_t* cellV = s.mccells + depth * MAX_FANOUT;
        int v = aFirst;
        for (int i = 0; i < aNc; i++) { ST(cellV[i], v); ST(pickedIdx[i], 0); v = s.vx_next[v]; }
        fN[depth] = n; fNc[depth] = aNc; fCi[depth] = 0;
        st = NEWCELL;
        continue;
      }
      if (st == POP) {
        if (depth == 0) return ret;
        depth--;
        st = RESUME;
        continue;
      }
      // a frame at work
      int32_t* cands = depth == 0 ? s.mc0 : s.mcbuf + depth * MAX_FANOUT;
      int32_t* pickedIdx = s.mcpick + depth * MAX_FANOUT;
      int32_t* cellV = s.mccells + depth * MAX_FANOUT;
      const int n = fN[depth], ncells = fNc[depth];
      int cellIndex = fCi[depth];
      int candidateIndex;
      bool picked = false;
      if (st == NEWCELL) {
        if (cellIndex < 0) { ret = false; st = POP; continue; }
        candidateIndex = pickedIdx[cellIndex];
      } else {  // RESUME: the subtree below candidate fCand[depth] has been tried
        if (panicCode) return false;
        candidateIndex = fCand[depth];
        if (ret) picked = true; else candidateIndex++;
      }
      bool descend = false;
      for (; !picked && candidateIndex < n; candidateIndex++) {
        bool used = false;  // pickedIndexSet == picks of the cells before cellIndex
        for (int j = 0; j < cellIndex; j++)
          if (pickedIdx[j] == candidateIndex) { used = true; break; }
        if (used) continue;
        const int candidate = cands[candidateIndex];
        const int vtx = cellV[cellIndex];
        if (d.p_level[candidate] == 1) {
          ST(d.binding[s.vx_cell[vtx]], candidate);
          picked = true;
          break;
        }
        fCand[depth] = candidateIndex;
        aFirst = s.vx_child[vtx]; aNc = s.vx_nch[vtx]; aIn = nullptr; aBase = d.p_child0[candidate]; aNcand = d.p_nchild[candidate];
        descend = true;
        break;
      }
      if (descend) { depth++; st = ENTER; continue; }
      if (picked) {
        ST(pickedIdx[cellIndex], candidateIndex);
        if (cellIndex == ncells - 1) {
          if (depth == 0 && pickedOut)
            for (int i = 0; i < ncells; i++) ST(pickedOut[i], cands[pickedIdx[i]]);
          ret = true; st = POP;
          continue;
        }
        fCi[depth] = cellIndex + 1;
      } else {  // every candidate of this cell failed: back to the previous cell, which moves on to its next candidate
        cellIndex--;
        if (cellIndex >= 0) { int v = pickedIdx[cellIndex]; hv_warp_sync(); ST(pickedIdx[cellIndex], v + 1); }
        fCi[depth] = cellIndex;
      }
      st = NEWCELL;
    }
  }

  // ---- the Schedule-time copy of the chain's free list (types.go:123-130, hived_algorithm.go:917-929)
  int sflChain;
  HIVED_DEV int32_t* sfl(int level) const { return s.sfl_data + d.fl_base[cl(sflChain, level)]; }
  HIVED_DEV_NOINLINE void sflCopy(int chain) {
    sflChain = chain;
    for (int l = 1; l < MAXL; l++) {
      int k = cl(chain, l);
      int n = l <= d.chain_top[chain] ? d.fl_len[k] : 0;
      ST(s.sfl_len[l], n);
      for (int i = lane; i < n; i += HIVED_WARPSZ) s.sfl_data[d.fl_base[k] + i] = d.fl_data[d.fl_base[k] + i];
    }
    hv_warp_sync();
  }
  HIVED_DEV_NOINLINE void sflRemove(int level, int cell) {  // types.go:78-95 on the copy
    int32_t* a = sfl(level);
    int n = s.sfl_len[level];
    int idx = firstIdx(n, [&](int i) { return a[i] == cell; });
    if (idx < 0) { panic(HIVED_ERR_PLATFORM); return; }
    int lastv = a[n - 1];
    hv_warp_sync();
    ST(a[idx], lastv);
    ST(s.sfl_len[level], n - 1);
  }

  // cell_allocation.go:34-80.  The reference recurses one level down per split; here one loop over the levels with
  // the loop index and the number of usable cells of every level in two small arrays (the usable cells themselves are
  // per-level rows of ba_buf already).
  HIVED_DEV_NOINLINE bool buddyAlloc(int vtx, int startLevel, bool ignoreSuggested) {
    const int cellLevel = d.v_level[s.vx_cell[vtx]];
    int fI[MAXL], fCnt[MAXL];
    int level = startLevel;
    bool ret = false;
    enum { ENTER = 0, LOOP = 1, RESUME = 2, POP = 3 };
    int st = ENTER;
    while (true) {
      if (st == ENTER) {
        if (level == cellLevel) {
          ST(s.vx_next[vtx], -1);
          const bool ok = mapVirtualCellsToPhysical(vtx, 1, sfl(level), 0, s.sfl_len[level], ignoreSuggested, 0, s.tmp_list);
          if (ok) sflRemove(level, s.tmp_list[0]);
          ret = ok; st = POP;
          continue;
        }
        if (level <= 1 || level >= MAXL) { ret = false; st = POP; continue; }  // (no level below to split into)
        int32_t* freeCells = s.ba_buf + (int64_t)level * d.S.maxLevelCount;
        const int nfree = getUsablePhysicalCells(sfl(level), 0, s.sfl_len[level], 1, ignoreSuggested, freeCells);
        if (nfree < 0) { ret = false; st = POP; continue; }
        fCnt[level] = nfree; fI[level] = 0;
        st = LOOP;
        continue;
      }
      if (st == POP) {
        if (level == startLevel) return ret;
        level++;  // back in the frame that split one of its cells
        st = RESUME;
        continue;
      }
      int32_t* freeCells = s.ba_buf + (int64_t)level * d.S.maxLevelCount;
      if (st == RESUME) {
        const int c = freeCells[fI[level]];
        if (ret) { sflRemove(level, c); ret = true; st = POP; continue; }
        if (panicCode) return false;
        ST(s.sfl_len[level - 1], 0);  // = nil
        fI[level]++;
        st = LOOP;
      }
      // LOOP: split the next usable cell of this level and try one level down
      if (fI[level] >= fCnt[level]) { ret = false; st = POP; continue; }
      {
        const int c = freeCells[fI[level]];
        int32_t* lower = sfl(level - 1);
        const int nl = s.sfl_len[level - 1];
        const int nc = d.p_nchild[c], c0 = d.p_child0[c];
        if (nl + nc > d.fl_cap[cl(sflChain, level - 1)]) { panic(HIVED_ERR_CAPACITY); return false; }  // (duplicates: see fl_append)
        for (int j = lane; j < nc; j += HIVED_WARPSZ) lower[nl + j] = c0 + j;
        hv_warp_sync();
        ST(s.sfl_len[level - 1], nl + nc);
        level--;
        st = ENTER;
      }
    }
  }

  // cell_allocation.go:82-150
  HIVED_DEV_NOINLINE bool safeRelaxedBuddyAlloc(int vtx, int* freeCellNum, int currentLevel, bool ignoreSuggested) {
    int top = sflChain >= 0 ? d.chain_top[sflChain] : 0;
    int splittableNum[MAXL];
    for (int i = 0; i < MAXL; i++) splittableNum[i] = 0;
    int splittableCell = -1;
    for (int i = top; i > currentLevel; i--) {
      splittableNum[i] = s.sfl_len[i] - freeCellNum[i];
      if (i < top && splittableCell >= 0) splittableNum[i] += splittableNum[i + 1] * d.p_nchild[splittableCell];
      if (splittableCell < 0 && s.sfl_len[i] > 0) splittableCell = sfl(i)[0];
      else if (splittableCell >= 0) splittableCell = d.p_child0[splittableCell];
      if (splittableNum[i] < 0) { panic(HIVED_ERR_PLATFORM); return false; }  // "VC Safety Broken"
    }
    for (int l = currentLevel + 1; l <= top; l++) {
      int cellNum = s.sfl_len[l];
      if (cellNum > splittableNum[l]) cellNum = splittableNum[l];
      if (cellNum > 0) {
        int32_t* split = s.ba_buf;  // level 0 row is otherwise unused
        int ns = 0;
        for (int i = 0; i < cellNum; i++) {
          int first = sfl(l)[0];
          ST(split[ns], first); ns++;
          sflRemove(l, first);
        }
        splittableNum[l] -= cellNum;
        for (int sl = l; sl > currentLevel; sl--) {
          // expand every cell of the split list into its children (in place, back to front)
          int total = 0;
          for (int i = 0; i < ns; i++) total += d.p_nchild[split[i]];
          if (total > d.S.maxLevelCount) { panic(HIVED_ERR_CAPACITY); return false; }
          int w = total;
          for (int i = ns - 1; i >= 0; i--) {
            int c = split[i], nc = d.p_nchild[c], c0 = d.p_child0[c];
            hv_warp_sync();
            for (int j = nc - 1; j >= 0; j--) { w--; ST(split[w], c0 + j); }
          }
          ns = total;
        }
        // freeList[currentLevel] = append(splitList, freeList[currentLevel]...)
        int32_t* cur = sfl(currentLevel);
        int nc = s.sfl_len[currentLevel];
        if (nc + ns > d.fl_cap[cl(sflChain, currentLevel)]) { panic(HIVED_ERR_CAPACITY); return false; }  // (duplicates: see fl_append)
        for (int i = nc - 1; i >= 0; i--) { int v = cur[i]; hv_warp_sync(); ST(cur[i + ns], v); }
        for (int i = 0; i < ns; i++) ST(cur[i], split[i]);
        ST(s.sfl_len[currentLevel], nc + ns);
        ST(s.vx_next[vtx], -1);
        bool ok = mapVirtualCellsToPhysical(vtx, 1, cur, 0, nc + ns, ignoreSuggested, 0, s.tmp_list);
        if (ok) { sflRemove(currentLevel, s.tmp_list[0]); return true; }
        if (panicCode) return false;
      }
    }
    return false;
  }

  // cell_allocation.go:152-197
  HIVED_DEV_NOINLINE bool mapVirtualPlacementToPhysical(int chain, bool ignoreSuggested) {
    int freeCellNum[MAXL];
    for (int l = 0; l < MAXL; l++) freeCellNum[l] = 0;
    if (paCount > 0) {
      if (chain < 0) { panic(HIVED_ERR_PLATFORM); return false; }  // nil free list: "VC Safety Broken"
      sharedEnter();  // held until the event (and its commit) is over
      for (int l = 0; l < MAXL; l++) freeCellNum[l] = d.chain_in_vc[chain] ? d.allVCFree[cl(chain, l)] : 0;
      sflCopy(chain);
    } else {
      sflChain = chain;
    }
    for (int i = 0; i < paCount; i++) {
      int vtx = s.pa_list[i];
      int level = d.v_level[s.vx_cell[vtx]];
      int l = level, top = d.chain_top[chain];
      for (; l <= top; l++)
        if (s.sfl_len[l] != 0) break;
      if (l > top) { panic(HIVED_ERR_PLATFORM); return false; }  // getLowestFreeCellLevel: "VC Safety Broken"
      if (!buddyAlloc(vtx, l, ignoreSuggested)) {
        if (panicCode) return false;
        if (!safeRelaxedBuddyAlloc(vtx, freeCellNum, level, ignoreSuggested)) return false;
      } else {
        freeCellNum[level]--;
      }
    }
    for (int g = 0; g < npCount; g++) {
      int head = s.np_head[g];
      int parentPhysical = d.v_pcell[d.v_parent[s.vx_cell[head]]];
      bool ok = mapVirtualCellsToPhysical(head, s.np_cnt[g], nullptr, d.p_child0[parentPhysical], d.p_nchild[parentPhysical],
                                          ignoreSuggested, 0, nullptr);
      if (!ok) return false;
    }
    return true;
  }

  // ======================================================================================
  // affinity groups (types.go:133-183; hived_algorithm.go:981-1222)
  // ======================================================================================
  HIVED_DEV int32_t* gphys(int g) const { return d.g_phys + (int64_t)g * d.S.LS; }
  HIVED_DEV int32_t* gvirt(int g) const { return d.g_virt + (int64_t)g * d.S.LS; }
  HIVED_DEV int32_t* gpods(int g) const { return d.g_pods + (int64_t)g * d.S.PS; }
  HIVED_DEV int32_t* gpre(int g) const { return d.g_pre + (int64_t)g * d.S.PS; }
  // The 32-word header record of a group is one coalesced load (lane = word); sums and searches over the member
  // tables (words 8.. = leaf numbers, 16.. = pod numbers, word 4 = #members) are warp reductions over that row
  // instead of loops of dependent loads.  (The 1-lane host emulation keeps the loops.)
#ifndef HIVED_EMU
  static_assert(GROUP_HDR_WORDS == HIVED_WARPSZ, "one header word per lane");
  HIVED_DEV int hdrWord(int g) const { return d.g_hdr[(int64_t)g * GROUP_HDR_WORDS + lane]; }
  HIVED_DEV int groupLeaves(int g) const {
    int w = hdrWord(g), n = hv_shfl(w, 4), up = hv_shfl(w, (lane + 8) & 31);
    return hv_reduce_add((lane >= 8 && lane < 8 + n) ? w * up : 0);
  }
  HIVED_DEV int groupPods(int g) const {
    int w = hdrWord(g), n = hv_shfl(w, 4);
    return hv_reduce_add((lane >= 16 && lane < 16 + n) ? w : 0);
  }
  HIVED_DEV void memberOffsets(int g, int m, int& leafOff, int& podOff) const {
    int w = hdrWord(g), up = hv_shfl(w, (lane + 8) & 31);
    leafOff = hv_reduce_add((lane >= 8 && lane < 8 + m) ? w * up : 0);
    podOff = hv_reduce_add((lane >= 16 && lane < 16 + m) ? w : 0);
  }
  HIVED_DEV int memberOf(int g, int leafNum) const {
    int w = hdrWord(g), n = hv_shfl(w, 4);
    unsigned hit = hv_ballot(lane >= 8 && lane < 8 + n && w == leafNum);
    return hit ? hv_ffs(hit) - 1 - 8 : -1;
  }
#else
  HIVED_DEV int groupLeaves(int g) const {
    int n = 0;
    for (int m = 0; m < d.g_nmem[g]; m++) n += d.g_mem_leaf[g * 8 + m] * d.g_mem_pods[g * 8 + m];
    return n;
  }
  HIVED_DEV int groupPods(int g) const {
    int n = 0;
    for (int m = 0; m < d.g_nmem[g]; m++) n += d.g_mem_pods[g * 8 + m];
    return n;
  }
  // slot offsets of member m: leaves before it / pods before it
  HIVED_DEV void memberOffsets(int g, int m, int& leafOff, int& podOff) const {
    leafOff = 0; podOff = 0;
    for (int i = 0; i < m; i++) { leafOff += d.g_mem_leaf[g * 8 + i] * d.g_mem_pods[g * 8 + i]; podOff += d.g_mem_pods[g * 8 + i]; }
  }
  HIVED_DEV int memberOf(int g, int leafNum) const {
    for (int m = 0; m < d.g_nmem[g]; m++) if (d.g_mem_leaf[g * 8 + m] == leafNum) return m;
    return -1;
  }
#endif
  // merge + sort the spec's members (types.go:157-160, hived_algorithm.go:775-778)
  HIVED_DEV static int mergeMembers(const hived_pod_spec_t& sp, int* leaf, int* pods) {
    int n = 0;
    for (int i = 0; i < sp.n_members; i++) {
      int ln = sp.member_leaf_num[i], pn = sp.member_pod_num[i];
      int j = 0;
      for (; j < n; j++) if (leaf[j] == ln) break;
      if (j < n) { pods[j] += pn; continue; }
      j = n++;
      while (j > 0 && leaf[j - 1] > ln) { leaf[j] = leaf[j - 1]; pods[j] = pods[j - 1]; j--; }
      leaf[j] = ln; pods[j] = pn;
    }
    return n;
  }
  // newAlgoAffinityGroup types.go:150-183
  HIVED_DEV int newGroup(int g, const hived_pod_spec_t& sp, int state, int* leaf, int* pods) {
    int n = mergeMembers(sp, leaf, pods);
    int nl = 0, np = 0;
    for (int m = 0; m < n; m++) { nl += leaf[m] * pods[m]; np += pods[m]; }
    hv_phase();
    if (lane == 0) {  // the header record (hived_dev.h), one sequence point for all of it
      d.g_state[g] = state;
      d.g_vc[g] = sp.vc;
      d.g_prio[g] = sp.priority;
      d.g_flags[g] = ((sp.flags & HIVED_SPEC_LAZY_PREEMPTION) ? GF_LAZY_ENABLE : 0) | GF_HAS_VIRTUAL;
      d.g_nmem[g] = n;
      d.g_npre[g] = 0;
      d.g_hdr[(int64_t)g * GROUP_HDR_WORDS + 6] = 0;  // no unit decomposition known (applyLean writes one)
      for (int m = 0; m < n; m++) { d.g_mem_leaf[g * 8 + m] = leaf[m]; d.g_mem_pods[g * 8 + m] = pods[m]; }
    }
    int32_t* ph = gphys(g); int32_t* vi = gvirt(g); int32_t* po = gpods(g);
    for (int i = lane; i < nl; i += HIVED_WARPSZ) { ph[i] = -1; vi[i] = -1; }
    for (int i = lane; i < np; i += HIVED_WARPSZ) po[i] = -1;
    hv_warp_sync();
    return n;
  }
  HIVED_DEV void eraseGroup(int g) { ST(d.g_state[g], HIVED_GROUP_NONE); }
  // delete(h.affinityGroups, g.name) for an object reached through a cell (cell.reservingOrReservedGroup): when the
  // object is a ghost, whichever group carries its name NOW leaves the map as well — and lives on as a ghost itself
  // while its own leaves name it (the shims keep name <-> id while a ghost of the id exists: hived.h "Id lifetime")
  HIVED_DEV void eraseGroupByName(int g) {
    if (g < d.S.maxGroups) { eraseGroup(g); return; }
    const int origin = d.g_hdr[(int64_t)g * GROUP_HDR_WORDS + GH_ORIGIN] - 1;
    eraseGroup(g);
    if (origin >= 0 && d.g_state[origin] != HIVED_GROUP_NONE) { ghostify(origin); eraseGroup(origin); }
  }
  // Object identity of an erased group.  The reference's cells point at *AlgoAffinityGroup objects (cell.usingGroup,
  // cell.reservingOrReservedGroup), its name map at whichever object carries the name now.  One path erases a group
  // from the map while its own leaves keep naming it: schedulePodFromExistingGroup treats every state but Allocated as
  // Preempting (hived_algorithm.go:671-707), so a pod of a group that is BEING PREEMPTED whose placement has a bad or
  // non-suggested node runs deletePreemptingAffinityGroup on it (:1114-1145) — the Reserving leaves go back to "the group
  // being preempted" (the group itself) and the name is freed; the next Schedule creates a NEW object under that name,
  // while the victims of whoever preempts those leaves later are still the OLD object's pods (utils.go:217).  Below the
  // ABI a group is its interned id, so the old incarnation moves to a ghost record and the leaves are re-pointed;
  // a ghost whose leaves no longer name it is garbage (the reference's GC) and its slot is reused.
  HIVED_DEV bool groupNamedByOwnLeaves(int g) const {
    const int32_t* ph = gphys(g);
    return firstIdx(groupLeaves(g), [&](int i) { const int c = ph[i]; return c >= 0 && (d.p_using[c] == g || d.p_resv[c] == g); }) >= 0;
  }
  HIVED_DEV_NOINLINE void ghostify(int g) {
    if (!groupNamedByOwnLeaves(g)) return;
    int gg = -1;
    for (int k = 0; k < GHOST_GROUPS && gg < 0; k++) {
      const int c = d.S.maxGroups + k;
      if (d.g_nmem[c] == 0 || !groupNamedByOwnLeaves(c)) gg = c;
    }
    if (gg < 0) { panic(HIVED_ERR_CAPACITY); return; }
    const int nl = groupLeaves(g), np = groupPods(g), npre = d.g_npre[g];
    hv_phase();
    // the name travels with the object: a ghost of a ghost keeps the first id
    const int origin = g >= d.S.maxGroups ? d.g_hdr[(int64_t)g * GROUP_HDR_WORDS + GH_ORIGIN] : g + 1;
    for (int w = lane; w < GROUP_HDR_WORDS; w += HIVED_WARPSZ)
      d.g_hdr[(int64_t)gg * GROUP_HDR_WORDS + w] = w == GH_ORIGIN ? origin : d.g_hdr[(int64_t)g * GROUP_HDR_WORDS + w];
    if (lane == 0 && origin > 0) d.g_hdr[(int64_t)(origin - 1) * GROUP_HDR_WORDS + GH_LINK] = gg + 1;
    for (int i = lane; i < nl; i += HIVED_WARPSZ) { gphys(gg)[i] = gphys(g)[i]; gvirt(gg)[i] = gvirt(g)[i]; }
    for (int i = lane; i < np; i += HIVED_WARPSZ) gpods(gg)[i] = gpods(g)[i];
    for (int i = lane; i < npre; i += HIVED_WARPSZ) gpre(gg)[i] = gpre(g)[i];
    hv_warp_sync();
    for (int i = lane; i < nl; i += HIVED_WARPSZ) {
      const int c = gphys(g)[i];
      if (c >= 0) { if (d.p_using[c] == g) d.p_using[c] = gg; if (d.p_resv[c] == g) d.p_resv[c] = gg; }
    }
    hv_warp_sync();
  }

  // hived_algorithm.go:1165-1191.  save != nullptr receives the original virtual placement.
  HIVED_DEV_NOINLINE void lazyPreemptAffinityGroup(int g, int32_t* save) {
    int nl = groupLeaves(g);
    bool had = (d.g_flags[g] & GF_HAS_VIRTUAL) != 0;
    if (had) {
      for (int i = 0; i < nl; i++) {
        int vLeaf = gvirt(g)[i];
        if (vLeaf >= 0) {
          int pLeaf = d.v_pcell[vLeaf];
          if (pLeaf < 0) { panic(HIVED_ERR_PLATFORM); return; }
          releaseLeafCell(pLeaf, d.g_vc[g]);
          allocateLeafCell(pLeaf, -1, OPP_PRIO, d.g_vc[g]);
        }
      }
    }
    if (save) {
      ST(save[0], had ? 1 : 0);  // word 0: non-nil marker
      for (int i = 0; i < nl; i++) ST(save[1 + i], had ? gvirt(g)[i] : -1);
    }
    int fl = d.g_flags[g];
    hv_warp_sync();
    ST(d.g_flags[g], (fl & ~GF_HAS_VIRTUAL) | GF_LAZY_PREEMPTED);
  }
  // hived_algorithm.go:1193-1201: every Used leaf below the cell, in depth-first order = ascending id (the leaves below
  // a cell are a contiguous range in child order, hived_topo.hpp fillTree)
  HIVED_DEV_NOINLINE void lazyPreemptCell(int vcell) {
    const int l0 = d.v_leaf0[vcell], nl = d.v_nleaf[vcell];
    for (int i = 0; i < nl; i++) {
      const int leaf = l0 + i;
      if (d.v_state[leaf] != HIVED_CELL_USED) continue;
      int pc = d.v_pcell[leaf];
      int g = pc >= 0 ? d.p_using[pc] : -1;
      if (g < 0) { panic(HIVED_ERR_PLATFORM); continue; }
      lazyPreemptAffinityGroup(g, nullptr);
    }
  }
  // hived_algorithm.go:1203-1222
  HIVED_DEV_NOINLINE void revertLazyPreempt(int g, const int32_t* save) {
    if (!save[0]) { panic(HIVED_ERR_PLATFORM); return; }  // nil placement indexed in the reference
    int nl = groupLeaves(g);
    for (int i = 0; i < nl; i++) {
      int pLeaf = gphys(g)[i];
      if (pLeaf < 0) continue;
      int vLeaf = save[1 + i];
      releaseLeafCell(pLeaf, d.g_vc[g]);
      allocateLeafCell(pLeaf, vLeaf, d.g_prio[g], d.g_vc[g]);
    }
    for (int i = 0; i < nl; i++) ST(gvirt(g)[i], save[1 + i]);
    int fl = d.g_flags[g];
    hv_warp_sync();
    ST(d.g_flags[g], (fl | GF_HAS_VIRTUAL) & ~GF_LAZY_PREEMPTED);
  }

  // ---- whole-gang release: the per-leaf loop of deleteAllocatedAffinityGroup for the common case (every leaf
  // Used, healthy, bound, guaranteed, not pinned), with lanes over the gang's leaves and one step per tree level
  // instead of one upward walk per leaf.  Equivalence with the sequential walks: leaf fields are independent;
  // a parent's priority is the max of its children (cell_allocation.go:422-441 keeps that invariant), it turns
  // Free iff all children are Free (utils.go:397-415) and is unbound iff no child stays bound
  // (cell_allocation.go:399-420) — all functions of the children's FINAL values, so each level is computed once
  // after the level below is complete (lanes sharing an ancestor write the same values).  Preassigned cells are
  // released in the order of their last leaf, as the sequential loop would.  false: nothing written.
  HIVED_DEV bool deleteGroupBatched(int g, int nl, int vc) {
    const int32_t* ph = gphys(g);
    bool bad = false;
    long long tq = pclock();
    for (int b0 = 0; b0 < nl; b0 += HIVED_WARPSZ) {
      int i = b0 + lane;
      bool ok = true;
      if (i < nl) {
        int L = ph[i];
        ok = L >= 0;
        int V = ok ? d.p_vcell[L] : -1;
        // (a leaf on a bad node is released like a healthy one except that it stays bound, releaseLeafCell :1340)
        ok = ok && V >= 0 && d.p_state[L] == HIVED_CELL_USED && d.p_prio[L] >= 0 && !(d.p_flags[L] & PF_PINNED_BIT);
        ok = ok && d.v_prio[V] != FREE_PRIO;
        if (ok) {
          int pre = d.v_pre[V];
          s.pl_v[i] = V; s.pl_v2[i] = pre; s.pl_p[i] = d.v_pcell[pre]; s.pl_p2[i] = L;
          ok = s.pl_p[i] >= 0;  // (an unbound preassigned cell above a bound leaf: the per-leaf code reports the reference's panic)
        }
      }
      if (hv_ballot(!ok)) bad = true;
    }
    if (bad) return false;
    hv_warp_sync();
    // With bad cells around, releasing one preassigned cell can re-bind doomed bad cells (tryBind/tryUnbindDoomedBadCell)
    // and so change the binding of ANOTHER preassigned cell that later leaves of the gang sit in: the sequential
    // order then matters.  One preassigned cell for the whole gang, or no bad node at all, rules that out.
    if (d.nbad[0] != 0 && firstIdx(nl, [&](int i) { return s.pl_v2[i] != s.pl_v2[0]; }) >= 0) return false;
    stat_add(ST_LEAVES, nl);
    // level 1: the leaves themselves (releaseLeafCell :1319-1352 + setCellState Free)
    for (int b0 = 0; b0 < nl; b0 += HIVED_WARPSZ) {
      int i = b0 + lane;
      bkMarkLeaves(i < nl, i < nl ? s.pl_v[i] : 0);
      if (i < nl) {
        int L = ph[i], V = s.pl_v[i];
        const bool healthy = d.p_healthy[L] != 0;
        d.p_using[L] = -1;
        d.v_prio[V] = FREE_PRIO; d.p_prio[L] = FREE_PRIO;
        if (healthy) { d.p_vcell[L] = -1; d.v_pcell[V] = -1; d.v_healthy[V] = 1; }  // unbindCell only "if pLeafCell.IsHealthy()"
        d.v_state[V] = HIVED_CELL_FREE;
        d.p_state[L] = HIVED_CELL_FREE;
      }
    }
    hv_warp_sync();
    return releaseAbove(nl, 2, vc);
  }
  // The levels above a set of released ITEMS (s.pl_p2 / s.pl_v: the physical / virtual cell of item i — leaf cells
  // for deleteGroupBatched, complete cells for leanDeleteMulti —, s.pl_v2 / s.pl_p: its preassigned cell, virtual /
  // physical), from startLevel up, then the release of the preassigned cells that became unused.
  HIVED_DEV bool releaseAbove(int nl, int startLevel, int vc) {
    for (int l = startLevel; l < AS; l++) {
      bool changedAny = false;
      for (int b0 = 0; b0 < nl; b0 += HIVED_WARPSZ) {
        int i = b0 + lane;
        const bool act = i < nl;
        const int L = act ? s.pl_p2[i] : 0, V = act ? s.pl_v[i] : 0;
        const int va = act ? d.v_anc[V * AS + l] : -1, pa = act ? d.p_anc[L * AS + l] : -1;
        const int ceil = (act && multi) ? d.v_level[s.pl_v2[i]] : AS;
        const bool actV = va >= 0, actP = pa >= 0 && l <= ceil;
        // every load of the step first (they overlap), the stores last
        const int vch = actV ? d.v_anc[V * AS + l - 1] : 0;
        int vOld = 0, vPc = -1, vchPc = 0, pOld = 0, pSt = 0, pVc = -1;
        if (actV) { vOld = d.v_prio[va]; vPc = d.v_pcell[va]; vchPc = d.v_pcell[vch]; }
        if (actP) { pOld = d.p_prio[pa]; pSt = d.p_state[pa]; pVc = d.p_vcell[pa]; }
        const int vPcFlags = vPc >= 0 ? d.p_flags[vPc] : PF_PINNED_BIT;
        int vmx, pmx;
        bool anyBound, anyNotFree;
        childrenSummary<true>(actV, va, vmx, anyBound);
        childrenSummary<false>(actP, pa, pmx, anyNotFree);
        bool changed = false;
        if (actV) {
          if (vOld != vmx) { d.v_prio[va] = vmx; changed = true; }
          if (!anyBound && vchPc < 0 && !(vPcFlags & PF_PINNED_BIT)) {
            d.p_vcell[vPc] = -1; d.v_pcell[va] = -1; d.v_state[va] = HIVED_CELL_FREE; d.v_healthy[va] = 1;
            changed = true;
          }
        }
        if (actP) {
          if (pOld != pmx) { d.p_prio[pa] = pmx; changed = true; }
          if (!anyNotFree) {
            if (pSt != HIVED_CELL_FREE) { d.p_state[pa] = HIVED_CELL_FREE; changed = true; }
            if (pVc >= 0) d.v_state[pVc] = HIVED_CELL_FREE;
          }
        }
        if (hv_ballot(changed)) changedAny = true;
      }
      hv_warp_sync();
      if (!changedAny) break;  // nothing moved at this level: the levels above keep their values
    }
    // hived_algorithm.go:1343-1347: a preassigned cell goes back once nothing in it is in real use
    bool anyRelease = false;
    for (int b0 = 0; b0 < nl; b0 += HIVED_WARPSZ) {
      int i = b0 + lane;
      bool c = i < nl && !(d.p_flags[s.pl_p[i]] & PF_PINNED_BIT) && d.v_prio[s.pl_v2[i]] < 0;
      if (hv_ballot(c)) anyRelease = true;
    }
    if (anyRelease) {
      for (int i = 0; i < nl; i++) {
        int pre = s.pl_v2[i], preP = s.pl_p[i];
        const int32_t* rest = s.pl_v2 + i + 1;
        if (firstIdx(nl - i - 1, [&](int j) { return rest[j] == pre; }) >= 0) continue;  // a later leaf sits in the same cell
        if (!(d.p_flags[preP] & PF_PINNED_BIT) && d.v_prio[pre] < 0 && !dm_contains(vc, preP)) releasePreassignedCell(preP, vc, false);
        if (panicCode) return true;
      }
    }
    return true;
  }

  // hived_algorithm.go:1043-1070
  HIVED_DEV void deleteAllocatedAffinityGroup(int g) {
    int nl = groupLeaves(g);
    int vc = d.g_vc[g];
    if (mgMode == 1 && mgDeleteNeedsShared(g, nl)) { mgStop = true; return; }
    if (leanDelete(g, nl, vc)) { eraseGroup(g); return; }
    path_add(PC_GENERAL_DELETE);
    if (deleteGroupBatched(g, nl, vc)) { eraseGroup(g); return; }
    const int32_t* ph = gphys(g);
    for (int i = 0; i < nl; i++) {
      int pLeaf = ph[i];
      if (pLeaf < 0) continue;
      ST(d.p_using[pLeaf], -1);
      const int ceil = ceilOf(d.p_vcell[pLeaf]);
      if (d.p_state[pLeaf] == HIVED_CELL_USED) {
        releaseLeafAndFree(pLeaf, vc);
      } else {
        setCellState(pLeaf, HIVED_CELL_RESERVED, ceil);
      }
    }
    // A group that is itself PREEMPTING can be deleted here (DeleteAllocatedPod of a pod bound under an earlier
    // incarnation of the name, hived_algorithm.go:272-296): its Reserved leaves keep naming the erased object
    // (cell.reservingOrReservedGroup), and a later preemptor / allocation on them cancels "its" preemption
    // (:731-742, :1001-1010) — the old object, not whoever carries the id by then (API fuzz seed 2385).
    ghostify(g);
    eraseGroup(g);
  }
  // utils.go:267-283
  HIVED_DEV int retrieveVirtualCell(int g, int pLeaf) const {
    const int32_t* ph = gphys(g);
    int i = firstIdx(groupLeaves(g), [&](int j) { return ph[j] == pLeaf; });
    return i < 0 ? -1 : gvirt(g)[i];
  }
  // hived_algorithm.go:1114-1145
  HIVED_DEV_NOINLINE void deletePreemptingAffinityGroup(int g) {
    int nl = groupLeaves(g);
    for (int i = 0; i < nl; i++) {
      int pLeaf = gphys(g)[i];
      releaseLeafCell(pLeaf, d.g_vc[g]);
      ST(d.p_resv[pLeaf], -1);
      if (d.p_state[pLeaf] == HIVED_CELL_RESERVING) {
        setCellState(pLeaf, HIVED_CELL_USED);
        int bg = d.p_using[pLeaf];
        int bv = -1;
        if (d.g_flags[bg] & GF_HAS_VIRTUAL) bv = retrieveVirtualCell(bg, pLeaf);
        allocateLeafCell(pLeaf, bv, d.g_prio[bg], d.g_vc[bg]);
      } else {
        setCellState(pLeaf, HIVED_CELL_FREE);
      }
    }
    ghostify(g);  // (only a group that was not Preempting can still be named by its leaves here)
    eraseGroupByName(g);
  }
  // hived_algorithm.go:1147-1163
  HIVED_DEV_NOINLINE void allocatePreemptingAffinityGroup(int g) {
    int nl = groupLeaves(g);
    for (int i = 0; i < nl; i++) {
      int pLeaf = gphys(g)[i];
      ST(d.p_resv[pLeaf], -1);
      ST(d.p_using[pLeaf], g);
      setCellState(pLeaf, HIVED_CELL_USED);
    }
    ST(d.g_state[g], HIVED_GROUP_ALLOCATED);
    ST(d.g_npre[g], 0);
  }
  // hived_algorithm.go:1072-1112
  HIVED_DEV_NOINLINE void createPreemptingAffinityGroup(int g, const hived_pod_spec_t& sp, const int32_t* phys, const int32_t* virt) {
    int gleaf[HIVED_MAX_MEMBERS], gpods_[HIVED_MAX_MEMBERS];
    newGroup(g, sp, HIVED_GROUP_PREEMPTING, gleaf, gpods_);
    int nl = groupLeaves(g);
    for (int i = 0; i < nl; i++) { ST(gphys(g)[i], phys[i]); ST(gvirt(g)[i], virt[i]); }
    for (int i = 0; i < nl; i++) {
      int pLeaf = phys[i], vLeaf = virt[i];
      if (d.p_state[pLeaf] == HIVED_CELL_USED) {
        int ug = d.p_using[pLeaf];
        releaseLeafCell(pLeaf, d.g_vc[ug]);
        ST(d.g_state[ug], HIVED_GROUP_BEING_PREEMPTED);
      }
      allocateLeafCell(pLeaf, vLeaf, sp.priority, sp.vc);
      ST(d.p_resv[pLeaf], g);
      if (d.p_state[pLeaf] == HIVED_CELL_USED) setCellState(pLeaf, HIVED_CELL_RESERVING);
      else setCellState(pLeaf, HIVED_CELL_RESERVED);
    }
    ST(gpre(g)[0], sp.pod);
    ST(d.g_npre[g], 1);
  }
  HIVED_DEV void addPreemptingPod(int g, int pod) {  // g.preemptingPods[pod.UID] = pod
    int n = d.g_npre[g];
    for (int i = 0; i < n; i++) if (gpre(g)[i] == pod) return;
    if (n >= d.S.PS) { panic(HIVED_ERR_CAPACITY); return; }
    hv_warp_sync();
    ST(gpre(g)[n], pod);
    ST(d.g_npre[g], n + 1);
  }

  // ======================================================================================
  // Schedule of a NEW affinity group (hived_algorithm.go:754-979)
  // ======================================================================================
  struct Req {
    int vc, pinned, chain, priority, group;
    bool ignoreSuggested;
    int nmem;
    int memLeaf[HIVED_MAX_MEMBERS], memPods[HIVED_MAX_MEMBERS];
    int nleaves;
  };
  int lzCount;
  bool freshPlacement;  // the last schedule() produced its placement in pl_p/pl_v (new group)
  int lastPodIndex;     // pod index of the last bind result (its row in the member's pod placements)
  // the essentials of the last result, kept on the SM so that the auto-commit does not read the record back from HBM
  int lastKind, lastNode, lastChain, lastFirstLeaf, lastHasVirtual, lastNmem;
  long long lastLeafOff;
  int lastVictims;  // number of victims found by the last collectPreemptionVictims
  int32_t lastMemLeaf[HIVED_MAX_MEMBERS], lastMemPods[HIVED_MAX_MEMBERS];

  // hived_algorithm.go:944-965
  HIVED_DEV void tryLazyPreempt(const int32_t* vleaves, int nleaves) {
    lzCount = 0;
    // fast path (inlined at the call site): no leaf of the placement is bound to a Used physical cell
    if (firstIdx(nleaves, [&](int i) { int pl = d.v_pcell[vleaves[i]]; return pl >= 0 && d.p_state[pl] == HIVED_CELL_USED; }) < 0) return;
    tryLazyPreemptSlow(vleaves, nleaves);
  }
  HIVED_DEV_NOINLINE void tryLazyPreemptSlow(const int32_t* vleaves, int nleaves) {
    for (int i = 0; i < nleaves; i++) {
      int pLeaf = d.v_pcell[vleaves[i]];
      if (pLeaf < 0) continue;
      if (d.p_state[pLeaf] == HIVED_CELL_USED) {
        int victim = d.p_using[pLeaf];
        if (victim >= 0 && (d.g_flags[victim] & GF_LAZY_ENABLE)) {
          int slot = -1;
          for (int j = 0; j < lzCount; j++) if (s.lz_group[j] == victim) { slot = j; break; }
          if (slot < 0) {
            if (lzCount >= d.S.LZ) { panic(HIVED_ERR_CAPACITY); return; }
            slot = lzCount++;
            ST(s.lz_group[slot], victim);
          }
          lazyPreemptAffinityGroup(victim, s.lz_save + (int64_t)slot * (d.S.LS + 1));
          if (panicCode) return;
        }
      }
    }
  }

  // ---- whole-placement mapping: toBindingPaths + mapVirtualPlacementToPhysical for the common case, lanes over
  // the placement's virtual leaves.  Preconditions (else false; only scratch was written): every leaf has a
  // bound virtual ancestor (no preassigned cell to allocate, hence no buddy allocation), no suggested-node
  // filter, and every unbound child of the physical cells searched is healthy with no opportunistic use.  Then
  // every candidate is usable, the stable sort by used[opportunistic] is the identity, no pick can fail, and the
  // backtracking search of cell_allocation.go:245-315 degenerates to: the r-th new virtual child (in order of
  // first appearance among the leaves) of a bound virtual cell gets the r-th unbound child of its physical cell,
  // and below that the j-th child vertex gets the j-th child — a rank/select per level, top-down.
  // Scratch: vx_stamp[x] == epochNow marks a virtual cell touched by this pass; binding[x] its physical cell
  // (for unbound x), vx_of[x] the number of its children mapped so far.
  HIVED_DEV bool mapPlacementBatched(const int32_t* vleaves, int nleaves, bool ignoreSuggested) {
    if (sugg != nullptr && !ignoreSuggested) return false;
    epochNow = d.epoch[cta] + 1;
    hv_warp_sync();
    ST(d.epoch[cta], epochNow);
    bool bad = false;
    int maxLs = 0;
    for (int b0 = 0; b0 < nleaves; b0 += HIVED_WARPSZ) {
      int i = b0 + lane;
      bool ok = true;
      int ls = 0;
      if (i < nleaves) {
        int v = vleaves[i];
        int pl = d.v_pcell[v];
        if (pl >= 0) {
          d.binding[v] = pl;
          ls = 1;
        } else {
          unsigned stop = 0, bound = 0;
#pragma unroll 4
          for (int l = 2; l < AS; l++) {  // no early exit: the loads of all levels overlap
            int a = d.v_anc[v * AS + l];
            int pc = a >= 0 ? d.v_pcell[a] : -1;
            if (a < 0 || pc >= 0) stop |= 1u << l;
            if (pc >= 0) bound |= 1u << l;
          }
          ls = stop ? hv_ffs(stop) - 1 : AS;
          ok = ls < AS && ((bound >> ls) & 1u);
        }
        s.pl_v2[i] = ls;
      }
      if (hv_ballot(!ok)) bad = true;
      ls = hv_reduce_max(ls);
      if (ls > maxLs) maxLs = ls;
    }
    if (bad) return false;
    hv_warp_sync();
    long long scanned = 0;
    for (int l = maxLs - 1; l >= 1; l--) {
      for (int b0 = 0; b0 < nleaves; b0 += HIVED_WARPSZ) {
        int i = b0 + lane;
        bool active = i < nleaves && l < s.pl_v2[i];
        int va = -1, vpar = -1, ppar = -1;
        bool topLevel = false;
        if (active) {
          int v = vleaves[i];
          va = d.v_anc[v * AS + l];
          vpar = d.v_anc[v * AS + l + 1];
          topLevel = l + 1 == s.pl_v2[i];
          ppar = topLevel ? d.v_pcell[vpar] : d.binding[vpar];
        }
        // first new child under a bound cell: one search over its physical cell's children
        bool firstTouch = active && topLevel && d.vx_stamp[vpar] != epochNow;
        unsigned same = hv_match(firstTouch ? vpar : -1 - lane);
        if (firstTouch) {
          if (hv_ffs(same) - 1 == lane) scanned += d.p_nchild[ppar];
          d.vx_stamp[vpar] = epochNow; d.vx_of[vpar] = 0;
        }
        hv_warp_sync();
        bool isNew = active && d.vx_stamp[va] != epochNow;
        unsigned grp = hv_match(active ? va : -1 - lane);
        bool leader = isNew && hv_ffs(grp) - 1 == lane;
        unsigned sib = hv_match(leader ? vpar : -1 - lane);
        int sel = -1;
        bool unusable = false;
        const int want = leader ? d.vx_of[vpar] + hv_popc(sib & hv_lanemask_lt()) : 0;
        if (leader && !topLevel && want < d.p_nchild[ppar]) sel = d.p_child0[ppar] + want;
        {  // below a bound cell: the (want)-th unbound child of its physical cell
          int t = selectUnboundPhysChild(leader && topLevel, ppar, want, unusable);
          if (leader && topLevel) sel = t;
        }
        if (leader && sel >= 0 && l > 1) scanned += d.p_nchild[sel];
        // below an unbound cell every child is unbound — unless an anomaly left a binding behind (a gang lazy-preempted
        // on a bad node keeps its bindings, hived_algorithm.go:1332-1335; Filtering-phase binds): the sequential search
        // would skip such a child, so the general path takes over (API fuzz on the synthetic cluster, seed 1087)
        const bool staleBound = leader && !topLevel && sel >= 0 && d.p_vcell[sel] >= 0;
        if (hv_ballot((leader && sel < 0) || staleBound) || unusable) return false;
        if (leader) {
          d.binding[va] = sel; d.vx_stamp[va] = epochNow; d.vx_of[va] = 0;
          if ((sib >> lane) <= 1u) d.vx_of[vpar] = d.vx_of[vpar] + hv_popc(sib);  // the last of the new siblings
        }
        hv_warp_sync();
      }
    }
    scanned = hv_reduce_add((int)scanned);
    stat_add(ST_FREE_CELLS, scanned);
    return true;
  }

  // hived_algorithm.go:898-942; intra_vc_scheduler.go:92-117
  HIVED_DEV bool scheduleGuaranteedAffinityGroup(const Req& r, int& reason, int& rcell) {
    int vset = r.pinned >= 0 ? d.vc_pinned_vset[r.vc * d.S.nPinned + r.pinned] : (r.chain >= 0 ? d.vc_chain_vset[r.vc * d.S.nChains + r.chain] : -1);
    int sched = vset >= 0 ? d.vset_sched[vset] : -1;
    if (sched < 0) { reason = HIVED_WAIT_NO_SCHEDULER | HIVED_WAIT_SCOPE_VC; rcell = -1; return false; }
    fastPlaced = false;
    if (!tasSchedule(sched, r.nmem, r.memLeaf, r.memPods, r.priority, r.ignoreSuggested, s.pl_v, reason, rcell)) {
      reason |= HIVED_WAIT_SCOPE_VC;
      return false;
    }
    long long tm0 = pclock();
    if (fastPlaced && planLean(fastSched, fastK, fastM)) {
      lzCount = 0;
      path_add(PC_FAST_MAP);
      stat_add(ST_CYC_MAP, pclock() - tm0);
      reason = 0; rcell = -1;
      return true;
    }
    if (mgMode == 1) { mgStop = true; return false; }  // the mapping may bind a preassigned cell (free lists)
    path_add(PC_GENERAL_MAP);
    tryLazyPreempt(s.pl_v, r.nleaves);
    if (panicCode) return false;
    bool mapped = mapPlacementBatched(s.pl_v, r.nleaves, r.ignoreSuggested);
    if (!mapped) {
      toBindingPaths(s.pl_v, r.nleaves);
      if (panicCode) return false;
      mapped = mapVirtualPlacementToPhysical(r.chain, r.ignoreSuggested);
    }
    stat_add(ST_CYC_MAP, pclock() - tm0);
    if (mapped) {
      // toPhysicalPlacement types.go:260-280
      for (int i = lane; i < r.nleaves; i += HIVED_WARPSZ) s.pl_p[i] = d.binding[s.pl_v[i]];
      hv_warp_sync();
      reason = 0; rcell = -1;
      return true;
    }
    if (panicCode) return false;
    for (int j = 0; j < lzCount; j++) revertLazyPreempt(s.lz_group[j], s.lz_save + (int64_t)j * (d.S.LS + 1));
    reason = HIVED_WAIT_MAPPING; rcell = -1;
    return false;
  }
  // hived_algorithm.go:967-979
  HIVED_DEV bool scheduleOpportunisticAffinityGroup(const Req& r, int& reason, int& rcell) {
    int sched = d.opp_sched[r.chain];
    if (!tasSchedule(sched, r.nmem, r.memLeaf, r.memPods, OPP_PRIO, r.ignoreSuggested, s.pl_p, reason, rcell)) {
      reason |= HIVED_WAIT_SCOPE_PHYSICAL;
      return false;
    }
    reason = 0; rcell = -1;
    return true;
  }
  // hived_algorithm.go:872-896; hasVirtual tells whether pl_v is meaningful
  HIVED_DEV bool handleSchedulingRequest(const Req& r, bool& hasVirtual, int& reason, int& rcell) {
    if (r.priority >= 0) { hasVirtual = true; return scheduleGuaranteedAffinityGroup(r, reason, rcell); }
    hasVirtual = false;
    return scheduleOpportunisticAffinityGroup(r, reason, rcell);
  }
  // hived_algorithm.go:798-829.  returns 1 placed, 0 not placed, <0 = -(user error code)
  HIVED_DEV int scheduleForLeafCellType(Req& r, int leafType, bool typeSpecified, bool& hasVirtual, int& reason, int& rcell) {
    bool vcHasType = false;
    reason = 0; rcell = -1;
    for (int i = 0; i < d.lt_cnt[leafType]; i++) {
      int chain = d.lt_chains[d.lt_off[leafType] + i];
      if (r.priority < 0 || d.vc_chain_vset[r.vc * d.S.nChains + chain] >= 0) {
        vcHasType = true;
        r.chain = chain;
        if (handleSchedulingRequest(r, hasVirtual, reason, rcell)) { reason = 0; return 1; }
        if (panicCode) return 0;
      }
    }
    if (typeSpecified && r.priority >= 0 && !vcHasType) return -HIVED_ERR_LEAF_TYPE_NOT_IN_VC;
    return 0;
  }
  // hived_algorithm.go:754-796 (+ validateSchedulingRequest :855-870)
  HIVED_DEV int scheduleNewAffinityGroup(const hived_pod_spec_t& sp, Req& r, bool& hasVirtual, int& reason, int& rcell) {
    r.vc = sp.vc; r.pinned = sp.pinned; r.chain = -1; r.priority = sp.priority; r.group = sp.group;
    r.ignoreSuggested = (sp.flags & HIVED_SPEC_IGNORE_SUGGESTED) != 0;
    r.nmem = mergeMembers(sp, r.memLeaf, r.memPods);
    r.nleaves = 0;
    for (int m = 0; m < r.nmem; m++) r.nleaves += r.memLeaf[m] * r.memPods[m];
    reason = 0; rcell = -1; hasVirtual = false;
    if (sp.vc < 0 || sp.vc >= d.S.nVCs) return -HIVED_ERR_UNKNOWN_VC;
    if (sp.pinned != -1) {
      if (sp.pinned < 0 || sp.pinned >= d.S.nPinned || d.vc_pinned_vset[sp.vc * d.S.nPinned + sp.pinned] < 0) return -HIVED_ERR_UNKNOWN_PINNED_CELL;
      if (sp.priority == OPP_PRIO) return -HIVED_ERR_OPPORTUNISTIC_PINNED;
      return handleSchedulingRequest(r, hasVirtual, reason, rcell) ? 1 : 0;
    }
    if (sp.leaf_type != -1) {
      if (sp.leaf_type < 0 || sp.leaf_type >= d.S.nLeafTypes || d.lt_cnt[sp.leaf_type] == 0) return -HIVED_ERR_LEAF_TYPE_NOT_IN_CLUSTER;
      return scheduleForLeafCellType(r, sp.leaf_type, true, hasVirtual, reason, rcell);
    }
    // any leaf cell type (:831-853): leaf types that own a chain, ascending
    int lastReason = 0, lastCell = -1;
    for (int lt = 0; lt < d.S.nLeafTypes; lt++) {
      if (d.lt_cnt[lt] == 0) continue;
      int tr, tc;
      int rc = scheduleForLeafCellType(r, lt, false, hasVirtual, tr, tc);
      if (rc != 0) { reason = 0; rcell = -1; return rc; }
      if (panicCode) return 0;
      if (tr != 0) { lastReason = tr; lastCell = tc; }
    }
    reason = lastReason; rcell = lastCell;
    return 0;
  }

  // ======================================================================================
  // results
  // ======================================================================================
  // utils.go:202-235.  victims written to the pool (pod id, node id) sorted by pod id; overlapping
  // preemptor groups (sorted by id) to s.lz_group, count returned through nOverlap.
  HIVED_DEV void collectPreemptionVictims(const int32_t* phys, int nleaves, hived_result_t* res, int& nOverlap) {
    nOverlap = 0;
    lastVictims = 0;
    // (victim_off / n_victims are 0 in the cleared record)
    // fast path (inlined at the call site): every cell of the placement is Free
    if (firstIdx(nleaves, [&](int i) { int c = phys[i]; return c >= 0 && d.p_state[c] != HIVED_CELL_FREE; }) < 0) return;
    collectPreemptionVictimsSlow(phys, nleaves, res, nOverlap);
  }
  HIVED_DEV_NOINLINE void collectPreemptionVictimsSlow(const int32_t* phys, int nleaves, hived_result_t* res, int& nOverlap) {
    int32_t* groups = s.tmp_list;  // using groups
    int ng = 0;
    int32_t* overlap = s.lz_group;  // lazy-preempt bookkeeping is dead by now
    long long start = poolOff;
    for (int i = 0; i < nleaves; i++) {
      int c = phys[i];
      if (c < 0) continue;
      int st = d.p_state[c];
      if (st == HIVED_CELL_USED || st == HIVED_CELL_RESERVING) {
        int g = d.p_using[c];
        if (g < 0) { panic(HIVED_ERR_PLATFORM); return; }  // GetUsingGroup() == nil dereferenced in the reference (utils.go:217)
        bool seen = false;
        for (int j = 0; j < ng; j++) if (groups[j] == g) { seen = true; break; }
        if (!seen) {
          if (ng >= d.S.maxLevelCount + MAX_FANOUT) { panic(HIVED_ERR_CAPACITY); return; }
          ST(groups[ng], g); ng++;
        }
      }
      if (st == HIVED_CELL_RESERVING || st == HIVED_CELL_RESERVED) {
        int g = d.p_resv[c];  // (-1 = nil: the reference adds it to the set all the same, utils.go:229, and dereferences
                              // it when it cancels the overlapping preemptions in the Preempting phase)
        bool seen = false;
        for (int j = 0; j < nOverlap; j++) if (overlap[j] == g) { seen = true; break; }
        if (!seen) {
          if (nOverlap >= d.S.LS) { panic(HIVED_ERR_CAPACITY); return; }
          ST(overlap[nOverlap], g); nOverlap++;
        }
      }
    }
    int nv = 0;
    for (int j = 0; j < ng; j++) {
      int g = groups[j], np = groupPods(g);
      for (int k = 0; k < np; k++) {
        int pod = gpods(g)[k];
        if (pod < 0) continue;
        if (poolOff + 2 > pool_cap) { panic(HIVED_ERR_CAPACITY); return; }
        poolOff += 2;
        int pos = nv;  // insert sorted by pod id
        while (pos > 0 && pool[start + 2 * (pos - 1)] > pod) {
          int a = pool[start + 2 * (pos - 1)], bb = pool[start + 2 * (pos - 1) + 1];
          hv_warp_sync();
          ST(pool[start + 2 * pos], a);
          ST(pool[start + 2 * pos + 1], bb);
          pos--;
        }
        ST(pool[start + 2 * pos], pod);
        ST(pool[start + 2 * pos + 1], d.pod_node[pod]);
        nv++;
      }
    }
    for (int i = 1; i < nOverlap; i++) {  // ascending group id
      int g = overlap[i], j = i - 1;
      while (j >= 0 && overlap[j] > g) { int v = overlap[j]; hv_warp_sync(); ST(overlap[j + 1], v); j--; }
      ST(overlap[j + 1], g);
    }
    ST(res->victim_off, nv ? (int)start : 0);
    ST(res->n_victims, nv);
    lastVictims = nv;
  }

  // generatePodScheduleResult / generateAffinityGroupBindInfo (utils.go:38-171): lanes over the gang's leaves
  // allowMissing: the group is an allocated one (utils.go:132-141: nil cells of such a group are reported, anything
  // else is "The first pod in group ... was allocated invalid resource")
  HIVED_DEV void emitBind(hived_result_t* res, int nmem, const int* memLeaf, const int* memPods, const int32_t* phys,
                          const int32_t* virt, bool hasVirtual, int curLeafNum, int curPodIndex, bool allowMissing) {
    int nl = 0, thisOff = -1, thisN = 0;
    for (int m = 0; m < nmem; m++) {
      if (lane == 0) { res->member_leaf_num[m] = memLeaf[m]; res->member_pod_num[m] = memPods[m]; }
      if (memLeaf[m] == curLeafNum && thisOff < 0) { thisOff = nl + curPodIndex * memLeaf[m]; thisN = memLeaf[m]; }
      nl += memLeaf[m] * memPods[m];
    }
    const long long base = poolOff;
    if (base + 3ll * nl > pool_cap) { panic(HIVED_ERR_CAPACITY); return; }
    bool bad = false;
    for (int b = 0; b < nl; b += HIVED_WARPSZ) {
      int k = b + lane;
      if (k < nl) {
        int pl = phys[k];
        if (pl < 0) {
          bad = true;  // a cell that left the spec: reported as a nil triple, completed by the shim (hived.h)
          pool[base + 3 * k] = HIVED_NIL_CELL; pool[base + 3 * k + 1] = HIVED_NIL_CELL; pool[base + 3 * k + 2] = HIVED_NIL_CELL;
        } else {
          int t = -1;
          if (hasVirtual) t = d.v_pretype[virt[k]];  // type of the virtual leaf's preassigned cell (static per cell)
          pool[base + 3 * k] = d.p_node[pl];
          pool[base + 3 * k + 1] = d.p_leafidx[pl];
          pool[base + 3 * k + 2] = t;
        }
      }
      bad = hv_ballot(bad) != 0;
      if (bad && !allowMissing) { panic(HIVED_ERR_PLATFORM); return; }
    }
    hv_warp_sync();
    if (thisOff < 0) { panic(HIVED_ERR_PLATFORM); return; }
    int first = phys[thisOff];
    if (bad) ST(res->incomplete, 1);
    lastLeafOff = base;
    int firstReal = first;  // PodPlacementInfo.PhysicalNode comes from the pod's first cell that still exists
    if (bad && first < 0) {
      int j = firstIdx(thisN, [&](int q) { return phys[thisOff + q] >= 0; });
      firstReal = j >= 0 ? phys[thisOff + j] : -1;
    }
    lastNode = firstReal >= 0 ? d.p_node[firstReal] : -1; lastChain = first >= 0 ? d.p_chain[first] : -1;
    lastFirstLeaf = first >= 0 ? d.p_leafidx[first] : -1;
    lastKind = HIVED_KIND_BIND; lastHasVirtual = hasVirtual ? 1 : 0; lastNmem = nmem;
    for (int m = 0; m < nmem; m++) { lastMemLeaf[m] = memLeaf[m]; lastMemPods[m] = memPods[m]; }
    if (lane == 0) {  // the fixed part of the record, one sequence point
      res->kind = HIVED_KIND_BIND;
      res->has_virtual = lastHasVirtual;
      res->pod_index = curPodIndex;
      res->n_members = nmem;
      res->leaf_off = (int)base;
      res->n_leaves = nl;
      res->this_off = (int)(base + 3 * thisOff);
      res->this_n = thisN;
      res->node = lastNode;
      res->chain = lastChain;
    }
    hv_warp_sync();
    poolOff = base + 3ll * nl;
  }

  // ======================================================================================
  // AddAllocatedPod / createAllocatedAffinityGroup (hived_algorithm.go:247-270, 981-1041, 1224-1290)
  // ======================================================================================
  // utils.go:347-378 through the (node, chain) -> leaves table
  HIVED_DEV_NOINLINE int findPhysicalLeafCellInChain(int chain, int node, int leafIdx) const {
    if (chain < 0 || node < 0) return -1;
    int k = node * d.S.nChains + chain;
    const int32_t* list = d.ncl_list + d.ncl_off[k];
    int i = firstIdx(d.ncl_cnt[k], [&](int j) { return leafIdx < 0 || d.p_leafidx[list[j]] == leafIdx; });
    return i < 0 ? -1 : list[i];
  }
  // utils.go:318-345
  HIVED_DEV_NOINLINE int findPhysicalLeafCell(int chain, int node, int leafIdx) const {
    int g = findPhysicalLeafCellInChain(chain, node, leafIdx);
    if (g >= 0) return g;
    for (int c = 0; c < d.S.nChains; c++)
      if (c != chain) { g = findPhysicalLeafCellInChain(c, node, leafIdx); if (g >= 0) return g; }
    return -1;
  }
  // cell_allocation.go:348-372 over a list (ptr) or a contiguous range: the first free-and-unbound cell,
  // else the first cell of minimal priority among those below p
  HIVED_DEV_NOINLINE int getLowestPriorityVirtualCell(const int32_t* list, int base, int n, int p) const {
    int freeIdx = firstIdx(n, [&](int i) { int vc = list ? list[i] : base + i; return d.v_prio[vc] == FREE_PRIO && d.v_pcell[vc] < 0; });
    if (freeIdx >= 0) return list ? list[freeIdx] : base + freeIdx;
    const int NONE = 0x7fffffff;
    int best = NONE;  // (priority + 2) * 4096 + index: minimal priority, then first position
    for (int b = 0; b < n; b += HIVED_WARPSZ) {
      int i = b + lane;
      if (i < n) {
        int vc = list ? list[i] : base + i;
        int q = d.v_prio[vc];
        if (q != FREE_PRIO && q < p && q < HIVED_MAX_GUARANTEED_PRIORITY) { int key = (q + 2) * 4096 + i; if (key < best) best = key; }
      }
    }
    best = hv_reduce_min(best);
    if (best == NONE) return -1;
    int idx = best & 4095;
    return list ? list[idx] : base + idx;
  }
  // cell_allocation.go:317-346.  vccl: pinned -> the vset's cells at the level; else the VC's preassigned roots
  HIVED_DEV_NOINLINE int mapPhysicalCellToVirtual(int c, int vc, int chain, int pinned, int preassignedLevel, int p) const {
    int lc = d.p_level[c];
    // first level (>= the cell's) whose ancestor is bound, or that is the preassigned level, or beyond the top
    unsigned m = levelMask(lc, AS, [&](int l) {
      int a = d.p_anc[c * AS + l];
      return a < 0 || d.p_vcell[a] >= 0 || l == preassignedLevel;
    });
    if (!m) return -1;
    int ls = hv_ffs(m) - 1;
    int a = d.p_anc[c * AS + ls];
    if (a < 0) return -1;  // ran past the top: hierarchies do not match
    int virt;
    if (d.p_vcell[a] >= 0) {
      virt = d.p_vcell[a];
    } else if (pinned >= 0) {
      int vset = d.vc_pinned_vset[vc * d.S.nPinned + pinned];
      int k = vset * MAXL + preassignedLevel;
      virt = getLowestPriorityVirtualCell(nullptr, d.v_lvl_base[k], d.v_lvl_cnt[k], p);
    } else {
      int k = vcl(vc, chain, preassignedLevel);
      virt = getLowestPriorityVirtualCell(d.pre_list + d.pre_off[k], 0, d.pre_cnt[k], p);
    }
    for (int i = ls - lc; i > 0 && virt >= 0; i--) virt = getLowestPriorityVirtualCell(nullptr, d.v_child0[virt], d.v_nchild[virt], p);
    return virt;
  }

  struct BindView {  // api.PodBindInfo in ids
    int node, first_leaf, chain, has_preassigned, n_members;
    const int32_t* member_leaf_num;
    const int32_t* member_pod_num;
    const int32_t* leaves;  // triples
    const int32_t* physIds;  // optional: the physical leaf cells themselves (auto-commit of a fresh placement)
    const int32_t* virtIds;  // optional, with physIds: the virtual leaf cells Schedule chose (their preassigned cell's
                             // level names the PreassignedCellTypes entry without reading the emitted triples back)
  };

  // (getAllocatedPodIndex, utils.go:291-304, runs in the shim for recovered pods — algorithm.py — and is the identity on
  // a PodBindInfo that Schedule has just produced, see processEvent)

  // ---- whole-gang commit: the per-leaf loop of createAllocatedAffinityGroup (below) for the common case, with
  // lanes over the gang's leaves.  Preconditions (else false, nothing written): a fresh placement (cells known,
  // slots in emission order), a guaranteed priority above everything on the leaves, every leaf under an already
  // bound preassigned cell — then no free-list work, lazy preemption or safety check can occur.
  // The sequential loop gives every not-yet-bound physical cell on a leaf's path the FIRST free unbound child
  // of its parent's virtual cell (mapPhysicalCellToVirtual / getLowestPriorityVirtualCell) and binds the path
  // before looking at the next leaf; so under one virtual cell the r-th new child (in order of first
  // appearance among the leaves) gets the r-th free unbound virtual child: a rank/select per level, top-down.
  // Afterwards priorities only rise (max per ancestor) and states only become Used.
  HIVED_DEV bool commitGroupBatched(const hived_pod_spec_t& sp, const BindView& b, int g, int gnmem, const int* gleaf, const int* gpods_) {
    const int p = sp.priority, chain = b.chain;
    long long tq0 = pclock();
    if (!b.physIds || !b.has_preassigned || p < 0 || sp.vc < 0 || sp.vc >= d.S.nVCs || chain < 0 || chain >= d.S.nChains) return false;
    if (sp.pinned != -1) {
      if (sp.pinned < 0 || sp.pinned >= d.S.nPinned || d.vc_pinned_vset[sp.vc * d.S.nPinned + sp.pinned] < 0) return false;
    } else if (d.vc_chain_vset[sp.vc * d.S.nChains + chain] < 0) {
      return false;
    }
    if (b.n_members != gnmem) return false;  // the group's merged members (newGroup), still in registers
    int nl = 0;
    for (int m = 0; m < b.n_members; m++) {
      if (b.member_leaf_num[m] != gleaf[m] || b.member_pod_num[m] != gpods_[m]) return false;
      nl += b.member_leaf_num[m] * b.member_pod_num[m];
    }
    const int top = d.chain_top[chain];
    bool bad = false;
    int maxLs = 0;
    for (int b0 = 0; b0 < nl; b0 += HIVED_WARPSZ) {
      int i = b0 + lane;
      bool ok = true;
      int ls = 0;
      if (i < nl) {
        int L = b.physIds[i];
        int preLevel = -1;
        if (b.virtIds) {  // cell types are distinct along a chain: the type emitted for this leaf names exactly this level
          preLevel = d.v_prelevel[b.virtIds[i]];
        } else {
          int t = b.leaves[3 * i + 2];
          if (t != -1) for (int l = 1; l <= top; l++) if (d.chain_lvl_type[cl(chain, l)] == t) preLevel = l;
        }
        ok = L >= 0 && preLevel >= 1;
        ok = ok && d.p_chain[L] == chain && d.p_prio[L] == FREE_PRIO;
        if (ok) {
          // first level whose ancestor is bound, or the preassigned level, or past the top (mapPhysicalCellToVirtual):
          // all levels loaded at once (no early exit, so the loads overlap), then a bit scan
          unsigned stop = 0, bound = 0;
#pragma unroll 4
          for (int l = 1; l < AS; l++) {
            int a = d.p_anc[L * AS + l];
            int pv = a >= 0 ? d.p_vcell[a] : -1;
            if (a < 0 || pv >= 0 || l == preLevel) stop |= 1u << l;
            if (pv >= 0) bound |= 1u << l;
          }
          ls = stop ? hv_ffs(stop) - 1 : AS;
          ok = ls < AS && ((bound >> ls) & 1u);
          if (ok && ls == 1) ok = d.v_prio[d.p_vcell[L]] == FREE_PRIO;
          s.pl_v2[i] = ls;
        }
      }
      if (hv_ballot(!ok)) bad = true;
      ls = hv_reduce_max(ls);
      if (ls > maxLs) maxLs = ls;
    }
    if (bad) return false;
    hv_warp_sync();
    // bind, top-down
    bool failed = false;
    for (int l = maxLs - 1; l >= 1 && !failed; l--) {
      for (int b0 = 0; b0 < nl && !failed; b0 += HIVED_WARPSZ) {
        int i = b0 + lane;
        bool active = i < nl && l < s.pl_v2[i];
        int pa = -1, pv = -1;
        bool isNew = false;
        if (active) {
          int L = b.physIds[i];
          pa = d.p_anc[L * AS + l];
          pv = d.p_vcell[d.p_anc[L * AS + l + 1]];
          isNew = d.p_vcell[pa] < 0;
        }
        unsigned grp = hv_match(active ? pa : -1 - lane);
        bool leader = active && isNew && hv_ffs(grp) - 1 == lane;
        unsigned sib = hv_match(leader ? pv : -1 - lane);
        int rank = hv_popc(sib & hv_lanemask_lt());
        int sel = selectFreeUnboundChild(leader, pv, rank);
        if (hv_ballot(leader && sel < 0)) { failed = true; break; }
        if (leader) { d.p_vcell[pa] = sel; d.v_pcell[sel] = pa; d.v_healthy[sel] = d.p_healthy[pa]; }
        hv_warp_sync();
      }
    }
    if (failed) {  // no free unbound virtual cell somewhere: undo the bindings, let the sequential loop decide
      hv_warp_sync();
      for (int b0 = 0; b0 < nl; b0 += HIVED_WARPSZ) {
        int i = b0 + lane;
        if (i < nl) {
          int L = b.physIds[i];
          for (int l = 1; l < s.pl_v2[i]; l++) {
            int pa = d.p_anc[L * AS + l];
            int v = d.p_vcell[pa];
            if (v >= 0) { d.p_vcell[pa] = -1; d.v_pcell[v] = -1; d.v_state[v] = HIVED_CELL_FREE; d.v_healthy[v] = 1; }
          }
        }
        hv_warp_sync();
      }
      return false;
    }
    // allocateLeafCell (raise) + using group + setCellState(Used), all leaves at once
    stat_add(ST_LEAVES, nl);
    int32_t* ph = gphys(g);
    int32_t* vi = gvirt(g);
    for (int b0 = 0; b0 < nl; b0 += HIVED_WARPSZ) {
      int i = b0 + lane;
      bkMarkLeaves(i < nl, i < nl ? d.p_vcell[b.physIds[i]] : 0);
      if (i < nl) {
        int L = b.physIds[i];
        int V = d.p_vcell[L];
        const int ceil = multi ? d.v_prelevel[V] : AS;
        for (int lb = 1; lb < AS; lb += 4) {  // all loads of four levels, then their stores
          int pa[4], va[4], vq[4], pq[4], bd[4];
#pragma unroll
          for (int k = 0; k < 4; k++) {
            int l = lb + k;
            pa[k] = l < AS ? d.p_anc[L * AS + l] : -1;
            va[k] = l < AS ? d.v_anc[V * AS + l] : -1;
            if (l > ceil) pa[k] = -1;
          }
#pragma unroll
          for (int k = 0; k < 4; k++) {
            vq[k] = va[k] >= 0 ? d.v_prio[va[k]] : p;
            pq[k] = pa[k] >= 0 ? d.p_prio[pa[k]] : p;
            bd[k] = pa[k] >= 0 ? d.p_vcell[pa[k]] : -1;
          }
#pragma unroll
          for (int k = 0; k < 4; k++) {
            if (vq[k] < p) d.v_prio[va[k]] = p;
            if (pa[k] >= 0) {
              if (pq[k] < p) d.p_prio[pa[k]] = p;
              d.p_state[pa[k]] = HIVED_CELL_USED;
              if (bd[k] >= 0) d.v_state[bd[k]] = HIVED_CELL_USED;
            }
          }
        }
        d.p_using[L] = g;
        ph[i] = L; vi[i] = V;
      }
    }
    hv_warp_sync();
    return true;
  }

  HIVED_DEV void createAllocatedAffinityGroup(const hived_pod_spec_t& sp, const BindView& b) {
    int g = sp.group;
    long long tq = pclock();
    int gleaf[HIVED_MAX_MEMBERS], gpods_[HIVED_MAX_MEMBERS];
    int gnmem = newGroup(g, sp, HIVED_GROUP_ALLOCATED, gleaf, gpods_);
    if (commitGroupBatched(sp, b, g, gnmem, gleaf, gpods_)) return;
    bool shouldLazyPreempt = false;
    bool hasVirtualFlag = true;
    int32_t* ph = gphys(g);
    int32_t* vi = gvirt(g);
    int k = 0;
    for (int m = 0; m < b.n_members; m++) {
      int leafNumber = b.member_leaf_num[m];
      int gm = memberOf(g, leafNumber);
      int leafOff = 0, podOff = 0;
      if (gm >= 0) memberOffsets(g, gm, leafOff, podOff);
      int gmPods = gm >= 0 ? d.g_mem_pods[g * 8 + gm] : 0;
      for (int podIndex = 0; podIndex < b.member_pod_num[m]; podIndex++) {
        int node = b.leaves[3 * k];
        for (int li = 0; li < leafNumber; li++, k++) {
          // findAllocatedLeafCell :1224-1290
          int pLeaf = b.physIds ? b.physIds[k] : findPhysicalLeafCell(b.chain, node, b.leaves[3 * k + 1]);
          if (pLeaf < 0) continue;  // not found in the spec: ignored
          int vLeaf = -1;
          int lazy = 1;  // 0 nil, 1 false, 2 true
          if (!b.has_preassigned) {
            lazy = 2;
          } else if (hasVirtualFlag && !shouldLazyPreempt) {
            int t = b.leaves[3 * k + 2];
            if (t != -1) {
              int chainOfLeaf = d.p_chain[pLeaf];
              int preLevel = -1;
              for (int l = 1; l <= d.chain_top[chainOfLeaf]; l++)
                if (d.chain_lvl_type[cl(chainOfLeaf, l)] == t) preLevel = l;
              if (preLevel >= 0 && sp.vc >= 0 && sp.vc < d.S.nVCs) {
                bool have;
                if (sp.pinned != -1) have = sp.pinned >= 0 && sp.pinned < d.S.nPinned && d.vc_pinned_vset[sp.vc * d.S.nPinned + sp.pinned] >= 0;
                else have = d.vc_chain_vset[sp.vc * d.S.nChains + chainOfLeaf] >= 0;
                if (have) vLeaf = mapPhysicalCellToVirtual(pLeaf, sp.vc, chainOfLeaf, sp.pinned != -1 ? sp.pinned : -1, preLevel, sp.priority);
              }
              lazy = vLeaf < 0 ? 2 : 1;
            } else {
              lazy = 0;
            }
          }
          if (gm < 0 || podIndex >= gmPods) { panic(HIVED_ERR_PLATFORM); return; }  // index out of range
          int slot = leafOff + podIndex * leafNumber + li;
          ST(ph[slot], pLeaf);
          if (lazy == 0) {
            hasVirtualFlag = false;
          } else if (vLeaf >= 0) {
            ST(vi[slot], vLeaf);
            if (inFreeCellList(pLeaf) && d.v_prio[d.v_pre[vLeaf]] > FREE_PRIO) lazyPreemptCell(d.v_pre[vLeaf]);
          } else {
            shouldLazyPreempt = shouldLazyPreempt || lazy == 2;
          }
          bool safetyOk = commitLeaf(pLeaf, vLeaf, sp.priority, sp.vc, g);
          if (!safetyOk) shouldLazyPreempt = true;
          if (panicCode) return;
        }
      }
    }
    if (!hasVirtualFlag) { int fl = d.g_flags[g]; hv_warp_sync(); ST(d.g_flags[g], fl & ~GF_HAS_VIRTUAL); }
    if (shouldLazyPreempt) lazyPreemptAffinityGroup(g, nullptr);
  }

  HIVED_DEV int addAllocatedPod(const hived_pod_spec_t& sp, const BindView& b, int podIndexFromInfo) {
    int g = sp.group;
    int podIndex = 0;
    if (d.g_state[g] != HIVED_GROUP_NONE) {
      if (d.g_state[g] == HIVED_GROUP_PREEMPTING) allocatePreemptingAffinityGroup(g);
      podIndex = podIndexFromInfo;
      if (podIndex == -1) return 0;
    } else {
      createAllocatedAffinityGroup(sp, b);
      if (panicCode) return 0;
    }
    long long tq = pclock();
    int m = memberOf(g, sp.leaf_num);
    if (m < 0 || podIndex < 0 || podIndex >= d.g_mem_pods[g * 8 + m]) { panic(HIVED_ERR_PLATFORM); return 0; }
    int leafOff, podOff;
    memberOffsets(g, m, leafOff, podOff);
    ST(gpods(g)[podOff + podIndex], sp.pod);
    ST(d.pod_node[sp.pod], b.node);
    return 0;
  }

  // hived_algorithm.go:272-296
  // res->pod_index of a DELETE_ALLOCATED event: the pod id that occupied the slot the call cleared, -1 when it cleared
  // nothing (the reference clears allocatedPods[leafNum][podIndex] whoever sits there, :287: the shims need to know
  // whether THEIR pod left the table, see hived.h "Id lifetime")
  HIVED_DEV void deleteAllocatedPod(int g, int leafNum, int podIndex, int evVc, hived_result_t* res) {
    long long tq = pclock();
    ST(res->pod_index, -1);
    if (g < 0 || g >= d.S.maxGroups || d.g_state[g] == HIVED_GROUP_NONE) return;
    (void)evVc;  // (the host routes a DELETE by the VC its group was scheduled under, hived_engine.hpp prepare())
    if (podIndex == -1) return;
    int m = memberOf(g, leafNum);
    if (m < 0 || podIndex < 0 || podIndex >= d.g_mem_pods[g * 8 + m]) { panic(HIVED_ERR_PLATFORM); return; }
    int leafOff, podOff;
    memberOffsets(g, m, leafOff, podOff);
    const int occupant = gpods(g)[podOff + podIndex];
    ST(gpods(g)[podOff + podIndex], -1);
    ST(res->pod_index, occupant);
    const int32_t* po = gpods(g);
    if (firstIdx(groupPods(g), [&](int i) { return po[i] >= 0; }) >= 0) return;
    deleteAllocatedAffinityGroup(g);
  }
  // hived_algorithm.go:229-245
  HIVED_DEV_NOINLINE void deleteUnallocatedPod(int g, int pod) {
    if (g < 0 || g >= d.S.maxGroups || d.g_state[g] != HIVED_GROUP_PREEMPTING) return;
    int n = d.g_npre[g];
    for (int i = 0; i < n; i++)
      if (gpre(g)[i] == pod) { int lastv = gpre(g)[n - 1]; hv_warp_sync(); ST(gpre(g)[i], lastv); n--; ST(d.g_npre[g], n); break; }
    if (n == 0) deletePreemptingAffinityGroup(g);
  }

  // ======================================================================================
  // Schedule (hived_algorithm.go:180-224, 655-752)
  // ======================================================================================
  HIVED_DEV int schedule(const hived_pod_spec_t& sp, int phase, hived_result_t* res) {
    int g = sp.group;
    prioMask |= (sp.priority >= -1 && sp.priority < 62) ? (1ull << (sp.priority + 1)) : (1ull << 62);
    bool havePlacement = false, hasVirtual = false;
    const int32_t* phys = nullptr;
    const int32_t* virt = nullptr;
    int nmem = 0, memLeaf[HIVED_MAX_MEMBERS], memPods[HIVED_MAX_MEMBERS];
    int podIndex = 0, reason = 0, rcell = -1;
    bool victimsCollected = false;
    freshPlacement = false;
    leanOn = false; fastPlaced = false;
    long long tq = pclock();
    if (d.g_state[g] != HIVED_GROUP_NONE) {
      // schedulePodFromExistingGroup :655-712
      int nl = groupLeaves(g);
      const int32_t* ph = gphys(g);
      // collectBadOrNonSuggestedNodes utils.go:175-200 (ignoreK8sSuggestedNodes is never set on a group)
      // (only a preempting group's answer depends on it)
      bool badOrNonSuggested = d.g_state[g] != HIVED_GROUP_ALLOCATED && firstIdx(nl, [&](int i) {
        int c = ph[i];
        return c >= 0 && (!d.p_healthy[c] || !node_suggested(d.p_node[c]));
      }) >= 0;
      nmem = d.g_nmem[g];
      for (int m = 0; m < nmem; m++) { memLeaf[m] = d.g_mem_leaf[g * 8 + m]; memPods[m] = d.g_mem_pods[g * 8 + m]; }
      if (d.g_state[g] == HIVED_GROUP_ALLOCATED) {
        havePlacement = true; phys = gphys(g); virt = gvirt(g); hasVirtual = (d.g_flags[g] & GF_HAS_VIRTUAL) != 0;
        int m = memberOf(g, sp.leaf_num);
        podIndex = -1;
        if (m >= 0) {
          int leafOff, podOff;
          memberOffsets(g, m, leafOff, podOff);
          const int32_t* po = gpods(g) + podOff;
          podIndex = firstIdx(d.g_mem_pods[g * 8 + m], [&](int i) { return po[i] < 0; });
        }
        if (podIndex == -1) return HIVED_ERR_TOO_MANY_PODS;
      } else {
        if (phase == HIVED_PHASE_PREEMPTING && badOrNonSuggested) {
          deletePreemptingAffinityGroup(g);
        } else {
          havePlacement = true; phys = gphys(g); virt = gvirt(g); hasVirtual = (d.g_flags[g] & GF_HAS_VIRTUAL) != 0;
          int nOverlap;
          collectPreemptionVictims(phys, nl, res, nOverlap);
          victimsCollected = true;
          addPreemptingPod(g, sp.pod);
        }
      }
      if (panicCode) return panicCode;
    }
    if (d.g_state[g] == HIVED_GROUP_NONE) {
      // schedulePodFromNewGroup :714-752
      Req r;
      int rc = scheduleNewAffinityGroup(sp, r, hasVirtual, reason, rcell);
      if (panicCode) return panicCode;
      if (mgStop) return 0;
      if (rc < 0) return -rc;
      nmem = r.nmem;
      for (int m = 0; m < nmem; m++) { memLeaf[m] = r.memLeaf[m]; memPods[m] = r.memPods[m]; }
      podIndex = 0;
      if (rc == 1) {
        havePlacement = true; phys = s.pl_p; virt = s.pl_v; freshPlacement = true;
        int nOverlap;
        tq = pclock();
        if (leanOn) { nOverlap = 0; lastVictims = 0; }  // planLean saw every cell of the placement Free
        else collectPreemptionVictims(phys, r.nleaves, res, nOverlap);
        victimsCollected = true;
        if (panicCode) return panicCode;
        if (phase == HIVED_PHASE_PREEMPTING) {
          for (int i = 0; i < nOverlap; i++) {
            if (s.lz_group[i] < 0) { panic(HIVED_ERR_PLATFORM); return panicCode; }  // nil *AlgoAffinityGroup dereferenced (:1116)
            deletePreemptingAffinityGroup(s.lz_group[i]);
          }
          if (lastVictims != 0) {
            if (!hasVirtual) { panic(HIVED_ERR_PLATFORM); return panicCode; }  // nil virtual placement indexed in the reference
            for (int i = 0; i < r.nleaves; i++) { ST(s.pl_p2[i], s.pl_p[i]); ST(s.pl_v2[i], s.pl_v[i]); }
            createPreemptingAffinityGroup(g, sp, s.pl_p2, s.pl_v2);
          }
        }
        if (panicCode) return panicCode;
      } else {
        havePlacement = false;
      }
    }
    // generatePodScheduleResult utils.go:38-79
    if (!havePlacement) {
      ST(res->kind, HIVED_KIND_WAIT);
      ST(res->wait_code, reason);
      ST(res->wait_cell, rcell);
      stat_add(ST_WAIT, 1);
      return 0;
    }
    if (victimsCollected && lastVictims > 0) {
      ST(res->kind, HIVED_KIND_PREEMPT);
      ST(res->has_virtual, hasVirtual ? 1 : 0);
      stat_add(ST_PREEMPT, 1);
      return 0;
    }
    long long te0 = pclock();
    emitBind(res, nmem, memLeaf, memPods, phys, virt, hasVirtual, sp.leaf_num, podIndex,
             d.g_state[g] == HIVED_GROUP_ALLOCATED || d.g_state[g] == HIVED_GROUP_BEING_PREEMPTED);
    lastPodIndex = podIndex;
    stat_add(ST_CYC_EMIT, pclock() - te0);
    stat_add(ST_BIND, 1);
    return panicCode;
  }

  // ======================================================================================
  // one event (leader warp).  aux: hived_bind_info_t + leaf triples for the explicit AddAllocatedPod.
  // ======================================================================================
  static constexpr int EV_SCHEDULE_ONLY = 16, EV_ADD_ALLOCATED = 17;

  // pkg/internal/utils.go:256-287 + capacity checks (the shim validates first; this is defensive)
  HIVED_DEV int validateSpec(const hived_pod_spec_t& sp) const {
    if (sp.group < 0 || sp.group >= d.S.maxGroups || sp.pod < 0 || sp.pod >= d.S.maxPods) return HIVED_ERR_CAPACITY;
    if (sp.priority < OPP_PRIO || sp.priority > HIVED_MAX_GUARANTEED_PRIORITY || sp.leaf_num <= 0) return HIVED_ERR_BAD_SPEC;
    if (sp.n_members <= 0 || sp.n_members > HIVED_MAX_MEMBERS) return HIVED_ERR_BAD_SPEC;
    bool in = false;
    long long leaves = 0, pods = 0;
    for (int i = 0; i < sp.n_members; i++) {
      if (sp.member_pod_num[i] <= 0 || sp.member_leaf_num[i] <= 0) return HIVED_ERR_BAD_SPEC;
      if (sp.member_leaf_num[i] == sp.leaf_num) in = true;
      leaves += (long long)sp.member_leaf_num[i] * sp.member_pod_num[i];
      pods += sp.member_pod_num[i];
    }
    if (!in) return HIVED_ERR_BAD_SPEC;
    if (leaves > d.S.LS || pods > d.S.PS) return HIVED_ERR_CAPACITY;
    return 0;
  }

  HIVED_DEV void processEvent(const hived_event_t& ev, hived_result_t* res, const uint32_t* suggPool, const int32_t* aux) {
    panicCode = 0;
    long long tev0 = pclock();
    {  // clearResult: one word per lane
      int32_t* w = reinterpret_cast<int32_t*>(res);
      const int iWait = (int)(offsetof(hived_result_t, wait_cell) / 4), iChain = (int)(offsetof(hived_result_t, chain) / 4),
                iNode = (int)(offsetof(hived_result_t, node) / 4);
      for (int i = lane; i < (int)(sizeof(hived_result_t) / 4); i += HIVED_WARPSZ) w[i] = (i == iWait || i == iChain || i == iNode) ? -1 : 0;
      hv_warp_sync();
    }
    sugg = (ev.suggested_off >= 0 && suggPool) ? suggPool + ev.suggested_off : nullptr;
    int rc = 0;
    int type = ev.type;
    { long long tq = tev0; dbg(13, tq); }
    if (type == HIVED_EV_SCHEDULE || type == EV_SCHEDULE_ONLY) {
      const hived_pod_spec_t& sp = ev.spec;
      rc = validateSpec(sp);
      const bool existing = rc == 0 && d.g_state[sp.group] != HIVED_GROUP_NONE;
      long long ts0 = pclock();
      lastKind = -1;
      if (rc == 0 && existing && type == HIVED_EV_SCHEDULE && leanPodOfGang(sp, res)) {
        stat_add(ST_SCHEDULE, 1);  // scheduled and recorded (the commit is part of the lean step)
      } else if (rc == 0) {
        rc = schedule(sp, ev.phase, res);
        if (mgStop) return;
        if (rc == 0) stat_add(ST_SCHEDULE, 1);  // Schedule calls that returned a result (a panic is not a decision)
      }
      if (existing) { stat_add(ST_CYC_SCHED_EXISTING, pclock() - ts0); stat_add(ST_N_SCHED_EXISTING, 1); }
      if (rc == 0 && type == HIVED_EV_SCHEDULE && lastKind == HIVED_KIND_BIND) {
        // the filterRoutine sequence: AddAllocatedPod with the PodBindInfo just produced
        BindView b;
        b.node = lastNode; b.first_leaf = lastFirstLeaf; b.chain = lastChain; b.has_preassigned = 1;
        b.n_members = lastNmem; b.member_leaf_num = lastMemLeaf; b.member_pod_num = lastMemPods;
        b.leaves = pool + lastLeafOff;
        // a fresh placement's cells are known; (node, index) identifies them uniquely when S.directLeaf
        b.physIds = (d.S.directLeaf && freshPlacement) ? s.pl_p : nullptr;
        b.virtIds = (b.physIds && lastHasVirtual) ? s.pl_v : nullptr;
        sugg = nullptr;
        long long ta0 = pclock();
        long long tq = ta0;
        // getAllocatedPodIndex (utils.go:291-304) on the PodBindInfo just produced finds the row that holds this
        // pod's node and first leaf index — the row Schedule emitted it from (leaf cells of a gang are distinct)
        int api = lastPodIndex;
        if (leanOn && freshPlacement) applyLean(sp, api, lastNode);
        else { if (!existing) path_add(PC_GENERAL_COMMIT); addAllocatedPod(sp, b, api); }
        stat_add(ST_CYC_COMMIT, pclock() - ta0);
        if (existing) { stat_add(ST_CYC_COMMIT_POD, pclock() - ta0); stat_add(ST_N_COMMIT_POD, 1); }
        rc = panicCode;
      }
    } else if (type == EV_ADD_ALLOCATED) {
      const hived_bind_info_t* bi = reinterpret_cast<const hived_bind_info_t*>(aux);
      BindView b;
      b.node = bi->node; b.first_leaf = bi->first_leaf; b.chain = bi->chain; b.has_preassigned = bi->has_preassigned;
      b.n_members = bi->n_members; b.member_leaf_num = bi->member_leaf_num; b.member_pod_num = bi->member_pod_num;
      b.leaves = aux + sizeof(hived_bind_info_t) / 4;
      b.physIds = nullptr;
      b.virtIds = nullptr;
      rc = validateSpec(ev.spec);
      if (rc == 0) { addAllocatedPod(ev.spec, b, ev.arg0); rc = panicCode; }
    } else if (type == HIVED_EV_DELETE_ALLOCATED) {
      long long td0 = pclock();
      deleteAllocatedPod(ev.spec.group, ev.spec.leaf_num, ev.arg0, ev.spec.vc, res);
      if (mgStop) return;
      stat_add(ST_CYC_DELETE, pclock() - td0);
      if (ev.spec.group >= 0 && ev.spec.group < d.S.maxGroups && d.g_state[ev.spec.group] != HIVED_GROUP_NONE) {
        stat_add(ST_CYC_DELETE_POD, pclock() - td0); stat_add(ST_N_DELETE_POD, 1);
      }
      rc = panicCode;
    } else if (mgMode == 1) {
      mgStop = true;  // (the host only partitions calm batches; anything else runs alone)
      return;
    } else if (type == HIVED_EV_DELETE_UNALLOCATED) {
      deleteUnallocatedPod(ev.spec.group, ev.spec.pod);
      rc = panicCode;
    } else if (type == HIVED_EV_NODE_HEALTH) {
      setNodeHealth(ev.arg0, ev.arg1 != 0);
      rc = panicCode;
    } else {
      rc = HIVED_ERR_PLATFORM;
    }
    ST(res->error, rc);
    stat_add(ST_CYC_TOTAL, pclock() - tev0);
  }

  // NewHivedAlgorithm's dynamic part: initPinnedCells + initBadNodes (hived_algorithm.go:437-464)
  HIVED_DEV_NOINLINE void initState(const int32_t* pinnedOrder, int nPinnedOrder, const int32_t* badOrder, int nBad) {
    panicCode = 0;
    sugg = nullptr;
    for (int i = 0; i < nPinnedOrder; i++) {
      int pi = pinnedOrder[i];
      allocatePreassignedCell(d.pin_pcell[pi], d.pin_vc[pi], false);
      bindCell(d.pin_pcell[pi], d.pin_vcell[pi]);
    }
    for (int i = 0; i < nBad; i++) setNodeHealth(badOrder[i], false);
  }

  // After a VC-parallel batch: priority and state of the physical cells ABOVE every bound preassigned
  // cell, recomputed bottom-up from their children (priority = max; state = Used iff a child is Used —
  // exact whenever no cell is Reserving/Reserved, which is what the host checks before going parallel).
  HIVED_DEV void repairSharedAncestors() {
    if (hv_is_runahead()) return;  // (launched with the events kernel's geometry)
    for (int l = 2; l <= d.S.maxLevels; l++) {
      for (int chain = 0; chain < d.S.nChains; chain++) {
        int base = d.p_lvl_base[cl(chain, l)], cnt = d.p_lvl_cnt[cl(chain, l)];
        for (int i = hv_tid(); i < cnt; i += hv_nth()) {
          int cell = base + i;
          bool under = false;
          for (int L = l; L < AS; L++) { int a = d.p_anc[cell * AS + L]; if (a >= 0 && d.p_vcell[a] >= 0) { under = true; break; } }
          if (under) continue;
          int mx = FREE_PRIO; bool anyUsed = false;
          int c0 = d.p_child0[cell], n = d.p_nchild[cell];
          for (int j = 0; j < n; j++) { int q = d.p_prio[c0 + j]; if (q > mx) mx = q; if (d.p_state[c0 + j] == HIVED_CELL_USED) anyUsed = true; }
          d.p_prio[cell] = mx;
          d.p_state[cell] = anyUsed ? HIVED_CELL_USED : HIVED_CELL_FREE;
        }
      }
      hv_cta_sync();
    }
  }

  // the CTA's main loop: leader warp walks its share of the ordered batch, the other warps serve view
  // passes.  own[0..nOwn): ascending indices of the events this CTA owns (nullptr: all of them).
  HIVED_DEV void run(const hived_event_t* events, int n, hived_result_t* results, const uint32_t* suggPool, const int32_t* aux,
                     const int32_t* initLists, int nPinnedOrder, int nBad, const int32_t* own, int nOwn) {
    if (hv_warp() == 0) {
      poolOff = smp()->pool_off;
      int initPanic = 0;
      if (initLists) { initState(initLists, nPinnedOrder, initLists + nPinnedOrder, nBad); initPanic = panicCode; }
      if (!own) nOwn = n;
      // the CTA's event indices travel through a 64-entry window in shared memory, refilled 32 at a time (lane =
      // entry): the index of the next event is never a dependent global load on the leader's path
      if (own) { for (int q = lane; q < 64; q += HIVED_WARPSZ) { const int idx = mgStart + q; if (idx < nOwn) smp()->own_win[idx & 63] = own[idx]; } }
      ST(smp()->bkc_sched, -1);
      hv_warp_sync();
      auto ownAt = [&](int kk) { return own ? smp()->own_win[kk & 63] : kk; };
      int stopK = nOwn;
      mgStop = false;
      for (int k = mgStart; k < nOwn; k++) {
        if (own && k > mgStart && (k & 31) == 0) {
          for (int q = lane; q < 32; q += HIVED_WARPSZ) { const int idx = k + 32 + q; if (idx < nOwn) smp()->own_win[idx & 63] = own[idx]; }
          hv_warp_sync();
        }
        int i = ownAt(k);
        if (lane == 0) hv_publish_smem(&smp()->lead_k, k);
        curEvent = i;
        sharedHeld = false;
        long long tq = pclock();
        // The events are streamed from HBM once.  Event k was requested while event k-1 ran (asynchronous 16-byte
        // copies into the other half of the double buffer: no register target, nothing waits at a call boundary);
        // wait for it, then request event k+1 and pull event k+2 towards L2/L1.
        constexpr int EVQ = (int)(sizeof(hived_event_t) / 16);
        int32_t* cur = smp()->ev_words[k & 1];
        if (k == mgStart) { for (int q = lane; q < EVQ; q += HIVED_WARPSZ) hv_cp_async16(cur + 4 * q, reinterpret_cast<const char*>(&events[i]) + 16 * q); }
        hv_cp_async_wait();
        hv_warp_sync();
        if (k + 1 < nOwn) {
          const char* nxt = reinterpret_cast<const char*>(&events[ownAt(k + 1)]);
          int32_t* dst = smp()->ev_words[(k + 1) & 1];
          for (int q = lane; q < EVQ; q += HIVED_WARPSZ) hv_cp_async16(dst + 4 * q, nxt + 16 * q);
        }
        if (k + 2 < nOwn) hv_prefetch(&events[ownAt(k + 2)]);
        dbg(14, tq);
        processEvent(*reinterpret_cast<const hived_event_t*>(cur), &results[i], suggPool, aux);
        if (mgStop) { hv_cp_async_wait(); stopK = k; break; }
        tq = pclock();
        if (multi) {
          int next = (k + 1 < nOwn) ? ownAt(k + 1) : 0x7fffffff;
          // release: only an event that touched the cluster-wide state publishes anything another CTA may read
          // (free lists, counters, and the cells it put into them — with everything this CTA wrote to those
          // cells in earlier events, the fence being cumulative).  Other events move the progress word on with a
          // plain store: the fence (MEMBAR + L1 invalidation) after every event kept the L1 cold.
          if (sharedHeld) hv_fence();
          if (lane == 0) hv_st_volatile(d.progress + cta, next);
          hv_warp_sync();
        }
        dbg(15, tq);
      }
      if (lane == 0) hv_publish_smem(&smp()->lead_k, 0x7fffffff);
      flushWork();
      ST(smp()->pool_off, poolOff);
      ST(smp()->stop_k, stopK);
      ST(smp()->panic, initPanic);
      ST(smp()->cmd, CMD_EXIT);
      hv_cta_sync();
    } else if (hv_is_runahead()) {
      if (!initLists) runAhead(events, n, own, nOwn);
    } else {
      while (true) {
        hv_cta_sync();
        if (smp()->cmd == CMD_EXIT) break;
        sugg = smp()->a_sugg;
        viewOp();
      }
    }
  }

#if defined(__CUDACC__) && !defined(HIVED_EMU)
  // ---- resident ("serve") mode: the per-call path without a launch per call (hived_cuda.cu bk_run_small) ----------
  // The leader polls a request slot in MAPPED HOST memory, runs the request's events (at most SERVE_MAX_EVENTS) and
  // writes results + pool words back to mapped host memory; the workers serve view passes as in run().  The kernel
  // leaves by itself after `idleSpins` empty polls (a resident kernel must not outlive the calls it serves: any
  // device-wide synchronisation elsewhere in the process would wait for it) or on a STOP request.
  // slot layout: see ServeSlot in hived_cuda.cu; all offsets in 32-bit words.
  HIVED_DEV void serve(volatile int32_t* slot, int seq0, int idleSpins, hived_result_t* stageRes, uint32_t* dSugg, int32_t* dAux,
                       int nPinnedOrder, int nBad) {
    (void)nPinnedOrder; (void)nBad;
    if (hv_warp() == 0) {
      int lastSeq = seq0;
      ST(smp()->bkc_sched, -1);
      while (true) {
        int seq = lastSeq, spins = 0;
        // header line: [0] seq  [1] n (0 = STOP)  [2] suggWords  [3] auxWords  [4] poolCap
        int hdr = 0;
        while (true) {
          hdr = lane < 8 ? slot[lane] : 0;
          seq = hv_shfl(hdr, 0);
          if (seq != lastSeq) break;
          if (++spins > idleSpins) break;
        }
        if (seq == lastSeq) break;  // idle: leave
        const int n = hv_shfl(hdr, 1), suggWords = hv_shfl(hdr, 2), auxWords = hv_shfl(hdr, 3);
        pool_cap = hv_shfl(hdr, 4);
        lastSeq = seq;
        if (n <= 0) break;  // STOP
        // payload: events at word SERVE_EV_OFF, then the suggested bitmaps, then aux
        const volatile int32_t* pay = slot + SERVE_EV_OFF;
        const int evWords = (int)(sizeof(hived_event_t) / 4);
        const volatile int32_t* hs = pay + SERVE_MAX_EVENTS * evWords;
        for (int i = lane; i < suggWords; i += HIVED_WARPSZ) dSugg[i] = (uint32_t)hs[i];
        const volatile int32_t* ha = hs + suggWords;
        for (int i = lane; i < auxWords; i += HIVED_WARPSZ) dAux[i] = ha[i];
        hv_warp_sync();
        poolOff = 0;
        for (int k = 0; k < n; k++) {
          int32_t* cur = smp()->ev_words[k & 1];
          for (int i = lane; i < evWords; i += HIVED_WARPSZ) cur[i] = pay[k * evWords + i];
          hv_warp_sync();
          curEvent = k;
          sharedHeld = false;
          processEvent(*reinterpret_cast<const hived_event_t*>(cur), &stageRes[k], suggWords > 0 ? dSugg : nullptr, auxWords > 0 ? dAux : nullptr);
        }
        flushWork();
        hv_warp_sync();
        // response: results at SERVE_RES_OFF, pool window after them, then [poolOff, panic]; `done` last
        volatile int32_t* out = slot + SERVE_RES_OFF;
        const int32_t* sr = reinterpret_cast<const int32_t*>(stageRes);
        const int resWords = n * (int)(sizeof(hived_result_t) / 4);
        for (int i = lane; i < resWords; i += HIVED_WARPSZ) out[i] = sr[i];
        volatile int32_t* op = out + SERVE_MAX_EVENTS * (int)(sizeof(hived_result_t) / 4);
        const long long used = poolOff < SERVE_POOL_WINDOW ? poolOff : SERVE_POOL_WINDOW;
        for (int i = lane; i < (int)used; i += HIVED_WARPSZ) op[i] = pool[i];
        if (lane == 0) { slot[SERVE_DONE_OFF + 1] = (int32_t)poolOff; slot[SERVE_DONE_OFF + 2] = (int32_t)(poolOff >> 32); }
        __threadfence_system();
        hv_warp_sync();
        if (lane == 0) slot[SERVE_DONE_OFF] = seq;
        hv_warp_sync();
      }
      ST(smp()->cmd, CMD_EXIT);
      hv_cta_sync();
      if (lane == 0) { __threadfence_system(); slot[SERVE_DONE_OFF + 3] = lastSeq; slot[SERVE_DONE_OFF + 4] = 1; }  // exited
    } else if (hv_is_runahead()) {
      return;
    } else {
      while (true) {
        hv_cta_sync();
        if (smp()->cmd == CMD_EXIT) break;
        sugg = smp()->a_sugg;
        viewOp();
      }
    }
  }
#endif
};

#ifdef HIVED_DEV_IN_CONSTANT
#undef d
#endif

}  // namespace hived
