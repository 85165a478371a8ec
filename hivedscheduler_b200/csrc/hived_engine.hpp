// Host side of the library behind include/hived.h: owns the flattened topology, the device memory
// and the staging buffers; every ABI call becomes an ordered batch of events executed by the device
// program (hived_core.h).  Included by exactly one translation unit per build:
//   hived_cuda.cu        -> libhived_cuda.so   (the product: CUDA backend, sm_100a, no host path)
//   tests/emu/hived_emu.cpp -> test-only 1-thread emulation of the same device program (HIVED_EMU)
// The backend supplies bk_* (memory) and launchProgram().
#pragma once
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/hived.h"
#include "../../include/hived_bench.h"
#include "../../include/hived_hash.h"
#include "../../include/hived_multigpu.h"
#include "hived_topo.hpp"
#define HIVED_TOPO_CONSTS
#include "hived_core.h"

namespace hived {

struct Engine;
// ---- backend hooks (defined by the including translation unit)
void* bk_alloc(size_t bytes);
void bk_free(void* p);
void bk_h2d(void* dst, const void* src, size_t bytes);
void bk_d2h(void* dst, const void* src, size_t bytes);
void bk_d2d(void* dst, const void* src, size_t bytes);
void bk_zero(void* dst, size_t bytes);
void bk_quiesce(Engine& e);  // stop a resident per-call kernel before the state is written from elsewhere (CUDA backend)
void bk_forget(Engine& e);   // the context is being destroyed (CUDA backend: it may own the device's constant bank)
int bk_init(int& device, std::string& err);  // device: in = requested ordinal, out = the one in use
void bk_use_device(int device);  // make `device` current for the calling thread (contexts on several GPUs in one process)
// runs the program over n staged events; returns 0 or a HIVED_ERR_* code
int launchProgram(Engine& e, int n, bool withInit);
// after a VC-parallel run: rewrite the per-CTA pool slices as one pool in event order (dPool2) and patch the
// offsets in dResults; *total = words used
int bk_canonicalise(Engine& e, int n, long long* total);
// the per-call path (one pod per call, batches of a few events): everything staged through one pinned host buffer,
// copies and kernel queued on the context's stream, ONE synchronisation.  Returns -1 when it does not apply.
int bk_run_small(Engine& e, const hived_event_t* events, int n, const uint32_t* suggPool, int64_t suggWords, const int32_t* aux,
                 int64_t auxWords, hived_result_t* res, int32_t* pool, int64_t poolCap);
void bk_flush_l2();

struct Buf {
  void* p = nullptr;
  size_t bytes = 0;
  void ensure(size_t need) {
    if (need <= bytes) return;
    if (p) bk_free(p);
    size_t cap = need + need / 2 + 256;
    p = bk_alloc(cap);
    bytes = p ? cap : 0;
    if (!p) failed = true;
  }
  bool failed = false;  // an allocation failed: the owner reports HIVED_ERR_CAPACITY instead of launching
  ~Buf() { if (p) bk_free(p); }
};

struct Engine {
  FlatTopo T;
  Dev dev{};
  hived_options_t opt{};
  std::string err;
  std::vector<void*> allocs;
  std::vector<std::pair<void*, size_t>> mutableRegions;  // for save/restore
  std::vector<void*> savedRegions;
  // staging (device side)
  Buf dEvents, dResults, dPool, dSugg, dAux, dInit, dScalars, dOwn;
  long long poolOff = 0;
  // ---- VC-parallel execution
  int nCtaMax = 1, launchCta = 1;
  std::vector<int32_t> ownOff;          // [launchCta + 1] into the owner-sorted index list (device: dOwn)
  std::vector<long long> poolBase;      // [launchCta + 1] pool slice of every CTA
  std::vector<long long> poolEnd;       // [launchCta] first unused word of every slice after the run
  std::vector<uint8_t> ownerOf;         // owner CTA of every event of the batch being prepared (MAX_CTAS <= 255)
  std::vector<char> nodeBadHost;        // host mirror of the node health (decides whether a batch may run VC-parallel)
  std::vector<int32_t> groupStamp;      // batch that last named a group id (the two-VCs check is per batch)
  int32_t batchStamp = 0;
  std::vector<int32_t> groupVcHost;     // VC under which a group id was last scheduled (-1: never): DELETE events are routed
                                        // by it, not by the VC field of the event (which hived_delete_allocated_pod leaves 0)
  int badCount = 0;
  uint64_t prioMaskHost = 0;
  bool everRecovered = false;
  long long multiBatches = 0;
  int nPinnedOrder = 0, nBad = 0;
  uint64_t hash = HIVED_FNV_OFFSET;
  bool hashing = true;                  // maintain `hash` over hived_process_events results (HIVED_OPT_NO_RESULT_HASH)
  bool canonicalDone = false;           // the last VC-parallel run's pool was already compacted into dPool2
  long long canonicalTotal = 0;
  Buf dPool2, dScan;
  float lastKernelMs = 0.f;
  double kernelMsTotal = 0.0;
  long long kernelLaunches = 0;
  void* stream = nullptr;

  ~Engine() {
    bk_quiesce(*this);
    bk_forget(*this);
    for (void* p : allocs) bk_free(p);
    for (void* p : savedRegions) bk_free(p);
  }

  template <typename TT>
  TT* allocFill(size_t count, TT init) {
    if (count == 0) count = 1;
    std::vector<TT> h(count, init);
    TT* p = (TT*)bk_alloc(count * sizeof(TT));
    if (!p) { allocFailed = true; return nullptr; }
    bk_h2d(p, h.data(), count * sizeof(TT));
    allocs.push_back(p);
    return p;
  }
  bool allocFailed = false;  // some device allocation of create() failed (reported as HIVED_ERR_CAPACITY)
  const int32_t* uploadStatic(const std::vector<int32_t>& v) {
    size_t count = v.empty() ? 1 : v.size();
    int32_t* p = (int32_t*)bk_alloc(count * sizeof(int32_t));
    if (!p) { allocFailed = true; return nullptr; }
    if (!v.empty()) bk_h2d(p, v.data(), v.size() * sizeof(int32_t));
    allocs.push_back(p);
    return p;
  }

  int create(const char* spec, const hived_options_t* o) {
    if (o) opt = *o;
    hashing = !(opt.flags & HIVED_OPT_NO_RESULT_HASH);
    if (opt.max_groups <= 0) opt.max_groups = 1 << 17;
    if (opt.max_pods <= 0) opt.max_pods = 1 << 20;
    if (opt.max_group_leaves <= 0) opt.max_group_leaves = 64;
    if (opt.max_group_pods <= 0) opt.max_group_pods = 8;
    deviceOrdinal = opt.device;
    int rc = bk_init(deviceOrdinal, err);
    if (rc) return rc;
    try {
      T = buildTopo(spec);
    } catch (const TopoError& e) {
      err = e.what();
      return e.code;
    } catch (const std::exception& e) {
      err = e.what();
      return HIVED_ERR_BAD_CONFIG;
    }
    DevSizes& S = dev.S;
    S.NP = T.NP; S.NV = T.NV; S.nChains = T.nChains; S.nVCs = T.nVCs; S.nLeafTypes = T.nLeafTypes; S.nPinned = T.nPinned;
    S.nNodes = T.nNodes; S.nVsets = T.nVsets; S.nScheds = T.nScheds;
    S.flTotal = T.flTotal; S.dmTotal = T.dmTotal; S.cvTotal = (int32_t)T.cv_init.size();
    S.maxGroups = opt.max_groups; S.maxPods = opt.max_pods; S.LS = opt.max_group_leaves; S.PS = opt.max_group_pods;
    S.VX = S.LS * MAXL + 16; S.LZ = S.LS < 64 ? S.LS : 64;
    S.maxLevelCount = T.maxLevelCount; S.maxViewN = T.maxViewN; S.bitmapWords = (T.nNodes + 31) / 32;
    S.maxLevels = T.maxLevels; S.maxNodeLeaves = T.maxNodeLeaves; S.AS = T.AS; S.directLeaf = T.uniqueLeafIdx ? 1 : 0;
#define X(name) dev.name = uploadStatic(T.name);
    HIVED_STATIC_ARRAYS(X)
#undef X
#define Y(name, count, init)                                                   \
  {                                                                            \
    size_t cnt_ = (size_t)(count);                                             \
    dev.name = allocFill<int32_t>(cnt_, (int32_t)(init));                      \
    mutableRegions.push_back({dev.name, (cnt_ ? cnt_ : 1) * sizeof(int32_t)}); \
  }
    HIVED_MUTABLE_ARRAYS(Y)
#undef Y
    auto oom = [&]() {
      err = "out of device memory while creating the context (see hived_options_t: the group tables grow with "
            "max_groups * max_group_leaves)";
      return HIVED_ERR_CAPACITY;
    };
    if (allocFailed) return oom();  // before anything is copied into a null array
    dev.g_state.b = dev.g_vc.b = dev.g_prio.b = dev.g_flags.b = dev.g_nmem.b = dev.g_npre.b = dev.g_hdr;
    dev.g_mem_leaf.b = dev.g_mem_pods.b = dev.g_hdr;
    {  // g_vc starts at -1
      std::vector<int32_t> hdr((size_t)(S.maxGroups + GHOST_GROUPS) * GROUP_HDR_WORDS, 0);
      for (int g = 0; g < S.maxGroups + GHOST_GROUPS; g++) hdr[(size_t)g * GROUP_HDR_WORDS + 1] = -1;
      bk_h2d(dev.g_hdr, hdr.data(), hdr.size() * 4);
    }
    dev.stats = allocFill<long long>(ST_COUNT, 0);
    mutableRegions.push_back({dev.stats, ST_COUNT * sizeof(long long)});
    dev.epoch = allocFill<int32_t>(MAX_CTAS, 1);
    mutableRegions.push_back({dev.epoch, MAX_CTAS * sizeof(int32_t)});
    dev.progress = allocFill<int32_t>(MAX_CTAS, 0);
    if (allocFailed) return oom();
    // one private scratch set per CTA (VC-parallel execution uses up to nCtaMax CTAs)
    nCtaMax = T.nVCs < 16 ? (T.nVCs > 0 ? T.nVCs : 1) : 16;
    if (const char* env = getenv("HIVED_NCTA")) { int v = atoi(env); if (v >= 1 && v <= MAX_CTAS) nCtaMax = v < nCtaMax ? v : nCtaMax; }
    {
      std::vector<Scratch> sc(nCtaMax);
      for (int c = 0; c < nCtaMax; c++) {
#define Z(name, count) sc[c].name = allocFill<int32_t>((size_t)(count), 0);
        HIVED_SCRATCH_ARRAYS(Z)
#undef Z
      }
      Scratch* dsc = (Scratch*)bk_alloc(sizeof(Scratch) * nCtaMax);
      if (!dsc || allocFailed) { if (dsc) bk_free(dsc); return oom(); }
      bk_h2d(dsc, sc.data(), sizeof(Scratch) * nCtaMax);
      allocs.push_back(dsc);
      dev.scratch = dsc;
    }
    groupVcHost.assign((size_t)S.maxGroups, -1);
    nodeBadHost.assign(T.nNodes > 0 ? T.nNodes : 1, 1);  // every node starts bad (hived_algorithm.go:453-464)
    badCount = T.nNodes;
    // initial dynamic state (hived_algorithm.go:108-145, 365-409)
    bk_h2d(dev.vcFree, T.vcFree.data(), T.vcFree.size() * 4);
    bk_h2d(dev.allVCFree, T.allVCFree.data(), T.allVCFree.size() * 4);
    bk_h2d(dev.totalLeft, T.totalLeft.data(), T.totalLeft.size() * 4);
    if (!T.fl_init_data.empty()) bk_h2d(dev.fl_data, T.fl_init_data.data(), T.fl_init_data.size() * 4);
    bk_h2d(dev.fl_len, T.fl_init_len.data(), T.fl_init_len.size() * 4);
    {
      std::vector<int32_t> flpos(T.NP ? T.NP : 1, -1);
      for (int c = 0; c < T.nChains; c++)
        for (int l = 1; l < MAXL; l++)
          for (int i = 0; i < T.fl_init_len[c * MAXL + l]; i++) flpos[T.fl_init_data[T.fl_base[c * MAXL + l] + i]] = i;
      bk_h2d(dev.p_flpos, flpos.data(), flpos.size() * 4);
    }
    if (!T.cv_init.empty()) bk_h2d(dev.cv, T.cv_init.data(), T.cv_init.size() * 4);
    // initPinnedCells + initBadNodes run on the device
    std::vector<int32_t> init = T.pinned_init_order;
    nPinnedOrder = (int)T.pinned_init_order.size();
    init.insert(init.end(), T.bad_init_order.begin(), T.bad_init_order.end());
    nBad = (int)T.bad_init_order.size();
    dInit.ensure((init.size() + 1) * 4);
    if (!init.empty()) bk_h2d(dInit.p, init.data(), init.size() * 4);
    dScalars.ensure(MAX_CTAS * 4 * sizeof(long long));
    dOwn.ensure(64);
    dPool.ensure(4096 * 4);
    dResults.ensure(sizeof(hived_result_t));
    dEvents.ensure(sizeof(hived_event_t));
    poolOff = 0;
    if (allocFailed || buffersFailed()) {
      err = "out of device memory while creating the context (see hived_options_t: the group tables grow with "
            "max_groups * max_group_leaves)";
      return HIVED_ERR_CAPACITY;
    }
    rc = launchProgram(*this, 0, true);
    if (rc) { if (err.empty()) err = "device initialisation failed"; return rc; }
    return 0;
  }

  // Decide how the batch runs and stage everything but the results.  A batch runs VC-parallel (one CTA per
  // group of VCs) only in the regime where VCs interact through nothing but the chain-wide free lists:
  // every node healthy, a single guaranteed priority ever used (so no preemption, no lazy preemption, no
  // opportunistic cells), no recovery calls, and only SCHEDULE / DELETE events with valid VC ids.
  int prepare(const hived_event_t* events, int n, int64_t poolCap) {
    launchCta = 1;
    batchStamp++;
    if (groupStamp.size() != groupVcHost.size()) groupStamp.assign(groupVcHost.size(), 0);
    uint64_t mask = prioMaskHost;
    bool simple = nCtaMax > 1 && n >= 256 && badCount == 0 && !everRecovered;
    // one pass over the events: regime flags, the owner CTA of every event and the pool words every owner may need
    const int C = nCtaMax < T.nVCs ? nCtaMax : T.nVCs;
    std::vector<int32_t> cnt(C + 1, 0);
    std::vector<long long> need(C, 0);
    ownerOf.resize((size_t)(n > 0 ? n : 1));
    for (int i = 0; i < n; i++) {
      const hived_event_t& ev = events[i];
      if (ev.type == HIVED_EV_SCHEDULE || ev.type == Core::EV_SCHEDULE_ONLY || ev.type == Core::EV_ADD_ALLOCATED) {
        int p = ev.spec.priority;
        mask |= (p >= -1 && p < 62) ? (1ull << (p + 1)) : (1ull << 62);
      }
      if (ev.type != HIVED_EV_SCHEDULE && ev.type != HIVED_EV_DELETE_ALLOCATED) simple = false;
      // the VC that owns the event: a SCHEDULE names it; a DELETE belongs to the VC its group was scheduled under
      // (the event's own VC field is optional, hived.h).  A group id seen under two VCs, or an unknown one: sequential.
      int evVc = ev.spec.vc;
      const int g = ev.spec.group;
      if (ev.type == HIVED_EV_SCHEDULE || ev.type == Core::EV_SCHEDULE_ONLY) {
        if (g >= 0 && g < (int)groupVcHost.size() && ev.spec.vc >= 0 && ev.spec.vc < T.nVCs) {
          // a group id that THIS batch has already used under another VC (ids are recycled, hived.h "Id lifetime": the
          // old incarnation's release and the new one's creation would meet in the same table row on two CTAs)
          if (groupStamp[g] == batchStamp && groupVcHost[g] >= 0 && groupVcHost[g] != ev.spec.vc) simple = false;
          groupVcHost[g] = ev.spec.vc;
          groupStamp[g] = batchStamp;
        }
      } else if (ev.type == HIVED_EV_DELETE_ALLOCATED) {
        evVc = (g >= 0 && g < (int)groupVcHost.size()) ? groupVcHost[g] : -1;
        if (evVc < 0) evVc = (ev.spec.vc >= 0 && ev.spec.vc < T.nVCs) ? ev.spec.vc : 0;  // unknown group: a no-op wherever it runs
        if (g >= 0 && g < (int)groupStamp.size()) groupStamp[g] = batchStamp;
      }
      if (evVc < 0 || evVc >= T.nVCs) simple = false;
      if (ev.type == Core::EV_ADD_ALLOCATED) everRecovered = true;
      if (simple) {
        int o = evVc % C;
        ownerOf[i] = (uint8_t)o;
        cnt[o + 1]++;
        if (ev.type == HIVED_EV_SCHEDULE) {
          long long leaves = 0;
          for (int m = 0; m < ev.spec.n_members && m < HIVED_MAX_MEMBERS; m++)
            leaves += (long long)ev.spec.member_leaf_num[m] * ev.spec.member_pod_num[m];
          need[o] += 3 * leaves;
        }
      }
    }
    prioMaskHost = mask;
    if ((mask & (mask - 1)) != 0 || (mask & 1)) simple = false;  // more than one priority, or opportunistic (-1)
    ownOff.assign(2, 0); ownOff[1] = n;
    poolBase.assign(2, 0); poolBase[1] = poolCap;
    if (simple) {
      long long total = 0;
      for (int c = 0; c < C; c++) total += need[c];
      if (total <= poolCap) {
        launchCta = C;
        ownOff.assign(C + 1, 0);
        for (int c = 0; c < C; c++) ownOff[c + 1] = ownOff[c] + cnt[c + 1];
        std::vector<int32_t> own(n), fill(ownOff.begin(), ownOff.end() - 1);
        for (int i = 0; i < n; i++) own[fill[ownerOf[i]]++] = i;
        dOwn.ensure((size_t)(n + C + 2) * 4);
        bk_h2d(dOwn.p, own.data(), (size_t)n * 4);
        bk_h2d((int32_t*)dOwn.p + n, ownOff.data(), (size_t)(C + 1) * 4);
        poolBase.assign(C + 1, 0);
        for (int c = 0; c < C; c++) poolBase[c + 1] = poolBase[c] + need[c];
        std::vector<int32_t> prog(MAX_CTAS, 0x7fffffff);
        for (int c = 0; c < C; c++) if (ownOff[c + 1] > ownOff[c]) prog[c] = own[ownOff[c]];
        bk_h2d(dev.progress, prog.data(), MAX_CTAS * 4);
        multiBatches++;
      }
    }
    dEvents.ensure((size_t)(n > 0 ? n : 1) * sizeof(hived_event_t));
    dResults.ensure((size_t)(n > 0 ? n : 1) * sizeof(hived_result_t));
    dPool.ensure((size_t)(poolCap > 0 ? poolCap : 1) * 4);
    if (n > 0) bk_h2d(dEvents.p, events, (size_t)n * sizeof(hived_event_t));
    poolCapWords = poolCap;
    stagedN = n;
    stagedEvents = events;
    return 0;
  }
  // health events change the host mirror (applied after the batch ran)
  void trackHealth(const hived_event_t* events, int n) {
    for (int i = 0; i < n; i++) {
      if (events[i].type != HIVED_EV_NODE_HEALTH) continue;
      int node = events[i].arg0;
      if (node < 0 || node >= T.nNodes) continue;
      char bad = events[i].arg1 ? 0 : 1;
      if (nodeBadHost[node] != bad) { nodeBadHost[node] = bad; badCount += bad ? 1 : -1; }
    }
  }
  // results + pool to the caller, in the canonical layout (pool slices in event order)
  int fetch(hived_result_t* res, int32_t* pool, int64_t poolCap, int64_t* used) {
    bk_use_device(deviceOrdinal);
    int n = stagedN;
    if (launchCta == 1) {
      if (n > 0) bk_d2h(res, dResults.p, (size_t)n * sizeof(hived_result_t));
      if (poolOff > poolCap) return HIVED_ERR_CAPACITY;
      if (poolOff > 0) bk_d2h(pool, dPool.p, (size_t)poolOff * 4);
      if (used) *used = poolOff;
      return 0;
    }
    // VC-parallel run: every CTA wrote into its own slice; compact the slices into event order on the device
    // (scan of the per-result word counts + gather) and copy the canonical pool straight into the caller's buffer
    if (!canonicalDone) {
      int rc = bk_canonicalise(*this, n, &canonicalTotal);
      if (rc) return rc;
      canonicalDone = true;
    }
    if (canonicalTotal > poolCap) return HIVED_ERR_CAPACITY;
    if (n > 0) bk_d2h(res, dResults.p, (size_t)n * sizeof(hived_result_t));
    if (canonicalTotal > 0) bk_d2h(pool, dPool2.p, (size_t)canonicalTotal * 4);
    poolOff = canonicalTotal;
    if (used) *used = canonicalTotal;
    return 0;
  }
  const hived_event_t* stagedEvents = nullptr;

  // stage + run a batch; host result/pool buffers are caller-owned
  int runBatch(const hived_event_t* events, int n, const uint32_t* suggPool, int64_t suggWords, const int32_t* aux,
               int64_t auxWords, hived_result_t* res, int32_t* pool, int64_t poolCap) {
    if (n <= 0) return 0;
    bk_use_device(deviceOrdinal);
    if (n <= SMALL_BATCH) {
      int rc = bk_run_small(*this, events, n, suggPool, suggWords, aux, auxWords, res, pool, poolCap);
      if (rc >= 0) { if (rc == 0) trackHealth(events, n); return rc; }
    }
    prepare(events, n, poolCap);
    hasSugg = suggPool != nullptr && suggWords > 0;
    if (hasSugg) { dSugg.ensure((size_t)suggWords * 4); bk_h2d(dSugg.p, suggPool, (size_t)suggWords * 4); }
    hasAux = aux != nullptr && auxWords > 0;
    if (hasAux) { dAux.ensure((size_t)auxWords * 4); bk_h2d(dAux.p, aux, (size_t)auxWords * 4); }
    poolOff = 0;
    canonicalDone = false;
    if (buffersFailed()) { err = "out of device memory while staging the batch"; return HIVED_ERR_CAPACITY; }
    int rc = launchProgram(*this, n, false);
    if (rc) return rc;
    trackHealth(events, n);
    return fetch(res, pool, poolCap, nullptr);
  }
  static constexpr int SMALL_BATCH = 8;
  // what prepare() decides per event, for bk_run_small (no device traffic)
  void notePriorities(const hived_event_t* events, int n) {
    for (int i = 0; i < n; i++) {
      const hived_event_t& ev = events[i];
      if (ev.type == HIVED_EV_SCHEDULE || ev.type == Core::EV_SCHEDULE_ONLY || ev.type == Core::EV_ADD_ALLOCATED) {
        int p = ev.spec.priority;
        prioMaskHost |= (p >= -1 && p < 62) ? (1ull << (p + 1)) : (1ull << 62);
      }
      if (ev.type == Core::EV_ADD_ALLOCATED) everRecovered = true;
      if ((ev.type == HIVED_EV_SCHEDULE || ev.type == Core::EV_SCHEDULE_ONLY) && ev.spec.group >= 0 &&
          ev.spec.group < (int)groupVcHost.size() && ev.spec.vc >= 0 && ev.spec.vc < T.nVCs)
        groupVcHost[ev.spec.group] = ev.spec.vc;
    }
  }
  bool buffersFailed() const {
    return dEvents.failed || dResults.failed || dPool.failed || dSugg.failed || dAux.failed || dInit.failed || dScalars.failed ||
           dOwn.failed || dPool2.failed || dScan.failed;
  }
  int deviceOrdinal = 0;
  bool hasSugg = false, hasAux = false;
  int64_t poolCapWords = 0;
  int stagedN = 0;
  int stage(const hived_event_t* events, int n, int64_t poolCap) {
    bk_use_device(deviceOrdinal);
    hasSugg = false; hasAux = false;
    return prepare(events, n, poolCap);
  }
  int runStaged() {
    bk_use_device(deviceOrdinal);
    poolOff = 0;
    canonicalDone = false;
    if (launchCta > 1) {  // the progress words were consumed by the previous run
      std::vector<int32_t> own(stagedN), prog(MAX_CTAS, 0x7fffffff);
      bk_d2h(own.data(), dOwn.p, (size_t)stagedN * 4);
      for (int c = 0; c < launchCta; c++) if (ownOff[c + 1] > ownOff[c]) prog[c] = own[ownOff[c]];
      bk_h2d(dev.progress, prog.data(), MAX_CTAS * 4);
    }
    return launchProgram(*this, stagedN, false);
  }

  // ---- multi-GPU partition of one calm batch (include/hived_multigpu.h) --------------------------------------
  // Every rank holds the whole cluster; rank r owns the VCs v with v % world == r and runs one CTA per owned VC.
  // VCs interact only through the chain-wide buddy free lists and counters (`sharedArrays`): a rank runs its
  // events up to the first one that may touch them (mgRun), the ranks agree on the smallest such event (min over
  // ranks: the caller's collective), its owner runs it alone (mgSolo) and ships the arrays to everybody else.
  int mgMode = 0, mgRank = 0, mgWorld = 1;
  std::vector<int32_t> mgCursor, mgLimit, mgStopOut, mgOwnHost;
  std::vector<long long> mgPoolCur;
  std::vector<std::pair<void*, size_t>> sharedArrays() {
    std::vector<std::pair<void*, size_t>> v;
    const size_t NP = (size_t)dev.S.NP * 4, LV = (size_t)dev.S.nChains * MAXL * 4;
    v.push_back({dev.p_split, NP}); v.push_back({dev.p_flpos, NP}); v.push_back({dev.p_bfpos, NP});
    v.push_back({dev.p_dmpos, NP}); v.push_back({dev.p_dmvc, NP});
    v.push_back({dev.vcFree, LV * dev.S.nVCs}); v.push_back({dev.allVCFree, LV}); v.push_back({dev.totalLeft, LV});
    v.push_back({dev.allVCDoomed, LV});
    v.push_back({dev.fl_data, (size_t)dev.S.flTotal * 4}); v.push_back({dev.fl_len, LV}); v.push_back({dev.fl_dup, LV});
    v.push_back({dev.bf_data, (size_t)dev.S.flTotal * 4}); v.push_back({dev.bf_len, LV});
    v.push_back({dev.dm_data, (size_t)dev.S.dmTotal * 4}); v.push_back({dev.dm_len, LV * dev.S.nVCs});
    return v;
  }
  int64_t mgSharedBytes() { int64_t t = 0; for (auto& r : sharedArrays()) t += (int64_t)((r.second + 15) & ~(size_t)15); return t; }
  void mgExportShared(void* dst) {
    bk_use_device(deviceOrdinal);
    char* o = (char*)dst;
    for (auto& r : sharedArrays()) { if (r.second) bk_d2d(o, r.first, r.second); o += (r.second + 15) & ~(size_t)15; }
  }
  void mgImportShared(const void* src) {
    bk_use_device(deviceOrdinal);
    bk_quiesce(*this);
    const char* o = (const char*)src;
    for (auto& r : sharedArrays()) { if (r.second) bk_d2d(r.first, o, r.second); o += (r.second + 15) & ~(size_t)15; }
  }
  int mgStage(const hived_event_t* events, int n, int64_t poolCap, int rank, int world) {
    bk_use_device(deviceOrdinal);
    if (world < 1 || rank < 0 || rank >= world) { err = "multi-GPU partition: bad rank/world"; return HIVED_ERR_BAD_SPEC; }
    if (badCount != 0 || everRecovered) { err = "multi-GPU partition: only calm batches (every node healthy, no recovery)"; return HIVED_ERR_BAD_SPEC; }
    batchStamp++;
    if (groupStamp.size() != groupVcHost.size()) groupStamp.assign(groupVcHost.size(), 0);
    uint64_t mask = prioMaskHost;
    const int C = (T.nVCs - rank + world - 1) / world > 0 ? (T.nVCs - rank + world - 1) / world : 0;
    if (C > MAX_CTAS) { err = "multi-GPU partition: more VCs per rank than CTAs"; return HIVED_ERR_CAPACITY; }
    const int CL = C > 0 ? C : 1;
    std::vector<std::vector<int32_t>> lists(CL);
    std::vector<long long> need(CL, 0);
    for (int i = 0; i < n; i++) {
      const hived_event_t& ev = events[i];
      if (ev.type != HIVED_EV_SCHEDULE && ev.type != HIVED_EV_DELETE_ALLOCATED) { err = "multi-GPU partition: only SCHEDULE / DELETE_ALLOCATED events"; return HIVED_ERR_BAD_SPEC; }
      int evVc = ev.spec.vc;
      const int g = ev.spec.group;
      if (ev.type == HIVED_EV_SCHEDULE) {
        int p = ev.spec.priority;
        mask |= (p >= -1 && p < 62) ? (1ull << (p + 1)) : (1ull << 62);
        if (g >= 0 && g < (int)groupVcHost.size() && evVc >= 0 && evVc < T.nVCs) {
          if (groupStamp[g] == batchStamp && groupVcHost[g] >= 0 && groupVcHost[g] != evVc) { err = "multi-GPU partition: a group id used under two VCs in one batch"; return HIVED_ERR_BAD_SPEC; }
          groupVcHost[g] = evVc;
          groupStamp[g] = batchStamp;
        }
      } else {
        if (g >= 0 && g < (int)groupStamp.size()) groupStamp[g] = batchStamp;
        evVc = (g >= 0 && g < (int)groupVcHost.size()) ? groupVcHost[g] : -1;
        if (evVc < 0) evVc = (ev.spec.vc >= 0 && ev.spec.vc < T.nVCs) ? ev.spec.vc : 0;
      }
      if (evVc < 0 || evVc >= T.nVCs) { err = "multi-GPU partition: event with an unknown VC"; return HIVED_ERR_BAD_SPEC; }
      if (evVc % world != rank) continue;
      const int c = evVc / world;
      lists[c].push_back(i);
      if (ev.type == HIVED_EV_SCHEDULE) {
        long long leaves = 0;
        for (int m = 0; m < ev.spec.n_members && m < HIVED_MAX_MEMBERS; m++) leaves += (long long)ev.spec.member_leaf_num[m] * ev.spec.member_pod_num[m];
        need[c] += 3 * leaves;
      }
    }
    prioMaskHost = mask;
    if ((mask & (mask - 1)) != 0 || (mask & 1)) { err = "multi-GPU partition: more than one priority in use"; return HIVED_ERR_BAD_SPEC; }
    launchCta = CL;
    ownOff.assign(CL + 1, 0);
    mgOwnHost.clear();
    for (int c = 0; c < CL; c++) { mgOwnHost.insert(mgOwnHost.end(), lists[c].begin(), lists[c].end()); ownOff[c + 1] = (int32_t)mgOwnHost.size(); }
    poolBase.assign(CL + 1, 0);
    for (int c = 0; c < CL; c++) poolBase[c + 1] = poolBase[c] + need[c];
    if (poolBase[CL] > poolCap) { err = "multi-GPU partition: pool too small"; return HIVED_ERR_CAPACITY; }
    dOwn.ensure((size_t)(n + CL + 2) * 4);
    if (!mgOwnHost.empty()) bk_h2d(dOwn.p, mgOwnHost.data(), mgOwnHost.size() * 4);
    bk_h2d((int32_t*)dOwn.p + n, ownOff.data(), (size_t)(CL + 1) * 4);
    dEvents.ensure((size_t)(n > 0 ? n : 1) * sizeof(hived_event_t));
    dResults.ensure((size_t)(n > 0 ? n : 1) * sizeof(hived_result_t));
    dPool.ensure((size_t)(poolCap > 0 ? poolCap : 1) * 4);
    if (buffersFailed()) { err = "out of device memory while staging the batch"; return HIVED_ERR_CAPACITY; }
    if (n > 0) bk_h2d(dEvents.p, events, (size_t)n * sizeof(hived_event_t));
    bk_zero(dResults.p, (size_t)(n > 0 ? n : 1) * sizeof(hived_result_t));  // events of other ranks stay all-zero here
    poolCapWords = poolCap;
    stagedN = n;
    stagedEvents = events;
    hasSugg = false; hasAux = false;
    canonicalDone = false;
    mgRank = rank; mgWorld = world;
    mgCursor.assign(CL, 0);
    mgPoolCur.assign(poolBase.begin(), poolBase.end() - 1);
    return 0;
  }
  // run the staged batch again (bench: after the scheduler state was rewound)
  int mgReset() {
    bk_use_device(deviceOrdinal);
    if (mgCursor.empty()) { err = "multi-GPU partition: nothing staged"; return HIVED_ERR_BAD_SPEC; }
    bk_zero(dResults.p, (size_t)(stagedN > 0 ? stagedN : 1) * sizeof(hived_result_t));
    mgCursor.assign(launchCta, 0);
    mgPoolCur.assign(poolBase.begin(), poolBase.end() - 1);
    canonicalDone = false;
    return 0;
  }
  // first pending event of every CTA's list; 0x7fffffff when the rank is through
  int mgNextStop() const {
    int mn = 0x7fffffff;
    for (int c = 0; c < launchCta; c++) {
      const int k = mgCursor[c], cnt = ownOff[c + 1] - ownOff[c];
      if (k < cnt && mgOwnHost[ownOff[c] + k] < mn) mn = mgOwnHost[ownOff[c] + k];
    }
    return mn;
  }
  int mgLaunch(int mode) {
    mgMode = mode;
    int rc = launchProgram(*this, stagedN, false);
    mgMode = 0;
    if (rc) return rc;
    for (int c = 0; c < launchCta; c++) { mgCursor[c] = mgStopOut[c]; mgPoolCur[c] = poolEnd[c]; }
    return 0;
  }
  // every CTA of this rank runs its events BELOW `horizon` until its next event that may touch the cluster-wide state.
  // *stopEvent = the first such event among this rank's events below the horizon (the CTA is parked before it), or
  // 0x7fffffff when every owned event below the horizon has run.  The horizon keeps the VCs moving together: without
  // one, a CTA runs on to its own next such event while the others stay parked at theirs, and the whole batch
  // degenerates to one VC at a time (measured: 8x slower than one GPU).
  int mgRun(int32_t horizon, int32_t* stopEvent) {
    bk_use_device(deviceOrdinal);
    mgLimit.assign(launchCta, 0);
    bool work = false;
    for (int c = 0; c < launchCta; c++) {
      const int32_t* lst = mgOwnHost.data() + ownOff[c];
      const int cnt = ownOff[c + 1] - ownOff[c];
      mgLimit[c] = (int32_t)(std::lower_bound(lst, lst + cnt, horizon) - lst);  // events of the list with index < horizon
      if (mgLimit[c] < mgCursor[c]) mgLimit[c] = mgCursor[c];
      if (mgLimit[c] > mgCursor[c]) work = true;
    }
    if (work) {
      int rc = mgLaunch(1);
      if (rc) return rc;
    }
    int mn = 0x7fffffff;
    for (int c = 0; c < launchCta; c++)
      if (mgCursor[c] < mgLimit[c] && mgOwnHost[ownOff[c] + mgCursor[c]] < mn) mn = mgOwnHost[ownOff[c] + mgCursor[c]];  // parked
    *stopEvent = mn;
    return 0;
  }
  // the event every rank stopped at or before runs alone on the cluster, on the rank that owns it
  int mgSolo(int eventIndex) {
    bk_use_device(deviceOrdinal);
    mgLimit.assign(mgCursor.begin(), mgCursor.end());
    int owner = -1;
    for (int c = 0; c < launchCta; c++) {
      const int k = mgCursor[c], cnt = ownOff[c + 1] - ownOff[c];
      if (k < cnt && mgOwnHost[ownOff[c] + k] == eventIndex) { owner = c; break; }
    }
    if (owner < 0) { err = "multi-GPU partition: this rank is not stopped at that event"; return HIVED_ERR_BAD_SPEC; }
    mgLimit[owner] = mgCursor[owner] + 1;
    return mgLaunch(2);
  }
  // after the last round: the cells above the bound preassigned cells are re-derived (as after a VC-parallel batch)
  int mgFinish() {
    bk_use_device(deviceOrdinal);
    mgMode = 3;
    int rc = launchProgram(*this, stagedN, false);
    mgMode = 0;
    poolEnd.assign(mgPoolCur.begin(), mgPoolCur.end());
    return rc;
  }

  void readArray(const int32_t* devPtr, std::vector<int32_t>& out, size_t count) {
    out.resize(count ? count : 1);
    bk_d2h(out.data(), devPtr, out.size() * 4);
  }
  void saveState() {
    bk_use_device(deviceOrdinal);
    if (savedRegions.empty())
      for (auto& r : mutableRegions) savedRegions.push_back(bk_alloc(r.second));
    for (size_t i = 0; i < mutableRegions.size(); i++) bk_d2d(savedRegions[i], mutableRegions[i].first, mutableRegions[i].second);
    savedHash = hash;
  }
  int restoreState() {
    if (savedRegions.empty()) return HIVED_ERR_PLATFORM;
    bk_quiesce(*this);
    for (size_t i = 0; i < mutableRegions.size(); i++) bk_d2d(mutableRegions[i].first, savedRegions[i], mutableRegions[i].second);
    hash = savedHash;
    return 0;
  }
  uint64_t savedHash = HIVED_FNV_OFFSET;
};

}  // namespace hived

// ================================================================================================
// C ABI
// ================================================================================================
struct hived_ctx {
  hived::Engine e;
};

static std::string g_hived_create_error;

extern "C" {

const char* hived_create_error(void) { return g_hived_create_error.c_str(); }

int hived_create(const char* spec_text, const hived_options_t* opt, hived_ctx** out) {
  *out = nullptr;
  auto ctx = std::make_unique<hived_ctx>();
  int rc = ctx->e.create(spec_text, opt);
  if (rc) { g_hived_create_error = ctx->e.err; return rc; }
  *out = ctx.release();
  return 0;
}
void hived_destroy(hived_ctx* ctx) { delete ctx; }
const char* hived_last_error(hived_ctx* ctx) { return ctx->e.err.c_str(); }

#define HIVED_TABLE(fn_num, fn_name, vec)                                                        \
  int32_t fn_num(hived_ctx* ctx) { return (int32_t)ctx->e.T.vec.size(); }                         \
  const char* fn_name(hived_ctx* ctx, int32_t id) {                                               \
    return (id >= 0 && id < (int32_t)ctx->e.T.vec.size()) ? ctx->e.T.vec[id].c_str() : nullptr;   \
  }
HIVED_TABLE(hived_num_nodes, hived_node_name, nodeNames)
HIVED_TABLE(hived_num_chains, hived_chain_name, chainNames)
HIVED_TABLE(hived_num_vcs, hived_vc_name, vcNames)
HIVED_TABLE(hived_num_leaf_types, hived_leaf_type_name, leafTypeNames)
HIVED_TABLE(hived_num_pinned, hived_pinned_name, pinnedNames)
HIVED_TABLE(hived_num_cell_types, hived_cell_type_name, cellTypeNames)
#undef HIVED_TABLE
int32_t hived_num_physical_cells(hived_ctx* ctx) { return ctx->e.T.NP; }
int32_t hived_num_virtual_cells(hived_ctx* ctx) { return ctx->e.T.NV; }
const char* hived_physical_cell_address(hived_ctx* ctx, int32_t c) { return (c >= 0 && c < ctx->e.T.NP) ? ctx->e.T.pAddr[c].c_str() : nullptr; }
const char* hived_virtual_cell_address(hived_ctx* ctx, int32_t c) { return (c >= 0 && c < ctx->e.T.NV) ? ctx->e.T.vAddr[c].c_str() : nullptr; }

int hived_vc_preassigned_cells(hived_ctx* ctx, int32_t vc, int32_t chain, int32_t level, int32_t* cells, int32_t cap, int32_t* n) {
  const hived::FlatTopo& T = ctx->e.T;
  *n = 0;
  if (vc < 0 || vc >= T.nVCs || chain < 0 || chain >= T.nChains || level < 1 || level >= hived::MAXL) return HIVED_ERR_PLATFORM;
  size_t k = ((size_t)vc * T.nChains + chain) * hived::MAXL + level;
  for (int i = 0; i < T.pre_cnt[k]; i++) {
    if (*n < cap) cells[*n] = T.pre_list[T.pre_off[k] + i];
    (*n)++;
  }
  return 0;
}

static int hived_run_one(hived_ctx* ctx, const hived_event_t& ev, const uint32_t* sugg, const int32_t* aux, int64_t auxWords,
                         hived_result_t* res, int32_t* pool, int64_t poolCap) {
  hived::Engine& e = ctx->e;
  hived_event_t copy = ev;
  copy.suggested_off = sugg ? 0 : -1;
  int rc = e.runBatch(&copy, 1, sugg, sugg ? e.dev.S.bitmapWords : 0, aux, auxWords, res, pool, poolCap);
  if (rc) return rc;
  if (res->error) {
    char buf[96];
    snprintf(buf, sizeof buf, "scheduler error %d (see HIVED_ERR_* in hived.h)", res->error);
    e.err = buf;
  }
  return res->error;
}

int hived_set_node_health(hived_ctx* ctx, int32_t node, int32_t healthy) {
  hived_event_t ev;
  memset(&ev, 0, sizeof ev);
  ev.type = HIVED_EV_NODE_HEALTH; ev.arg0 = node; ev.arg1 = healthy;
  hived_result_t res; int32_t pool[4];
  return hived_run_one(ctx, ev, nullptr, nullptr, 0, &res, pool, 4);
}

int hived_schedule(hived_ctx* ctx, const hived_pod_spec_t* spec, const uint32_t* suggested, int32_t phase, hived_result_t* res,
                   int32_t* pool, int32_t pool_cap) {
  hived_event_t ev;
  memset(&ev, 0, sizeof ev);
  ev.type = hived::Core::EV_SCHEDULE_ONLY; ev.phase = phase; ev.spec = *spec;
  int rc = hived_run_one(ctx, ev, suggested, nullptr, 0, res, pool, pool_cap);
  if (rc == 0) ctx->e.hash = hived_hash_result(ctx->e.hash, res, pool);
  return rc;
}

int hived_add_allocated_pod(hived_ctx* ctx, const hived_pod_spec_t* spec, const hived_bind_info_t* info, const int32_t* leaves,
                            int32_t pod_index) {
  hived_event_t ev;
  memset(&ev, 0, sizeof ev);
  ev.type = hived::Core::EV_ADD_ALLOCATED; ev.arg0 = pod_index; ev.spec = *spec;
  std::vector<int32_t> aux(sizeof(hived_bind_info_t) / 4 + 3 * (size_t)info->n_leaves);
  memcpy(aux.data(), info, sizeof(hived_bind_info_t));
  if (info->n_leaves > 0) memcpy(aux.data() + sizeof(hived_bind_info_t) / 4, leaves, 3 * (size_t)info->n_leaves * 4);
  hived_result_t res; int32_t pool[4];
  return hived_run_one(ctx, ev, nullptr, aux.data(), (int64_t)aux.size(), &res, pool, 4);
}

int hived_delete_allocated_pod_ex(hived_ctx* ctx, int32_t group, int32_t leaf_num, int32_t pod_index, int32_t* removed_pod) {
  hived_event_t ev;
  memset(&ev, 0, sizeof ev);
  ev.type = HIVED_EV_DELETE_ALLOCATED; ev.arg0 = pod_index; ev.spec.group = group; ev.spec.leaf_num = leaf_num;
  hived_result_t res; int32_t pool[4];
  res.pod_index = -1;
  int rc = hived_run_one(ctx, ev, nullptr, nullptr, 0, &res, pool, 4);
  if (removed_pod) *removed_pod = res.pod_index;
  return rc;
}
int hived_delete_allocated_pod(hived_ctx* ctx, int32_t group, int32_t leaf_num, int32_t pod_index) {
  return hived_delete_allocated_pod_ex(ctx, group, leaf_num, pod_index, nullptr);
}

int hived_delete_unallocated_pod(hived_ctx* ctx, int32_t group, int32_t pod) {
  hived_event_t ev;
  memset(&ev, 0, sizeof ev);
  ev.type = HIVED_EV_DELETE_UNALLOCATED; ev.spec.group = group; ev.spec.pod = pod;
  hived_result_t res; int32_t pool[4];
  return hived_run_one(ctx, ev, nullptr, nullptr, 0, &res, pool, 4);
}

int hived_process_events(hived_ctx* ctx, const hived_event_t* events, int32_t n, const uint32_t* suggested_pool,
                         int64_t suggested_words, hived_result_t* res, int32_t* pool, int64_t pool_cap) {
  hived::Engine& e = ctx->e;
  int rc = e.runBatch(events, n, suggested_pool, suggested_words, nullptr, 0, res, pool, pool_cap);
  if (rc) return rc;
  bool noted = false;
  for (int32_t i = 0; i < n; i++) {
    if (e.hashing && events[i].type == HIVED_EV_SCHEDULE) e.hash = hived_hash_result(e.hash, &res[i], pool);
    if (res[i].error == HIVED_ERR_CAPACITY) { e.err = "capacity exceeded (result pool or hived_options_t)"; return HIVED_ERR_CAPACITY; }
    if (res[i].error >= 100 && !noted) {  // per-event platform errors stay in the results; the text names the first
      char buf[128];
      snprintf(buf, sizeof buf, "event %d failed with platform error %d (see hived_result_t.error of every event)", (int)i, (int)res[i].error);
      e.err = buf;
      noted = true;
    }
  }
  return 0;
}

int hived_get_group(hived_ctx* ctx, int32_t group, hived_group_info_t* out) {
  memset(out, 0, sizeof *out);
  hived::Engine& e = ctx->e;
  if (group < 0 || group >= e.dev.S.maxGroups) return 0;
  int32_t hdr[hived::GROUP_HDR_WORDS];
  hived::bk_d2h(hdr, e.dev.g_hdr + (size_t)group * hived::GROUP_HDR_WORDS, sizeof hdr);
  int32_t v[5] = {hdr[0], hdr[1], hdr[2], hdr[3], hdr[5]};
  if (v[0] == HIVED_GROUP_NONE) {
    // an erased object of this id that cells may still name (Core::ghostify): the shims keep the id (hived.h "Id lifetime").
    // Every cell is looked at, like the reference's pointers would be: a ghost that was itself erased by name
    // (Core::eraseGroupByName) has state NONE but its cells still name it, and a later erase through them hits this id.
    const int32_t G = e.dev.S.maxGroups;
    std::vector<int32_t> usingG, resv, gh;
    e.readArray(e.dev.p_using, usingG, e.T.NP); e.readArray(e.dev.p_resv, resv, e.T.NP);
    e.readArray(e.dev.g_hdr + (size_t)G * hived::GROUP_HDR_WORDS, gh, (size_t)hived::GHOST_GROUPS * hived::GROUP_HDR_WORDS);
    auto names = [&](int32_t s) {
      if (s == group) return true;
      return s >= G && s < G + hived::GHOST_GROUPS && gh[(size_t)(s - G) * hived::GROUP_HDR_WORDS + hived::GH_ORIGIN] == group + 1;
    };
    for (int c = 0; c < e.T.NP && !out->referenced; c++)
      if (names(usingG[c]) || names(resv[c])) out->referenced = 1;
    return 0;
  }
  out->state = v[0]; out->vc = v[1]; out->priority = v[2];
  out->has_virtual = (v[3] & hived::GF_HAS_VIRTUAL) ? 1 : 0;
  out->n_preempting_pods = v[0] == HIVED_GROUP_PREEMPTING ? v[4] : 0;
  return 0;
}

int hived_get_group_placement(hived_ctx* ctx, int32_t group, hived_group_placement_t* out, int32_t* phys, int32_t* virt,
                              int32_t leaf_cap, int32_t* pods, int32_t pod_cap, int32_t* preempting, int32_t preempting_cap) {
  memset(out, 0, sizeof *out);
  hived::Engine& e = ctx->e;
  if (group < 0 || group >= e.dev.S.maxGroups) return 0;
  int32_t hdr[hived::GROUP_HDR_WORDS];
  hived::bk_d2h(hdr, e.dev.g_hdr + (size_t)group * hived::GROUP_HDR_WORDS, sizeof hdr);
  if (hdr[0] == HIVED_GROUP_NONE) return 0;
  out->state = hdr[0];
  out->n_members = hdr[4];
  for (int m = 0; m < hdr[4] && m < HIVED_MAX_MEMBERS; m++) {
    out->member_leaf_num[m] = hdr[8 + m];
    out->member_pod_num[m] = hdr[16 + m];
    out->n_leaves += hdr[8 + m] * hdr[16 + m];
    out->n_pods += hdr[16 + m];
  }
  out->has_virtual = (hdr[3] & hived::GF_HAS_VIRTUAL) ? 1 : 0;
  out->lazy_preempted = (hdr[3] & hived::GF_LAZY_PREEMPTED) ? 1 : 0;
  const int nl = out->n_leaves < leaf_cap ? out->n_leaves : leaf_cap;
  if (nl > 0 && phys) hived::bk_d2h(phys, e.dev.g_phys + (size_t)group * e.dev.S.LS, (size_t)nl * 4);
  if (nl > 0 && virt) {
    hived::bk_d2h(virt, e.dev.g_virt + (size_t)group * e.dev.S.LS, (size_t)nl * 4);
    if (!out->has_virtual) for (int i = 0; i < nl; i++) virt[i] = -1;  // virtualLeafCellPlacement == nil
  }
  const int np = out->n_pods < pod_cap ? out->n_pods : pod_cap;
  if (np > 0 && pods) hived::bk_d2h(pods, e.dev.g_pods + (size_t)group * e.dev.S.PS, (size_t)np * 4);
  if (out->state == HIVED_GROUP_PREEMPTING) {
    out->n_preempting = hdr[5];
    const int n = hdr[5] < preempting_cap ? hdr[5] : preempting_cap;
    if (n > 0 && preempting) {
      hived::bk_d2h(preempting, e.dev.g_pre + (size_t)group * e.dev.S.PS, (size_t)n * 4);
      std::sort(preempting, preempting + n);
    }
  }
  return 0;
}

int32_t hived_list_groups(hived_ctx* ctx, int32_t* ids, int32_t cap) {
  hived::Engine& e = ctx->e;
  const int32_t G = e.dev.S.maxGroups;
  std::vector<int32_t> hdr((size_t)G * hived::GROUP_HDR_WORDS);
  hived::bk_d2h(hdr.data(), e.dev.g_hdr, hdr.size() * 4);
  int32_t n = 0;
  for (int32_t g = 0; g < G; g++) {
    if (hdr[(size_t)g * hived::GROUP_HDR_WORDS] == HIVED_GROUP_NONE) continue;
    if (ids && n < cap) ids[n] = g;
    n++;
  }
  return n;
}

int hived_physical_cell_info(hived_ctx* ctx, int32_t c, hived_cell_info_t* out) {
  const hived::FlatTopo& T = ctx->e.T;
  memset(out, 0xff, sizeof *out);
  if (c < 0 || c >= T.NP) return HIVED_ERR_PLATFORM;
  const int chain = T.p_chain[c], level = T.p_level[c];
  out->cell_type = T.chain_lvl_type[(size_t)chain * hived::MAXL + level];
  out->is_node_level = (T.p_flags[c] & hived::PF_NODE_LEVEL) ? 1 : 0;
  out->leaf_type = T.chain_leaftype[chain];
  out->node = level == 1 ? T.p_node[c] : -1;
  out->leaf_index = level == 1 ? T.p_leafidx[c] : -1;
  out->vc = -1; out->preassigned = -1; out->pinned = -1;
  if (T.p_flags[c] & hived::PF_PINNED)
    for (int i = 0; i < T.nPinned; i++) if (T.pin_pcell[i] == c) out->pinned = i;
  return 0;
}

int hived_virtual_cell_info(hived_ctx* ctx, int32_t c, hived_cell_info_t* out) {
  const hived::FlatTopo& T = ctx->e.T;
  memset(out, 0xff, sizeof *out);
  if (c < 0 || c >= T.NV) return HIVED_ERR_PLATFORM;
  const int chain = T.v_chain[c], level = T.v_level[c];
  out->cell_type = T.chain_lvl_type[(size_t)chain * hived::MAXL + level];
  out->is_node_level = (T.v_flags[c] & hived::PF_NODE_LEVEL) ? 1 : 0;
  out->leaf_type = T.chain_leaftype[chain];
  out->node = -1; out->leaf_index = -1;
  out->vc = T.v_vc[c];
  out->preassigned = T.v_pre[c];
  out->pinned = T.vs_pinned[T.v_vset[c]];
  return 0;
}

int hived_snapshot_physical(hived_ctx* ctx, hived_cell_status_t* out, int32_t cap) {
  hived::Engine& e = ctx->e;
  int n = e.T.NP;
  if (cap < n) return HIVED_ERR_CAPACITY;
  std::vector<int32_t> prio, state, healthy, vcell, split, flpos;
  e.readArray(e.dev.p_prio, prio, n); e.readArray(e.dev.p_state, state, n); e.readArray(e.dev.p_healthy, healthy, n);
  e.readArray(e.dev.p_vcell, vcell, n); e.readArray(e.dev.p_split, split, n);
  for (int i = 0; i < n; i++) {
    out[i].priority = prio[i]; out[i].state = state[i]; out[i].healthy = healthy[i]; out[i].peer = vcell[i];
    out[i].level = e.T.p_level[i]; out[i].chain = e.T.p_chain[i]; out[i].parent = e.T.p_parent[i];
    // inFreeCellList (utils.go:381-391) on the snapshot
    bool inFree;
    int c = i;
    while (true) {
      if (vcell[c] >= 0 || split[c]) { inFree = false; break; }
      int par = e.T.p_parent[c];
      if (par < 0 || split[par]) { inFree = true; break; }
      c = par;
    }
    out[i].flags = (split[i] ? 1 : 0) | ((e.T.p_flags[i] & hived::PF_PINNED) ? 2 : 0) | (inFree ? 4 : 0);
  }
  return 0;
}

int hived_snapshot_virtual(hived_ctx* ctx, hived_cell_status_t* out, int32_t cap) {
  hived::Engine& e = ctx->e;
  int n = e.T.NV;
  if (cap < n) return HIVED_ERR_CAPACITY;
  std::vector<int32_t> prio, state, healthy, pcell;
  e.readArray(e.dev.v_prio, prio, n); e.readArray(e.dev.v_state, state, n); e.readArray(e.dev.v_healthy, healthy, n);
  e.readArray(e.dev.v_pcell, pcell, n);
  for (int i = 0; i < n; i++) {
    out[i].priority = prio[i]; out[i].state = state[i]; out[i].healthy = healthy[i]; out[i].peer = pcell[i];
    out[i].level = e.T.v_level[i]; out[i].chain = e.T.v_chain[i]; out[i].parent = e.T.v_parent[i];
    out[i].flags = e.T.v_parent[i] < 0 ? 1 : 0;
  }
  return 0;
}

int hived_get_stats(hived_ctx* ctx, hived_stats_t* out) {
  memset(out, 0, sizeof *out);
  hived::Engine& e = ctx->e;
  long long st[hived::ST_COUNT];
  hived::bk_d2h(st, e.dev.stats, sizeof st);
  out->schedule_events = st[hived::ST_SCHEDULE]; out->bind_results = st[hived::ST_BIND]; out->wait_results = st[hived::ST_WAIT];
  out->preempt_results = st[hived::ST_PREEMPT]; out->view_nodes_scanned = st[hived::ST_VIEW_NODES];
  out->leaves_committed = st[hived::ST_LEAVES]; out->free_cells_scanned = st[hived::ST_FREE_CELLS]; out->pods_placed = st[hived::ST_PODS];
  long long K = __builtin_popcountll((unsigned long long)st[hived::ST_PRIO_MASK]);
  if (K < 1) K = 1;
  long long L = e.T.maxLevels;
  out->algorithmic_bytes = st[hived::ST_VIEW_NODES] * (36 + 4 * K) + st[hived::ST_PODS] * 64 + st[hived::ST_FREE_CELLS] * 12 +
                           st[hived::ST_LEAVES] * 16 * L * (1 + K);
  return 0;
}

uint64_t hived_result_hash(hived_ctx* ctx) { return ctx->e.hash; }

// ---- measurement hooks (include/hived_bench.h)
int hived_bench_save_state(hived_ctx* ctx) { ctx->e.saveState(); return 0; }
int hived_bench_restore_state(hived_ctx* ctx) { return ctx->e.restoreState(); }
int hived_bench_stage_events(hived_ctx* ctx, const hived_event_t* events, int32_t n, int64_t pool_cap) { return ctx->e.stage(events, n, pool_cap); }
int hived_bench_run_staged(hived_ctx* ctx) { return ctx->e.runStaged(); }
int hived_bench_fetch_results(hived_ctx* ctx, hived_result_t* res, int32_t* pool, int64_t pool_cap, int64_t* pool_used) {
  hived::Engine& e = ctx->e;
  return e.fetch(res, pool, pool_cap, pool_used);
}
// ---- include/hived_multigpu.h
int hived_mg_stage(hived_ctx* ctx, const hived_event_t* events, int32_t n, int64_t pool_cap, int32_t rank, int32_t world) {
  return ctx->e.mgStage(events, n, pool_cap, rank, world);
}
int hived_mg_reset(hived_ctx* ctx) { return ctx->e.mgReset(); }
int hived_mg_run(hived_ctx* ctx, int32_t* stop_event) { return ctx->e.mgRun(0x7fffffff, stop_event); }
int hived_mg_run_window(hived_ctx* ctx, int32_t horizon, int32_t* stop_event) { return ctx->e.mgRun(horizon, stop_event); }
int hived_mg_solo(hived_ctx* ctx, int32_t event_index) { return ctx->e.mgSolo(event_index); }
int64_t hived_mg_shared_bytes(hived_ctx* ctx) { return ctx->e.mgSharedBytes(); }
int hived_mg_export_shared(hived_ctx* ctx, void* buf) { ctx->e.mgExportShared(buf); return 0; }
int hived_mg_import_shared(hived_ctx* ctx, const void* buf) { ctx->e.mgImportShared(buf); return 0; }
int hived_mg_finish(hived_ctx* ctx) { return ctx->e.mgFinish(); }
int hived_mg_chain_hash(const hived_event_t* events, int32_t n, int32_t world, const hived_result_t* const* res,
                        const int32_t* const* pools, uint64_t seed, uint64_t* out) {
  uint64_t h = seed;
  for (int i = 0; i < n; i++) {
    if (events[i].type != HIVED_EV_SCHEDULE) continue;
    const int vc = events[i].spec.vc;
    if (vc < 0 || world < 1) return HIVED_ERR_BAD_SPEC;
    const int r = vc % world;
    h = hived_hash_result(h, &res[r][i], pools[r]);
  }
  *out = h;
  return 0;
}
int hived_bench_num_ctas(hived_ctx* ctx) { return ctx->e.launchCta; }
int hived_bench_set_result_hash(hived_ctx* ctx, int on) { ctx->e.hashing = on != 0; return 0; }
int hived_bench_flush_l2(hived_ctx*) { hived::bk_flush_l2(); return 0; }
/* out[0..7): SM cycles in view pass, leaf search, mapping, result emission, commit, delete, all events */
int hived_bench_phase_cycles(hived_ctx* ctx, int64_t* out) {
  long long st[hived::ST_COUNT];
  hived::bk_d2h(st, ctx->e.dev.stats, sizeof st);
  for (int i = 0; i < 15; i++) out[i] = st[hived::ST_CYC_VIEW + i];
  return 0;
}
int hived_bench_debug_cycles(hived_ctx* ctx, int64_t* out) {
  long long st[hived::ST_COUNT];
  hived::bk_d2h(st, ctx->e.dev.stats, sizeof st);
  for (int i = 0; i < 16; i++) out[i] = st[hived::ST_DBG0 + i];
  return 0;
}
/* out[0..PC_COUNT): how many scheduling passes / commits / deletes took the fast and the general paths (hived_dev.h PC_*) */
int hived_bench_path_counters(hived_ctx* ctx, int64_t* out) {
  long long st[hived::ST_COUNT];
  hived::bk_d2h(st, ctx->e.dev.stats, sizeof st);
  for (int i = 0; i < hived::PC_COUNT; i++) out[i] = st[hived::ST_PATH0 + i];
  return hived::PC_COUNT;
}
/* test hook: a hash of every cluster view's persisted order (cell addresses in order; order-independent across views).
   The order is state that no result shows until a tie is broken by it. */
uint64_t hived_debug_view_hash(hived_ctx* ctx) {
  hived::Engine& e = ctx->e;
  const hived::FlatTopo& T = e.T;
  std::vector<int32_t> cv, valid, head, cnt, next;
  e.readArray(e.dev.cv, cv, T.cv_init.size());
  e.readArray(e.dev.bk_valid, valid, T.nScheds);
  e.readArray(e.dev.bk_head, head, (size_t)T.nScheds * hived::BK_STRIDE);
  e.readArray(e.dev.bk_cnt, cnt, (size_t)T.nScheds * hived::BK_STRIDE);
  e.readArray(e.dev.vn_next, next, T.NV);
  uint64_t total = 0;
  for (int s = 0; s < T.nScheds; s++) {
    std::vector<int32_t> order;
    if (valid[s]) {
      for (int u = T.s_maxleaf[s]; u >= 0; u--)
        for (int x = head[(size_t)s * hived::BK_STRIDE + u]; x >= 0; x = next[x]) order.push_back(x);
    } else {
      for (int i = 0; i < T.s_n[s]; i++) order.push_back(cv[T.s_off[s] + i]);
    }
    uint64_t h = HIVED_FNV_OFFSET;
    for (int32_t c : order) {
      const std::string& a = T.s_virtual[s] ? T.vAddr[c] : T.pAddr[c];
      for (char ch : a) { h ^= (uint8_t)ch; h *= HIVED_FNV_PRIME; }
      h ^= 0xff; h *= HIVED_FNV_PRIME;
    }
    total += h;
  }
  return total;
}
/* test hook: the scheduler state that decides LATER calls and that neither a result nor a cell snapshot shows, in the
   canonical encoding of include/hived_bench.h (tagged sections, zeros and missing map entries omitted).  Derived the
   way the device program reads it: the used-leaf counters from the leaf priorities plus the recorded drift
   (noteDelta), the opportunistic count of a physical cell from p_usedopp, a ghost group record as its origin id. */
int64_t hived_debug_state(hived_ctx* ctx, int32_t* out, int64_t cap) {
  hived::Engine& e = ctx->e;
  const hived::FlatTopo& T = e.T;
  const auto& S = e.dev.S;
  using hived::MAXL;
  const size_t CL = (size_t)S.nChains * MAXL, VCL = (size_t)S.nVCs * CL;
  std::vector<int32_t> fl, fll, bf, bfl, dm, dml, vcf, allf, tl, ad;
  e.readArray(e.dev.fl_data, fl, S.flTotal); e.readArray(e.dev.fl_len, fll, CL);
  e.readArray(e.dev.bf_data, bf, S.flTotal); e.readArray(e.dev.bf_len, bfl, CL);
  e.readArray(e.dev.dm_data, dm, S.dmTotal); e.readArray(e.dev.dm_len, dml, VCL);
  e.readArray(e.dev.vcFree, vcf, VCL); e.readArray(e.dev.allVCFree, allf, CL);
  e.readArray(e.dev.totalLeft, tl, CL); e.readArray(e.dev.allVCDoomed, ad, CL);
  std::vector<int32_t> o;
  auto list = [&](std::initializer_list<int32_t> head, const std::vector<int32_t>& data, int32_t base, int32_t n) {
    if (n == 0) return;
    o.insert(o.end(), head); o.push_back(n);
    for (int32_t i = 0; i < n; i++) o.push_back(data[(size_t)base + i]);
  };
  for (int c = 0; c < S.nChains; c++)
    for (int l = 1; l < MAXL; l++) list({HIVED_DS_FREE, c, l}, fl, T.fl_base[c * MAXL + l], fll[c * MAXL + l]);
  for (int c = 0; c < S.nChains; c++)
    for (int l = 1; l < MAXL; l++) list({HIVED_DS_BAD_FREE, c, l}, bf, T.fl_base[c * MAXL + l], bfl[c * MAXL + l]);
  for (int v = 0; v < S.nVCs; v++)
    for (int c = 0; c < S.nChains; c++)
      for (int l = 1; l < MAXL; l++) {
        const size_t k = ((size_t)v * S.nChains + c) * MAXL + l;
        list({HIVED_DS_DOOMED_BAD, v, c, l}, dm, T.dm_base[k], dml[k]);
      }
  for (int v = 0; v < S.nVCs; v++)
    for (int c = 0; c < S.nChains; c++) {
      if (!T.vc_chain_counter[(size_t)v * S.nChains + c]) continue;
      for (int l = 1; l < MAXL; l++) {
        const int32_t x = vcf[((size_t)v * S.nChains + c) * MAXL + l];
        if (x) o.insert(o.end(), {HIVED_DS_VC_FREE, v, c, l, x});
      }
    }
  const std::pair<int32_t, const std::vector<int32_t>*> perChain[] = {
      {HIVED_DS_ALL_VC_FREE, &allf}, {HIVED_DS_TOTAL_LEFT, &tl}, {HIVED_DS_ALL_VC_DOOMED, &ad}};
  for (const auto& t : perChain)
    for (int c = 0; c < S.nChains; c++)
      for (int l = 1; l < MAXL; l++) {
        const int32_t x = (*t.second)[c * MAXL + l];
        if (x) o.insert(o.end(), {t.first, c, l, x});
      }
  // used-leaf counters: (priority, count) per cell, ascending priority
  auto used = [&](bool virt, int n, int32_t tag) {
    std::vector<int32_t> prio, dprio, dcnt, opp;
    e.readArray(virt ? e.dev.v_prio : e.dev.p_prio, prio, n);
    e.readArray(virt ? e.dev.v_dprio : e.dev.p_dprio, dprio, (size_t)n * hived::DELTA_SLOTS);
    e.readArray(virt ? e.dev.v_dcnt : e.dev.p_dcnt, dcnt, (size_t)n * hived::DELTA_SLOTS);
    if (!virt) e.readArray(e.dev.p_usedopp, opp, n);
    const std::vector<int32_t>& level = virt ? T.v_level : T.p_level;
    const std::vector<int32_t>& parent = virt ? T.v_parent : T.p_parent;
    std::vector<std::map<int32_t, int32_t>> m(n);
    for (int c = 0; c < n; c++) {
      if (level[c] != 1 || prio[c] == hived::FREE_PRIO) continue;
      if (!virt && prio[c] == hived::OPP_PRIO) continue;  // counted by p_usedopp
      for (int a = c; a >= 0; a = parent[a]) m[a][prio[c]]++;
    }
    for (int c = 0; c < n; c++) {
      for (int i = 0; i < hived::DELTA_SLOTS; i++) {
        const int32_t p = dprio[(size_t)c * hived::DELTA_SLOTS + i];
        if (p == hived::DELTA_EMPTY || (!virt && p == hived::OPP_PRIO)) continue;
        m[c][p] += dcnt[(size_t)c * hived::DELTA_SLOTS + i];
      }
      if (!virt) m[c][hived::OPP_PRIO] += opp[c];
      int32_t k = 0;
      for (const auto& kv : m[c]) k += kv.second != 0;
      if (k == 0) continue;
      o.insert(o.end(), {tag, c, k});
      for (const auto& kv : m[c]) if (kv.second != 0) o.insert(o.end(), {kv.first, kv.second});
    }
  };
  used(false, T.NP, HIVED_DS_USED_PHYSICAL);
  used(true, T.NV, HIVED_DS_USED_VIRTUAL);
  // using / reserving group of every physical cell: (id, live); a ghost record stands for the object its id named
  {
    std::vector<int32_t> usingG, resv, hdr;
    e.readArray(e.dev.p_using, usingG, T.NP); e.readArray(e.dev.p_resv, resv, T.NP);
    e.readArray(e.dev.g_hdr, hdr, (size_t)(S.maxGroups + hived::GHOST_GROUPS) * hived::GROUP_HDR_WORDS);
    auto group = [&](int32_t tag, int c, int32_t g) {
      if (g < 0) return;
      const int32_t* h = hdr.data() + (size_t)g * hived::GROUP_HDR_WORDS;
      if (g < S.maxGroups) o.insert(o.end(), {tag, c, g, h[0] != HIVED_GROUP_NONE ? 1 : 0});
      else o.insert(o.end(), {tag, c, h[hived::GH_ORIGIN] - 1, 0});
    };
    for (int c = 0; c < T.NP; c++) group(HIVED_DS_USING_GROUP, c, usingG[c]);
    for (int c = 0; c < T.NP; c++) group(HIVED_DS_RESERVING_GROUP, c, resv[c]);
  }
  {
    std::vector<int32_t> bad;
    e.readArray(e.dev.node_bad, bad, S.nNodes);
    for (int i = 0; i < S.nNodes; i++) if (bad[i]) o.insert(o.end(), {HIVED_DS_BAD_NODE, i});
  }
  for (size_t i = 0; i < o.size() && (int64_t)i < cap; i++) out[i] = o[i];
  return (int64_t)o.size();
}
double hived_bench_last_kernel_ms(hived_ctx* ctx) { return ctx->e.lastKernelMs; }
double hived_bench_total_kernel_ms(hived_ctx* ctx) { return ctx->e.kernelMsTotal; }
int64_t hived_bench_kernel_launches(hived_ctx* ctx) { return ctx->e.kernelLaunches; }

}  // extern "C"

#include "hived_ingest.hpp"
#include "hived_frontend.hpp"
