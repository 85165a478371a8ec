// TEST INFRASTRUCTURE — exposes the CPU oracle (hived_oracle.cpp) through the same C ABI as the
// product (include/hived.h) so tests and the CPU-baseline leg of bench.py can drive both with one
// harness.  The adapter converts ids <-> the strings the reference works with; in particular
// Schedule() receives suggestedNodes as node-name strings and builds the string set per call like
// the reference does (hived_algorithm.go:190-193).
#include <algorithm>
#include <cstring>
#include <memory>
#include <set>
#include <string>
#include <vector>

#include "../include/hived.h"
#include "../include/hived_bench.h"
#include "../include/hived_hash.h"
#include "hived_oracle.hpp"

using namespace hived_oracle;

struct hived_ctx {
  std::unique_ptr<HivedAlgorithm> h;
  hived_options_t opt{};
  std::string err;
  std::unordered_map<std::string, int32_t> cellTypeIds, chainIds;
  std::set<int32_t> priorities;
  int32_t maxLevels = 0;
  uint64_t hash = HIVED_FNV_OFFSET;
  int64_t schedule_events = 0, binds = 0, waits = 0, preempts = 0;
};

static std::string g_create_error;

static std::string groupName(int32_t id) { return "g" + std::to_string(id); }

static PodSchedulingSpec toSpec(hived_ctx* ctx, const hived_pod_spec_t* sp) {
  HivedAlgorithm& h = *ctx->h;
  PodSchedulingSpec s;
  s.virtualCluster = (sp->vc >= 0 && sp->vc < (int32_t)h.vcNames.size()) ? h.vcNames[sp->vc] : "<unknown-vc>";
  s.priority = sp->priority;
  if (sp->pinned == -1)
    s.pinnedCellId = "";
  else
    s.pinnedCellId = (sp->pinned >= 0 && sp->pinned < (int32_t)h.pinnedNames.size()) ? h.pinnedNames[sp->pinned] : "<unknown-pinned-cell>";
  if (sp->leaf_type == -1)
    s.leafCellType = "";
  else
    s.leafCellType = (sp->leaf_type >= 0 && sp->leaf_type < (int32_t)h.leafTypeNames.size()) ? h.leafTypeNames[sp->leaf_type] : "<unknown-leaf-type>";
  s.leafCellNumber = sp->leaf_num;
  s.lazyPreemptionEnable = (sp->flags & HIVED_SPEC_LAZY_PREEMPTION) != 0;
  s.ignoreK8sSuggestedNodes = (sp->flags & HIVED_SPEC_IGNORE_SUGGESTED) != 0;
  s.groupName = groupName(sp->group);
  s.groupId = sp->group;
  for (int32_t i = 0; i < sp->n_members; i++) s.members.push_back({sp->member_pod_num[i], sp->member_leaf_num[i]});
  return s;
}

// pkg/internal/utils.go:256-287 restated defensively (the shim validates first)
static void validateSpec(hived_ctx* ctx, const hived_pod_spec_t* sp) {
  if (sp->group < 0 || sp->group >= ctx->opt.max_groups || sp->pod < 0 || sp->pod >= ctx->opt.max_pods)
    throw Panic("group or pod id exceeds hived_options_t", HIVED_ERR_CAPACITY);
  if (sp->priority < HIVED_OPPORTUNISTIC_PRIORITY) throw BadRequest(HIVED_ERR_BAD_SPEC, "Priority is less than -1");
  if (sp->priority > HIVED_MAX_GUARANTEED_PRIORITY) throw BadRequest(HIVED_ERR_BAD_SPEC, "Priority is greater than 1000");
  if (sp->leaf_num <= 0) throw BadRequest(HIVED_ERR_BAD_SPEC, "LeafCellNumber is non-positive");
  if (sp->n_members <= 0 || sp->n_members > HIVED_MAX_MEMBERS) throw BadRequest(HIVED_ERR_BAD_SPEC, "bad member count");
  bool in = false;
  int64_t leaves = 0, pods = 0;
  for (int32_t i = 0; i < sp->n_members; i++) {
    if (sp->member_pod_num[i] <= 0) throw BadRequest(HIVED_ERR_BAD_SPEC, "AffinityGroup.Members has non-positive PodNumber");
    if (sp->member_leaf_num[i] <= 0) throw BadRequest(HIVED_ERR_BAD_SPEC, "AffinityGroup.Members has non-positive LeafCellNumber");
    if (sp->member_leaf_num[i] == sp->leaf_num) in = true;
    leaves += (int64_t)sp->member_leaf_num[i] * sp->member_pod_num[i];
    pods += sp->member_pod_num[i];
  }
  if (!in) throw BadRequest(HIVED_ERR_BAD_SPEC, "AffinityGroup.Members does not contains current Pod");
  if (leaves > ctx->opt.max_group_leaves || pods > ctx->opt.max_group_pods)
    throw Panic("affinity group exceeds hived_options_t capacity", HIVED_ERR_CAPACITY);
}

static void clearResult(hived_result_t* r) {
  memset(r, 0, sizeof(*r));
  r->wait_cell = -1;
  r->chain = -1;
  r->node = -1;
}

// utils.go:291-304
static int32_t getAllocatedPodIndex(const PodBindInfo& info, int32_t leafCellNum) {
  for (auto& gms : info.affinityGroupBindInfo) {
    if ((int32_t)gms[0].physicalLeafCellIndices.size() == leafCellNum) {
      for (size_t podIndex = 0; podIndex < gms.size(); podIndex++) {
        const PodPlacementInfo& pl = gms[podIndex];
        if (pl.physicalNode == info.node) {
          for (int32_t g : pl.physicalLeafCellIndices)
            if (!info.leafCellIsolation.empty() && g == info.leafCellIsolation[0]) return (int32_t)podIndex;
        }
      }
    }
  }
  return -1;
}

template <typename F>
static int guarded(hived_ctx* ctx, F&& f) {
  try {
    f();
    return 0;
  } catch (const BadRequest& e) {
    ctx->err = e.what();
    return e.code;
  } catch (const Panic& e) {
    ctx->err = e.what();
    return e.code;
  } catch (const std::exception& e) {
    ctx->err = std::string("panic: ") + e.what();
    return HIVED_ERR_PLATFORM;
  }
}

// fills res/pool from the oracle's ScheduleResult; returns words consumed or throws on capacity
static int64_t emitResult(hived_ctx* ctx, const hived_pod_spec_t* sp, const ScheduleResult& r, hived_result_t* res,
                          int32_t* pool, int64_t off, int64_t cap) {
  HivedAlgorithm& h = *ctx->h;
  int64_t start = off;
  res->kind = r.kind;
  res->pod_index = r.podIndex;
  res->has_virtual = r.virtual_.nil ? 0 : 1;
  if (r.kind == HIVED_KIND_WAIT) {
    res->wait_code = r.wait.code;
    res->wait_cell = r.wait.cell ? r.wait.cell->id : -1;
    return 0;
  }
  if (r.kind == HIVED_KIND_PREEMPT) {
    res->victim_off = (int32_t)off;
    res->n_victims = (int32_t)r.victims.size();
    if (off + 2 * (int64_t)r.victims.size() > cap) throw Panic("result pool too small", HIVED_ERR_CAPACITY);
    for (auto& v : r.victims) {
      pool[off++] = v.first->id;
      pool[off++] = v.second;
    }
    return off - start;
  }
  const PodBindInfo& info = r.bindInfo;
  res->chain = ctx->chainIds.count(info.cellChain) ? ctx->chainIds[info.cellChain] : -1;
  res->node = h.nodeIds.count(info.node) ? h.nodeIds[info.node] : -1;
  res->leaf_off = (int32_t)off;
  int32_t m = 0, nLeaves = 0;
  for (auto& lk : r.physical.m) {
    if (m >= HIVED_MAX_MEMBERS) throw Panic("too many members", HIVED_ERR_CAPACITY);
    res->member_leaf_num[m] = lk.first;
    res->member_pod_num[m] = (int32_t)lk.second.size();
    const auto& gms = info.affinityGroupBindInfo[m];
    for (size_t p = 0; p < gms.size(); p++) {
      if (lk.first == sp->leaf_num && (int32_t)p == r.podIndex) {
        res->this_off = (int32_t)off;
        res->this_n = lk.first;
      }
      if (off + 3 * (int64_t)lk.first > cap) throw Panic("result pool too small", HIVED_ERR_CAPACITY);
      for (int32_t j = 0; j < lk.first; j++) {
        if (gms[p].physicalLeafCellIndices[j] == HIVED_NIL_CELL && gms[p].preassignedCellTypes[j] == kNilCellType) {
          pool[off++] = HIVED_NIL_CELL; pool[off++] = HIVED_NIL_CELL; pool[off++] = HIVED_NIL_CELL;  // hived.h: incomplete
          nLeaves++;
          continue;
        }
        pool[off++] = h.nodeIds.count(gms[p].physicalNode) ? h.nodeIds[gms[p].physicalNode] : -1;
        pool[off++] = gms[p].physicalLeafCellIndices[j];
        const std::string& t = gms[p].preassignedCellTypes[j];
        pool[off++] = t.empty() ? -1 : ctx->cellTypeIds.at(t);
        nLeaves++;
      }
    }
    m++;
  }
  res->n_members = m;
  res->n_leaves = nLeaves;
  res->incomplete = info.incomplete ? 1 : 0;
  return off - start;
}

static PodBindInfo toBindInfo(hived_ctx* ctx, const hived_bind_info_t* bi, const int32_t* leaves) {
  HivedAlgorithm& h = *ctx->h;
  PodBindInfo info;
  auto nodeName = [&](int32_t id) -> std::string {
    return (id >= 0 && id < (int32_t)h.nodeNames.size()) ? h.nodeNames[id] : "<unknown-node>";
  };
  info.node = nodeName(bi->node);
  info.leafCellIsolation = {bi->first_leaf};
  info.cellChain = (bi->chain >= 0 && bi->chain < (int32_t)h.chainNames.size()) ? h.chainNames[bi->chain] : "<unknown-chain>";
  int64_t k = 0;
  for (int32_t m = 0; m < bi->n_members; m++) {
    std::vector<PodPlacementInfo> gms(bi->member_pod_num[m]);
    for (auto& pl : gms) {
      pl.preassignedNil = bi->has_preassigned == 0;
      for (int32_t j = 0; j < bi->member_leaf_num[m]; j++) {
        if (j == 0) pl.physicalNode = nodeName(leaves[3 * k]);
        pl.physicalLeafCellIndices.push_back(leaves[3 * k + 1]);
        int32_t t = leaves[3 * k + 2];
        pl.preassignedCellTypes.push_back(t == -1 ? "" : (t >= 0 && t < (int32_t)h.cellTypeNames.size()) ? h.cellTypeNames[t] : "<unknown-cell-type>");
        k++;
      }
    }
    info.affinityGroupBindInfo.push_back(gms);
  }
  return info;
}

static std::vector<std::string> suggestedNames(hived_ctx* ctx, const uint32_t* bitmap) {
  HivedAlgorithm& h = *ctx->h;
  std::vector<std::string> out;
  int32_t n = (int32_t)h.nodeNames.size();
  out.reserve(n);
  for (int32_t i = 0; i < n; i++)
    if (bitmap == nullptr || (bitmap[i >> 5] >> (i & 31)) & 1u) out.push_back(h.nodeNames[i]);
  return out;
}

// Schedule (+ optional AddAllocatedPod on bind, the filterRoutine sequence)
static void scheduleOne(hived_ctx* ctx, const hived_pod_spec_t* sp, const uint32_t* suggested, int32_t phase,
                        bool autoCommit, hived_result_t* res, int32_t* pool, int64_t& off, int64_t cap) {
  validateSpec(ctx, sp);
  PodSchedulingSpec s = toSpec(ctx, sp);
  ctx->priorities.insert(sp->priority);
  std::vector<std::string> names = suggestedNames(ctx, suggested);
  ScheduleResult r = ctx->h->Schedule(s, sp->pod, names, phase == HIVED_PHASE_PREEMPTING);
  off += emitResult(ctx, sp, r, res, pool, off, cap);
  ctx->schedule_events++;
  if (r.kind == HIVED_KIND_BIND) ctx->binds++;
  if (r.kind == HIVED_KIND_WAIT) ctx->waits++;
  if (r.kind == HIVED_KIND_PREEMPT) ctx->preempts++;
  if (autoCommit && r.kind == HIVED_KIND_BIND) {
    int32_t podIndex = getAllocatedPodIndex(r.bindInfo, sp->leaf_num);
    ctx->h->AddAllocatedPod(s, r.bindInfo, sp->pod, res->node, podIndex);
  }
}

extern "C" {

const char* hived_backend(void) { return "cpu-oracle"; }
const char* hived_create_error(void) { return g_create_error.c_str(); }

int hived_create(const char* spec_text, const hived_options_t* opt, hived_ctx** out) {
  *out = nullptr;
  auto ctx = std::make_unique<hived_ctx>();
  if (opt) ctx->opt = *opt;
  if (ctx->opt.max_groups <= 0) ctx->opt.max_groups = 1 << 20;
  if (ctx->opt.max_pods <= 0) ctx->opt.max_pods = 1 << 22;
  if (ctx->opt.max_group_leaves <= 0) ctx->opt.max_group_leaves = 1 << 20;
  if (ctx->opt.max_group_pods <= 0) ctx->opt.max_group_pods = 1 << 20;
  try {
    ctx->h = std::make_unique<HivedAlgorithm>(spec_text);
  } catch (const Panic& e) {
    g_create_error = e.what();
    return e.code >= 100 ? (e.code == HIVED_ERR_PLATFORM ? HIVED_ERR_BAD_CONFIG : e.code) : HIVED_ERR_BAD_CONFIG;
  } catch (const std::exception& e) {
    g_create_error = e.what();
    return HIVED_ERR_BAD_CONFIG;
  }
  HivedAlgorithm& h = *ctx->h;
  for (size_t i = 0; i < h.cellTypeNames.size(); i++) ctx->cellTypeIds[h.cellTypeNames[i]] = (int32_t)i;
  for (size_t i = 0; i < h.chainNames.size(); i++) ctx->chainIds[h.chainNames[i]] = (int32_t)i;
  for (auto& kv : h.fullCellList) ctx->maxLevels = std::max(ctx->maxLevels, kv.second.len());
  *out = ctx.release();
  return 0;
}

void hived_destroy(hived_ctx* ctx) { delete ctx; }
const char* hived_last_error(hived_ctx* ctx) { return ctx->err.c_str(); }

#define TABLE(fn_num, fn_name, vec)                                                       \
  int32_t fn_num(hived_ctx* ctx) { return (int32_t)ctx->h->vec.size(); }                   \
  const char* fn_name(hived_ctx* ctx, int32_t id) {                                        \
    return (id >= 0 && id < (int32_t)ctx->h->vec.size()) ? ctx->h->vec[id].c_str() : nullptr; \
  }
TABLE(hived_num_nodes, hived_node_name, nodeNames)
TABLE(hived_num_chains, hived_chain_name, chainNames)
TABLE(hived_num_vcs, hived_vc_name, vcNames)
TABLE(hived_num_leaf_types, hived_leaf_type_name, leafTypeNames)
TABLE(hived_num_pinned, hived_pinned_name, pinnedNames)
TABLE(hived_num_cell_types, hived_cell_type_name, cellTypeNames)
#undef TABLE

int32_t hived_num_physical_cells(hived_ctx* ctx) { return (int32_t)ctx->h->physicalCells.size(); }
int32_t hived_num_virtual_cells(hived_ctx* ctx) { return (int32_t)ctx->h->virtualCells.size(); }
const char* hived_physical_cell_address(hived_ctx* ctx, int32_t cell) {
  return (cell >= 0 && cell < (int32_t)ctx->h->physicalCells.size()) ? ctx->h->physicalCells[cell]->address.c_str() : nullptr;
}
const char* hived_virtual_cell_address(hived_ctx* ctx, int32_t cell) {
  return (cell >= 0 && cell < (int32_t)ctx->h->virtualCells.size()) ? ctx->h->virtualCells[cell]->address.c_str() : nullptr;
}

int hived_vc_preassigned_cells(hived_ctx* ctx, int32_t vc, int32_t chain, int32_t level, int32_t* cells, int32_t cap, int32_t* n) {
  HivedAlgorithm& h = *ctx->h;
  *n = 0;
  if (vc < 0 || vc >= (int32_t)h.vcNames.size() || chain < 0 || chain >= (int32_t)h.chainNames.size()) return HIVED_ERR_PLATFORM;
  auto& npc = h.vcSchedulers[h.vcNames[vc]]->nonPinnedPreassignedCells;
  auto it = npc.find(h.chainNames[chain]);
  if (it == npc.end()) return 0;
  for (Cell* c : it->second.at(level)) {
    if (*n < cap) cells[*n] = c->id;
    (*n)++;
  }
  return 0;
}

int hived_set_node_health(hived_ctx* ctx, int32_t node, int32_t healthy) {
  return guarded(ctx, [&] {
    if (node < 0 || node >= (int32_t)ctx->h->nodeNames.size()) return;  // unknown node: no cell matches (no-op)
    if (healthy)
      ctx->h->setHealthyNode(ctx->h->nodeNames[node]);
    else
      ctx->h->setBadNode(ctx->h->nodeNames[node]);
  });
}

int hived_schedule(hived_ctx* ctx, const hived_pod_spec_t* spec, const uint32_t* suggested, int32_t phase,
                   hived_result_t* res, int32_t* pool, int32_t pool_cap) {
  clearResult(res);
  int64_t off = 0;
  int rc = guarded(ctx, [&] { scheduleOne(ctx, spec, suggested, phase, false, res, pool, off, pool_cap); });
  res->error = rc;
  if (rc == 0) ctx->hash = hived_hash_result(ctx->hash, res, pool);
  return rc;
}

int hived_add_allocated_pod(hived_ctx* ctx, const hived_pod_spec_t* spec, const hived_bind_info_t* info,
                            const int32_t* leaves, int32_t pod_index) {
  return guarded(ctx, [&] {
    validateSpec(ctx, spec);
    PodSchedulingSpec s = toSpec(ctx, spec);
    PodBindInfo bi = toBindInfo(ctx, info, leaves);
    ctx->h->AddAllocatedPod(s, bi, spec->pod, info->node, pod_index);
  });
}

int hived_delete_allocated_pod_ex(hived_ctx* ctx, int32_t group, int32_t leaf_num, int32_t pod_index, int32_t* removed_pod) {
  int rc = guarded(ctx, [&] { ctx->h->DeleteAllocatedPod(groupName(group), leaf_num, pod_index); });
  if (removed_pod) *removed_pod = ctx->h->lastRemovedPod;
  return rc;
}
int hived_delete_allocated_pod(hived_ctx* ctx, int32_t group, int32_t leaf_num, int32_t pod_index) {
  return hived_delete_allocated_pod_ex(ctx, group, leaf_num, pod_index, nullptr);
}

int hived_delete_unallocated_pod(hived_ctx* ctx, int32_t group, int32_t pod) {
  return guarded(ctx, [&] { ctx->h->DeleteUnallocatedPod(groupName(group), pod); });
}

int hived_process_events(hived_ctx* ctx, const hived_event_t* events, int32_t n, const uint32_t* suggested_pool,
                         int64_t suggested_words, hived_result_t* res, int32_t* pool, int64_t pool_cap) {
  (void)suggested_words;
  int64_t off = 0;
  for (int32_t i = 0; i < n; i++) {
    const hived_event_t& ev = events[i];
    hived_result_t* r = &res[i];
    clearResult(r);
    int rc = 0;
    switch (ev.type) {
      case HIVED_EV_SCHEDULE: {
        const uint32_t* sugg = (ev.suggested_off >= 0 && suggested_pool) ? suggested_pool + ev.suggested_off : nullptr;
        rc = guarded(ctx, [&] { scheduleOne(ctx, &ev.spec, sugg, ev.phase, true, r, pool, off, pool_cap); });
        r->error = rc;
        ctx->hash = hived_hash_result(ctx->hash, r, pool);
        break;
      }
      case HIVED_EV_DELETE_ALLOCATED:
        r->pod_index = -1;
        rc = hived_delete_allocated_pod_ex(ctx, ev.spec.group, ev.spec.leaf_num, ev.arg0, &r->pod_index);
        break;
      case HIVED_EV_DELETE_UNALLOCATED:
        rc = hived_delete_unallocated_pod(ctx, ev.spec.group, ev.spec.pod);
        break;
      case HIVED_EV_NODE_HEALTH:
        rc = hived_set_node_health(ctx, ev.arg0, ev.arg1);
        break;
      default:
        rc = HIVED_ERR_PLATFORM;
        ctx->err = "unknown event type";
    }
    r->error = rc;
    if (rc == HIVED_ERR_CAPACITY) return rc;
  }
  return 0;
}

int hived_get_group(hived_ctx* ctx, int32_t group, hived_group_info_t* out) {
  memset(out, 0, sizeof(*out));
  auto it = ctx->h->affinityGroups.find(groupName(group));
  if (it == ctx->h->affinityGroups.end()) {
    // an erased object of this name that a cell still points at (the reference can erase it BY NAME later)
    const std::string name = groupName(group);
    for (Cell* c : ctx->h->physicalCells)
      if ((c->usingGroup && c->usingGroup->name == name) || (c->reservingOrReservedGroup && c->reservingOrReservedGroup->name == name)) {
        out->referenced = 1;
        break;
      }
    return 0;
  }
  Group* g = it->second;
  out->state = g->state;
  out->vc = -1;
  for (size_t i = 0; i < ctx->h->vcNames.size(); i++)
    if (ctx->h->vcNames[i] == g->vc) out->vc = (int32_t)i;
  out->priority = g->priority;
  out->has_virtual = g->virtualPlacement.nil ? 0 : 1;
  out->n_preempting_pods = (int32_t)g->preemptingPods.size();
  return 0;
}

// AlgoAffinityGroup.ToAffinityGroup raw material (types.go:187-214)
int hived_get_group_placement(hived_ctx* ctx, int32_t group, hived_group_placement_t* out, int32_t* phys, int32_t* virt,
                              int32_t leaf_cap, int32_t* pods, int32_t pod_cap, int32_t* preempting, int32_t preempting_cap) {
  memset(out, 0, sizeof(*out));
  auto it = ctx->h->affinityGroups.find(groupName(group));
  if (it == ctx->h->affinityGroups.end()) return 0;
  Group* g = it->second;
  out->state = g->state;
  out->has_virtual = g->virtualPlacement.nil ? 0 : 1;
  out->lazy_preempted = g->lazyPreempted ? 1 : 0;
  int32_t k = 0, pk = 0;
  for (auto& kv : g->totalPodNums) {  // ascending leaf number
    int32_t m = out->n_members++;
    if (m < HIVED_MAX_MEMBERS) { out->member_leaf_num[m] = kv.first; out->member_pod_num[m] = kv.second; }
    for (int32_t p = 0; p < kv.second; p++) {
      for (int32_t l = 0; l < kv.first; l++, k++) {
        if (k >= leaf_cap) continue;
        Cell* pc = nullptr; Cell* vc = nullptr;
        auto pit = g->physicalPlacement.m.find(kv.first);
        if (pit != g->physicalPlacement.m.end() && p < (int32_t)pit->second.size() && l < (int32_t)pit->second[p].size()) pc = pit->second[p][l];
        if (!g->virtualPlacement.nil) {
          auto vit = g->virtualPlacement.m.find(kv.first);
          if (vit != g->virtualPlacement.m.end() && p < (int32_t)vit->second.size() && l < (int32_t)vit->second[p].size()) vc = vit->second[p][l];
        }
        if (phys) phys[k] = pc ? pc->id : -1;
        if (virt) virt[k] = vc ? vc->id : -1;
      }
      if (pk < pod_cap && pods) {
        auto ait = g->allocatedPods.find(kv.first);
        Pod* pod = (ait != g->allocatedPods.end() && p < (int32_t)ait->second.size()) ? ait->second[p] : nullptr;
        pods[pk] = pod ? pod->id : -1;
      }
      pk++;
    }
  }
  out->n_leaves = k;
  out->n_pods = pk;
  if (g->state == groupPreempting) {
    out->n_preempting = (int32_t)g->preemptingPods.size();
    int32_t i = 0;
    for (auto& kv : g->preemptingPods) { if (i < preempting_cap && preempting) preempting[i] = kv.first; i++; }
  }
  return 0;
}

int32_t hived_list_groups(hived_ctx* ctx, int32_t* ids, int32_t cap) {
  std::vector<int32_t> v;
  for (auto& kv : ctx->h->affinityGroups) v.push_back(kv.second->id);
  std::sort(v.begin(), v.end());
  for (size_t i = 0; i < v.size() && (int32_t)i < cap; i++) if (ids) ids[i] = v[i];
  return (int32_t)v.size();
}

static void fillInfo(hived_ctx* ctx, Cell* c, hived_cell_info_t* out) {
  HivedAlgorithm& h = *ctx->h;
  memset(out, 0xff, sizeof(*out));
  out->cell_type = ctx->cellTypeIds.count(c->cellType) ? ctx->cellTypeIds[c->cellType] : -1;
  out->is_node_level = c->isNodeLevel ? 1 : 0;
  out->leaf_type = -1;
  for (auto& kv : h.cellChains)  // leaf type -> chains
    for (auto& ch : kv.second)
      if (ch == c->chain)
        for (size_t i = 0; i < h.leafTypeNames.size(); i++) if (h.leafTypeNames[i] == kv.first) out->leaf_type = (int32_t)i;
  out->node = -1; out->leaf_index = -1; out->vc = -1; out->preassigned = -1; out->pinned = -1;
  if (c->physical) {
    if (c->level == 1 && !c->nodes.empty()) {
      out->node = h.nodeIds.count(c->nodes[0]) ? h.nodeIds[c->nodes[0]] : -1;
      out->leaf_index = c->leafCellIndices.empty() ? -1 : c->leafCellIndices[0];
    }
    if (c->pinned && c->virtualCell)  // a pinned cell stays bound to its virtual cell, which carries the id
      for (size_t i = 0; i < h.pinnedNames.size(); i++) if (h.pinnedNames[i] == c->virtualCell->pid) out->pinned = (int32_t)i;
  } else {
    for (size_t i = 0; i < h.vcNames.size(); i++) if (h.vcNames[i] == c->vc) out->vc = (int32_t)i;
    out->preassigned = c->preassignedCell ? c->preassignedCell->id : -1;
    if (!c->pid.empty())
      for (size_t i = 0; i < h.pinnedNames.size(); i++) if (h.pinnedNames[i] == c->pid) out->pinned = (int32_t)i;
  }
}
int hived_physical_cell_info(hived_ctx* ctx, int32_t cell, hived_cell_info_t* out) {
  if (cell < 0 || cell >= (int32_t)ctx->h->physicalCells.size()) { memset(out, 0xff, sizeof(*out)); return HIVED_ERR_PLATFORM; }
  fillInfo(ctx, ctx->h->physicalCells[cell], out);
  return 0;
}
int hived_virtual_cell_info(hived_ctx* ctx, int32_t cell, hived_cell_info_t* out) {
  if (cell < 0 || cell >= (int32_t)ctx->h->virtualCells.size()) { memset(out, 0xff, sizeof(*out)); return HIVED_ERR_PLATFORM; }
  fillInfo(ctx, ctx->h->virtualCells[cell], out);
  return 0;
}

static void fillStatus(hived_ctx* ctx, Cell* c, hived_cell_status_t* s) {
  s->priority = c->priority;
  s->state = c->state;
  s->healthy = c->healthy ? 1 : 0;
  s->level = c->level;
  s->chain = ctx->chainIds.count(c->chain) ? ctx->chainIds[c->chain] : -1;
  s->parent = c->parent ? c->parent->id : -1;
  if (c->physical) {
    s->peer = c->virtualCell ? c->virtualCell->id : -1;
    s->flags = (c->split ? 1 : 0) | (c->pinned ? 2 : 0) | (inFreeCellList(c) ? 4 : 0);
  } else {
    s->peer = c->physicalCell ? c->physicalCell->id : -1;
    s->flags = c->parent == nullptr ? 1 : 0;
  }
}

int hived_snapshot_physical(hived_ctx* ctx, hived_cell_status_t* out, int32_t cap) {
  int32_t n = (int32_t)ctx->h->physicalCells.size();
  if (cap < n) return HIVED_ERR_CAPACITY;
  for (int32_t i = 0; i < n; i++) fillStatus(ctx, ctx->h->physicalCells[i], &out[i]);
  return 0;
}

int hived_snapshot_virtual(hived_ctx* ctx, hived_cell_status_t* out, int32_t cap) {
  int32_t n = (int32_t)ctx->h->virtualCells.size();
  if (cap < n) return HIVED_ERR_CAPACITY;
  for (int32_t i = 0; i < n; i++) fillStatus(ctx, ctx->h->virtualCells[i], &out[i]);
  return 0;
}

int hived_get_stats(hived_ctx* ctx, hived_stats_t* out) {
  memset(out, 0, sizeof(*out));
  const Stats& st = ctx->h->stats;
  out->schedule_events = ctx->schedule_events;
  out->bind_results = ctx->binds;
  out->wait_results = ctx->waits;
  out->preempt_results = ctx->preempts;
  out->view_nodes_scanned = st.view_nodes_scanned;
  out->leaves_committed = st.leaves_committed;
  out->free_cells_scanned = st.free_cells_scanned;
  out->pods_placed = st.pods_placed;
  int64_t K = (int64_t)std::max<size_t>(1, ctx->priorities.size());
  int64_t L = ctx->maxLevels;
  out->algorithmic_bytes = st.view_nodes_scanned * (36 + 4 * K) + st.pods_placed * 64 + st.free_cells_scanned * 12 +
                           st.leaves_committed * 16 * L * (1 + K);
  return 0;
}

uint64_t hived_result_hash(hived_ctx* ctx) { return ctx->hash; }

/* test hook (same definition as the device library's): a hash of every cluster view's persisted order */
uint64_t hived_debug_view_hash(hived_ctx* ctx) {
  uint64_t total = 0;
  auto one = [&](const TopologyAwareScheduler* t) {
    uint64_t h = HIVED_FNV_OFFSET;
    for (const Node* n : t->cv) {
      for (char ch : n->c->address) { h ^= (uint8_t)ch; h *= HIVED_FNV_PRIME; }
      h ^= 0xff; h *= HIVED_FNV_PRIME;
    }
    total += h;
  };
  for (auto& kv : ctx->h->vcSchedulers) {
    for (auto& s : kv.second->nonPinnedCellSchedulers) one(s.second);
    for (auto& s : kv.second->pinnedCellSchedulers) one(s.second);
  }
  for (auto& s : ctx->h->opportunisticSchedulers) one(s.second);
  return total;
}

/* test hook (same encoding as the device library's, include/hived_bench.h): the lists, counters, used-leaf maps, cell
   groups and bad nodes that decide later calls */
int64_t hived_debug_state(hived_ctx* ctx, int32_t* out, int64_t cap) {
  HivedAlgorithm& h = *ctx->h;
  std::vector<int32_t> o;
  const int nC = (int)h.chainNames.size(), nV = (int)h.vcNames.size();
  auto lists = [&](std::initializer_list<int32_t> head, const ChainCellList& ccl) {
    for (const auto& kv : ccl.m) {
      if (kv.second.empty()) continue;
      o.insert(o.end(), head); o.push_back(kv.first); o.push_back((int32_t)kv.second.size());
      for (const Cell* c : kv.second) o.push_back(c->id);
    }
  };
  auto counters = [&](std::initializer_list<int32_t> head, const std::map<int32_t, int32_t>& m) {
    for (const auto& kv : m) {
      if (kv.second == 0) continue;
      o.insert(o.end(), head); o.push_back(kv.first); o.push_back(kv.second);
    }
  };
  for (int c = 0; c < nC; c++) {
    auto it = h.freeCellList.find(h.chainNames[c]);
    if (it != h.freeCellList.end()) lists({HIVED_DS_FREE, c}, it->second);
  }
  for (int c = 0; c < nC; c++) {
    auto it = h.badFreeCells.find(h.chainNames[c]);
    if (it != h.badFreeCells.end()) lists({HIVED_DS_BAD_FREE, c}, it->second);
  }
  for (int v = 0; v < nV; v++) {
    auto vt = h.vcDoomedBadCells.find(h.vcNames[v]);
    if (vt == h.vcDoomedBadCells.end()) continue;
    for (int c = 0; c < nC; c++) {
      auto it = vt->second.find(h.chainNames[c]);
      if (it != vt->second.end()) lists({HIVED_DS_DOOMED_BAD, v, c}, it->second);
    }
  }
  for (int v = 0; v < nV; v++) {
    auto vt = h.vcFreeCellNum.find(h.vcNames[v]);
    if (vt == h.vcFreeCellNum.end()) continue;
    for (int c = 0; c < nC; c++) {
      auto it = vt->second.find(h.chainNames[c]);
      if (it != vt->second.end()) counters({HIVED_DS_VC_FREE, v, c}, it->second);
    }
  }
  const std::pair<int32_t, const std::map<std::string, std::map<int32_t, int32_t>>*> perChain[] = {
      {HIVED_DS_ALL_VC_FREE, &h.allVCFreeCellNum}, {HIVED_DS_TOTAL_LEFT, &h.totalLeftCellNum},
      {HIVED_DS_ALL_VC_DOOMED, &h.allVCDoomedBadCellNum}};
  for (const auto& t : perChain)
    for (int c = 0; c < nC; c++) {
      auto it = t.second->find(h.chainNames[c]);
      if (it != t.second->end()) counters({t.first, c}, it->second);
    }
  auto used = [&](const std::vector<Cell*>& cells, int32_t tag) {
    for (const Cell* c : cells) {
      int32_t k = 0;
      for (const auto& kv : c->used) k += kv.second != 0;
      if (k == 0) continue;
      o.insert(o.end(), {tag, c->id, k});
      for (const auto& kv : c->used) if (kv.second != 0) o.insert(o.end(), {kv.first, kv.second});
    }
  };
  used(h.physicalCells, HIVED_DS_USED_PHYSICAL);
  used(h.virtualCells, HIVED_DS_USED_VIRTUAL);
  auto group = [&](int32_t tag, const Cell* c, const Group* g) {
    if (g == nullptr) return;
    auto it = h.affinityGroups.find(g->name);
    o.insert(o.end(), {tag, c->id, g->id, it != h.affinityGroups.end() && it->second == g ? 1 : 0});
  };
  for (const Cell* c : h.physicalCells) group(HIVED_DS_USING_GROUP, c, c->usingGroup);
  for (const Cell* c : h.physicalCells) group(HIVED_DS_RESERVING_GROUP, c, c->reservingOrReservedGroup);
  for (int i = 0; i < (int)h.nodeNames.size(); i++)
    if (h.badNodes.count(h.nodeNames[i])) o.insert(o.end(), {HIVED_DS_BAD_NODE, i});
  for (size_t i = 0; i < o.size() && (int64_t)i < cap; i++) out[i] = o[i];
  return (int64_t)o.size();
}

}  // extern "C"
