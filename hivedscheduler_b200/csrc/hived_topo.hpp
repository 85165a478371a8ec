// Host-side flattener: HIVEDSPEC text -> flat SoA arrays (the HBM-resident layout of DESIGN.md).
//
// Runs once at hived_create.  It plays the role of the reference's ParseConfig + constructors
// (pkg/algorithm/config.go:442-477, :111-246, :248-413) and of the static part of
// NewHivedAlgorithm (hived_algorithm.go:108-145: scheduler/cluster-view construction,
// topology_aware_scheduler.go:158-179), but instead of a pointer forest it emits integer arrays:
//   * cells of one (chain, level) are contiguous in construction (pre-order) order, so the
//     children of a cell and all leaves below a cell are contiguous id ranges;
//   * every Go-map iteration site is given the canonical order documented in include/hived.h.
// Pure C++ (no CUDA): the product uploads the arrays to the GPU; tests/emu reuses it.
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <functional>
#include <map>
#include <set>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

namespace hived {

constexpr int MAXL = 16;            // levels per chain are 1..MAXL-1
constexpr int MAX_NODE_LEAVES = 64; // leaves below one cluster-view node
constexpr int MAX_FANOUT = 64;      // children per cell
constexpr int FL_DUP_SLACK = 16;    // duplicate entries a free-list segment can hold (see fl_cap)
constexpr int DM_STALE_SLACK = 16;  // stale entries a doomed-bad segment can hold beyond the VC's preassigned cells (dm_cap)

struct TopoError : std::runtime_error {
  int code;
  TopoError(const std::string& m, int c = 101) : std::runtime_error(m), code(c) {}
};

struct FlatTopo {
  // ---- names (interning tables of include/hived.h)
  std::vector<std::string> cellTypeNames, leafTypeNames, chainNames, vcNames, pinnedNames, nodeNames;
  std::vector<std::string> pAddr, vAddr;
  int32_t NP = 0, NV = 0, nChains = 0, nVCs = 0, nLeafTypes = 0, nPinned = 0, nNodes = 0, nVsets = 0, nScheds = 0;

  // ---- physical cells [NP]
  std::vector<int32_t> p_parent, p_child0, p_nchild, p_level, p_chain, p_leaf0, p_nleaf, p_node, p_leafidx, p_flags;
  std::vector<int32_t> p_nodes_off, p_nodes_cnt, nodes_flat;  // node ids below a cell
  std::vector<int32_t> p_anc, v_anc;                          // [N * AS] ancestor per level
  int32_t AS = 1;
  bool uniqueLeafIdx = true;  // no two leaf cells of one (node, chain) share a leaf index
  // ---- virtual cells [NV]
  std::vector<int32_t> v_parent, v_child0, v_nchild, v_level, v_chain, v_leaf0, v_nleaf, v_vc, v_pre, v_vset, v_flags;
  std::vector<int32_t> v_pretype, v_prelevel;  // level of a virtual cell's preassigned (top) cell and that level's cell type id

  // ---- per chain
  std::vector<int32_t> chain_top, chain_leaftype;         // [nChains]
  std::vector<int32_t> chain_lvl_type, chain_lvl_leafnum; // [nChains*MAXL] cell type id / #leaves at level
  std::vector<int32_t> chain_lvl_nchild;                  // [nChains*MAXL] fan-out of level-l cells
  std::vector<int32_t> p_lvl_base, p_lvl_cnt;             // [nChains*MAXL] id range of fullCellList[chain][level]
  std::vector<int32_t> chain_in_vc;                       // [nChains] some VC owns cells of the chain
  std::vector<int32_t> lt_off, lt_cnt, lt_chains;         // chains of a leaf type, descending name order
  // ---- virtual cell sets: (vc, chain) non-pinned or (vc, pinned id)
  std::vector<int32_t> vs_vc, vs_chain, vs_pinned, vs_top;  // [nVsets]
  std::vector<int32_t> v_lvl_base, v_lvl_cnt;               // [nVsets*MAXL]
  std::vector<int32_t> vc_chain_vset;                       // [nVCs*nChains] or -1
  std::vector<int32_t> vc_pinned_vset;                      // [nVCs*nPinned] or -1
  std::vector<int32_t> pre_off, pre_cnt, pre_list;          // [nVCs*nChains*MAXL] preassigned roots per level
  std::vector<int32_t> vc_chain_counter;                    // [nVCs*nChains] vcFreeCellNum[vc] has the chain
  std::vector<int32_t> pin_pcell, pin_vcell, pin_vc;        // [nPinned]
  // ---- schedulers (cluster views)
  std::vector<int32_t> s_off, s_n, s_cross, s_chain, s_virtual, s_maxleaf;  // [nScheds]
  // bucketed (incremental) cluster views: s_level = level of the view cells, s_vc = owning VC (-1: physical view),
  // s_fast = 1 when every view cell is a virtual cell of that one level with the same number (<= 32) of leaf cells
  // laid out uniformly (the level-l cells below a view cell are aligned runs of chain_lvl_leafnum[l] leaves)
  std::vector<int32_t> s_level, s_vc, s_fast;
  std::vector<int32_t> s_cell0, s_leaf0;  // fast views: the view cells are the ids s_cell0 + i, their leaves s_leaf0 + i * L + j
  std::vector<int32_t> cv_init;                                             // initial view order (cell ids)
  std::vector<int32_t> vset_sched, opp_sched;                               // [nVsets], [nChains]
  // ---- node -> leaves per chain (findPhysicalLeafCellInChain without the linear scan)
  std::vector<int32_t> ncl_off, ncl_cnt, ncl_list;  // [nNodes*nChains]
  // ---- initial dynamic state
  std::vector<int32_t> vcFree, allVCFree, totalLeft;  // [nVCs*nChains*MAXL], [nChains*MAXL] x2
  std::vector<int32_t> fl_base, fl_cap;               // [nChains*MAXL] free-list segments (cap = #cells)
  std::vector<int32_t> fl_init_len, fl_init_data;     // initial free lists (top cells)
  int32_t flTotal = 0;
  std::vector<int32_t> dm_base, dm_cap;  // [nVCs*nChains*MAXL] doomed-bad list segments
  int32_t dmTotal = 0;
  int32_t maxFanout = 1, maxLevelCount = 1, maxViewN = 1, maxChainFree = 1, maxNodeLeaves = 1, maxLevels = 1;
  // initPinnedCells order: (vc asc, pinned id asc) pairs
  std::vector<int32_t> pinned_init_order;
  // initBadNodes order (every node once, hived_algorithm.go:453-464)
  std::vector<int32_t> bad_init_order;
};

enum : int32_t { PF_AT_OR_ABOVE_NODE = 1, PF_NODE_LEVEL = 2, PF_PINNED = 4 };

namespace detail {

struct TypeSpec { std::string child; int32_t n = 0; bool node = false; };
struct Elem {  // cellChainElement, config.go:34-43
  int32_t level = 0; std::string child; int32_t childNumber = 0; bool hasNode = false, isMultiNodes = false;
  std::string leafType; int32_t leafNum = 0;
};
struct PSpec { std::string type, addr, pid; std::vector<PSpec> ch; };
struct VCSpec { std::vector<std::pair<std::string, int32_t>> cells; std::vector<std::string> pinned; };

struct Tok {
  std::istringstream in;
  explicit Tok(const std::string& s) : in(s) {}
  std::string s() { std::string t; if (!(in >> t)) throw TopoError("HIVEDSPEC: unexpected end"); return t; }
  int32_t i() {
    std::string t = s(); char* e = nullptr; long v = strtol(t.c_str(), &e, 10);
    if (*e) throw TopoError("HIVEDSPEC: expected integer, got " + t); return (int32_t)v;
  }
  void expect(const char* w) { std::string t = s(); if (t != w) throw TopoError(std::string("HIVEDSPEC: expected ") + w + " got " + t); }
};

inline void readP(Tok& tk, PSpec& p, int depth) {
  if (tk.i() != depth) throw TopoError("HIVEDSPEC: bad depth");
  p.type = tk.s(); p.addr = tk.s(); p.pid = tk.s(); if (p.pid == "-") p.pid.clear();
  int32_t n = tk.i(); p.ch.resize(n);
  for (auto& c : p.ch) readP(tk, c, depth + 1);
}

inline std::string lastSeg(const std::string& a) { size_t p = a.rfind('/'); return p == std::string::npos ? a : a.substr(p + 1); }
inline int32_t toInt(const std::string& s) {
  char* e = nullptr; long v = strtol(s.c_str(), &e, 10);
  if (s.empty() || *e) throw TopoError("leaf cell address is not an integer index: " + s); return (int32_t)v;
}

// a cell while building (one struct for both forests)
struct BCell {
  int32_t parent = -1, level = 0, chain = -1, vset = -1, pre = -1, node = -1, leafidx = -1, flags = 0, type = -1;
  std::vector<int32_t> children, nodes;
  std::string addr;
  int32_t finalId = -1, leaf0 = -1, nleaf = 0;
};

}  // namespace detail

inline FlatTopo buildTopo(const std::string& text) {
  using namespace detail;
  FlatTopo T;
  // ------------------------------------------------------------------ parse
  Tok tk(text);
  tk.expect("HIVEDSPEC"); tk.expect("1"); tk.expect("celltypes");
  std::map<std::string, TypeSpec> types;
  for (int32_t n = tk.i(), k = 0; k < n; k++) { std::string nm = tk.s(); TypeSpec t; t.child = tk.s(); t.n = tk.i(); t.node = tk.i() != 0; types[nm] = t; }
  tk.expect("physicalcells");
  std::vector<PSpec> pcs(tk.i());
  for (auto& p : pcs) readP(tk, p, 0);
  tk.expect("virtualclusters");
  std::map<std::string, VCSpec> vcs;
  for (int32_t n = tk.i(), k = 0; k < n; k++) {
    tk.expect("vc"); std::string nm = tk.s(); int32_t nv = tk.i(), np = tk.i(); VCSpec v;
    for (int32_t j = 0; j < nv; j++) { std::string t = tk.s(); int32_t c = tk.i(); v.cells.push_back({t, c}); }
    for (int32_t j = 0; j < np; j++) v.pinned.push_back(tk.s());
    vcs[nm] = v;
  }
  tk.expect("end");

  // ------------------------------------------------------------------ cell chain elements (config.go:59-109)
  std::map<std::string, Elem> el;
  std::function<void(const std::string&)> addChain = [&](const std::string& ct) {
    if (el.count(ct)) return;
    auto it = types.find(ct);
    if (it == types.end()) { Elem e; e.level = 1; e.leafType = ct; e.leafNum = 1; el[ct] = e; return; }
    addChain(it->second.child);
    const Elem c = el[it->second.child];
    Elem e; e.level = c.level + 1; e.child = it->second.child; e.childNumber = it->second.n;
    e.hasNode = c.hasNode || it->second.node; e.isMultiNodes = c.hasNode; e.leafType = c.leafType; e.leafNum = c.leafNum * it->second.n;
    if (e.level >= MAXL) throw TopoError("cell chain deeper than MAXL levels");
    el[ct] = e;
  };
  for (auto& kv : types) addChain(kv.first);

  // ------------------------------------------------------------------ id tables
  {
    std::set<std::string> tset, lset, cset, pset;
    for (auto& kv : el) { tset.insert(kv.first); if (kv.second.level == 1) lset.insert(kv.first); }
    for (auto& p : pcs) cset.insert(p.type);
    std::function<void(const PSpec&)> pins = [&](const PSpec& p) { if (!p.pid.empty()) pset.insert(p.pid); for (auto& c : p.ch) pins(c); };
    for (auto& p : pcs) pins(p);
    T.cellTypeNames.assign(tset.begin(), tset.end()); T.leafTypeNames.assign(lset.begin(), lset.end());
    T.chainNames.assign(cset.begin(), cset.end()); T.pinnedNames.assign(pset.begin(), pset.end());
    for (auto& kv : vcs) T.vcNames.push_back(kv.first);
  }
  auto idOf = [](const std::vector<std::string>& v, const std::string& s) -> int32_t {
    auto it = std::lower_bound(v.begin(), v.end(), s); return (it != v.end() && *it == s) ? (int32_t)(it - v.begin()) : -1;
  };
  T.nChains = (int32_t)T.chainNames.size(); T.nVCs = (int32_t)T.vcNames.size(); T.nLeafTypes = (int32_t)T.leafTypeNames.size();
  T.nPinned = (int32_t)T.pinnedNames.size();
  std::map<std::string, int32_t> nodeIds;

  // ------------------------------------------------------------------ physical forest (config.go:141-246)
  std::vector<BCell> P;
  std::vector<std::vector<std::vector<int32_t>>> pLvl(T.nChains, std::vector<std::vector<int32_t>>(MAXL));  // fullCellList
  std::vector<std::vector<int32_t>> pTops(T.nChains);
  std::map<std::string, int32_t> pinnedCell;  // pid -> building index
  std::function<int32_t(const PSpec&, const std::string&, int32_t, int32_t)> buildP =
      [&](const PSpec& sp, const std::string& ct, int32_t chain, int32_t curNode) -> int32_t {
    auto eit = el.find(ct);
    if (eit == el.end()) throw TopoError("cellType " + ct + " not found in cell types definition");
    const Elem& ce = eit->second;
    if (ce.hasNode && !ce.isMultiNodes) {
      std::string nn = lastSeg(sp.addr);
      auto nit = nodeIds.find(nn);
      if (nit == nodeIds.end()) { nit = nodeIds.insert({nn, (int32_t)T.nodeNames.size()}).first; T.nodeNames.push_back(nn); }
      curNode = nit->second;
    }
    int32_t me = (int32_t)P.size();
    P.emplace_back();
    P[me].level = ce.level; P[me].chain = chain; P[me].addr = sp.addr; P[me].type = idOf(T.cellTypeNames, ct);
    P[me].flags = (ce.hasNode ? PF_AT_OR_ABOVE_NODE : 0) | ((ce.hasNode && !ce.isMultiNodes) ? PF_NODE_LEVEL : 0);
    pLvl[chain][ce.level].push_back(me);
    if (!sp.pid.empty()) { pinnedCell[sp.pid] = me; P[me].flags |= PF_PINNED; }
    if (ce.level == 1) { P[me].nodes = {curNode}; P[me].leafidx = toInt(lastSeg(sp.addr)); return me; }
    std::vector<int32_t> nodes;
    for (auto& chs : sp.ch) {
      int32_t c = buildP(chs, ce.child, chain, curNode);
      P[c].parent = me; P[me].children.push_back(c);
      if (ce.isMultiNodes) nodes.insert(nodes.end(), P[c].nodes.begin(), P[c].nodes.end());
    }
    if (!ce.isMultiNodes) nodes = {curNode};
    P[me].nodes = nodes;
    return me;
  };
  for (auto& sp : pcs) {
    int32_t chain = idOf(T.chainNames, sp.type);
    auto eit = el.find(sp.type);
    if (eit == el.end()) throw TopoError("cellType " + sp.type + " in PhysicalCells is not found in cell types definition");
    if (!eit->second.hasNode) throw TopoError("top cell must be node-level or above: " + sp.type);
    pTops[chain].push_back(buildP(sp, sp.type, chain, -1));
  }
  T.nNodes = (int32_t)T.nodeNames.size();

  // ------------------------------------------------------------------ virtual forests (config.go:332-413)
  // vsets: for each VC (asc): non-pinned chains (asc) then pinned ids (asc)
  std::vector<BCell> V;
  struct VSetB { int32_t vc, chain, pinned; std::vector<std::vector<int32_t>> lvl; std::vector<std::vector<int32_t>> pre; };
  std::vector<VSetB> vsets;
  T.vc_chain_vset.assign((size_t)T.nVCs * T.nChains, -1);
  T.vc_pinned_vset.assign((size_t)T.nVCs * std::max(1, T.nPinned), -1);
  T.vc_chain_counter.assign((size_t)T.nVCs * T.nChains, 0);
  T.vcFree.assign((size_t)T.nVCs * T.nChains * MAXL, 0);
  T.pin_pcell.assign(T.nPinned, -1); T.pin_vcell.assign(T.nPinned, -1); T.pin_vc.assign(T.nPinned, -1);
  std::vector<int32_t> pinPhysB(T.nPinned, -1);
  std::function<int32_t(const std::string&, const std::string&, int32_t, int32_t&, int32_t)> buildV =
      [&](const std::string& ct, const std::string& addr, int32_t vsi, int32_t& root, int32_t vc) -> int32_t {
    const Elem& ce = el.at(ct);
    int32_t me = (int32_t)V.size();
    V.emplace_back();
    V[me].level = ce.level; V[me].chain = vsets[vsi].chain; V[me].vset = vsi; V[me].addr = addr; V[me].type = idOf(T.cellTypeNames, ct);
    V[me].flags = (ce.hasNode ? PF_AT_OR_ABOVE_NODE : 0) | ((ce.hasNode && !ce.isMultiNodes) ? PF_NODE_LEVEL : 0);
    vsets[vsi].lvl[ce.level].push_back(me);
    if (root < 0) root = me;
    V[me].pre = root;
    if (ce.level == 1) return me;
    size_t slashes = std::count(addr.begin(), addr.end(), '/');
    int32_t offset = slashes == 1 ? 0 : toInt(lastSeg(addr)) * ce.childNumber;
    for (int32_t i = 0; i < ce.childNumber; i++) {
      int32_t c = buildV(ce.child, addr + "/" + std::to_string(offset + i), vsi, root, vc);
      V[c].parent = me; V[me].children.push_back(c);
    }
    return me;
  };
  for (int32_t vc = 0; vc < T.nVCs; vc++) {
    const VCSpec& spec = vcs[T.vcNames[vc]];
    // pre-create the vsets of this VC in canonical order
    std::set<int32_t> chainsOfVc;
    for (auto& c : spec.cells) {
      std::string ch = c.first.substr(0, c.first.find('.'));
      int32_t cid = idOf(T.chainNames, ch);
      if (cid < 0) throw TopoError("Illegal initial VC assignment: Chain " + ch + " does not exists in physical cluster");
      // a spec with cellNumber 0 creates the counter key but no cells, hence no scheduler (config.go:379-391)
      if (c.second > 0) chainsOfVc.insert(cid);
    }
    for (int32_t cid : chainsOfVc) {
      T.vc_chain_vset[(size_t)vc * T.nChains + cid] = (int32_t)vsets.size();
      vsets.push_back({vc, cid, -1, std::vector<std::vector<int32_t>>(MAXL), std::vector<std::vector<int32_t>>(MAXL)});
    }
    std::vector<std::string> pins = spec.pinned;
    std::vector<std::string> pinsSorted = pins; std::sort(pinsSorted.begin(), pinsSorted.end());
    for (auto& pid : pinsSorted) {
      int32_t pi = idOf(T.pinnedNames, pid);
      if (pi < 0 || !pinnedCell.count(pid)) throw TopoError("pinned cell not found in physicalCells: VC: " + T.vcNames[vc] + ", ID: " + pid);
      T.vc_pinned_vset[(size_t)vc * T.nPinned + pi] = (int32_t)vsets.size();
      vsets.push_back({vc, P[pinnedCell[pid]].chain, pi, std::vector<std::vector<int32_t>>(MAXL), std::vector<std::vector<int32_t>>(MAXL)});
    }
    int32_t numCells = 0;
    for (auto& c : spec.cells) {
      std::string ch = c.first.substr(0, c.first.find('.'));
      size_t lp = c.first.rfind('.');
      std::string rootType = lp == std::string::npos ? c.first : c.first.substr(lp + 1);
      auto rit = el.find(rootType);
      if (rit == el.end()) throw TopoError("cellType " + rootType + " in VirtualCells is not found in cell types definition");
      int32_t cid = idOf(T.chainNames, ch);
      int32_t vsi = T.vc_chain_vset[(size_t)vc * T.nChains + cid];
      T.vc_chain_counter[(size_t)vc * T.nChains + cid] = 1;
      T.vcFree[((size_t)vc * T.nChains + cid) * MAXL + rit->second.level] += c.second;
      for (int32_t i = 0; i < c.second; i++) {
        int32_t root = -1;
        int32_t r = buildV(rootType, T.vcNames[vc] + "/" + std::to_string(numCells), vsi, root, vc);
        vsets[vsi].pre[V[r].level].push_back(r);
        numCells++;
      }
    }
    for (auto& pid : pins) {  // config order decides the addresses vc/<k>
      int32_t pi = idOf(T.pinnedNames, pid);
      int32_t pcB = pinnedCell[pid];
      std::string child = T.chainNames[P[pcB].chain];
      while (el.at(child).level > P[pcB].level) child = el.at(child).child;
      int32_t cid = P[pcB].chain;
      T.vc_chain_counter[(size_t)vc * T.nChains + cid] = 1;
      T.vcFree[((size_t)vc * T.nChains + cid) * MAXL + P[pcB].level] += 1;
      int32_t vsi = T.vc_pinned_vset[(size_t)vc * T.nPinned + pi];
      int32_t root = -1;
      int32_t r = buildV(child, T.vcNames[vc] + "/" + std::to_string(numCells), vsi, root, vc);
      pinPhysB[pi] = pcB; T.pin_vcell[pi] = r; T.pin_vc[pi] = vc;
      numCells++;
    }
  }
  T.nVsets = (int32_t)vsets.size();

  // ------------------------------------------------------------------ final ids (include/hived.h)
  T.p_lvl_base.assign((size_t)T.nChains * MAXL, 0); T.p_lvl_cnt.assign((size_t)T.nChains * MAXL, 0);
  T.chain_top.assign(T.nChains, 0);
  {
    int32_t id = 0;
    for (int32_t c = 0; c < T.nChains; c++)
      for (int32_t l = 1; l < MAXL; l++) {
        T.p_lvl_base[c * MAXL + l] = id; T.p_lvl_cnt[c * MAXL + l] = (int32_t)pLvl[c][l].size();
        if (!pLvl[c][l].empty()) T.chain_top[c] = l;
        for (int32_t b : pLvl[c][l]) P[b].finalId = id++;
      }
    T.NP = id;
  }
  T.v_lvl_base.assign((size_t)T.nVsets * MAXL, 0); T.v_lvl_cnt.assign((size_t)T.nVsets * MAXL, 0);
  T.vs_vc.resize(T.nVsets); T.vs_chain.resize(T.nVsets); T.vs_pinned.resize(T.nVsets); T.vs_top.assign(T.nVsets, 0);
  {
    int32_t id = 0;
    for (int32_t s = 0; s < T.nVsets; s++) {
      T.vs_vc[s] = vsets[s].vc; T.vs_chain[s] = vsets[s].chain; T.vs_pinned[s] = vsets[s].pinned;
      for (int32_t l = 1; l < MAXL; l++) {
        T.v_lvl_base[s * MAXL + l] = id; T.v_lvl_cnt[s * MAXL + l] = (int32_t)vsets[s].lvl[l].size();
        if (!vsets[s].lvl[l].empty()) T.vs_top[s] = l;
        for (int32_t b : vsets[s].lvl[l]) V[b].finalId = id++;
      }
    }
    T.NV = id;
  }
  auto fillTree = [&](std::vector<BCell>& B, int32_t N, std::vector<int32_t>& parent, std::vector<int32_t>& child0,
                      std::vector<int32_t>& nchild, std::vector<int32_t>& level, std::vector<int32_t>& chain,
                      std::vector<int32_t>& leaf0, std::vector<int32_t>& nleaf, std::vector<std::string>& addr) {
    parent.assign(N, -1); child0.assign(N, -1); nchild.assign(N, 0); level.assign(N, 0); chain.assign(N, -1);
    leaf0.assign(N, -1); nleaf.assign(N, 0); addr.assign(N, "");
    // leaves below a cell: contiguous final ids at level 1 (pre-order construction)
    std::function<void(int32_t)> leaves = [&](int32_t b) {
      if (B[b].level == 1) { B[b].leaf0 = B[b].finalId; B[b].nleaf = 1; return; }
      for (int32_t c : B[b].children) leaves(c);
      B[b].leaf0 = B[B[b].children.front()].leaf0; B[b].nleaf = 0;
      for (int32_t c : B[b].children) {
        if (B[c].leaf0 != B[b].leaf0 + B[b].nleaf) throw TopoError("internal: leaves of a cell are not contiguous");
        B[b].nleaf += B[c].nleaf;
      }
    };
    for (size_t b = 0; b < B.size(); b++) if (B[b].parent < 0) leaves((int32_t)b);
    for (auto& bc : B) {
      int32_t i = bc.finalId;
      parent[i] = bc.parent < 0 ? -1 : B[bc.parent].finalId;
      nchild[i] = (int32_t)bc.children.size();
      if ((int32_t)bc.children.size() > T.maxFanout) T.maxFanout = (int32_t)bc.children.size();
      if (!bc.children.empty()) {
        child0[i] = B[bc.children[0]].finalId;
        for (size_t k = 0; k < bc.children.size(); k++)
          if (B[bc.children[k]].finalId != child0[i] + (int32_t)k) throw TopoError("internal: children of a cell are not contiguous");
      }
      level[i] = bc.level; chain[i] = bc.chain; leaf0[i] = bc.leaf0; nleaf[i] = bc.nleaf; addr[i] = bc.addr;
    }
  };
  fillTree(P, T.NP, T.p_parent, T.p_child0, T.p_nchild, T.p_level, T.p_chain, T.p_leaf0, T.p_nleaf, T.pAddr);
  fillTree(V, T.NV, T.v_parent, T.v_child0, T.v_nchild, T.v_level, T.v_chain, T.v_leaf0, T.v_nleaf, T.vAddr);
  if (T.maxFanout > MAX_FANOUT) throw TopoError("a cell has more than MAX_FANOUT children", 102);
  T.p_node.assign(T.NP, -1); T.p_leafidx.assign(T.NP, -1); T.p_flags.assign(T.NP, 0);
  T.p_nodes_off.assign(T.NP, 0); T.p_nodes_cnt.assign(T.NP, 0);
  for (auto& bc : P) {
    int32_t i = bc.finalId;
    T.p_flags[i] = bc.flags; T.p_leafidx[i] = bc.leafidx;
    T.p_nodes_off[i] = (int32_t)T.nodes_flat.size(); T.p_nodes_cnt[i] = (int32_t)bc.nodes.size();
    T.nodes_flat.insert(T.nodes_flat.end(), bc.nodes.begin(), bc.nodes.end());
    if (bc.nodes.size() == 1) T.p_node[i] = bc.nodes[0];
  }
  T.v_vc.assign(T.NV, -1); T.v_pre.assign(T.NV, -1); T.v_vset.assign(T.NV, -1); T.v_flags.assign(T.NV, 0);
  for (auto& bc : V) {
    int32_t i = bc.finalId;
    T.v_vc[i] = vsets[bc.vset].vc; T.v_pre[i] = V[bc.pre].finalId; T.v_vset[i] = bc.vset; T.v_flags[i] = bc.flags;
  }
  for (int32_t pi = 0; pi < T.nPinned; pi++) {
    if (pinPhysB[pi] >= 0) { T.pin_pcell[pi] = P[pinPhysB[pi]].finalId; T.pin_vcell[pi] = V[T.pin_vcell[pi]].finalId; }
    else if (pinnedCell.count(T.pinnedNames[pi])) T.pin_pcell[pi] = P[pinnedCell[T.pinnedNames[pi]]].finalId;  // pinned but owned by no VC
  }

  // ------------------------------------------------------------------ chain tables (config.go:415-440)
  T.chain_leaftype.assign(T.nChains, -1);
  T.chain_lvl_type.assign((size_t)T.nChains * MAXL, -1); T.chain_lvl_leafnum.assign((size_t)T.nChains * MAXL, 0);
  T.chain_lvl_nchild.assign((size_t)T.nChains * MAXL, 0);
  for (int32_t c = 0; c < T.nChains; c++) {
    const Elem* ce = &el.at(T.chainNames[c]);
    std::string nm = T.chainNames[c];
    T.chain_leaftype[c] = idOf(T.leafTypeNames, ce->leafType);
    while (true) {
      T.chain_lvl_type[c * MAXL + ce->level] = idOf(T.cellTypeNames, nm);
      T.chain_lvl_leafnum[c * MAXL + ce->level] = ce->leafNum;
      // len(fullCellList[chain][l][0].GetChildren()) — of the first cell actually built
      if (!pLvl[c][ce->level].empty()) T.chain_lvl_nchild[c * MAXL + ce->level] = (int32_t)P[pLvl[c][ce->level][0]].children.size();
      if (ce->level > T.maxLevels) T.maxLevels = ce->level;
      auto nit = el.find(ce->child);
      if (nit == el.end()) break;
      nm = ce->child; ce = &nit->second;
    }
  }
  // PreassignedCellTypes of a virtual cell (utils.go:150-153): level of its preassigned cell and that level's type
  T.v_prelevel.assign(std::max(1, T.NV), 0); T.v_pretype.assign(std::max(1, T.NV), -1);
  for (int32_t i = 0; i < T.NV; i++) {
    int32_t pre = T.v_pre[i];
    if (pre < 0) continue;
    T.v_prelevel[i] = T.v_level[pre];
    T.v_pretype[i] = T.chain_lvl_type[(size_t)T.v_chain[i] * MAXL + T.v_level[pre]];
  }
  // ancestor tables: anc[cell * AS + l] = the ancestor of `cell` at level l (the cell itself at its own
  // level, -1 below it or above its tree's top) — turns every leaf-to-root walk into independent loads
  T.AS = T.maxLevels + 1;
  T.p_anc.assign((size_t)std::max(1, T.NP) * T.AS, -1);
  for (int32_t i = 0; i < T.NP; i++)
    for (int32_t c = i; c >= 0; c = T.p_parent[c]) T.p_anc[(size_t)i * T.AS + T.p_level[c]] = c;
  T.v_anc.assign((size_t)std::max(1, T.NV) * T.AS, -1);
  for (int32_t i = 0; i < T.NV; i++)
    for (int32_t c = i; c >= 0; c = T.v_parent[c]) T.v_anc[(size_t)i * T.AS + T.v_level[c]] = c;
  T.lt_off.assign(T.nLeafTypes, 0); T.lt_cnt.assign(T.nLeafTypes, 0);
  for (int32_t lt = 0; lt < T.nLeafTypes; lt++) {
    T.lt_off[lt] = (int32_t)T.lt_chains.size();
    for (int32_t c = T.nChains - 1; c >= 0; c--)  // descending chain name
      if (T.chain_leaftype[c] == lt) { T.lt_chains.push_back(c); T.lt_cnt[lt]++; }
  }

  // ------------------------------------------------------------------ preassigned lists, counters (hived_algorithm.go:365-409)
  T.pre_off.assign((size_t)T.nVCs * T.nChains * MAXL, 0); T.pre_cnt.assign((size_t)T.nVCs * T.nChains * MAXL, 0);
  for (int32_t s = 0; s < T.nVsets; s++) {
    if (vsets[s].pinned >= 0) continue;
    for (int32_t l = 1; l < MAXL; l++) {
      size_t k = ((size_t)vsets[s].vc * T.nChains + vsets[s].chain) * MAXL + l;
      T.pre_off[k] = (int32_t)T.pre_list.size(); T.pre_cnt[k] = (int32_t)vsets[s].pre[l].size();
      for (int32_t b : vsets[s].pre[l]) T.pre_list.push_back(V[b].finalId);
    }
  }
  T.allVCFree.assign((size_t)T.nChains * MAXL, 0); T.totalLeft.assign((size_t)T.nChains * MAXL, 0); T.chain_in_vc.assign(T.nChains, 0);
  for (int32_t vc = 0; vc < T.nVCs; vc++)
    for (int32_t c = 0; c < T.nChains; c++)
      if (T.vc_chain_counter[(size_t)vc * T.nChains + c]) {
        T.chain_in_vc[c] = 1;
        for (int32_t l = 1; l < MAXL; l++) T.allVCFree[c * MAXL + l] += T.vcFree[((size_t)vc * T.nChains + c) * MAXL + l];
      }
  for (int32_t c = 0; c < T.nChains; c++) {
    if (!T.chain_in_vc[c]) continue;
    int32_t top = T.chain_top[c];
    int32_t available = T.p_lvl_cnt[c * MAXL + top];
    T.totalLeft[c * MAXL + top] = available;
    for (int32_t l = top; l >= 1; l--) {
      int32_t left = available - T.allVCFree[c * MAXL + l];
      if (left < 0)
        throw TopoError("Illegal initial VC assignment: Insufficient physical cells at chain " + T.chainNames[c] + " level " +
                        std::to_string(l) + ": " + std::to_string(T.allVCFree[c * MAXL + l]) + " needed, " + std::to_string(available) + " available");
      if (l > 1) {
        int32_t childNum = T.chain_lvl_nchild[c * MAXL + l];
        available = left * childNum;
        T.totalLeft[c * MAXL + l - 1] = T.totalLeft[c * MAXL + l] * childNum;
      }
    }
  }

  // ------------------------------------------------------------------ list segments
  T.fl_base.assign((size_t)T.nChains * MAXL, 0); T.fl_cap.assign((size_t)T.nChains * MAXL, 0);
  T.fl_init_len.assign((size_t)T.nChains * MAXL, 0);
  for (int32_t c = 0; c < T.nChains; c++) {
    int32_t chainTotal = 0;
    for (int32_t l = 1; l < MAXL; l++) {
      // the reference's free list is a slice: releasing a preassigned cell that is already free appends it AGAIN
      // (addCellToFreeList, hived_algorithm.go:1530-1565 — reachable once Filtering-phase binds have made its counters
      // drift), so a segment has room for FL_DUP_SLACK duplicates beyond the cells of its level (hived_core.h fl_append)
      const int32_t cap = T.p_lvl_cnt[c * MAXL + l] > 0 ? T.p_lvl_cnt[c * MAXL + l] + FL_DUP_SLACK : 0;
      T.fl_base[c * MAXL + l] = T.flTotal; T.fl_cap[c * MAXL + l] = cap;
      T.flTotal += cap; chainTotal += cap;
      if (cap > T.maxLevelCount) T.maxLevelCount = cap;
    }
    if (chainTotal > T.maxChainFree) T.maxChainFree = chainTotal;
  }
  T.fl_init_data.assign(T.flTotal, -1);
  for (int32_t c = 0; c < T.nChains; c++) {
    int32_t top = T.chain_top[c];
    for (int32_t b : pTops[c]) T.fl_init_data[T.fl_base[c * MAXL + top] + T.fl_init_len[c * MAXL + top]++] = P[b].finalId;
  }
  T.dm_base.assign((size_t)T.nVCs * T.nChains * MAXL, 0); T.dm_cap.assign((size_t)T.nVCs * T.nChains * MAXL, 0);
  for (size_t k = 0; k < T.dm_base.size(); k++) {
    // doomed bad cells bound now (at most one per preassigned cell) plus stale entries (hived_core.h dm_append)
    const int32_t cap = T.pre_cnt[k] > 0 ? T.pre_cnt[k] + DM_STALE_SLACK : 0;
    T.dm_base[k] = T.dmTotal; T.dm_cap[k] = cap; T.dmTotal += cap;
  }

  // ------------------------------------------------------------------ cluster views (topology_aware_scheduler.go:158-198)
  auto makeView = [&](std::vector<BCell>& B, const std::vector<std::vector<int32_t>>& lvl, int32_t top, bool cross, int32_t chain, bool isVirtual) -> int32_t {
    int32_t sid = (int32_t)T.s_off.size();
    int32_t l = 1;
    for (; l <= top; l++) {
      if (lvl[l].empty()) throw TopoError("internal: empty level in a cell list");
      if (B[lvl[l][0]].flags & PF_AT_OR_ABOVE_NODE) break;
    }
    T.s_off.push_back((int32_t)T.cv_init.size());
    std::set<int32_t> inView;  // building indices of view cells
    int32_t n = 0, maxleaf = 1;
    for (; l >= 1; l--) {
      if (l >= MAXL) continue;
      for (int32_t b : lvl[l]) {
        int32_t a = b;  // ancestorNoHigherThanNode
        while (!(B[a].flags & PF_AT_OR_ABOVE_NODE) && B[a].parent >= 0) a = B[a].parent;
        if (!inView.count(a)) {
          inView.insert(b); T.cv_init.push_back(B[b].finalId); n++;
          if (B[b].nleaf > maxleaf) maxleaf = B[b].nleaf;
        }
      }
    }
    if (maxleaf > MAX_NODE_LEAVES) throw TopoError("a cluster-view node has more than MAX_NODE_LEAVES leaf cells", 102);
    if (maxleaf > T.maxNodeLeaves) T.maxNodeLeaves = maxleaf;
    if (n > T.maxViewN) T.maxViewN = n;
    T.s_n.push_back(n); T.s_cross.push_back(cross ? 1 : 0); T.s_chain.push_back(chain); T.s_virtual.push_back(isVirtual ? 1 : 0);
    T.s_maxleaf.push_back(maxleaf);
    // ---- eligibility for the bucketed view (hived_core.h: fastPlace)
    int32_t viewLevel = -1, vc = -1;
    bool fast = isVirtual && n > 0 && maxleaf <= 32;
    const int32_t off = T.s_off.back();
    for (int32_t i = 0; i < n && fast; i++) {
      int32_t c = T.cv_init[off + i];
      if (i == 0) { viewLevel = T.v_level[c]; vc = T.v_vc[c]; }
      if (T.v_level[c] != viewLevel || T.v_nleaf[c] != maxleaf || T.v_vc[c] != vc) fast = false;
      for (int32_t l = 1; l < viewLevel && fast; l++) {
        int32_t sl = T.chain_lvl_leafnum[(size_t)chain * MAXL + l];
        if (sl <= 0 || maxleaf % sl) { fast = false; break; }
        for (int32_t j = 0; j < maxleaf; j++) {
          int32_t leaf = T.v_leaf0[c] + j, first = T.v_leaf0[c] + j / sl * sl;
          if (T.v_anc[(size_t)leaf * T.AS + l] != T.v_anc[(size_t)first * T.AS + l]) fast = false;
          if (j % sl == 0 && j > 0 && T.v_anc[(size_t)leaf * T.AS + l] == T.v_anc[(size_t)(leaf - 1) * T.AS + l]) fast = false;
        }
      }
    }
    int32_t cell0 = n > 0 ? T.cv_init[off] : 0, leaf0 = (isVirtual && n > 0) ? T.v_leaf0[T.cv_init[off]] : 0;
    for (int32_t i = 0; i < n && fast; i++)
      if (T.cv_init[off + i] != cell0 + i || T.v_leaf0[cell0 + i] != leaf0 + i * maxleaf) fast = false;
    for (int32_t l = 2; l <= T.chain_top[chain] && fast; l++)
      if (T.chain_lvl_nchild[(size_t)chain * MAXL + l] > 32) fast = false;  // child masks are 32 bits wide
    T.s_cell0.push_back(cell0); T.s_leaf0.push_back(leaf0);
    if (isVirtual && n > 0 && viewLevel < 0) viewLevel = T.v_level[T.cv_init[off]];
    T.s_level.push_back(viewLevel); T.s_vc.push_back(isVirtual ? vc : -1); T.s_fast.push_back(fast ? 1 : 0);
    return sid;
  };
  T.vset_sched.assign(T.nVsets, -1);
  for (int32_t s = 0; s < T.nVsets; s++) T.vset_sched[s] = makeView(V, vsets[s].lvl, T.vs_top[s], true, vsets[s].chain, true);
  T.opp_sched.assign(T.nChains, -1);
  for (int32_t c = 0; c < T.nChains; c++) T.opp_sched[c] = makeView(P, pLvl[c], T.chain_top[c], false, c, false);
  T.nScheds = (int32_t)T.s_off.size();

  // ------------------------------------------------------------------ node -> leaves per chain
  T.ncl_off.assign((size_t)T.nNodes * T.nChains, 0); T.ncl_cnt.assign((size_t)T.nNodes * T.nChains, 0);
  {
    std::vector<std::vector<int32_t>> tmp((size_t)T.nNodes * T.nChains);
    for (int32_t c = 0; c < T.nChains; c++)
      for (int32_t b : pLvl[c][1]) tmp[(size_t)P[b].nodes[0] * T.nChains + c].push_back(P[b].finalId);
    for (size_t k = 0; k < tmp.size(); k++) {
      std::set<int32_t> seenIdx;
      for (int32_t leaf : tmp[k]) if (!seenIdx.insert(T.p_leafidx[leaf]).second) T.uniqueLeafIdx = false;
      T.ncl_off[k] = (int32_t)T.ncl_list.size(); T.ncl_cnt[k] = (int32_t)tmp[k].size();
      T.ncl_list.insert(T.ncl_list.end(), tmp[k].begin(), tmp[k].end());
    }
  }
  // ------------------------------------------------------------------ init orders
  for (int32_t vc = 0; vc < T.nVCs; vc++)
    for (int32_t pi = 0; pi < T.nPinned; pi++)
      if (T.vc_pinned_vset[(size_t)vc * T.nPinned + pi] >= 0) T.pinned_init_order.push_back(pi);
  {
    std::vector<char> seen(T.nNodes, 0);
    for (int32_t c = 0; c < T.nChains; c++)
      for (int32_t b : pTops[c])
        for (int32_t n : P[b].nodes)
          if (!seen[n]) { seen[n] = 1; T.bad_init_order.push_back(n); }
  }
  return T;
}

}  // namespace hived
