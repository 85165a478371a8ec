"""Scheduler state that decides later calls but that no result or cell snapshot shows, read through the test hooks of
include/hived_bench.h (hived_debug_state) and the group inspection calls of include/hived.h, so that two
implementations can be compared after every call and a difference is named where it arises rather than many
operations later.

    state(lib, ctx)            -> {item key: value} decoded from hived_debug_state
    group_tables(lib, ctx)     -> {group id: (state, members, leaves, pods, preempting, has_virtual, lazy_preempted)}
    diff(a, b)                 -> None, or the first differing item in words
"""
import ctypes as C

from hivedscheduler_b200 import _cabi

# section tags (include/hived_bench.h HIVED_DS_*)
FREE, BAD_FREE, DOOMED_BAD, VC_FREE, ALL_VC_FREE, TOTAL_LEFT, ALL_VC_DOOMED = 1, 2, 3, 4, 5, 6, 7
USED_PHYSICAL, USED_VIRTUAL, USING_GROUP, RESERVING_GROUP, BAD_NODE = 8, 9, 10, 11, 12

# the reference's names of the sections, for diff()
_NAMES = {FREE: "freeCellList", BAD_FREE: "badFreeCells", DOOMED_BAD: "vcDoomedBadCells", VC_FREE: "vcFreeCellNum",
          ALL_VC_FREE: "allVCFreeCellNum", TOTAL_LEFT: "totalLeftCellNum", ALL_VC_DOOMED: "allVCDoomedBadCellNum",
          USED_PHYSICAL: "physical usedLeafCellNumAtPriorities", USED_VIRTUAL: "virtual usedLeafCellNumAtPriorities",
          USING_GROUP: "usingGroup", RESERVING_GROUP: "reservingOrReservedGroup", BAD_NODE: "badNodes",
          "group": "affinity group"}
# words of a section's key (after the tag), and whether a list or a counted tuple follows
_KEY_WORDS = {FREE: 2, BAD_FREE: 2, DOOMED_BAD: 3, VC_FREE: 3, ALL_VC_FREE: 2, TOTAL_LEFT: 2, ALL_VC_DOOMED: 2,
              USED_PHYSICAL: 1, USED_VIRTUAL: 1, USING_GROUP: 1, RESERVING_GROUP: 1, BAD_NODE: 1}
_KEY_FIELDS = {FREE: ("chain", "level"), BAD_FREE: ("chain", "level"), DOOMED_BAD: ("vc", "chain", "level"),
               VC_FREE: ("vc", "chain", "level"), ALL_VC_FREE: ("chain", "level"), TOTAL_LEFT: ("chain", "level"),
               ALL_VC_DOOMED: ("chain", "level"), USED_PHYSICAL: ("cell",), USED_VIRTUAL: ("cell",),
               USING_GROUP: ("cell",), RESERVING_GROUP: ("cell",), BAD_NODE: ("node",), "group": ("id",)}


def _bind(lib):
    if getattr(lib, "_hidden_state_bound", False):
        return
    lib.hived_debug_state.restype = C.c_int64
    lib.hived_debug_state.argtypes = [C.c_void_p, C.POINTER(C.c_int32), C.c_int64]
    lib._hidden_state_bound = True


def raw(lib, ctx):
    """The words of hived_debug_state."""
    _bind(lib)
    n = lib.hived_debug_state(ctx, None, 0)
    buf = (C.c_int32 * max(n, 1))()
    assert lib.hived_debug_state(ctx, buf, n) == n
    return list(buf[:n])


def decode(words):
    """{(tag, *key): value}: a tuple of cells for the lists, ((priority, count), ...) for the used maps, (group, live)
    for the cell groups, the count for the counters, True for a bad node.  Raises ValueError on a malformed encoding
    (an unknown tag, a section out of order or twice, a truncated list)."""
    out, i, n, last = {}, 0, len(words), None
    while i < n:
        tag = words[i]
        if tag not in _KEY_WORDS:
            raise ValueError("unknown section tag %d at word %d" % (tag, i))
        kw = _KEY_WORDS[tag]
        key = (tag,) + tuple(words[i + 1:i + 1 + kw])
        i += 1 + kw
        if tag in (FREE, BAD_FREE, DOOMED_BAD):
            cnt = words[i]
            val = tuple(words[i + 1:i + 1 + cnt])
            i += 1 + cnt
        elif tag in (USED_PHYSICAL, USED_VIRTUAL):
            cnt = words[i]
            flat = words[i + 1:i + 1 + 2 * cnt]
            val = tuple(zip(flat[0::2], flat[1::2]))
            i += 1 + 2 * cnt
        elif tag in (USING_GROUP, RESERVING_GROUP):
            val = tuple(words[i:i + 2])
            i += 2
        elif tag == BAD_NODE:
            val = True
        else:
            val = words[i]
            i += 1
        if i > n:
            raise ValueError("section %r runs past the end of the encoding" % (key,))
        if last is not None and key <= last:
            raise ValueError("section %r out of order or repeated after %r" % (key, last))
        last = key
        out[key] = val
    return out


def state(lib, ctx):
    return decode(raw(lib, ctx))


def group_tables(lib, ctx):
    """Every group hived_list_groups names, with its placement as hived_get_group_placement reports it."""
    n = lib.hived_list_groups(ctx, None, 0)
    ids = (C.c_int32 * max(n, 1))()
    assert lib.hived_list_groups(ctx, ids, n) == n
    out = {}
    for g in ids[:n]:
        gp = _cabi.GroupPlacement()
        assert lib.hived_get_group_placement(ctx, g, C.byref(gp), None, None, 0, None, 0, None, 0) == 0
        nl, npods, npre = gp.n_leaves, gp.n_pods, gp.n_preempting
        phys, virt = (C.c_int32 * max(nl, 1))(), (C.c_int32 * max(nl, 1))()
        pods, pre = (C.c_int32 * max(npods, 1))(), (C.c_int32 * max(npre, 1))()
        assert lib.hived_get_group_placement(ctx, g, C.byref(gp), phys, virt, nl, pods, npods, pre, npre) == 0
        m = gp.n_members
        out[("group", g)] = (gp.state, tuple(zip(gp.member_leaf_num[:m], gp.member_pod_num[:m])),
                             tuple(zip(phys[:nl], virt[:nl])), tuple(pods[:npods]), tuple(pre[:npre]),
                             gp.has_virtual, gp.lazy_preempted)
    return out


def full(lib, ctx, group_names=None, pod_names=None):
    """state() and group_tables() in one dict.  Two callers that intern names on their own (the HivedAlgorithm shim
    recycles ids as it sees fit) compare by name: group_names / pod_names map an id to the name it stands for."""
    s = state(lib, ctx)
    s.update(group_tables(lib, ctx))
    if group_names is None and pod_names is None:
        return s
    gn = (lambda g: group_names[g] if 0 <= g < len(group_names) else g) if group_names is not None else (lambda g: g)
    pn = (lambda p: pod_names[p] if 0 <= p < len(pod_names) else p) if pod_names is not None else (lambda p: p)
    out = {}
    for k, v in s.items():
        if k[0] in (USING_GROUP, RESERVING_GROUP):
            v = (gn(v[0]), v[1])
        elif k[0] == "group":
            k = ("group", gn(k[1]))
            v = v[:3] + (tuple(pn(p) for p in v[3]), tuple(pn(p) for p in v[4])) + v[5:]
        out[k] = v
    return out


def _where(key):
    tag = key[0]
    fields = _KEY_FIELDS[tag]
    if tag in (FREE, BAD_FREE, DOOMED_BAD, VC_FREE, ALL_VC_FREE, TOTAL_LEFT, ALL_VC_DOOMED):
        return _NAMES[tag] + "".join("[%s %d]" % f for f in zip(fields, key[1:]))
    return "%s of %s" % (_NAMES[tag], " ".join("%s %s" % f for f in zip(fields, key[1:])))


def _show(key, v):
    if v is None:
        return "absent"
    if key[0] in (USED_PHYSICAL, USED_VIRTUAL):
        return "{%s}" % ", ".join("%d: %d" % pc for pc in v)
    if key[0] in (USING_GROUP, RESERVING_GROUP):
        return "group %s%s" % (v[0], "" if v[1] else " (not the group its name maps to)")
    if key[0] == "group":
        return "(state %d, members %r, (phys, virt) leaves %r, pods %r, preempting %r, has_virtual %d, lazy_preempted %d)" % v
    return repr(v)


def diff(a, b, names=("a", "b")):
    """None if the two decoded states are equal, else the first differing item in words (keys in encoding order)."""
    if a == b:
        return None

    def order(k):
        return (1, str(k[1])) if k[0] == "group" else (0, k)

    for key in sorted(set(a) | set(b), key=order):
        va, vb = a.get(key), b.get(key)
        if va == vb:
            continue
        where = _where(key)
        if key[0] in (FREE, BAD_FREE, DOOMED_BAD) and va is not None and vb is not None:
            if len(va) != len(vb):
                return "%s length: %d != %d (%s %r, %s %r)" % (where, len(va), len(vb), names[0], va, names[1], vb)
            i = next(i for i in range(len(va)) if va[i] != vb[i])
            return "%s position %d: %d != %d" % (where, i, va[i], vb[i])
        return "%s: %s != %s" % (where, _show(key, va), _show(key, vb))
    return None
