#!/usr/bin/env python
"""Generates tests/golden/hived_algorithm_test.json from the reference's own test file and fixture.

Needs a checkout of microsoft/hivedscheduler; the tests only read the committed JSON:

    python tests/golden/make_fixture.py <hivedscheduler checkout>

Extracted verbatim (data only, no code) from
  pkg/algorithm/hived_algorithm_test.go
    group1..group34 (:66-170), pss (:172-542), casesThatShouldSucceed/Fail/BeLazyPreempted,
    casesForStatefulPreemption (:544-560), expectedBindInfos (:566-592), expectedPreemptInfos (:594-602),
    deletedPreemptorGroups (:604-608)
  example/config/design/hivedscheduler.yaml (the cluster the vectors are defined on)
The scenario (call order, config edits, assertions) is restated in tests/golden_scenario.py.
"""
import json
import os
import re
import sys

import yaml

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hived_algorithm_test.json")


def main(ref):
    src = open(os.path.join(ref, "pkg/algorithm/hived_algorithm_test.go")).read()
    # ---- affinity group specs
    groups = {}
    for m in re.finditer(r'Name:\s+"(group\d+)",\s*Members:\s*\[\]api\.AffinityGroupMemberSpec\{(.*?)\},\n', src):
        members = [{"podNumber": int(a), "leafCellNumber": int(b)}
                   for a, b in re.findall(r"\{PodNumber: (\d+), LeafCellNumber: (\d+)\}", m.group(2))]
        groups[m.group(1)] = {"name": m.group(1), "members": members}
    assert len(groups) == 34, len(groups)
    # ---- pod scheduling specs
    pss_src = src[src.index("var pss = map[types.UID]api.PodSchedulingSpec{"):src.index("var casesThatShouldSucceed")]
    pss = {}
    for m in re.finditer(r'"(pod\d+)": \{(.*?)\n\t\}', pss_src, re.S):
        body = m.group(2)

        def field(name, default=None, conv=str):
            mm = re.search(r"\b%s:\s+([^,\n]+)," % name, body)
            if not mm:
                return default
            v = mm.group(1).strip()
            if conv is str:
                return v.strip('"')
            if conv is bool:
                return v == "true"
            return conv(v)

        pss[m.group(1)] = {
            "virtualCluster": field("VirtualCluster", ""),
            "priority": field("Priority", 0, int),
            "pinnedCellId": field("PinnedCellId", ""),
            "leafCellType": field("LeafCellType", ""),
            "leafCellNumber": field("LeafCellNumber", 0, int),
            "gangReleaseEnable": field("GangReleaseEnable", False, bool),
            "lazyPreemptionEnable": field("LazyPreemptionEnable", False, bool),
            # Go zero value: the test marshals the struct, so an unset field is an explicit `false`
            "ignoreK8sSuggestedNodes": field("IgnoreK8sSuggestedNodes", False, bool),
            "affinityGroup": groups[field("AffinityGroup")],
        }
    assert len(pss) == 46, len(pss)

    def str_list(name):
        mm = re.search(r"var %s = \[\]string\{(.*?)\n\}" % name, src, re.S)
        return re.findall(r'"([^"]+)"', mm.group(1))

    fail_src = re.search(r"var casesThatShouldFail = \[\]\[\]string\{(.*?)\n\}", src, re.S).group(1)
    cases_fail = [re.findall(r'"([^"]+)"', g) for g in re.findall(r"\{([^{}]*)\}", fail_src)]
    bind_src = re.search(r"var expectedBindInfos = map\[string\]result\{(.*?)\n\}", src, re.S).group(1)
    expected_bind = {}
    for mm in re.finditer(r'"(pod\d+)":\s+\{node: "([^"]+)", leafCellIsolation: \[\]int32\{([^}]*)\}\}', bind_src):
        expected_bind[mm.group(1)] = {"node": mm.group(2),
                                      "leafCellIsolation": [int(x) for x in mm.group(3).split(",") if x.strip()]}
    assert len(expected_bind) == 25, len(expected_bind)
    pre_src = re.search(r"var expectedPreemptInfos = map\[string\]common\.Set\{(.*?)\n\}", src, re.S).group(1)
    expected_preempt = {mm.group(1): re.findall(r'"([^"]+)"', mm.group(2))
                        for mm in re.finditer(r'"(pod\d+)": common\.NewSet\(([^)]*)\)', pre_src)}
    assert len(expected_preempt) == 7
    del_src = re.search(r"var deletedPreemptorGroups = map\[string\]\[\]string\{(.*?)\n\}", src, re.S).group(1)
    deleted = {mm.group(1): re.findall(r'"([^"]+)"', mm.group(2))
               for mm in re.finditer(r'"(pod\d+)": \{([^}]*)\}', del_src)}
    design = yaml.safe_load(open(os.path.join(ref, "example/config/design/hivedscheduler.yaml")))
    out = {
        "source": "microsoft/hivedscheduler pkg/algorithm/hived_algorithm_test.go + example/config/design/hivedscheduler.yaml",
        "design_config": {"physicalCluster": design["physicalCluster"], "virtualClusters": design["virtualClusters"]},
        "pss": pss,
        "casesThatShouldSucceed": str_list("casesThatShouldSucceed"),
        "casesThatShouldFail": cases_fail,
        "casesThatShouldBeLazyPreempted": str_list("casesThatShouldBeLazyPreempted"),
        "casesForStatefulPreemption": str_list("casesForStatefulPreemption"),
        "expectedBindInfos": expected_bind,
        "expectedPreemptInfos": expected_preempt,
        "deletedPreemptorGroups": deleted,
    }
    with open(OUT, "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print("wrote", OUT, "pods:", len(pss), "bind vectors:", len(expected_bind))


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: make_fixture.py <hivedscheduler checkout>")
    sys.exit(main(sys.argv[1]))
