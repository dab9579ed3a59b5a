"""Strategy layer: lenient XML, trees, relay-control truth tables (golden rows from the reference's
logs), schedule slicing with tails, native (C++) vs Python cross-check."""
import glob
import os

import pytest

from adapcc_b200.constants import (ALLREDUCE, BOARDCAST, REDUCE, RELAY_BYPASS, RELAY_FORWARD, TR_HAS_LOCAL,
                                   TR_IN_BCAST, TR_IN_REDUCE, TR_PUBLISH, TR_WANT_RESULT)
from adapcc_b200.strategy import (Strategy, make_strategy, participants, relay_control, slice_bounds, tree_role,
                                  work_items, xmlio)
from adapcc_b200.strategy.schedule import default_chunk_bytes


def test_lenient_xml_accepts_missing_attribute_space(strategy4_xml):
    import xml.etree.ElementTree as ET

    with pytest.raises(ET.ParseError):
        ET.fromstring(strategy4_xml)                      # stock parser rejects the reference dialect
    doc = xmlio.parse(strategy4_xml)
    assert doc.tag == "trees" and len(doc.find_all("root")) == 4
    first = doc.find_all("root")[0].children[0]
    assert first.attrs == {"id": "1", "ip": "10.0.0.1"}


def test_xml_roundtrip_and_comments():
    txt = '<?xml version="1.0"?><!-- c --><graph version="1"><server id="0" ip="a"><nic id="0"><gpu id="3"/></nic></server></graph>'
    doc = xmlio.parse(txt)
    again = xmlio.parse(xmlio.dumps(doc))
    assert [n.tag for n in again.iter()] == ["graph", "server", "nic", "gpu"]
    assert again.find("server").find("nic").find("gpu").attrs["id"] == "3"
    with pytest.raises(xmlio.XmlError):
        xmlio.parse("<a><b></a")


def test_all_reference_strategy_files_parse(reference_strategy_dir):
    files = sorted(glob.glob(os.path.join(reference_strategy_dir, "*.xml")))
    assert len(files) >= 16
    for f in files:
        s = Strategy.from_file(f, max_trees=64) if False else Strategy.from_xml(open(f).read(), max_trees=64)
        assert s.trees and all(t.root >= 0 for t in s.trees)
        for t in s.trees:
            assert len(set(t.nodes)) == len(t.nodes)


def test_strategy_roles_and_world_pruning(strategy4_xml):
    s = Strategy.from_xml(strategy4_xml)
    assert [t.root for t in s.trees] == [0, 2, 3, 1]
    assert s.trees[0].kids(0) == [1, 2] and s.trees[0].kids(2) == [3]
    # BASELINE config 1: the 4-GPU file at world_size=2 -> ranks 2,3 are contracted out
    s2 = Strategy.from_xml(strategy4_xml, world=2)
    assert all(set(t.nodes) == {0, 1} for t in s2.trees)
    assert [t.root for t in s2.trees] == [0, 1, 0, 1]
    s2.validate(world=2)
    back = Strategy.from_xml(s2.to_xml())
    assert [t.parent for t in back.trees] == [t.parent for t in s2.trees]


GOLDEN = {   # rank -> (recv, local, kernel, send)
    "all": {0: (1, 1, 1, 0), 1: (1, 1, 1, 1), 2: (0, 1, 0, 1), 3: (0, 1, 0, 1)},      # log/primitive:139-146
    "0,2": {0: (1, 1, 1, 0), 1: (1, 0, 0, 1), 2: (0, 1, 0, 1), 3: (0, 0, 0, 0)},      # log/training:150-159
}


def test_relay_control_matches_reference_logs(strategy_test_xml):
    t = Strategy.from_xml(strategy_test_xml).trees[0]
    for r, want in GOLDEN["all"].items():
        assert relay_control(t, r, [0, 1, 2, 3]).as_tuple() == want
    for r, want in GOLDEN["0,2"].items():
        assert relay_control(t, r, [0, 2]).as_tuple() == want
    assert relay_control(t, 1, [0, 2]).active_recvs == [2]


def test_native_relay_control_and_roles_match_python(strategy_test_xml, strategy4_xml):
    from adapcc_b200.runtime.native import native_relay_control, native_tree_role

    for xml, world in [(strategy_test_xml, 4), (strategy4_xml, 4), (strategy4_xml, 2), (strategy4_xml, 3)]:
        s = Strategy.from_xml(xml, world)
        subsets = [list(range(world)), [0], [world - 1], [0, world - 1]]
        for ti, t in enumerate(s.trees):
            for act in subsets:
                for r in range(world):
                    n = native_relay_control(xml, world, ti, r, act)
                    p = relay_control(t, r, act)
                    assert (n["has_recv"], n["has_local"], n["has_kernel"], n["has_send"]) == tuple(map(bool, p.as_tuple()))
                    assert n["active_recvs"] == p.active_recvs
                    for prim in (ALLREDUCE, REDUCE, BOARDCAST):
                        for mode in (RELAY_FORWARD, RELAY_BYPASS):
                            nr = native_tree_role(xml, world, ti, r, act, prim, mode)
                            pr = tree_role(t, r, act, prim, mode)
                            assert (nr["parent"], nr["flags"], nr["children"]) == (pr.parent, pr.flags, pr.children), \
                                (world, ti, act, r, prim, mode)


def test_tree_roles_forward_vs_bypass(strategy_test_xml):
    t = Strategy.from_xml(strategy_test_xml).trees[0]          # 0 <- 1 <- {2, 3}
    fwd = tree_role(t, 1, [0, 2], ALLREDUCE, RELAY_FORWARD)    # inactive rank 1 forwards 2's data
    assert fwd.has(TR_IN_REDUCE) and not fwd.has(TR_HAS_LOCAL) and fwd.children == [2] and fwd.parent == 0
    assert fwd.has(TR_PUBLISH) and fwd.has(TR_IN_BCAST) and not fwd.has(TR_WANT_RESULT)
    byp = tree_role(t, 1, [0, 2], ALLREDUCE, RELAY_BYPASS)     # NVSwitch: nobody routes through 1
    assert not byp.any()
    assert tree_role(t, 2, [0, 2], ALLREDUCE, RELAY_BYPASS).parent == 0
    assert tree_role(t, 0, [0, 2], ALLREDUCE, RELAY_BYPASS).children == [2]
    s = Strategy.from_xml(strategy_test_xml)
    assert participants(s, 4, [0, 2], ALLREDUCE, RELAY_FORWARD) == [0, 1, 2, 3]   # 3 is tree 1's (inactive) root
    s.trees = s.trees[:1]
    assert participants(s, 4, [0, 2], ALLREDUCE, RELAY_FORWARD) == [0, 1, 2]
    assert participants(s, 4, [0, 2], ALLREDUCE, RELAY_BYPASS) == [0, 2]
    # inactive root: first active node is promoted
    assert tree_role(t, 1, [1, 3], REDUCE, RELAY_BYPASS).parent == -1


def test_work_items_cover_every_element_once():
    for count, trees, chunk, isz in [(16, 1, 8, 4), (4097000, 4, 4 << 20, 4), (138357544, 3, 4 << 20, 4),
                                     (1001, 4, 64, 2), (7, 8, 16, 4), (0, 2, 16, 4)]:
        items = work_items(count, trees, chunk, isz)
        covered = sorted((it.start, it.start + it.length) for it in items)
        pos = 0
        for a, b in covered:
            assert a == pos and b > a
            pos = b
        assert pos == count                     # reference drops tails (log/training: 4 097 000 -> 3 chunks)
        b = slice_bounds(count, trees, isz)
        assert b[0] == 0 and b[-1] == count and all(x <= y for x, y in zip(b, b[1:]))


def test_default_chunk_rule():
    assert default_chunk_bytes(553430176) == 4 * 1024 * 1024          # log/training:135
    assert default_chunk_bytes(64) == 16
    assert default_chunk_bytes(4 * 1000 * 1000) == 1000000 // 16 * 16


def test_generated_strategies_are_spanning():
    for world in (2, 3, 4, 8):
        for shape in ("binary", "chain", "star"):
            s = make_strategy(world, 4, shape)
            s.validate(world)
            assert len({t.root for t in s.trees}) == len(s.trees)


def test_python_and_native_parsers_agree_under_fuzzing():
    """Differential fuzz of the two lenient strategy readers (strategy/xmlio.py and csrc/schedule.cpp): well-formed
    dialect variants, truncations, deletions, duplicated chunks and garbage. Whenever both accept, the relay-control
    rows must be identical; the native reader must never accept something whose result differs, and never crash."""
    import random

    from adapcc_b200.runtime.native import NativeError, native_relay_control
    from adapcc_b200.strategy import Strategy, make_strategy
    from adapcc_b200.strategy.relay import relay_control

    rng = random.Random(11)

    def mangle(xml):
        c = rng.random()
        if c < 0.25:
            return xml.replace('" ip=', '"ip=').replace('" id=', '"id=')        # the reference's missing-space dialect
        if c < 0.4:
            return xml.replace(">", ">\n\t ").replace(" id=", "   id=")
        if c < 0.55:
            return xml[: rng.randrange(1, len(xml))]
        if c < 0.7:
            x = list(xml)
            for _ in range(rng.randint(1, 5)):
                del x[rng.randrange(len(x))]
            return "".join(x)
        if c < 0.8:
            i = rng.randrange(len(xml))
            j = min(len(xml), i + rng.randint(1, 40))
            return xml[:j] + xml[i:j] + xml[j:]
        if c < 0.9:
            i = rng.randrange(len(xml))
            return xml[:i] + "".join(rng.choice("<>/\"'= \n&;!-") for _ in range(rng.randint(1, 8))) + xml[i:]
        return xml

    agree = 0
    for _ in range(400):
        world = rng.choice([2, 3, 4, 8, 16])
        deg = rng.choice([1, 2, 4])
        xml = mangle(make_strategy(world, deg, rng.choice(["chain", "binary", "star"])).to_xml(compact=rng.random() < 0.5))
        active = sorted(rng.sample(range(world), rng.randint(1, world)))
        rank, tree = rng.randrange(world), rng.randrange(deg)
        py = nat = None
        try:
            st = Strategy.from_xml(xml, world)
            st.validate(world)
            if tree < len(st.trees):
                rc = relay_control(st.trees[tree], rank, active)
                py = (bool(rc.has_recv), bool(rc.has_local), bool(rc.has_kernel), bool(rc.has_send),
                      sorted(rc.active_recvs), len(st.trees))
        except Exception:                                                     # noqa: BLE001  any rejection counts
            py = None
        try:
            r = native_relay_control(xml, world, tree, rank, active)
            nat = (r["has_recv"], r["has_local"], r["has_kernel"], r["has_send"], sorted(r["active_recvs"]), r["n_trees"])
        except NativeError:
            nat = None
        if py is not None:
            assert nat == py, (py, nat, xml[:300])
            agree += 1
    assert agree > 150


def test_native_reader_accepts_every_shipped_and_reference_strategy_file(reference_strategy_dir):
    """csrc/schedule.cpp against all strategy XML files of this repo and of the reference, including the
    reference's malformed-attribute dialect: same number of trees as the Python reader."""
    import glob

    from adapcc_b200.runtime.native import native_relay_control

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    files = sorted(glob.glob(os.path.join(root, "strategy", "*.xml")))
    files += sorted(glob.glob(os.path.join(reference_strategy_dir, "*.xml")))
    assert len(files) >= 36
    for f in files:
        xml = open(f).read()
        s = Strategy.from_xml(xml)
        world = len(s.ranks())
        r = native_relay_control(xml, world, 0, s.trees[0].root, list(range(world)))
        assert r["n_trees"] == len(s.trees), f
