"""CPU: the oracle and the host mirror against the answers of the reference's OWN compiled code (StaticGStore, SPARQLEngine,
Planner and config loader behind C shims, see oracle/Makefile).  Those answers are committed: tests/golden/ref_checks.json
(made by tests/golden/make_ref_checks.py) and tests/golden/ref_engine_lubm{1,2}.json (make_ref_engine.py), so every check
here runs without the reference tree."""
import hashlib
import json
import os

import numpy as np
import pytest

import random_bgp as R
import sparql_mini as M
from conftest import PLANS, load_query
from oracle import oracle as O
from oracle import ref as REF
from wukong_b200 import host

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def gold():
    return json.load(open(os.path.join(HERE, "golden", "ref_checks.json")))


def table_digest(t):
    t = M.sort_rows(np.asarray(t, dtype=np.uint32))
    return hashlib.sha256(t.tobytes()).hexdigest()


def split_key(k):
    """-> (vid, pid, dir) of a raw ikey_t"""
    return k >> 18, (k >> 1) & 0x1FFFF, k & 1


def occupied_keys(v):
    """keys of the occupied slots of a header array (slot 7 of every bucket is the chain pointer)"""
    idx = np.arange(v.shape[0])
    return v[(idx % 8 != 7) & (v[:, 0] != 0), 0]


def keys_digest(keys):
    return hashlib.sha256(np.sort(np.asarray(keys, dtype=np.uint64)).tobytes()).hexdigest()


def edge_lists_digest(keys, edges_of):
    """sha256 over every key's edge list in key order; index lists (vid 0) follow hash-map iteration in the reference, a set
    is the contract, so they are sorted first"""
    h = hashlib.sha256()
    for k in sorted(int(x) for x in keys):
        e = np.asarray(edges_of(k), dtype=np.uint32)
        if k >> 18 == 0:
            e = np.sort(e)
        h.update(np.array([k, e.size], dtype=np.uint64).tobytes())
        h.update(e.tobytes())
    return h.hexdigest()


def check_store(o, want):
    """an oracle store against the reference's build of the same triples: segment table, key set and every key's edge list"""
    ov, oe = o.vertices(), o.edges()
    assert ov.shape[0] == want["num_slots"]
    assert sorted([x.index, x.dir, x.pid, x.num_keys, x.num_buckets, x.bucket_start, x.num_edges, x.edge_start]
                  for x in o.segs()) == want["segs"]
    keys = occupied_keys(ov)
    assert keys_digest(keys) == want["keys_sha256"]
    assert oe.shape[0] == want["num_edges"]
    idx = np.arange(ov.shape[0])
    ptr = dict(zip(ov[:, 0][(idx % 8 != 7) & (ov[:, 0] != 0)].tolist(), ov[:, 1][(idx % 8 != 7) & (ov[:, 0] != 0)].tolist()))

    def edges_of(k):
        p = ptr[k]
        size, off = p & ((1 << 28) - 1), (p >> 28) & ((1 << 34) - 1)
        return oe[off:off + size]
    assert edge_lists_digest(keys, edges_of) == want["edges_sha256"]
    return keys


def test_store_matches_reference_store(lubm1, gold):
    """segment table, key set and every key's edge list: the reference's StaticGStore::init + GStore::get_edges"""
    o = O.Store.build(lubm1, kvstore_bytes=1 << 30, num_engines=1, gpu_ext_mode=False)
    keys = check_store(o, gold["store_lubm1"])
    assert int(((keys >> np.uint64(18)) == 0).sum()) > 30           # index lists
    # the product host builder is bit-identical to the oracle (test_host_builder.py), hence pinned through it
    hs = host.HostStore(lubm1, kvstore_bytes=1 << 30, gpu_ext_extents=False)
    assert np.array_equal(hs.vertices(), o.vertices()) and np.array_equal(hs.edges(), o.edges())


def special_queries():
    """plans beyond the workload files, by name"""
    univ0 = M.lubm_str2id("<http://www.University0.edu>")
    P = {n: i for i, n in enumerate(M.LUBM_INDEX)}
    return {
        # const_to_known in the middle of a plan (sparql.hpp:144-186): departments of graduate students that belong to University0
        "const_to_known": ([(P[M.UB + "GraduateStudent>"], 1, 0, -1), (-1, P[M.UB + "memberOf>"], 1, -2),
                            (univ0, P[M.UB + "subOrganizationOf>"], 0, -2), (-2, P[M.UB + "name>"], 1, -3)], 3, [-1, -3]),
        # known_to_unknown through the type index (pid == TYPE_ID && d == IN, sparql.hpp:339-340): professors -> their types ->
        # every instance of those types
        "type_index": ([(P[M.UB + "FullProfessor>"], 1, 0, -1), (-1, 1, 1, -2), (-2, 1, 0, -3)], 3, [-1, -2, -3]),
    }


STATUS_QUERIES = [([(-1, 5, 1, -2)], 2, [-1]), ([(18, 1, 0, -1), (M.lubm_str2id("<http://www.University0.edu>"), 7, 0, -2)], 2, [-1]),
                  ([(18, 5, 0, -1)], 1, [-1]), ([(18, 1, 0, -1)], 1, [])]


def test_engine_matches_reference_engine(ostore1, gold):
    """Q1-Q7 x 3 plan sets x mt 1/3, blind, DISTINCT / OFFSET / LIMIT, error codes: SPARQLEngine vs the oracle"""
    G = gold["engine_lubm1"]
    for q in range(1, 8):
        for plan in PLANS:
            pats, nvars, req, _ = load_query(q, plan)
            g = G["q%d_%s" % (q, plan)]
            for mt in (1, 3):
                want = g["mt%d" % mt]
                got = O.run_query([ostore1], pats, nvars, req, mt_factor=mt)
                assert want["rc"] == got.status == 0 and got.rows == want["rows"], (q, plan, mt)
                if got.rows:
                    assert got.cols == want["cols"] and table_digest(got.table) == want["sha256"], (q, plan, mt)
            assert g["blind_rows"] == got.rows
            wd = O.run_query([ostore1], pats, nvars, req, distinct=True, offset=1, limit=40)
            assert wd.rows == g["distinct"]["rows"], (q, plan)
            assert wd.rows == 0 or hashlib.sha256(np.ascontiguousarray(wd.table).tobytes()).hexdigest() == g["distinct"]["sha256"]
    for name, (pats, nvars, req) in special_queries().items():
        want = O.run_query([ostore1], pats, nvars, req)
        assert G[name]["rc"] == 0 and G[name]["rows"] == want.rows > 0, name
        assert table_digest(want.table) == G[name]["sha256"], name
    assert G["type_index"]["rows"] > 1000
    assert G["status"] == [O.run_query([ostore1], p, nv, rq).status for p, nv, rq in STATUS_QUERIES]


@pytest.mark.parametrize("gseed", [3, 11, 12])
def test_random_graph_matches_reference_engine(gold, gseed):
    """random graphs (hubs, self loops, duplicates, multi-typed vertices) and 60 random plans each, chains of every primitive,
    through the reference engine"""
    tr, meta = R.graph(gseed, nv=300, ntriples=2500)
    npreds = meta["num_normal_preds"]
    ost = O.Store.build(tr, kvstore_bytes=8 << 20, num_engines=2, num_normal_preds=npreds)
    checked = 0
    for qseed in range(60):
        planned, _, nvars, req = R.query(7000 + 100 * gseed + qseed, tr, meta)
        name = "g%d_q%d" % (gseed, qseed)
        if O.run_query([ost], planned, nvars, req, blind=True).rows > 200_000:
            assert name not in gold["random_graphs"]
            continue
        g = gold["random_graphs"][name]
        want = O.run_query([ost], planned, nvars, req)
        assert g["rc"] == want.status == 0 and g["rows"] == want.rows, (qseed, planned)
        if want.rows:
            assert table_digest(want.table) == g["sha256"], (qseed, planned)
        wd = O.run_query([ost], planned, nvars, req, distinct=True)
        d = g["distinct"]
        assert d["rc"] == 0 and d["rows"] == wd.rows, (qseed, planned)
        assert wd.rows == 0 or hashlib.sha256(np.ascontiguousarray(wd.table).tobytes()).hexdigest() == d["sha256"], (qseed, planned)
        checked += 1
    assert checked >= 45


@pytest.mark.parametrize("which", [1, 2])
def test_oracle_matches_reference_engine_fixture(ostore1, ostore2, which):
    """the reference engine's answers on LUBM-1 (seed 1) and LUBM-2 (seed 7), committed as row counts + digests of the sorted
    tables"""
    G = json.load(open(os.path.join(HERE, "golden", "ref_engine_lubm%d.json" % which)))
    ostore1 = ostore1 if which == 1 else ostore2
    assert G["queries"]
    for name, e in G["queries"].items():
        q, plan = int(name.split("_")[0][1:]), name.split("_", 1)[1]
        pats, nvars, req, _ = load_query(q, plan)
        got = O.run_query([ostore1], pats, nvars, req)
        assert got.status == 0 and got.rows == e["rows"], name
        if got.rows:
            assert table_digest(got.table) == e["sha256"], name
        d = O.run_query([ostore1], pats, nvars, req, distinct=True, offset=1, limit=40)
        assert d.rows == e["distinct_rows"] and (d.rows == 0 or hashlib.sha256(d.table.tobytes()).hexdigest() == e["distinct_sha256"]), name


# comments, blank lines, braces, reordering, every direction token, more plan lines than patterns
ODD_FMT = "# plan\n{\n 3 <\n\n1 >>\n  2 <<\n4 >\n5 <\n6 >\n1 >\n}\n9 >\n"
BAD_FMTS = ("1 <\n", "", "# nothing\n")          # fewer plan lines than patterns


def test_set_plan_matches_reference_planner(gold):
    """Planner::set_plan + set_direction (core/planner.hpp:1647-1754) vs the oracle's restatement and the independent Python
    reader (the C++ host mirror is held to the same reader in test_host_surface.py)"""
    from conftest import WORKLOADS
    G = gold["set_plan"]
    norm = lambda plan: None if plan is None else [tuple(p) for p in plan]   # noqa: E731
    for q in range(1, 8):
        for plan in PLANS:
            planned, _, _, raw = load_query(q, plan)
            fmt = open(os.path.join(WORKLOADS, plan, "lubm_q%d.fmt" % q)).read()
            assert norm(G["q%d_%s" % (q, plan)]) == planned == O.set_plan(raw, fmt), (q, plan)
    raw = load_query(7, "osdi16_plan")[3]
    assert norm(G["q7_odd_fmt"]) == O.set_plan(raw, ODD_FMT) == M.apply_plan(raw, ODD_FMT)
    assert G["q7_bad_fmts"] == [None] * len(BAD_FMTS)
    for bad in BAD_FMTS:
        with pytest.raises(ValueError):
            O.set_plan(raw, bad)


TYPE_INDEX_PLAN = [(18, 1, 0, -1), (-1, 5, 0, -2), (-2, 1, 1, -3), (-3, 1, 0, -4)]
SPLITS = ((2, 0), (3, 2), (8, 1))


def split_table():
    return np.random.default_rng(5).integers(1 << 17, 1 << 31, (5000, 3), dtype=np.uint32)


def test_fork_join_decisions_and_split_match_reference(gold):
    """row a15: which steps exchange (SPARQLEngine::need_fork_join + the replicate rule of dispatch) and how rows are split
    (generate_sub_query), against the product's host-side exchange planner and the `row[col] % n` rule of its kernels"""
    from wukong_b200 import capi
    G = gold["fork_join"]
    for q in range(1, 8):
        for plan in PLANS:
            pats, nvars, _, _ = load_query(q, plan)
            rc, want = G["q%d_%s" % (q, plan)]
            assert rc == 0 and want == capi.plan_exchanges(pats, nvars), (q, plan, want)
    # a type-index lookup of a bound variable is replicated
    rc, want = G["type_index"]
    assert rc == 0 and want == capi.plan_exchanges(TYPE_INDEX_PLAN, 4) and -2 in want
    tbl = split_table()
    for n, col in SPLITS:
        parts = G["split"]["n%d_col%d" % (n, col)]
        assert len(parts) == n
        for i in range(n):
            # same rows, original order
            assert parts[i] == hashlib.sha256(np.ascontiguousarray(tbl[tbl[:, col] % n == i]).tobytes()).hexdigest(), (n, col, i)


def test_sharded_store_matches_reference_store(lubm1, gold):
    """server 1 of 2 (OUT edges with the subject's owner, IN edges with the object's, index lists of local vertices only):
    the reference's partition + StaticGStore::init against the oracle's per-server build"""
    o = O.Store.build(lubm1, num_servers=2, sid=1, kvstore_bytes=1 << 30, num_engines=1, gpu_ext_mode=False)
    check_store(o, gold["store_lubm1_server1_of_2"])


@pytest.mark.parametrize("n", [2, 3])
def test_simulated_reference_cluster(lubm1, gold, n):
    """n shard stores built by the reference (refs_build with the loader's owner rule) and one reference engine per shard; the
    plan is driven by execute_one_pattern / need_fork_join / generate_sub_query exactly as execute_patterns does, with an
    in-process work list instead of the transport.  Answers must equal the brute-force joiner's and the oracle's cluster's."""
    oshards = [O.Store.build(lubm1, num_servers=n, sid=i, kvstore_bytes=32 << 20, num_engines=2) for i in range(n)]
    for q in range(1, 8):
        for plan in PLANS:
            pats, nvars, req, raw = load_query(q, plan)
            bf = M.bruteforce_bgp(lubm1, raw, req)
            g = gold["cluster"]["n%d_q%d_%s" % (n, q, plan)]
            assert g["rc"] == 0 and g["rows"] == bf.shape[0], (n, q, plan)
            if g["rows"]:
                assert g["sha256"] == table_digest(bf), (n, q, plan)
            mine = O.run_query(oshards, pats, nvars, req)
            assert mine.status == 0 and mine.rows == g["rows"]


CONFIG_CASES = [
    "# general\nglobal_num_proxies              4\nglobal_num_engines              16\nglobal_data_port_base           5500\n"
    "global_ctrl_port_base           9576\nglobal_mt_threshold             8\nglobal_enable_workstealing      0\n"
    "global_stealing_pattern         0\nglobal_enable_planner           1\nglobal_generate_statistics      1\n"
    "global_enable_vattr             0\nglobal_silent                   1\n\n# kvstore\n"
    "global_input_folder             /path/to/input/rdfdata/id_lubm_40/\nglobal_memstore_size_gb         40\n"
    "global_est_load_factor          55\n\n# RDMA\nglobal_rdma_buf_size_mb         128\nglobal_rdma_rbf_size_mb         32\n"
    "global_use_rdma                 1\nglobal_rdma_threshold           300\nglobal_enable_caching           0\n\n# GPU\n"
    "global_num_gpus                 0\nglobal_gpu_rdma_buf_size_mb     64\nglobal_gpu_rbuf_size_mb         32\n"
    "global_gpu_kvcache_size_gb      10\nglobal_gpu_key_blk_size_mb      16\nglobal_gpu_value_blk_size_mb    4\n"
    "global_gpu_enable_pipeline      1\n"]
CONFIG_CASES += [CONFIG_CASES[0].replace("global_mt_threshold             8", "global_mt_threshold             64"),  # clamped to num_engines
                 "global_num_engines 4\n# c\n\nglobal_input_folder /a/b\nglobal_mt_threshold 2\nglobal_silent 0\nfoo_bar 3\nglobal_num_engines 6\n",
                 "global_input_folder x/\nglobal_est_load_factor 35\nglobal_gpu_rbuf_size_mb 4096\nglobal_enable_planner 0 trailing words\n"]
CONFIG_RELOADS = ["", "global_silent 0 global_mt_threshold 100 global_num_engines 99 global_use_rdma 1 global_enable_planner 0",
                  "global_rdma_threshold 7\nglobal_enable_caching 1\nglobal_memstore_size_gb 1"]


def test_config_loader_matches_reference(gold, tmp_path):
    """load_config(fname, nsrvs) + reload_config(str) of the host mirror (csrc/host/global.hpp) against the reference's own
    (core/config.hpp:42-230, non-GPU build, no RDMA device): every Global item, for the reference's sample config, for files
    that leave items at their defaults, repeat keys, carry unknown keys and comment lines, and for reloads that try to change
    immutable items"""
    for i, text in enumerate(CONFIG_CASES):
        f = tmp_path / ("c%d.cfg" % i)
        f.write_text(text)
        for j, nsrvs in enumerate((1, 3)):
            for k, rl in enumerate(CONFIG_RELOADS):
                want = gold["config"][i][j][k]
                got = host.load_config(str(f), nsrvs, rl)
                assert got == want, (i, nsrvs, rl, {x: (want[x], got[x]) for x in want if want[x] != got[x]})
    assert host.load_config(str(tmp_path / "missing.cfg"), 1) is None


def plan_tree_cases():
    """(pattern-group tree, .fmt text) pairs: the union / optional workloads, and hand-made blocks"""
    from conftest import ROOT
    X, Y, S, UG, MAS, DOC = -1, -2, -1, -2, -3, -4
    T, NAME, WORKS, UGD, MASD, DOCD = 1, 8, 9, 2, 11, 12
    grp = lambda pats, unions=(), optionals=(): ([(s, p, 1, o) for (s, p, o) in pats], list(unions), list(optionals))   # noqa: E731
    def fmt(rel):
        return open(os.path.join(ROOT, "workloads", "lubm", rel)).read()
    return [
        (grp([], unions=[grp([(X, T, 20), (X, NAME, Y)]), grp([(X, T, 21), (X, NAME, Y)])]), fmt("union/manual_plan/q1.fmt")),
        (grp([(X, WORKS, 131072 + 5)], unions=[grp([(X, T, 22), (X, NAME, Y)]), grp([(X, T, 23), (X, NAME, Y)]), grp([(X, T, 24), (X, NAME, Y)])]),
         fmt("union/manual_plan/q4.fmt")),
        (grp([(S, UGD, UG)], optionals=[grp([(S, DOCD, DOC)])]), fmt("optional/manual_plan/q1.fmt")),
        (grp([(S, UGD, UG)], optionals=[grp([(S, MASD, MAS), (MAS, NAME, 131072 + 9)]), grp([(S, DOCD, DOC)])]), fmt("optional/manual_plan/q3.fmt")),
        # own lines before, between and after the blocks; an optional nested in a union; upper / lower case keywords
        (grp([(X, T, 20), (X, NAME, Y), (X, WORKS, -3)],
             unions=[grp([(X, UGD, -4)], optionals=[grp([(-4, NAME, -5)])]), grp([(X, MASD, -4)])],
             optionals=[grp([(X, DOCD, -6), (-6, NAME, -7)])]),
         "2 <\nunion {\n 1 >\n OPTIONAL {\n  1 <\n }\n}\n1 >\nUnion{\n 1 <<\n}\n3 >\noptional {\n 2 <\n 1 >>\n}\n"),
        # the second block lists fewer lines than it has patterns: refused for that block only
        (grp([(X, T, 20)], unions=[grp([(X, NAME, Y)]), grp([(X, NAME, Y), (X, WORKS, -3)])]), "1 <\nUNION {\n 1 >\n}\nUNION {\n 1 >\n}\n"),
        # the group itself lists fewer lines than it has patterns: no plan
        (grp([(X, T, 20), (X, NAME, Y)], unions=[grp([(X, WORKS, -3)])]), "1 <\nUNION {\n 1 >\n}\n"),
    ]


def test_set_plan_with_union_and_optional_blocks(gold):
    """.fmt plans with UNION { } / OPTIONAL { } blocks (core/planner.hpp:1722-1738): the host mirror's Planner::set_plan on
    pattern-group trees against the reference's own, for the union / optional workloads (workloads/lubm/{union,optional}), a
    nested block, blocks interleaved with the group's own lines, a sub-plan the block refuses, and refused plans"""
    cases = plan_tree_cases()
    wants = gold["set_plan_tree"]
    assert len(wants) == len(cases)
    for (group, text), want in zip(cases, wants):
        got = host.set_plan_tree(REF.encode_group(group), text)
        assert (got is None) == (want is None), (group, text)
        if want is not None:
            assert got == want, (group, text, REF.decode_group(want)[0], REF.decode_group(got)[0])
    # at least one of each outcome was seen
    assert wants[0] is not None and wants[-1] is None
