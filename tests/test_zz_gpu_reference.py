"""GPU: the engine against the answers of the reference's OWN compiled code (the file name sorts last for historical
reasons), all of them committed under tests/golden/ (made from oracle/_ref by make_ref_engine.py and make_ref_checks.py):

* the reference engine's answers on LUBM-1 and LUBM-2 (ref_engine_lubm{1,2}.json);
* a store BUILT BY THE REFERENCE (StaticGStore::init, CPU build with many 256-bucket ext extents, unsorted index lists),
  uploaded as is with wk_store_create and queried on the GPU (ref_store_lubm1_head.npz);
* the reference engine's answers on a random graph (ref_checks.json)."""
import os

import numpy as np
import pytest

import sparql_mini as M
from conftest import PLANS, load_query, rows_equal
from oracle import oracle as O
from wukong_b200 import capi

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def eng1(gstore1):
    e = capi.Engine(gstore1, rbuf_bytes=64 << 20)
    yield e
    e.close()


@pytest.fixture(scope="module")
def eng2(gstore2):
    e = capi.Engine(gstore2, rbuf_bytes=64 << 20)
    yield e
    e.close()


@pytest.mark.parametrize("which", [1, 2])
def test_matches_reference_engine_fixture(eng1, eng2, which):
    """the answers of the reference's OWN compiled engine on this dataset (tests/golden/ref_engine_lubm1.json, produced by
    tests/golden/make_ref_engine.py from oracle/_ref): row counts and digests of the sorted tables, exact tables under DISTINCT"""
    import hashlib
    import json
    import os
    G = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_engine_lubm%d.json" % which)))
    eng1 = eng1 if which == 1 else eng2
    for name, e in G["queries"].items():
        q, plan = int(name.split("_")[0][1:]), name.split("_", 1)[1]
        pats, nvars, req, _ = load_query(q, plan)
        rc, rows, cols, tbl = eng1.query(pats, nvars, req)
        assert rc == 0 and rows == e["rows"], name
        if rows:
            assert hashlib.sha256(M.sort_rows(tbl).tobytes()).hexdigest() == e["sha256"], name
        rc, rows, cols, tbl = eng1.query(pats, nvars, req, distinct=True, offset=1, limit=40)
        assert rc == 0 and rows == e["distinct_rows"], name
        if rows:
            assert hashlib.sha256(np.ascontiguousarray(tbl).tobytes()).hexdigest() == e["distinct_sha256"], name


LUBM_HEAD = 10000     # the first triples of LUBM-1: a reference-built store of all of it does not fit a small test vector


def reference_built_store():
    """the store arrays the reference's StaticGStore::init builds for lubm1[:LUBM_HEAD] (tests/golden/ref_store_lubm1_head.npz,
    made by tests/golden/make_ref_checks.py from oracle/_ref; only the occupied header slots are stored)"""
    z = np.load(os.path.join(HERE, "golden", "ref_store_lubm1_head.npz"))
    v = np.zeros((int(z["num_slots"][0]), 2), dtype=np.uint64)
    v[z["slots"], 0], v[z["slots"], 1] = z["keys"], z["ptrs"]
    return v, z["edges"], z["segs"]


def test_reference_built_store_runs_on_the_gpu(lubm1):
    """a store BUILT BY THE REFERENCE (CPU build with many 256-bucket ext extents, unsorted index lists) uploaded as is with
    wk_store_create and queried on the GPU: Q1-Q7 x 3 plan sets against the oracle on the same triples"""
    tr = lubm1[:LUBM_HEAD]
    ost = O.Store.build(tr, kvstore_bytes=32 << 20, num_engines=4)
    v, e, rsegs = reference_built_store()
    segs = []
    for r in rsegs:
        m = capi.SegMeta()
        m.index, m.dir, m.pid = int(r[0]), int(r[1]), int(r[2])
        m.num_keys, m.num_buckets, m.bucket_start, m.num_edges, m.edge_start = (int(x) for x in r[3:8])
        m.ext_start, m.ext_num = int(r[9]), int(r[10])        # first extent only (informational: probes follow chain pointers)
        segs.append(m)
    v = v[: (v.shape[0] // 8) * 8]      # GStore's slot count need not be a multiple of 8; no bucket id reaches the partial tail
    gst = capi.Store(v, e, segs)
    eng = capi.Engine(gst, rbuf_bytes=64 << 20)
    nonempty = 0
    for q in range(1, 8):
        for plan in PLANS:
            pats, nvars, req, _ = load_query(q, plan)
            want = O.run_query([ost], pats, nvars, req)
            rc, rows, cols, tbl = eng.query(pats, nvars, req)
            assert rc == 0 and rows == want.rows, (q, plan)
            if rows:
                nonempty += 1
                assert rows_equal(tbl, want.table), (q, plan)
    assert nonempty == 18          # Q3 has no answer on these triples
    s, p, o = (int(x) for x in tr[4321])
    assert np.array_equal(gst.get_edges(s, p, O.OUT), ost.get_edges(s, p, O.OUT))
    eng.close()
    gst.close()


def test_random_graph_against_live_reference_engine():
    """a random graph (tests/random_bgp.py) answered by the GPU engine and by the reference's compiled engine (its answers are
    committed in tests/golden/ref_checks.json, made by tests/golden/make_ref_checks.py)"""
    import hashlib
    import json
    import random_bgp as R
    gold = json.load(open(os.path.join(HERE, "golden", "ref_checks.json")))["gpu_random_graph"]
    tr, meta = R.graph(0, nv=400, ntriples=4000)
    npreds = meta["num_normal_preds"]
    gst = capi.Store.build(tr, npreds)
    eng = capi.Engine(gst, rbuf_bytes=256 << 20)
    checked = 0
    for qseed in range(40):
        planned, _, nvars, req = R.query(qseed, tr, meta)
        rc, rows, cols, tbl = eng.query(planned, nvars, req)
        if rc == capi.WK_ERR_RBUF_OVERFLOW or rows > 300_000:
            continue
        g = gold["q%d" % qseed]
        assert rc == 0 and g["rc"] == 0 and g["rows"] == rows, (qseed, planned)
        assert rows == 0 or hashlib.sha256(M.sort_rows(tbl).tobytes()).hexdigest() == g["sha256"], (qseed, planned)
        checked += 1
    assert checked >= 30
    eng.close()
    gst.close()
