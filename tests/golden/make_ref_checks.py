"""Generates tests/golden/ref_checks.json and tests/golden/ref_store_lubm1_head.npz from the reference's OWN compiled code
(oracle/_ref, built by `make -C oracle ref`): the answers the tests in test_reference_pin.py, test_zz_gpu_reference.py and
test_integration_binding.py hold the oracle and the GPU engine to, so that those tests run without the reference tree.

    make -C oracle ref && python tests/golden/make_ref_checks.py
"""
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

import random_bgp as R  # noqa: E402
import test_reference_pin as T  # noqa: E402
from conftest import PLANS, WORKLOADS, load_query  # noqa: E402
from oracle import oracle as O  # noqa: E402
from oracle import ref as REF  # noqa: E402
from wukong_b200 import datagen  # noqa: E402


def ref_store(rs):
    keys = T.occupied_keys(rs.vertices())
    return {"num_slots": int(rs.num_slots), "segs": sorted([int(v) for v in r[:8]] for r in rs.segs()),
            "keys_sha256": T.keys_digest(keys), "num_edges": int(rs.edges().shape[0]),
            "edges_sha256": T.edge_lists_digest(keys, lambda k: rs.get_edges(*T.split_key(k)))}


def answer(rc, rows, t):
    return {"rc": rc, "rows": rows, "sha256": T.table_digest(t) if rows else None}


def exact(rows, t):
    return {"rows": rows, "sha256": hashlib.sha256(np.ascontiguousarray(t).tobytes()).hexdigest() if rows else None}


def main():
    from wukong_b200 import build
    build.build_all()                # oracle/_ref/libwukong_ref_gpu.so links against libwukong_b200.so
    if not REF.build() or not REF.gpu_binding_available():
        sys.exit("oracle/_ref is not built: run `make -C oracle ref` with REFERENCE pointing at the reference tree")
    G = {"source": "the reference's StaticGStore, SPARQLEngine, Planner and config loader compiled by oracle/Makefile `ref`"}
    lubm1 = datagen.lubm(1, seed=1)
    ref1 = REF.RefStore(lubm1)
    G["store_lubm1"] = ref_store(ref1)
    G["store_lubm1_server1_of_2"] = ref_store(REF.RefStore(lubm1, num_servers=2, sid=1))

    eng = {}
    for q in range(1, 8):
        for plan in PLANS:
            pats, nvars, req, _ = load_query(q, plan)
            e = {}
            for mt in (1, 3):
                rc, rows, cols, t = ref1.query(pats, nvars, req, mt_factor=mt)
                e["mt%d" % mt] = dict(answer(rc, rows, t), cols=cols)
            e["blind_rows"] = ref1.query(pats, nvars, req, blind=True)[1]
            rc, rows, _, t = ref1.query(pats, nvars, req, distinct=True, offset=1, limit=40)
            e["distinct"] = exact(rows, t)
            eng["q%d_%s" % (q, plan)] = e
    for name, (pats, nvars, req) in T.special_queries().items():
        rc, rows, _, t = ref1.query(pats, nvars, req)
        eng[name] = answer(rc, rows, t)
    eng["status"] = [ref1.query(p, nv, rq)[0] for p, nv, rq in T.STATUS_QUERIES]
    G["engine_lubm1"] = eng

    rnd = {}
    for gseed in (3, 11, 12):
        tr, meta = R.graph(gseed, nv=300, ntriples=2500)
        rs = REF.RefStore(tr, num_normal_preds=meta["num_normal_preds"])
        ost = O.Store.build(tr, kvstore_bytes=8 << 20, num_engines=2, num_normal_preds=meta["num_normal_preds"])
        for qseed in range(60):
            planned, _, nvars, req = R.query(7000 + 100 * gseed + qseed, tr, meta)
            if O.run_query([ost], planned, nvars, req, blind=True).rows > 200_000:
                continue
            rc, rows, _, t = rs.query(planned, nvars, req)
            e = answer(rc, rows, t)
            rc, rows, _, t = rs.query(planned, nvars, req, distinct=True)
            e["distinct"] = dict(exact(rows, t), rc=rc)
            rnd["g%d_q%d" % (gseed, qseed)] = e
    G["random_graphs"] = rnd

    plans = {}
    for q in range(1, 8):
        for plan in PLANS:
            _, _, _, raw = load_query(q, plan)
            plans["q%d_%s" % (q, plan)] = REF.set_plan(raw, open(os.path.join(WORKLOADS, plan, "lubm_q%d.fmt" % q)).read())
    raw = load_query(7, "osdi16_plan")[3]
    plans["q7_odd_fmt"] = REF.set_plan(raw, T.ODD_FMT)
    plans["q7_bad_fmts"] = [REF.set_plan(raw, bad) for bad in T.BAD_FMTS]
    G["set_plan"] = plans
    G["set_plan_tree"] = [(lambda w: None if w is None else REF.encode_group(w))(REF.set_plan_tree(g, text))
                          for g, text in T.plan_tree_cases()]

    fork = {}
    for q in range(1, 8):
        for plan in PLANS:
            pats, nvars, _, _ = load_query(q, plan)
            fork["q%d_%s" % (q, plan)] = ref1.fork_plan(pats, nvars, 4)
    fork["type_index"] = ref1.fork_plan(T.TYPE_INDEX_PLAN, 4, 3)
    tbl = T.split_table()
    fork["split"] = {"n%d_col%d" % (n, col): [hashlib.sha256(p.tobytes()).hexdigest() for p in ref1.split(tbl, col, n)]
                     for n, col in T.SPLITS}
    G["fork_join"] = fork

    cl = {}
    for n in (2, 3):
        shards = [REF.RefStore(lubm1, num_servers=n, sid=i) for i in range(n)]
        for q in range(1, 8):
            for plan in PLANS:
                pats, nvars, req, _ = load_query(q, plan)
                rc, rows, _, t = REF.cluster_query(shards, pats, nvars, req)
                cl["n%d_q%d_%s" % (n, q, plan)] = answer(rc, rows, t)
    G["cluster"] = cl

    import tempfile
    cfg = []
    with tempfile.TemporaryDirectory() as d:
        for i, text in enumerate(T.CONFIG_CASES):
            f = os.path.join(d, "c%d.cfg" % i)
            open(f, "w").write(text)
            cfg.append([[REF.load_config(f, nsrvs, rl) for rl in T.CONFIG_RELOADS] for nsrvs in (1, 3)])
    G["config"] = cfg

    # test_zz_gpu_reference.py: a random graph answered by the reference engine
    tr, meta = R.graph(0, nv=400, ntriples=4000)
    rs = REF.RefStore(tr, num_normal_preds=meta["num_normal_preds"])
    ost = O.Store.build(tr, kvstore_bytes=8 << 20, num_normal_preds=meta["num_normal_preds"])
    G["gpu_random_graph"] = {}
    for qseed in range(40):
        planned, _, nvars, req = R.query(qseed, tr, meta)
        if O.run_query([ost], planned, nvars, req, blind=True).rows > 300_000:
            continue
        rc, rows, _, t = rs.query(planned, nvars, req)
        G["gpu_random_graph"]["q%d" % qseed] = answer(rc, rows, t)

    # test_integration_binding.py: edge lists of the store of the -DUSE_GPU build
    import test_integration_binding as IB
    g = REF.RefGpuEngine(lubm1)
    G["gpu_build_edges"] = [hashlib.sha256(np.sort(g.get_edges(*k)).tobytes()).hexdigest() for k in IB.probe_keys(lubm1)]

    # test_zz_gpu_reference.py: the store arrays the reference builds for the first LUBM_HEAD triples of LUBM-1
    import test_zz_gpu_reference as Z
    rs = REF.RefStore(lubm1[:Z.LUBM_HEAD])
    v = rs.vertices()
    slots = np.nonzero(v[:, 0])[0]
    np.savez_compressed(os.path.join(HERE, "ref_store_lubm1_head.npz"), num_slots=np.array([v.shape[0]], dtype=np.uint64),
                        slots=slots.astype(np.uint32), keys=v[slots, 0], ptrs=v[slots, 1], edges=rs.edges(), segs=rs.segs())
    with open(os.path.join(HERE, "ref_checks.json"), "w") as f:
        json.dump(G, f, indent=0, sort_keys=True)
    print("wrote ref_checks.json and ref_store_lubm1_head.npz")


if __name__ == "__main__":
    main()
