"""The drop-in binding of INTEGRATION.md, compiled: integration/gpu_engine_cuda.hpp (the replacement `GPUEngineCuda` whose
bodies call the C ABI) against the reference's OWN core/gpu/gpu_engine.hpp, gpu_mem.hpp, gpu_cache.hpp, gpu_stream.hpp and
query.hpp under -DUSE_GPU, none of them edited (oracle/ref_gpu_engine_shim.cpp, `make -C oracle ref`).
CPU: it compiles, links against libwukong_b200.so and exports the driver.  GPU: the reference's GPUEngine::execute_one_pattern,
driven like GPUAgent::execute_sparql_query drives it, answers Q1-Q7 x 3 plan sets on LUBM-1 exactly like the oracle."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, load_query, rows_equal
from oracle import ref as REF

PLANS = ("osdi16_plan", "optimal2560_plan", "optimal10240_plan")


def _ensure_built():
    if os.path.isdir("/root/reference/core"):
        from wukong_b200 import build
        build.build_all()
        subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "ref"], stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    if not REF.gpu_binding_available():
        pytest.skip("oracle/_ref/libwukong_ref_gpu.so is built where the reference tree exists")


def test_binding_compiles_against_the_reference_and_links_against_the_abi():
    _ensure_built()
    out = subprocess.run(["nm", "-D", REF.GPU_LIB], capture_output=True, text=True, check=True).stdout
    undefined = {l.split()[-1] for l in out.splitlines() if " U wk_" in l}
    defined = {l.split()[-1] for l in out.splitlines() if " T " in l}
    assert "refg_query" in defined
    # the replacement backend reaches the engine through the C ABI and nothing else of this repository
    assert {"wk_store_create", "wk_engine_create", "wk_table_upload", "wk_known_to_unknown", "wk_known_to_known", "wk_known_to_const",
            "wk_table_download", "wk_engine_destroy", "wk_store_destroy"} <= undefined, undefined
    abi = subprocess.run(["nm", "-D", os.path.join(ROOT, "wukong_b200", "libwukong_b200.so")], capture_output=True, text=True, check=True).stdout
    exported = {l.split()[-1] for l in abi.splitlines() if " T " in l}
    assert undefined <= exported, undefined - exported
    # the reference's own classes are inside (GPUEngine's dispatch itself is inlined into the driver at -O2)
    syms = subprocess.run(["nm", "-C", REF.GPU_LIB], capture_output=True, text=True, check=True).stdout
    for name in ("GPUEngineCuda::GPUEngineCuda(int, GPUCache*, GPUMem*, GPUStreamPool*)", "GPUEngineCuda::finish_step", "GPUCache::GPUCache",
                 "GPUMem::GPUMem"):
        assert name in syms, name
    assert ctypes.CDLL(REF.GPU_LIB).refg_query is not None        # loads (libwukong_b200.so and libcudart resolve)


def probe_keys(tr):
    """(vid, pid, dir): three index lists, the OUT lists of 200 random subjects and the IN lists of 200 random objects"""
    from oracle import oracle as O
    rng = np.random.default_rng(11)
    return [(0, 1, O.IN), (0, 5, O.IN), (0, 7, O.OUT)] + [(int(s), int(p), O.OUT) for s, p, _ in tr[rng.integers(0, tr.shape[0], 200)]] + \
           [(int(o), int(p), O.IN) for _, p, o in tr[rng.integers(0, tr.shape[0], 200)]]


def test_store_of_the_gpu_flavoured_build_probes_like_the_oracle():
    """CPU: the library's store comes from the reference's StaticGStore::init compiled under -DUSE_GPU (other extent sizing, fixed
    extent array in rdf_seg_meta_t); its probe must give what the oracle's store gives.  The reference's edge lists are
    committed as digests (tests/golden/ref_checks.json, made by tests/golden/make_ref_checks.py from oracle/_ref)."""
    import hashlib
    import json
    from oracle import oracle as O
    from wukong_b200 import datagen
    tr = datagen.lubm(1, seed=1)
    st = O.Store.build(tr, kvstore_bytes=32 << 20, num_engines=4)
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "ref_checks.json")))["gpu_build_edges"]
    keys = probe_keys(tr)
    assert len(gold) == len(keys)
    for (vid, pid, d), want in zip(keys, gold):
        got = np.sort(st.get_edges(vid, pid, d))
        assert hashlib.sha256(np.ascontiguousarray(got, dtype=np.uint32).tobytes()).hexdigest() == want, (vid, pid, d)


def _binding_order(pats):
    """column of every variable in the pattern phase's raw table: the order in which the plan binds them"""
    col = {}
    for s, p, d, o in pats:
        for v in (s, o):
            if v < 0 and v not in col:
                col[v] = len(col)
    return col


@pytest.mark.gpu
def test_reference_gpu_engine_over_the_binding_matches_oracle():
    from oracle import oracle as O
    from wukong_b200 import datagen
    _ensure_built()
    tr = datagen.lubm(1, seed=1)
    st = O.Store.build(tr, kvstore_bytes=32 << 20, num_engines=4)
    eng = REF.RefGpuEngine(tr)
    for plan in PLANS:
        for q in range(1, 8):
            pats, nvars, req, _ = load_query(q, plan)
            want = O.run_query([st], pats, nvars, req)
            rc, rows, cols, tbl = eng.query(pats, nvars, req)
            assert rc == 0 and want.status == 0, (q, plan, rc)
            assert rows == want.rows, (q, plan, rows, want.rows)
            if rows:
                col = _binding_order(pats)
                got = tbl[:, [col[v] for v in req]]
                assert rows_equal(got, want.table), (q, plan)
            rc, rows_b, _, _ = eng.query(pats, nvars, req, blind=True)
            assert rc == 0 and rows_b == want.rows
