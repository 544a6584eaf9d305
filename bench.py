#!/usr/bin/env python
"""bench.py -- LUBM Q1-Q7 queries/sec (geomean) on B200, with roofline and CPU baseline.

Contract (see DESIGN.md, Measurement):
  step     = one pass over the query mix Q1..Q7 (each query executed once)
  N = 1    : LUBM-2560 on one GPU (BASELINE config 3)
  N > 1    : LUBM-10240 sharded by vid % N over the N GPUs (BASELINE config 4, optimal10240_plan), exchange through
             the single-pass peer-memory push over NVLink; `replicas` (LUBM-2560 on every GPU) and the single-GPU run of
             the same LUBM-10240 store are secondary keys of the same line.  --mode replicas restores round 1's default.
  value    = geomean over Q1..Q7 of 1 / mean latency, blind mode (= the reference's global_silent=1 protocol), store and
             plan resident in HBM: CUDA events on the engine's stream for every query that runs as kernel launches; light
             queries answered by the RESIDENT server kernel have no launch to bracket with events, so their term is the
             host wall clock of the blind call (an upper bound of the device time; the in-kernel %globaltimer span is
             reported beside it)
  e2e      = same metric through the public C-ABI call wk_query_execute with HOST buffers: the plan goes host->device
             inside the call, the projected result table comes back device->host into pinned memory inside the timed
             region (non-blind)
  roofline = the dominant kernel (largest share of device time): algorithmic bytes (SURVEY.md 8d) / CUDA-event duration
             vs the measured HBM peak in MEASURED_PEAKS.json
  cpu_baseline / --impl reference : the reference's OWN engine (oracle/_ref) on the host cores this process may use
             (sched_getaffinity capped by the cgroup CPU quota), best mt_factor per heavy query from a sweep, blind and
             non-blind latencies; `value` of the reference line is the NON-blind geomean (= its `e2e.value`, as the contract
             asks: the CPU engine's result is in host memory either way), `value_blind` the blind one, so that e2e/e2e and
             value/value_blind each compare equal work.
  parity   = at full scale: an order-independent digest of every query's non-blind table from the GPU engine equals the
             CPU arm's digest of its own table (not only the row counts).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

HEAVY = (1, 2, 3, 7)
LIGHT = (4, 5, 6)
QUERIES = (1, 2, 3, 4, 5, 6, 7)


def geomean(xs):
    xs = [max(float(x), 1e-12) for x in xs]
    return math.exp(sum(math.log(x) for x in xs) / len(xs))


def load_plans(plan):
    from conftest import load_query
    return {q: load_query(q, plan)[:3] for q in QUERIES}


class ClockSampler(threading.Thread):
    """SM clock and clock-event (throttle) reasons of one GPU sampled DURING the timed region: NVML in this process every 25 ms
    (the counters nvidia-smi prints; a subprocess of nvidia-smi -lms needs seconds to deliver its first line on an 8-GPU
    host, longer than a sharded run's timed region), falling back to `nvidia-smi -lms 20` when pynvml is missing."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    BITS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        cvd = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        try:
            ids = [int(x) for x in cvd.split(",") if x.strip() != ""]
            if ids and index < len(ids):
                self.index = ids[index]
        except ValueError:
            pass
        self.rows = []          # (time, sm MHz, max MHz, set of reasons)
        self.proc = None
        self.t_mark = None
        self.source = None
        self.quit = threading.Event()

    def run_nvml(self):
        import pynvml as N
        N.nvmlInit()
        h = N.nvmlDeviceGetHandleByIndex(self.index)
        mx = float(N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM))
        get = getattr(N, "nvmlDeviceGetCurrentClocksEventReasons", None) or N.nvmlDeviceGetCurrentClocksThrottleReasons
        self.source = "nvml"
        while not self.quit.is_set():
            sm = float(N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM))
            bits = int(get(h))
            self.rows.append((time.time(), sm, mx, {nm for nm, b in self.BITS if bits & b}))
            self.quit.wait(0.025)

    def run_smi(self):
        self.source = "nvidia-smi"
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits", "-lms", "20"],
                                     stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(",")]
            try:
                self.rows.append((time.time(), float(r[1]), float(r[2]), {nm for i, nm in enumerate(names) if r[5 + i].lower().startswith("active")}))
            except Exception:
                continue

    def run(self):
        try:
            self.run_nvml()
        except Exception:
            try:
                self.run_smi()
            except Exception:
                pass

    def stop(self):
        self.quit.set()
        if self.proc:
            self.proc.terminate()
        self.join(timeout=2)
        rows = list(self.rows)
        timed = [r for r in rows if self.t_mark is not None and r[0] >= self.t_mark]
        use = timed if timed else rows      # the statistics are those of the timed region whenever a sample fell into it
        sm = [r[1] for r in use]
        reasons = set()
        for r in use:
            reasons |= r[3]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": (max(r[2] for r in use) if use else None),
                "reasons": sorted(reasons), "samples": len(rows), "samples_in_timed_region": len(timed), "source": self.source,
                "note": "sampled from the start of warm-up to the end of the timed region (NVML every 25 ms); sm_mhz / reasons over the "
                        "samples inside the timed region when there are any"}


LOAD_FACTORS = (55, 45, 35, 25)   # Global::est_load_factor (global.hpp:99-104) and its fallbacks for small datasets


def host_cpus():
    """CPUs this process may really use: the affinity mask capped by the cgroup CPU quota (a lease of a GPU box often owns a
    share of the host); physical cores among them from /proc/cpuinfo."""
    aff = sorted(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else list(range(os.cpu_count() or 1))
    usable = len(aff)
    quota = None
    try:
        txt = open("/sys/fs/cgroup/cpu.max").read().split()
        if txt and txt[0] != "max":
            quota = float(txt[0]) / float(txt[1])
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    if quota:
        usable = max(1, min(usable, int(math.ceil(quota))))
    cores = set()
    try:
        cpu, phys, core = None, 0, None
        for line in open("/proc/cpuinfo"):
            if line.startswith("processor"):
                cpu = int(line.split(":")[1])
            elif line.startswith("physical id"):
                phys = int(line.split(":")[1])
            elif line.startswith("core id"):
                core = int(line.split(":")[1])
                if cpu in aff:
                    cores.add((phys, core))
    except Exception:
        pass
    return {"affinity": len(aff), "cgroup_quota": quota, "usable": usable, "physical_cores": len(cores) or None}


def mt_candidates(threads):
    """mt_factor values tried for the heavy queries (the reference's mt_factor knob, sparql.hpp:1064-1089): 16..128 and the
    usable CPU count, without oversubscribing the CPUs more than twice"""
    c = sorted({m for m in (16, 32, 64, 128, threads) if m <= max(2 * threads, 16)})
    return c or [threads]


def build_dataset(args):
    """host arm: triples -> store arrays with the host builder (csrc/store/host_builder.cpp)"""
    from wukong_b200 import datagen, host
    t0 = time.time()
    tr = datagen.lubm(args.scale, seed=args.seed)
    t1 = time.time()
    hs, lf = None, None
    for lf in LOAD_FACTORS:      # a segment that outgrows its single 15 % ext extent (meta.hpp:38-40) needs a sparser header
        try:
            hs = host.HostStore(tr, est_load_factor=lf)
            break
        except RuntimeError:
            if lf == LOAD_FACTORS[-1]:
                raise
    t2 = time.time()
    info = {"triples": int(tr.shape[0]), "keys": int(hs.num_keys), "gen_s": round(t1 - t0, 2), "build_s": round(t2 - t1, 2),
            "store_build": "host", "est_load_factor": lf, "header_mb": round(hs.num_slots * 16 / 1e6, 1), "edges_mb": round(hs.num_edges * 4 / 1e6, 1)}
    return tr, hs, info


class DeviceBuiltStore:
    """the arrays of a device-built store copied back for the CPU baseline (same accessors as host.HostStore)"""

    def __init__(self, gst):
        self._v, self._e = gst.download()
        self._s = gst.segs()

    def vertices(self): return self._v
    def edges(self): return self._e
    def segs(self): return self._s


def build_dataset_device(args, device, num_servers=1, sid=0):
    """triples -> store directly in HBM (wk_store_build: sort / dedup / partition / insert on the GPU)"""
    from wukong_b200 import capi, datagen
    t0 = time.time()
    if num_servers > 1:
        tr = datagen.lubm_shard(args.scale, num_servers, sid, seed=args.seed)
    else:
        tr = datagen.lubm(args.scale, seed=args.seed)
    t1 = time.time()
    gst, lf = None, None
    for lf in LOAD_FACTORS:
        try:
            gst = capi.Store.build(tr, datagen.LUBM_NUM_NORMAL_PREDS, num_servers=num_servers, sid=sid, est_load_factor=lf, device=device)
            break
        except capi.WukongError as ex:
            if ex.code != capi.WK_ERR_STORE_FULL or lf == LOAD_FACTORS[-1]:
                raise
    t2 = time.time()
    st = gst.build_stats
    info = {"triples": int(tr.shape[0]), "keys": int(st["num_keys"]), "gen_s": round(t1 - t0, 2), "build_s": round(t2 - t1, 2),
            "store_build": "device", "est_load_factor": lf, "build_ms": {k: round(st[k], 1) for k in ("ms_upload", "ms_sort", "ms_insert", "ms_total")},
            "header_mb": round(st["num_slots"] * 16 / 1e6, 1), "edges_mb": round(st["num_edges"] * 4 / 1e6, 1)}
    return tr, gst, info


def cpu_engine_kind(args):
    """which CPU engine times the path: "reference" = the reference's OWN SPARQLEngine (core/engine/sparql.hpp), compiled in
    oracle/_ref behind C shims (oracle/Makefile `ref`), probing the same store arrays through its own GStore code;
    "port" = the oracle restatement (when oracle/_ref was never built, i.e. no reference tree was available)."""
    from oracle import ref as REF
    want = getattr(args, "cpu_engine", "auto")
    if want == "port":
        return "port"
    if REF.available():
        return "reference"
    if want == "reference":
        raise RuntimeError("oracle/_ref/libwukong_ref.so is missing: run `make -C oracle ref` where /root/reference exists")
    return "port"


class CpuEngine:
    """the CPU arm over one set of store arrays (adopted once).  Heavy queries run as mt_factor index slices on host threads
    (the reference's mt_factor replicas, sparql.hpp:1064-1089), light queries single-threaded; the timed region is the pattern
    phase + merge + final_process (non-blind) or the pattern phase + merge (blind = global_silent)."""

    def __init__(self, hs, kind):
        self.kind = kind
        self.best_mt = {}
        if kind == "reference":
            from oracle import ref as REF
            self.rs = REF.RefStore.adopt(hs.vertices(), hs.edges(), hs.segs(), num_normal_preds=31)
        else:
            from oracle import oracle as O
            self.ost = O.Store.wrap(hs.vertices(), hs.edges(), hs.segs())

    def _run(self, pats, nvars, req, reps, mt, threaded, blind, digest=False):
        """-> (mean us over reps, rows, digest or None); one untimed repetition first when reps > 1"""
        from oracle import ref as REF
        if self.kind == "reference":
            n = reps + (1 if reps > 1 else 0)
            r = self.rs.time_query(pats, nvars, req, reps=n, mt_factor=mt, threaded=threaded, blind=blind, digest=digest)
            assert r[0] == 0, r[0]
            us = r[1][1:] if reps > 1 else r[1]
            return float(np.mean(us)), int(r[2]), (r[3] if digest else None)
        from oracle import oracle as O
        us, res = [], None
        for i in range(reps + (1 if reps > 1 else 0)):
            res = O.run_query([self.ost], pats, nvars, req, mt_factor=mt, blind=blind, threaded=threaded)
            assert res.status == 0
            if reps == 1 or i > 0:
                us.append(res.usec)
        dg = REF.table_digest(res.table) if (digest and not blind) else None
        return float(np.mean(us)), int(res.rows), dg

    def sweep(self, plans, threads):
        """pick the best mt_factor per heavy query (one non-blind run per candidate)"""
        for q in HEAVY:
            pats, nvars, req = plans[q]
            best = None
            for mt in mt_candidates(threads):
                us, _, _ = self._run(pats, nvars, req, 1, mt, True, False)
                if best is None or us < best[0]:
                    best = (us, mt)
            self.best_mt[q] = best[1]
        return dict(self.best_mt)

    def times(self, plans, threads, heavy_reps, light_reps, digest=False):
        """-> {q: dict(non_blind_us, blind_us, rows, mt, digest)}"""
        if not self.best_mt:
            self.sweep(plans, threads)
        out = {}
        for q in QUERIES:
            pats, nvars, req = plans[q]
            heavy = q in HEAVY
            reps = heavy_reps if heavy else light_reps
            mt = self.best_mt[q] if heavy else 1
            nb, rows, dg = self._run(pats, nvars, req, reps, mt, heavy, False, digest=digest)
            bl, rows_b, _ = self._run(pats, nvars, req, reps, mt, heavy, True)
            assert rows_b == rows, (q, rows, rows_b)
            out[q] = {"non_blind_us": nb, "blind_us": bl, "rows": rows, "mt": mt, "digest": dg}
        return out


CPU_ENGINE_NOTE = {"reference": "the reference's own SPARQLEngine + GStore probe (core/engine/sparql.hpp, core/store/gstore.hpp) compiled "
                                "in oracle/_ref with std-based stand-ins for Boost/TBB/ZeroMQ, over the product-built store arrays",
                   "port": "oracle restatement of the reference engine (oracle/_ref not built)"}


def published_baseline(args):
    """BASELINE.md 1: the reference's own published geomean for this exact metric and config (LUBM-2560, Q1-Q7, OSDI16
    fixed plans, 1 node, 2 x 12-core Xeon E5-2650 v4; docs/performance/S1C24-LUBM2560-20181203.md:417-425): 4 253 us -> 235 q/s.
    Other scales / plan sets have no published counterpart."""
    if args.scale == 2560 and args.plan == "osdi16_plan":
        return 235.0
    return None


def vs_published(value, args):
    b = published_baseline(args)
    return (value / b) if b else None


def peak_hbm():
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(pk["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


NVLINK_PEAK_GBS = 770.0   # B200_PROFILING.md: measured peer copy per direction per GPU on this pool (900 nominal)


def workload_name(args, world, sharded):
    w = "LUBM-%d Q1-Q7 (%s), seeded LUBM-shaped generator" % (args.scale, args.plan)
    if sharded:
        w += ", store sharded by vid %% %d" % world
    return w


def cpu_sample_note(threads, best_mt, kind, heavy_reps, light_reps):
    return ("same store arrays; Q1,Q2,Q3,Q7 %dx on host threads with the best mt_factor of a sweep over %s (%s), Q4-Q6 %dx single "
            "thread; blind = pattern phase + merge, non-blind = + final_process; engine: %s"
            % (heavy_reps, mt_candidates(threads), ", ".join("q%d:%d" % (q, m) for q, m in sorted(best_mt.items())), light_reps,
               CPU_ENGINE_NOTE[kind]))


def run_reference(args, rank, world):
    """the reference arm: the reference's CPU engine on the same config as the GPU arm at this N"""
    if rank != 0:
        return
    # the store arrays the CPU engine probes (input data, outside the timed region): built on the GPU when there is one (seconds
    # and one copy back instead of minutes and a second copy of the triples in host memory at LUBM-10240), else by the host builder
    hs = None
    try:
        from wukong_b200 import capi
        if args.store_build == "device" and capi.device_count() > 0:
            tr, gst, info = build_dataset_device(args, 0)
            del tr
            hs = DeviceBuiltStore(gst)
            gst.close()
    except Exception as ex:   # noqa: BLE001
        print("device-side store build for the CPU arm failed (%r): host builder" % (ex,), file=sys.stderr)
        hs = None
    if hs is None:
        tr, hs, info = build_dataset(args)
        del tr
    plans = load_plans(args.plan)
    cpus = host_cpus()
    threads = args.cpu_threads or cpus["usable"]
    kind = cpu_engine_kind(args)
    cpu = CpuEngine(hs, kind)
    t_start = time.time()
    best_mt = cpu.sweep(plans, threads)
    nb = {q: [] for q in QUERIES}
    bl = {q: [] for q in QUERIES}
    rows = {}
    # each step = one bounded pass: heavy queries once (blind and non-blind) on the host threads, light queries 50x
    for it in range(args.warmup + args.steps):
        res = cpu.times(plans, threads, 1, 50)
        if it >= args.warmup:
            for q in QUERIES:
                nb[q].append(res[q]["non_blind_us"])
                bl[q].append(res[q]["blind_us"])
                rows[q] = res[q]["rows"]
    nb_mean = {q: float(np.mean(nb[q])) for q in QUERIES}
    bl_mean = {q: float(np.mean(bl[q])) for q in QUERIES}
    # the contract gives the reference line ONE number (value == e2e.value): the non-blind one, i.e. the work the GPU arm's e2e
    # does (the headline ratio is e2e / e2e); the blind geomean (the work of the GPU arm's `value`) rides along as value_blind
    value = geomean([1e6 / nb_mean[q] for q in QUERIES])
    value_blind = geomean([1e6 / bl_mean[q] for q in QUERIES])
    e2e = value
    sharded = args.gpus > 1 and args.mode == "sharded"
    line = {"impl": "reference", "metric": "lubm_q1_q7_geomean_queries_per_sec", "value": value, "unit": "queries/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": sum(nb_mean.values()) / 1e3, "higher_is_better": True, "scaling": "strong" if sharded else "weak",
            "vs_baseline": vs_published(value, args), "value_blind": value_blind,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": workload_name(args, args.gpus, sharded), "triples": info["triples"],
                       "value_mode": "non-blind: pattern phase + merge + final_process (value_blind: without final_process, global_silent)",
                       "note": "CPU arm: one host, whole store in host memory (the GPU arm at N > 1 shards the same dataset)"},
            "cpu_baseline": {"value": value, "unit": "queries/s", "cores": threads, "kind": kind, "host_cpus": cpus,
                             "mt_factor": {"q%d" % q: m for q, m in best_mt.items()},
                             "sample": "per step: " + cpu_sample_note(threads, best_mt, kind, 1, 50)},
            "e2e": {"value": e2e, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "latency_us": {"blind": {"q%d" % q: round(bl_mean[q], 2) for q in QUERIES},
                           "non_blind": {"q%d" % q: round(nb_mean[q], 2) for q in QUERIES}},
            "rows": {"q%d" % q: rows[q] for q in QUERIES},
            "wall_s": round(time.time() - t_start, 1)}
    emit(line)


def setup_group(args, eng, rank, world, dist):
    from wukong_b200 import capi
    if args.exchange == "p2p":
        allh = [None] * world
        dist.all_gather_object(allh, eng.p2p_export(world, rank))
        eng.p2p_import(b"".join(allh))
        # peers' store arrays: const-start (light) plans are answered in place by the constant's owner over NVLink loads
        blobs = [None] * world
        dist.all_gather_object(blobs, eng.p2p_export_store())
        eng.p2p_import_store(blobs)
        dist.barrier()
    else:
        uid = [capi.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        eng.comm_init(world, rank, uid[0])


class SpinBarrier:
    """Host barrier with a release skew of about a microsecond: one generation counter per rank in a shared-memory file, spun
    on.  dist.barrier() alone lets the ranks leave tens of microseconds apart, which a query of 10-20 us then absorbs as waiting
    time on whichever rank left first (every collective query ends when its slowest rank ends)."""

    def __init__(self, rank, world, dist):
        self.rank, self.dist, self.gen, self.a = rank, dist, 0, None
        name = [None]
        if rank == 0:
            try:
                path = "/dev/shm/wk_bench_%d_%d" % (os.getpid(), time.time_ns())
                np.zeros(world * 8, dtype=np.int64).tofile(path)
                name[0] = path
            except OSError:
                name[0] = None
        dist.broadcast_object_list(name, src=0)
        if name[0]:
            self.a = np.memmap(name[0], dtype=np.int64, mode="r+")
            self.slots = self.a[::8]
        dist.barrier()
        if rank == 0 and name[0]:
            os.unlink(name[0])

    def wait(self):
        self.dist.barrier()
        if self.a is None:
            return
        self.gen = int(self.a[self.rank * 8]) + 1     # the native timer (host.ShardedTimer) advances the same counters
        g = self.gen
        self.a[self.rank * 8] = g
        t0 = time.monotonic()
        while (self.slots < g).any():
            if time.monotonic() - t0 > 120:
                raise RuntimeError("spin barrier timed out")


def run_sharded(args, rank, world, local_rank, dist):
    """vid % N sharded store; before every step whose start variable is not local the table is bucketised by owner and pushed
    over NVLink (or exchanged through NCCL).  Strong scaling: the dataset is fixed, every query is answered by all ranks together."""
    import torch
    from wukong_b200 import capi, datagen, host
    t0 = time.time()
    if args.store_build == "device":
        tr, gst, binfo = build_dataset_device(args, local_rank, num_servers=world, sid=rank)
    else:
        tr = datagen.lubm_shard(args.scale, world, rank, seed=args.seed)
        gst = host.HostStore(tr, num_servers=world, sid=rank).upload(local_rank)
        binfo = {}
    t1 = time.time()
    shard_triples = int(tr.shape[0])
    del tr
    rbuf = (args.rbuf_mb << 20) if args.rbuf_mb else max(256 << 20, min(8 << 30, shard_triples * 8))
    rb = torch.tensor([rbuf], device="cuda", dtype=torch.int64)     # the pushers check the owners' capacity: same on every rank
    dist.all_reduce(rb, op=dist.ReduceOp.MAX)
    rbuf = int(rb.item())
    eng = capi.Engine(gst, rbuf_bytes=rbuf)
    setup_group(args, eng, rank, world, dist)
    plans = load_plans(args.plan)
    out_tbl, _keep = capi.pinned_array(min(rbuf // 4, 1 << 26))
    bar = SpinBarrier(rank, world, dist)
    sampler = ClockSampler(local_rank)
    sampler.start()
    rows, nb_words = {}, {}
    for _ in range(args.warmup):
        for q in QUERIES:
            pats, nvars, req = plans[q]
            rc, r, c, _ = eng.query_sharded(pats, nvars, req, blind=True)
            assert rc == 0, rc
            rows[q] = r
            rc, r2, c2, _ = eng.query_sharded(pats, nvars, req, out=out_tbl)
            assert rc == 0 and r2 == r, (rc, r2, r)
            nb_words[q] = r2 * c2
    launches0 = eng.launch_count()
    st0 = eng.comm_stats()
    bytes0 = eng.get_option(capi.WK_INFO_COMM_BYTES_PUSHED) if args.exchange == "p2p" else 0
    eng.sync(); dist.barrier(); torch.cuda.synchronize()
    t_region0 = time.time()
    sampler.t_mark = t_region0
    eng.set_profiling(1)
    dev_us = {q: [] for q in QUERIES}
    wall_us = {q: [] for q in QUERIES}
    e2e_us = {q: [] for q in QUERIES}
    srv_ns = {q: [] for q in QUERIES}
    resident = {}
    # native timed calls (wkh_time_query_sharded): the L2 flush must be over on EVERY rank before anyone starts -- a rank still
    # flushing would make its peers' exchange waits absorb its flush -- so: flush, stream sync, spin barrier, clock, query
    timer = host.ShardedTimer(eng, bar.a, rank, world)
    bar.wait()
    for _ in range(args.steps):
        for q in QUERIES:
            pats, nvars, req = plans[q]
            w, d, r, c, res, ns = timer.time(pats, nvars, req, blind=True)
            assert r == rows[q] and d > 0, (q, r, rows[q], d)
            resident[q] = res
            wall_us[q].append(w)
            # a light plan answered by the resident servers has no launch to bracket with events: its term is the wall clock
            # of the call (doorbell -> record), like at N = 1
            dev_us[q].append(d)
            srv_ns[q].append(ns)
    eng.set_profiling(0)
    stats = eng.comm_stats()       # communication of the K blind steps (the end-to-end pass below repeats the same exchanges)
    bytes_pushed = (eng.get_option(capi.WK_INFO_COMM_BYTES_PUSHED) - bytes0) if args.exchange == "p2p" else 0
    # end to end: non-blind, every rank receives its share of the projected table in pinned host memory
    for _ in range(args.steps):
        for q in QUERIES:
            pats, nvars, req = plans[q]
            w, _, r, c, _, _ = timer.time(pats, nvars, req, blind=False, table=out_tbl)
            assert r == rows[q], (q, r, rows[q])
            e2e_us[q].append(w)
    eng.sync(); dist.barrier(); torch.cuda.synchronize()
    t_region = time.time() - t_region0
    clocks = sampler.stop()
    launches = eng.launch_count() - launches0
    # ---- per-step pass (CUDA events per step and per exchange): where the time goes, NVLink GB/s of the exchanges ----------
    eng.set_profiling(2)
    agg = {}
    for _ in range(max(3, min(args.steps, 5))):
        for q in HEAVY:   # light plans run in place on the constant's owner: no common step list
            pats, nvars, req = plans[q]
            eng.flush_l2(); eng.sync(); dist.barrier()
            rc, _, _, _ = eng.query_sharded(pats, nvars, req, blind=True)
            assert rc == 0
            for i, sst in enumerate(eng.step_stats()):
                a = agg.setdefault((q, i, sst["kind"]), {"us": [], "bytes": sst["algo_bytes"], "in_rows": sst["in_rows"],
                                                         "out_rows": sst["out_rows"]})
                a["us"].append(sst["device_us"])
    eng.set_profiling(0)
    keys = sorted(agg.keys())
    steps_table, exch = [], None
    nk = torch.tensor([len(keys), -len(keys)], device="cuda", dtype=torch.int64)
    dist.all_reduce(nk, op=dist.ReduceOp.MAX)
    if keys and int(nk[0].item()) == -int(nk[1].item()):          # the same step list on every rank
        h = torch.tensor([[float(np.mean(agg[k]["us"])) if agg[k]["us"] else 0.0, float(agg[k]["bytes"]), float(agg[k]["in_rows"]),
                           float(agg[k]["out_rows"])] for k in keys], device="cuda", dtype=torch.float64).reshape(-1, 4)
        h_us = h[:, 0].clone()
        dist.all_reduce(h_us, op=dist.ReduceOp.MAX)            # a step is over when the slowest rank is
        h_sum = h[:, 1:].clone()
        dist.all_reduce(h_sum, op=dist.ReduceOp.SUM)           # bytes and rows: all ranks together
        h_us, h_sum = h_us.cpu().numpy(), h_sum.cpu().numpy()
        xb, xus = 0.0, 0.0
        for i, k in enumerate(keys):
            us = float(h_us[i])
            gbs = (h_sum[i, 0] / us / 1e3) if us > 0 else None
            steps_table.append({"q": k[0], "step": k[1], "kind": k[2], "in_rows_all_ranks": int(h_sum[i, 1]), "out_rows_all_ranks": int(h_sum[i, 2]),
                                "algo_bytes_all_ranks": int(h_sum[i, 0]), "device_us_max_rank": round(us, 2),
                                "gbs_all_ranks": round(gbs, 1) if gbs else None})
            if k[2] == "exchange":
                xb += h_sum[i, 0]
                xus += us
        if xus > 0:
            per_gpu = xb / world / xus / 1e3
            exch = {"nvlink_bytes_per_step_all_ranks": int(xb), "exchange_us_per_step": round(xus, 1),
                    "achieved_gbs_per_gpu_per_direction": round(per_gpu, 1), "peak_gbs": NVLINK_PEAK_GBS,
                    "frac": round(per_gpu / NVLINK_PEAK_GBS, 4),
                    "note": "bytes stored into peers' buffers (4*C*rows pushed, SURVEY 8d) / summed ready->push->wait time of the heavy queries' "
                            "exchanges, barriers included; peak = measured peer copy per direction (B200_PROFILING.md), 900 GB/s nominal"}
    t = torch.tensor([np.mean(dev_us[q]) for q in QUERIES] + [np.mean(wall_us[q]) for q in QUERIES] + [np.mean(e2e_us[q]) for q in QUERIES] +
                     [1.0 if resident.get(q) else 0.0 for q in QUERIES], device="cuda", dtype=torch.float64)
    # samples far off their query's median (a descheduled host thread stalls every rank of a collective query): reported, not removed
    outl = torch.tensor([float(sum(1 for x in dev_us[q] if x > 3.0 * float(np.median(dev_us[q])))) for q in QUERIES] +
                        [float(np.median(dev_us[q])) for q in QUERIES], device="cuda", dtype=torch.float64)
    dist.all_reduce(outl, op=dist.ReduceOp.MAX)
    outl = outl.cpu().numpy()
    # per rank, for the record: blind wall clock and in-kernel span of the server request of the light plans (owner vs waiting peers)
    per_rank = torch.zeros((world, 2 * len(LIGHT)), device="cuda", dtype=torch.float64)
    per_rank[rank] = torch.tensor([np.mean(wall_us[q]) for q in LIGHT] + [np.mean(srv_ns[q]) / 1e3 for q in LIGHT], dtype=torch.float64)
    dist.all_reduce(per_rank, op=dist.ReduceOp.SUM)
    per_rank = per_rank.cpu().numpy()
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    lat = t.cpu().numpy()
    rr = torch.tensor([rows[q] for q in QUERIES] + [stats["rows_sent"] - st0["rows_sent"], launches, bytes_pushed, sum(nb_words.values()) * 4],
                      device="cuda", dtype=torch.int64)
    dist.all_reduce(rr, op=dist.ReduceOp.SUM)
    rr = rr.cpu().numpy()
    nx = stats["exchanges"] - st0["exchanges"]
    eng.close()
    gst.close()
    line = None
    if rank == 0:
        dev_mean, wall_mean, e2e_mean, res = lat[:7], lat[7:14], lat[14:21], lat[21:28]
        value = geomean(1e6 / dev_mean)
        par = ("single-pass bucketise + peer-memory push over NVLink (CUDA IPC, remote atomic reservations); light plans in place on the "
               "constant's owner through peer loads") if args.exchange == "p2p" else "NCCL all-to-all(v)"
        line = {"metric": "lubm_q1_q7_geomean_queries_per_sec", "value": value, "unit": "queries/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(dev_mean.sum() / 1e3), "higher_is_better": True,
                "scaling": "strong", "vs_baseline": vs_published(value, args), "dtype": "u32", "data": "synthetic",
                "config": {"workload": workload_name(args, world, True),
                           "parallelism": "sharded x%d, %s before non-local steps" % (world, par),
                           "l2": "flushed before every timed query (384 MB memset + 256 MB read-back, outside the timed region)",
                           "value_mode": "blind (row count only), shards resident in HBM, max over ranks; CUDA events, except light plans answered "
                                         "in place by the resident servers (no launch on any rank: wall clock of the call, doorbell -> record)",
                           "e2e_mode": "non-blind: every rank's share of the projected table D2H into pinned memory, host wall clock, max over ranks",
                           "barrier": "L2 flush, stream sync, shared-memory spin barrier, then the clock: all in native code (wkh_time_query_sharded)"},
                "e2e": {"value": geomean(1e6 / e2e_mean), "unit": "queries/s", "h2d_bytes_per_step": 584 * world,
                        "d2h_bytes_per_step": int(rr[10]) + 32 * len(QUERIES) * world},
                "gpu_launches": int(rr[8]), "clocks": clocks,
                "latency_us": {"device": {"q%d" % q: round(float(dev_mean[i]), 2) for i, q in enumerate(QUERIES)},
                               "wall": {"q%d" % q: round(float(wall_mean[i]), 2) for i, q in enumerate(QUERIES)},
                               "e2e": {"q%d" % q: round(float(e2e_mean[i]), 2) for i, q in enumerate(QUERIES)},
                               "device_median": {"q%d" % q: round(float(outl[7 + i]), 2) for i, q in enumerate(QUERIES)},
                               "samples_over_3x_median": {"q%d" % q: int(outl[i]) for i, q in enumerate(QUERIES)}},
                "light_path": {"resident_servers": {"q%d" % q: bool(res[i] > 0) for i, q in enumerate(QUERIES)},
                               "per_rank": {"q%d" % q: {"wall_us": [round(float(x), 2) for x in per_rank[:, j]],
                                                        "server_us": [round(float(x), 2) for x in per_rank[:, len(LIGHT) + j]]}
                                            for j, q in enumerate(LIGHT)},
                               "note": "in-place plans: the constant's owner walks the shards through peer loads, the other ranks wait for its "
                                       "verdict; server_us = in-kernel span of that rank's server request (0: launch path)"},
                "rows": {"q%d" % q: int(rr[i]) for i, q in enumerate(QUERIES)},
                "comm": {"rows_pushed_all_ranks": int(rr[7]), "bytes_pushed_all_ranks": int(rr[9]),
                         "bytes_pushed_per_step_all_ranks": int(rr[9] // max(1, args.steps)),
                         "exchanges_per_rank": int(nx), "nvlink": exch},
                "steps_table": steps_table,
                "dataset": {"shard_triples_rank0": shard_triples, "gen_build_s": round(t1 - t0, 1), "build": binfo.get("build_ms")},
                "timed_region_s": round(t_region, 2)}
    return line


def run_single(args, rank, world, local_rank, dist, cpu_arm=True):
    """one GPU per rank, the whole store on each (N = 1, or replicas at N > 1).  Returns the line on rank 0."""
    from wukong_b200 import capi, host
    from oracle import ref as REF
    hs = None
    if args.store_build == "device":
        tr, gst, info = build_dataset_device(args, local_rank)
    else:
        tr, hs, info = build_dataset(args)
        gst = hs.upload(local_rank)
    del tr
    plans = load_plans(args.plan)
    rbuf = (args.rbuf_mb << 20) if args.rbuf_mb else max(256 << 20, min(8 << 30, int(info["triples"]) * 8))
    eng = capi.Engine(gst, rbuf_bytes=rbuf)
    out_tbl, _keep = capi.pinned_array(min(rbuf // 4, 1 << 28))

    def barrier():
        eng.sync()
        if dist is not None:
            import torch
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    # ---- warm-up ---------------------------------------------------------------------------------
    rows = {}
    for _ in range(args.warmup):
        for q in QUERIES:
            pats, nvars, req = plans[q]
            _, _, r, c = host.time_query(eng, pats, nvars, req, 1, blind=False, table=out_tbl, flush=True)
            rows[q] = (r, c)
    launches0 = eng.launch_count()
    barrier()
    t_region0 = time.time()
    sampler.t_mark = t_region0
    # ---- timed: device-resident (value) and end-to-end (e2e), K steps, L2 flushed between queries ----
    dev_us = {q: [] for q in QUERIES}      # CUDA events (launch paths) or the server's in-kernel span (resident light queries)
    blind_wall_us = {q: [] for q in QUERIES}
    e2e_us = {q: [] for q in QUERIES}
    resident = {}
    blind_rows = {}
    eng.set_profiling(1)
    for _ in range(args.steps):
        for q in QUERIES:
            pats, nvars, req = plans[q]
            w, d, blind_rows[q], _ = host.time_query(eng, pats, nvars, req, 1, blind=True, flush=True, device_times=True)
            dev_us[q].append(float(d[0]))
            blind_wall_us[q].append(float(w[0]))
            resident[q] = bool(eng.get_option(capi.WK_INFO_LAST_RESIDENT))
    eng.set_profiling(0)
    dump = args.dump_outputs if rank == 0 else ""
    tables = {}
    for step in range(args.steps):
        for q in QUERIES:
            pats, nvars, req = plans[q]
            w, _, r, c = host.time_query(eng, pats, nvars, req, 1, blind=False, table=out_tbl, flush=True)
            e2e_us[q].append(float(w[0]))
            if dump and step == args.steps - 1:     # the next query overwrites out_tbl; its clock starts after this copy
                tables[q] = out_tbl[: r * c].reshape(r, c).copy()
    barrier()
    t_region = time.time() - t_region0
    clocks = sampler.stop()
    launches = eng.launch_count() - launches0
    if dump:
        dump_outputs(dump, tables, blind_rows)

    # ---- the tables themselves (not only their sizes): digest of every query's non-blind result -----------------
    digests = {}
    for q in QUERIES:
        pats, nvars, req = plans[q]
        rc, r, c, tbl = eng.query(pats, nvars, req, out=out_tbl)
        assert rc == 0 and r == rows[q][0]
        digests[q] = REF.table_digest(tbl) if r else 0

    # ---- roofline of the dominant kernel (per-step CUDA events; separate pass) ---------------------------
    eng.set_profiling(2)
    agg = {}
    for _ in range(max(3, min(args.steps, 10))):
        for q in QUERIES:
            pats, nvars, req = plans[q]
            eng.flush_l2()
            rc, _, _, _ = eng.query(pats, nvars, req, blind=True)
            assert rc == 0
            for i, sst in enumerate(eng.step_stats()):
                a = agg.setdefault((q, i, sst["kind"]), {"us": [], "bytes": sst["algo_bytes"], "in_rows": sst["in_rows"],
                                                         "out_rows": sst["out_rows"], "in_cols": sst["in_cols"]})
                a["us"].append(sst["device_us"])
    eng.set_profiling(0)
    kern = [(k, v) for k, v in agg.items() if k[2] in ("k2u", "k2k", "k2c", "filter") and np.mean(v["us"]) > 0]
    roof = None
    roof_expand = None
    steps_table = []
    for k, v in sorted(agg.items()):
        us = float(np.mean(v["us"])) if v["us"] else 0.0
        steps_table.append({"q": k[0], "step": k[1], "kind": k[2], "in_rows": int(v["in_rows"]), "out_rows": int(v["out_rows"]),
                            "algo_bytes": int(v["bytes"]), "device_us": round(us, 2),
                            "gbs": round(v["bytes"] / us / 1e3, 1) if us > 0 else None})
    if kern:
        (kq, ki, kk), v = max(kern, key=lambda kv: float(np.mean(kv[1]["us"])))
        peak, peak_src = peak_hbm()

        def roof_of(kq, ki, kk, v):
            us = float(np.mean(v["us"]))
            ach = v["bytes"] / us / 1e3   # GB/s
            tr_ = ncu_traffic(args, kq, ki, kk)
            return {"bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                    "traffic": int(tr_) if tr_ else None,
                    "kernel": "%s (q%d step %d: %d rows x %d cols -> %d rows)" % (kk, kq, ki, v["in_rows"], v["in_cols"], v["out_rows"]),
                    "algo_bytes_per_launch": int(v["bytes"]), "us_per_launch": round(us, 2), "peak_source": peak_src}
        roof = roof_of(kq, ki, kk, v)
        if roof["traffic"] is not None and roof["traffic"] < 0.5 * roof["algo_bytes_per_launch"]:
            roof["note"] = "this step probes a few thousand hot keys: most algorithmic bytes are L2 hits, not DRAM traffic"
        # the expand (known_to_unknown) launch with the largest device time: north_star's "expand-kernel HBM GB/s"
        k2u = [(k, v2) for k, v2 in kern if k[2] == "k2u"]
        if k2u:
            (eq, ei, ek), ev = max(k2u, key=lambda kv: float(np.mean(kv[1]["us"])))
            roof_expand = roof_of(eq, ei, ek, ev)

    # ---- reduce over ranks (max latency), compute the metric ----------------------------------------------------
    # value term per query: CUDA-event time, except for light queries answered by the resident server (no launch to bracket):
    # the host wall clock of the blind call, which contains the doorbell and the reply crossing PCIe
    val_us = np.array([np.mean(blind_wall_us[q]) if resident.get(q) else np.mean(dev_us[q]) for q in QUERIES])
    e2e_mean = np.array([np.mean(e2e_us[q]) for q in QUERIES])
    if dist is not None:
        import torch
        t = torch.tensor(np.concatenate([val_us, e2e_mean]), device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        arr = t.cpu().numpy()
        val_us, e2e_mean = arr[:7], arr[7:]
    # replicas: every rank answers its own stream of queries => whole-job rate = world x per-replica rate
    value = geomean(world * 1e6 / val_us)
    e2e = geomean(world * 1e6 / e2e_mean)
    d2h = sum(rows[q][0] * rows[q][1] * 4 + 32 for q in QUERIES)
    h2d = sum((448 if resident.get(q) else len(plans[q][0]) * 16 + len(plans[q][2]) * 4) for q in QUERIES)

    line = {"metric": "lubm_q1_q7_geomean_queries_per_sec", "value": value, "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(val_us.sum() / 1e3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": vs_published(value, args), "dtype": "u32", "data": "synthetic",
            "config": {"workload": workload_name(args, world, False),
                       "triples": info["triples"], "keys": info["keys"], "store_mb": info["header_mb"] + info["edges_mb"],
                       "parallelism": "replicas x%d" % world if world > 1 else "single GPU",
                       "l2": "flushed before every timed query (384 MB memset + 256 MB read-back, outside the timed region)",
                       "value_mode": "blind (row count only), device-resident; CUDA events, except light queries answered by the resident "
                                     "server kernel: host wall clock of the blind call",
                       "e2e_mode": "non-blind, table D2H into pinned memory, host wall clock"},
            "e2e": {"value": e2e, "unit": "queries/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "roofline_expand": roof_expand,
            "latency_us": {"value_term": {"q%d" % q: round(float(val_us[i]), 2) for i, q in enumerate(QUERIES)},
                           "device": {"q%d" % q: round(float(np.mean(dev_us[q])), 2) for q in QUERIES},
                           "blind_wall": {"q%d" % q: round(float(np.mean(blind_wall_us[q])), 2) for q in QUERIES},
                           "e2e": {"q%d" % q: round(float(e2e_mean[i]), 2) for i, q in enumerate(QUERIES)}},
            "light_path": {"resident_server": {"q%d" % q: bool(resident.get(q)) for q in QUERIES},
                           "note": "device = in-kernel %globaltimer span (request acquired -> record stored) for resident queries"},
            "rows": {"q%d" % q: int(rows[q][0]) for q in QUERIES}, "steps_table": steps_table,
            "dataset": info, "timed_region_s": round(t_region, 2)}
    if rank == 0 and cpu_arm and not args.no_cpu_baseline:
        cpus = host_cpus()
        threads = args.cpu_threads or cpus["usable"]
        kind = cpu_engine_kind(args)
        cpu = CpuEngine(hs if hs is not None else DeviceBuiltStore(gst), kind)
        res = cpu.times(plans, threads, 3, 200, digest=True)
        for q in QUERIES:
            assert res[q]["rows"] == rows[q][0], "GPU and CPU engine disagree on q%d rows: %d vs %d" % (q, rows[q][0], res[q]["rows"])
            assert res[q]["digest"] == digests[q], "GPU and CPU engine disagree on the CONTENT of q%d's table" % q
        line["parity"] = {"checked": "order-independent 64-bit digest (sum over rows of a mix of the row's words) of every query's "
                                     "non-blind table, GPU engine vs CPU arm, at full scale", "queries": len(QUERIES), "match": True,
                          "digests": {"q%d" % q: "%016x" % digests[q] for q in QUERIES}}
        line["cpu_baseline"] = {"value": geomean([1e6 / res[q]["blind_us"] for q in QUERIES]), "unit": "queries/s", "cores": threads,
                                "kind": kind, "host_cpus": cpus, "mt_factor": {"q%d" % q: m for q, m in cpu.best_mt.items()},
                                "e2e_value": geomean([1e6 / res[q]["non_blind_us"] for q in QUERIES]),
                                "sample": cpu_sample_note(threads, cpu.best_mt, kind, 3, 200),
                                "latency_us": {"blind": {"q%d" % q: round(res[q]["blind_us"], 2) for q in QUERIES},
                                               "non_blind": {"q%d" % q: round(res[q]["non_blind_us"], 2) for q in QUERIES}}}
    eng.close()
    gst.close()
    return line if rank == 0 else None


DUMP_BYTES = 64 * 10**6


def dump_outputs(d, tables, rows):
    """--dump-outputs: what the end-to-end path handed back in the last timed step, so that two builds can be compared output
    for output.  DIR/q<N>.npy is query N's result table as float64 (exact for every 32-bit id) with its rows in lexicographic
    order (the engine returns them in no fixed order); a query without an answer has no file.  DIR/rows.npy holds the row
    counts of Q1..Q7.  Should the tables exceed 64 MB in all, each keeps the same fraction of its sorted rows (at least one),
    drawn with a fixed seed."""
    import sparql_mini as M
    os.makedirs(d, exist_ok=True)
    total = 8 * sum(t.size for t in tables.values())
    frac = min(1.0, (DUMP_BYTES - 4096 * (len(tables) + 1)) / total) if total else 1.0
    for q, t in sorted(tables.items()):
        if t.size == 0:
            continue
        t = M.sort_rows(t)
        if frac < 1.0:
            keep = max(1, int(t.shape[0] * frac))
            t = t[np.sort(np.random.default_rng(q).choice(t.shape[0], keep, replace=False))]
        np.save(os.path.join(d, "q%d.npy" % q), t.astype(np.float64))
    np.save(os.path.join(d, "rows.npy"), np.array([rows[q] for q in QUERIES], dtype=np.float64))


def ncu_traffic(args, q, step, kind):
    """DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum) of this launch from the committed ncu --set full
    capture of the same command (profiles/ncu_traffic.json, see profiles/README.md); None when no capture of this workload /
    kernel is committed"""
    try:
        tab = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        key = "lubm%d_%s" % (args.scale, args.plan)
        return tab.get(key, {}).get("q%d_step%d_%s" % (q, step, kind))
    except Exception:
        return None


_RESULT_FD = None


def claim_stdout():
    """Libraries (NCCL prints its version banner) write to fd 1; the contract is ONE JSON line on stdout.
    Point fd 1 at stderr for the whole run and keep the real stdout for the result line."""
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    import faulthandler
    faulthandler.enable()     # a crash in native code leaves the Python stack on stderr
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="wukong_b200")
    ap.add_argument("--scale", type=int, default=0, help="number of universities (LUBM-<scale>); default 2560 (10240 for N > 1 sharded)")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--plan", default="", help="plan set; default osdi16_plan (optimal10240_plan for N > 1 sharded)")
    ap.add_argument("--rbuf-mb", type=int, default=0)
    ap.add_argument("--cpu-threads", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-engine", default="auto", choices=["auto", "reference", "port"],
                    help="CPU arm: the reference's own engine compiled in oracle/_ref, or the oracle port (auto: reference when built)")
    ap.add_argument("--store-build", default="device", choices=["device", "host"],
                    help="build the graph store on the GPU (wk_store_build) or with the host builder + upload")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "nccl"], help="sharded mode: peer-memory push or NCCL all-to-all(v)")
    ap.add_argument("--mode", default="auto", choices=["auto", "replicas", "sharded"],
                    help="N>1: sharded (vid %% N, exchange over NVLink; the default) or replicas (whole store per GPU, weak scaling)")
    ap.add_argument("--no-secondary", action="store_true", help="N>1 sharded: skip the single-GPU run of the same store and the replicas run")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the result tables of the last end-to-end step as DIR/q<N>.npy (float64, rows "
                         "sorted; no file for a query without an answer) and the row counts as DIR/rows.npy; one GPU or replicas only")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.mode == "auto":
        args.mode = "sharded" if args.gpus > 1 else "replicas"
    sharded = args.gpus > 1 and args.mode == "sharded"
    if args.dump_outputs and (sharded or args.impl == "reference"):
        ap.error("--dump-outputs writes the GPU path's tables of one GPU or of replicas, not of the sharded mode or the reference arm")
    if not args.scale:
        args.scale = 10240 if sharded else 2560     # BASELINE configs 4 and 3
    if not args.plan:
        args.plan = "optimal10240_plan" if sharded else "osdi16_plan"
    if world > 1:   # torchrun pins OMP_NUM_THREADS=1; the host-side store build is OpenMP-parallel
        os.environ["OMP_NUM_THREADS"] = str(max(1, (os.cpu_count() or 1) // world))

    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    from wukong_b200 import capi
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
        if rank != 0:
            ge.build()   # libraries exist by now; loads them
    if capi.device_count() < 1:
        raise RuntimeError("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")

    if world > 1 and args.mode == "sharded":
        line = run_sharded(args, rank, world, local_rank, dist)
        if not args.no_secondary:
            # (a) the same store on ONE GPU (rank 0): the strong-scaling denominator; (b) replicas of BASELINE config 3
            import copy
            sec = {}
            try:
                single = None
                if rank == 0:
                    single = run_single(args, 0, 1, local_rank, None, cpu_arm=False)
                if rank == 0 and single:
                    sec["single_gpu_same_store"] = {"value": single["value"], "latency_us": single["latency_us"]["value_term"],
                                                    "rows": single["rows"], "config": single["config"]["workload"]}
            except Exception as ex:   # noqa: BLE001
                sec["single_gpu_same_store"] = {"error": repr(ex)[:300]}
            dist.barrier()
            try:
                a2 = copy.copy(args)
                a2.scale, a2.plan, a2.mode = 2560, "osdi16_plan", "replicas"
                rep = run_single(a2, rank, world, local_rank, dist, cpu_arm=False)
                if rank == 0 and rep:
                    sec["replicas"] = {"value": rep["value"], "e2e": rep["e2e"]["value"], "config": rep["config"]["workload"],
                                       "parallelism": rep["config"]["parallelism"], "latency_us": rep["latency_us"]["value_term"]}
            except Exception as ex:   # noqa: BLE001
                sec["replicas"] = {"error": repr(ex)[:300]}
            if rank == 0:
                line["secondary"] = sec
        if rank == 0:
            emit(line)
        dist.barrier()
        dist.destroy_process_group()
        return
    line = run_single(args, rank, world, local_rank, dist)
    if rank == 0:
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
