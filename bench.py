#!/usr/bin/env python
"""bench.py — the reference's headline metric on B200: simulated-ms/sec (and msgs/sec) of
GSFSignature, 131 072 nodes (BASELINE.json), through the C ABI of wittgenstein_b200.

A "step" is one `network.runMs(STEP_MS)` window of one continuing simulation (the reference drives
its runs the same way: ProgressPerTime.java:79-95 calls runMs in a loop).  W warm-up steps, then
exactly K timed steps:
  value  = K*STEP_MS / device time (CUDA events on the engine's stream; max over ranks)
  e2e    = same metric through the public API with host buffers: every step also reads back what the
           reference's callers read after each runMs (per-node signature count + the 5 node counters)
           and writes/reads the control block — a fresh, identically seeded network, wall clock.
  roofline: dominant kernel of the timed region (per-kernel CUDA-event timing in a third identical
           pass), algorithmic bytes / its time, against MEASURED_PEAKS.json.
  cpu_baseline: the CPU oracle (C++ restatement of the reference engine, 1 thread like the reference)
           on a bounded sample of the same workload.
--impl reference times the reference's CPU path (the oracle port; the Java reference cannot run here:
no JVM) on the host cores with the same step definition.
--dump-outputs DIR writes the state the timed network holds after its last step (what a caller reads back) as .npy files,
so that two builds can be compared output for output on identical, seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

AWS_NB, AWS_NL = "AWS_SPEED=GAUSSIAN_TOR=0.33", "AwsRegionNetworkLatency"


def gsf_params(n):
    # GSFSignature.newProtocol() ratios (GSFSignature.java:684-697): threshold .85, dead .10, pairing 4,
    # level timeout 50, period 20, 10 accelerated calls, AWS regions + uniform speed + 33 % Tor
    return dict(node_count=n, threshold=int(0.85 * n), pairing_time=4, timeout_per_level_ms=50, period_duration_ms=20,
                accelerated_calls_count=10, nodes_down=int(0.10 * n), node_builder_name=AWS_NB, network_latency_name=AWS_NL)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        import statistics

        sm = [int(r[0]) for r in self.rows if r and r[0].isdigit()]
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def metric_name(n):
    return f"simulated-ms/sec, GSFSignature {n:,} nodes"


def workload_name(n):
    return (f"GSFSignature {n} nodes, threshold {int(.85*n)}, {int(.1*n)} dead, pairing 4, level timeout 50, period 20, "
            f"10 accelerated calls, {AWS_NB}, {AWS_NL}, seed 0")


def host_info():
    model = "unknown"
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                model = ln.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"cpu_model": model, "cores_total": os.cpu_count()}


SHARD = None  # (dist, rank, world, local) when the ranks of this job are node-id shards of ONE simulation


def make_gsf(n, seed):
    from wittgenstein_b200 import GSFSignature, GSFSignatureParameters

    if SHARD is not None:
        from wittgenstein_b200.sharded import DistributedGSFSignature

        dist, rank, world, local = SHARD
        p = DistributedGSFSignature(GSFSignatureParameters(**gsf_params(n)), dist, rank, world, local)
    else:
        p = GSFSignature(GSFSignatureParameters(**gsf_params(n)))
    p.network().set_seed(seed)
    t0 = time.time()
    p.init()
    p.network().msgs_size()  # sync
    return p, time.time() - t0


def state_digests(p, lo=None, hi=None):
    """blake2b digests of a protocol object's state (rows [lo, hi) of an oracle / unsharded object; all rows of a shard)"""
    import hashlib

    import numpy as np

    def dg(a):
        a = np.ascontiguousarray(a if lo is None else a[lo:hi])
        return hashlib.blake2b(a.tobytes(), digest_size=16).hexdigest()

    net = p if hasattr(p, "counters") else p.network()
    cnt = net.counters()
    out = {"counters": dg(cnt.T)}
    for k, v in p.scalars().items():
        out["scalar_" + k] = dg(v)
    out["verified"] = dg(p.verified())
    rows = p.level_rows if hasattr(p, "level_rows") else p.rows
    out["rows1"] = dg(rows(1))
    out["rows2"] = dg(rows(2))
    for k, v in p.level_scalars().items():
        out["level_" + k] = dg(v)
    return out


DUMP_LIMIT_BYTES = 64 << 20


def gsf_outputs(p):
    """What a caller reads back after runMs on a GSFSignature object (engine, shard or oracle): the per-node scalars, the 5
    node counters and a fixed, seeded sample of verifiedSignatures rows (the whole bitmap is N^2/8 bytes), each row as its
    32-bit words so that float64 holds them exactly."""
    import numpy as np

    q = getattr(p, "local", p)
    net = q if hasattr(q, "counters") else q.network()
    out = {"scalar_" + k: v for k, v in q.scalars().items()}
    out["counters"] = net.counters()
    ver = q.verified()
    rows = max(1, min(256, len(ver), (16 << 20) // (ver.shape[1] * 2 * 8)))
    idx = np.sort(np.random.default_rng(0).choice(len(ver), rows, replace=False))
    out["verified_sample_rows"] = idx
    out["verified_sample"] = np.ascontiguousarray(ver[idx]).view(np.uint32)
    return out


def casper_outputs(p):
    """What a caller reads back after runMs on a CasperIMD object (engine, shard or oracle): node state (the 64-bit
    attestation hash as its 32-bit words) and the 5 node counters."""
    import numpy as np

    q = getattr(p, "local", p)
    net = q if hasattr(q, "counters") else q.network()
    out = {"node_" + k: v for k, v in q.node_state().items()}
    out["node_att_hash"] = out["node_att_hash"].view(np.uint32).reshape(-1, 2)
    out["counters"] = net.counters()
    return out


def dump_outputs(d, arrays):
    """--dump-outputs: each array as <d>/<name>.npy in float64 (exact for the engine's integer state)."""
    import numpy as np

    total = sum(a.size * 8 for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(d, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(d, k + ".npy"), np.asarray(a, np.float64))


def event_counts(st0, st1):
    return {k: st1[k] - st0[k] for k in ("deliveries", "tasks", "cond_runs", "draws", "eval_entries", "eval_words", "updates",
                                         "cycles", "sends", "multi_sends", "send_words", "events", "update_words", "reevaluated")}


def algorithmic_bytes(ev):
    """DESIGN.md §6: minimal traffic per event type of this engine's layout (bytes)."""
    b = {}
    b["k_cond_scan"] = 20 * ev["eval_entries"] + 24 * ev["reevaluated"] + 64 * ev["cond_runs"]   # entry + stamp; re-scored: counters + 2 row words
    b["k_cond_score"] = 8 * ev["eval_words"]                                                  # payload, verified, indivVerified blocks
    b["k_cond_select"] = 4 * ev["eval_entries"] + 24 * ev["eval_entries"] // 2 + 64 * ev["cond_runs"]  # scores; about half the entries move
    b["k_node"] = (96 * ev["deliveries"] + 8 * (ev["send_words"] + ev["update_words"]) + 48 * (ev["sends"] + ev["multi_sends"])
                   + 128 * ev["updates"] + 64 * ev["cycles"])
    b["k_emit"] = (48 + 32 + 4) * (ev["sends"] + ev["multi_sends"] + ev["cycles"] + ev["cond_runs"])
    b["k_ms_scatter"] = (32 + 32 + 4) * (ev["sends"] + ev["multi_sends"] + ev["cycles"] + ev["cond_runs"])
    return b


def cpu_baseline_and_parity(n, args):
    """Oracle over the first windows of the run (bounded CPU time), then the GPU over exactly the same windows with
    the same runMs slicing, then a bit-exact comparison of the two states (time, rd state, msgs.size(), the 5 node
    counters, per-node scalars, verifiedSignatures and the per-level rows and scalars).  Node-sharded job: rank 0 runs the
    oracle, every rank runs its shard over the window and reports digests of its rows; rank 0 compares them with the
    digests of the oracle's corresponding rows."""
    from tests import parity as par

    rank = SHARD[1] if SHARD is not None else 0
    o, cpu, sim, step = None, None, 0, 10
    if rank == 0:
        from tests.oracle_lib import OracleGSF

        n_cpu = feasible_cpu_nodes(min(args.cpu_nodes, n), args.cpu_max_nodes)
        g = gsf_params(n_cpu)
        o = OracleGSF(n_cpu, g["threshold"], 4, 50, 20, 10, g["nodes_down"], AWS_NB, AWS_NL)
        t0 = time.time()
        o.init_fast(min(64, os.cpu_count() or 1))  # init is threaded (and untimed); runMs below is single-threaded
        init_s = time.time() - t0
        wall = 0.0
        st0 = o.stats()
        while wall < args.cpu_budget_s and sim < 4000:
            wall += o.run_timed(step, 1)
            sim += step
        st1 = o.stats()
        msgs = (st1["deliveries"] - st0["deliveries"]) + (st1["tasks"] - st0["tasks"]) + (st1["cond_runs"] - st0["cond_runs"])
        cpu = {"value": sim / wall, "unit": "simulated-ms/s", "cores": 1, "kind": "port",
               "sample": f"oracle (C++ restatement, 1 thread), GSFSignature {n_cpu} nodes, first {sim} simulated ms in {wall:.1f} s "
                         f"(init {init_s:.1f} s excluded)", "msgs_per_s": msgs / wall, "nodes": n_cpu, "sim_ms": sim, "host": host_info()}
        if n_cpu != n:
            cpu["note"] = f"host memory too small for the oracle at {n} nodes: ran {n_cpu}; no parity check at the metric size"
            sim = 0
    if SHARD is not None:
        box = [sim]
        SHARD[0].broadcast_object_list(box, src=0)
        sim = box[0]
    if sim == 0:
        return cpu, None
    p, _ = make_gsf(n, 0)
    net = p.network()
    net.timer_start()
    for _ in range(sim // step):
        net.run_ms(step)
    pm = net.timer_stop_ms()
    parity = None
    if SHARD is None:
        cpu["gpu_same_window"] = {"value": sim / (pm / 1000.0), "unit": "simulated-ms/s",
                                  "window": f"[0,{sim}] ms, runMs({step}) slicing, device-timed"}
        bad = par.compare_gsf(p, o, f"t={sim}", full=True)
    else:
        dist, _, world, _ = SHARD
        mine = {"range": net.shard_range(), "time": net.time, "rng": net.rng_state(), "msgs": net.msgs_size(), "ms": pm,
                "digests": state_digests(p.local)}
        allr = [None] * world
        dist.all_gather_object(allr, mine)
        bad = []
        if rank == 0:
            cpu["gpu_same_window"] = {"value": sim / (max(r["ms"] for r in allr) / 1000.0), "unit": "simulated-ms/s",
                                      "window": f"[0,{sim}] ms, runMs({step}) slicing, device-timed, max over shards"}
            if sum(r["msgs"] for r in allr) != o.msgs_live():
                bad.append(f"msgs.size() {sum(r['msgs'] for r in allr)} vs {o.msgs_live()}")
            for q, r in enumerate(allr):
                if r["time"] != o.time or r["rng"] != o.rng_state():
                    bad.append(f"shard {q}: time / rd state differ")
                n0, nl = r["range"]
                want = state_digests(o, n0, n0 + nl)
                bad += [f"shard {q}: {k} differs" for k in want if want[k] != r["digests"][k]]
    if rank == 0:
        parity = {"nodes": n, "t": sim, "slicing": f"runMs({step})", "status": "bit-exact" if not bad else "MISMATCH",
                  "compared": "time, rd state, msgs.size(), 5 node counters, node scalars, verifiedSignatures, level rows + scalars"
                              + (" (per shard, as digests)" if SHARD is not None else "")}
        if bad:
            parity["mismatches"] = bad[:8]
    del p, net
    return cpu, parity


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed ncu capture
    (profiles/r02_traffic.json, written by scripts/ncu_traffic.py from an `ncu --set full` page); None if absent."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        return t.get(kernel, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


def feasible_cpu_nodes(n, cap):
    """largest power-of-two node count <= n whose oracle state (peer tables: 4 N^2 bytes) fits in host RAM"""
    import psutil

    avail = psutil.virtual_memory().available
    while n > 1024 and (n * n * 4 * 1.5 > avail * 0.7 or n > cap):
        n //= 2
    return n


def run_reference(args):
    """--impl reference: the reference's CPU path.  The Java engine cannot run here (no JVM/gradle/jars:
    SURVEY.md §8c), so this times the oracle port with the same step definition on a bounded sample."""
    n = args.nodes
    n = feasible_cpu_nodes(n, args.cpu_max_nodes)
    from tests.oracle_lib import OracleGSF

    g = gsf_params(n)
    o = OracleGSF(n, g["threshold"], 4, 50, 20, 10, g["nodes_down"], AWS_NB, AWS_NL)
    o.init_fast(min(64, os.cpu_count() or 1))
    step_ms = args.ref_step_ms
    w = OracleGSF(1024, 870, 4, 50, 20, 10, 102, AWS_NB, AWS_NL)  # warm-up steps on a throw-away small network
    w.init()
    for _ in range(args.warmup):
        w.run_timed(step_ms, 1)
    del w
    wall = o.run_timed(step_ms, args.steps)
    val = args.steps * step_ms / wall
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, gsf_outputs(o))
    line = {"impl": "reference", "metric": metric_name(args.nodes), "value": val, "unit": "simulated-ms/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000 * wall / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u64 bitmaps / int32", "data": "synthetic",
            "config": {"workload": workload_name(args.nodes),
                       "sample": f"{n} nodes; step = runMs({step_ms}) of one run from t=0, timed window [0,{args.steps*step_ms}] ms "
                                 "(the cheapest part of the run for the CPU engine: its cost per tick grows with the queues); the b200 "
                                 "arm reports the same window as e2e_same_window_as_reference",
                       "host": host_info(),
                       "note": "reference = C++ oracle port, 1 thread (the reference engine is single-threaded: Network.java:10); "
                               "Java reference not runnable here (no JVM)"},
            "cpu_baseline": {"value": val, "unit": "simulated-ms/s", "cores": 1, "kind": "port",
                             "sample": f"{args.steps} x runMs({step_ms}) from t=0 at {n} nodes (init threaded and untimed)"},
            "e2e": {"value": val, "unit": "simulated-ms/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


CASPER_NB, CASPER_NL = "RANDOM_SPEED=CONSTANT_TOR=0.00", "NetworkLatencyByDistanceWJitter"


def casper_cfg():
    # SURVEY.md §8d config #4: CasperParemeters(64, false, 5, 256, 1000, 1, RANDOM builder, ByDistanceWJitter) -> 16 390 nodes
    return dict(cycle_length=64, random_on_ties=False, block_producers_count=5, attesters_per_round=256,
                block_construction_time=1000, attestation_construction_time=1, node_builder_name=CASPER_NB,
                network_latency_name=CASPER_NL)


def casper_oracle():
    from tests.oracle_lib import OracleCasper

    c = casper_cfg()
    o = OracleCasper(c["cycle_length"], False, c["block_producers_count"], c["attesters_per_round"], 1000, 1, CASPER_NB, CASPER_NL)
    o.init(0)
    return o


def casper_workload(K, W):
    return (f"CasperIMD 16390 nodes (64-slot cycles, 5 producers incl. ByzBlockProducerWF(0), 256 attesters per slot), {CASPER_NB}, "
            f"{CASPER_NL}; step = runMs(8000) = one slot of one run; {W} warm-up slots then {K} timed slots of the same network")


def run_casper_reference(args):
    o = casper_oracle()
    K, W = args.steps, args.warmup
    for _ in range(W):
        o.run_ms(8000)
    d0 = o.deliveries()
    wall = o.run_timed(8000 * K, 8000)
    val = 8000 * K / wall
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, casper_outputs(o))
    print(json.dumps({"impl": "reference", "metric": "simulated-ms/sec, CasperIMD 16,390 nodes", "value": val, "unit": "simulated-ms/s",
                      "n_gpus": args.gpus, "steps": K, "warmup": W, "ms_per_step": 1000 * wall / K, "higher_is_better": True,
                      "scaling": "weak", "vs_baseline": None, "dtype": "u64 bitmaps / int32", "data": "synthetic",
                      "config": {"workload": casper_workload(K, W), "note": "reference = C++ oracle port, 1 thread; Java reference not runnable here (no JVM)"},
                      "msgs_per_s": (o.deliveries() - d0) / wall,
                      "cpu_baseline": {"value": val, "unit": "simulated-ms/s", "cores": 1, "kind": "port", "sample": f"slots {W}..{W+K} of the run"},
                      "e2e": {"value": val, "unit": "simulated-ms/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def run_casper(args, rank, world, local, dist, barrier, max_over_ranks, sum_over_ranks):
    """--workload casper: SURVEY.md §8d config #4 on the device engine.  N > 1: ONE simulation, node ids sharded over the ranks'
    GPUs (BASELINE config #4: "node-sharded across 4xB200"; `--mode replicas`: independent seeds instead)."""
    import torch

    from wittgenstein_b200 import CasperIMD, CasperParemeters

    K, W = args.steps, args.warmup
    sharded = world > 1 and args.mode != "replicas"
    if sharded:
        sum_over_ranks_job = sum_over_ranks
        sum_over_ranks = lambda x: x  # noqa: E731  one run: its simulated time is not multiplied by the ranks

    def make():
        if sharded:
            from wittgenstein_b200.sharded import DistributedCasperIMD

            p = DistributedCasperIMD(CasperParemeters(**casper_cfg()), dist, rank, world, local, tunables={"casper_votes": (K + W) // 64 + 3})
            p.init(0)
            return p
        p = CasperIMD(CasperParemeters(**casper_cfg()))
        p.network().set_seed(rank)
        p.network().set_tunable("casper_votes", (K + W) // 64 + 3)
        p.init(0)
        return p

    # pass 1: device-timed
    p = make()
    net = p.network()
    for _ in range(W):
        net.run_ms(8000)
    st0 = net.stats()
    sampler = ClockSampler(local)
    barrier()
    torch.cuda.synchronize()
    sampler.start()
    net.timer_start()
    for _ in range(K):
        net.run_ms(8000)
    dev_ms = max_over_ranks(net.timer_stop_ms())
    torch.cuda.synchronize()
    barrier()
    sampler.stop_flag = True
    st1 = net.stats()
    heads_end = p.heads()
    nblocks = len(p.blocks()["height"])
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, casper_outputs(p))
    del p, net
    # pass 2: end to end with the read-backs a caller makes after every slot (heads + the five node counters)
    p = make()
    net = p.network()
    for _ in range(W):
        net.run_ms(8000)
    barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    d2h = 0
    for _ in range(K):
        net.run_ms(8000)
        heads = p.heads()
        cnt = net.counters()
        d2h = heads.nbytes + cnt.nbytes
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    assert (heads == heads_end).all(), "e2e pass diverged from the device-timed pass"
    del p, net
    # pass 3: per-kernel timing
    prof = {}
    if not args.no_profile:
        p = make()
        net = p.network()
        for _ in range(W):
            net.run_ms(8000)
        net.profile_enable(True)
        for _ in range(K):
            net.run_ms(8000)
        prof = net.profile_read()
        net.profile_enable(False)
        del p, net
    cpu = None
    if rank == 0 and not args.no_cpu:
        o = casper_oracle()
        t1 = time.time()
        wall = o.run_timed(8000 * 6, 8000)
        cpu = {"value": 48000 / wall, "unit": "simulated-ms/s", "cores": 1, "kind": "port",
               "sample": f"oracle (C++ restatement, 1 thread), same configuration, slots 0..6 ({o.deliveries()} deliveries) in {wall:.1f} s",
               "msgs_per_s": o.deliveries() / wall}
        del o
    deliveries = st1["deliveries"] - st0["deliveries"]
    tasks = st1["tasks"] - st0["tasks"]
    parity_unsharded = None
    if sharded:  # every shard's heads against the unsharded engine on the same slots (which the -m gpu tests pin on the oracle)
        deliveries, tasks = sum_over_ranks_job(deliveries), sum_over_ranks_job(tasks)
        ps = make()
        for _ in range(W + K):
            ps.network().run_ms(8000)
        got = ps.all_heads()
        nb_sh = len(ps.blocks()["height"])
        del ps
        if rank == 0:
            pu = CasperIMD(CasperParemeters(**casper_cfg()))
            pu.network().set_tunable("casper_votes", (K + W) // 64 + 3)
            pu.init(0)
            for _ in range(W + K):
                pu.network().run_ms(8000)
            parity_unsharded = bool((pu.heads() == got).all() and len(pu.blocks()["height"]) == nb_sh)
            del pu
    value = sum_over_ranks(K * 8000) / (dev_ms / 1000.0)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    line = {"metric": "simulated-ms/sec, CasperIMD 16,390 nodes", "value": value, "unit": "simulated-ms/s", "n_gpus": world, "steps": K,
            "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True, "scaling": "strong" if sharded else "weak", "vs_baseline": None,
            "dtype": "u64 bitmaps / int32", "data": "synthetic",
            "config": {"workload": casper_workload(K, W),
                       "parallelism": "1 GPU" if world == 1 else (f"node-sharded: ONE simulation, {world} contiguous ranges of node ids, replicated block / attestation "
                                                                  "tables, per-pass exchanges as peer stores over NVLink" if sharded else f"{world} independent seeded replicas"),
                       "l2": "launch-bound: ~340 non-empty milliseconds per slot, ~12 k deliveries each; working set (attestation bitmaps 200 MB) exceeds L2",
                       "blocks_at_end": nblocks},
            "msgs_per_s": sum_over_ranks(deliveries + tasks) / (dev_ms / 1000.0),
            "e2e": {"value": sum_over_ranks(K * 8000) / e2e_s, "unit": "simulated-ms/s", "h2d_bytes_per_step": 6000, "d2h_bytes_per_step": int(d2h + 18000)},
            "gpu_launches": int(st1["kernel_launches"] - st0["kernel_launches"]), "clocks": sampler.summary()}
    if prof:
        kname, (kms, kcnt) = max(prof.items(), key=lambda kv: kv[1][0])
        total_ms = sum(v[0] for v in prof.values())
        ab = 104 * deliveries  # SURVEY.md §8d: Casper deliver = 96 B + 8 B bitmap RMW
        line["roofline"] = {"bound": "hbm", "kernel": "whole tick pipeline (no kernel dominates: each is at its launch floor)",
                            "achieved": ab / (dev_ms / 1000.0) / 1e9, "peak": peak, "unit": "GB/s", "frac": ab / (dev_ms / 1000.0) / 1e9 / peak,
                            "traffic": None, "peak_source": "measured" if peaks else "fallback", "top_kernel": kname,
                            "share_of_step": kms / total_ms, "kernel_ms": {k: round(v[0], 3) for k, v in prof.items() if v[1]},
                            "ticks": int(prof.get("k_begin", (0, 0))[1])}
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if parity_unsharded is not None:
        line["parity_sharded_vs_unsharded"] = "heads and block count identical" if parity_unsharded else "MISMATCH"
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    if parity_unsharded is False:
        sys.exit(3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="gsf", choices=["gsf", "casper"])
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=22)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--nodes", type=int, default=131072)
    ap.add_argument("--step-ms", type=int, default=0, help="0: ceil(run length / steps)")
    ap.add_argument("--ref-step-ms", type=int, default=20)
    ap.add_argument("--cpu-nodes", type=int, default=131072)
    ap.add_argument("--cpu-max-nodes", type=int, default=131072)
    ap.add_argument("--cpu-budget-s", type=float, default=20.0)
    ap.add_argument("--mode", default="auto", choices=["auto", "sharded", "weak", "replicas"],
                    help="N > 1: sharded = ONE simulation of --nodes nodes, node ids sharded over the GPUs (default; strong scaling); "
                         "weak = one sharded simulation of --weak-nodes-per-gpu x N nodes (BASELINE config #5); replicas = N independent seeds")
    ap.add_argument("--weak-nodes-per-gpu", type=int, default=32768)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the timed network holds after its last step as DIR/<name>.npy "
                         "(float64; with several ranks, rank 0's network or shard)")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        if rank == 0:
            run_casper_reference(args) if args.workload == "casper" else run_reference(args)
        return

    import torch

    import __graft_entry__ as g

    if rank == 0:
        g.build()
    from wittgenstein_b200.replicas import Replicas

    rep = Replicas("nccl")
    dist = rep.dist
    barrier, max_over_ranks, sum_over_ranks = rep.barrier, rep.max_over_ranks, rep.sum_over_ranks

    if args.workload == "casper":
        run_casper(args, rank, world, local, dist, barrier, max_over_ranks, sum_over_ranks)
        return

    global SHARD
    n, K, W = args.nodes, args.steps, args.warmup
    mode = args.mode if args.mode != "auto" else ("sharded" if world > 1 else "replicas")
    if world == 1:
        mode = "single" if args.mode != "weak" else "weak"
    sharded = world > 1 and mode in ("sharded", "weak")
    if mode == "weak":
        n = args.weak_nodes_per_gpu * world
    if sharded:
        SHARD = (dist, rank, world, local)
        seed = 0  # one simulation: every shard is configured identically
        jobs = 1
    else:
        seed = rank  # replicas: rank r simulates seed r (RunMultipleTimes.java:44-48 runs seeds one after the other)
        jobs = world

    def total(x):  # whole-job count of something every rank holds a share of
        return sum_over_ranks(x) if world > 1 else x

    # ---- warm-up: the whole run on a throw-away network of the same configuration (module load, graph
    #      instantiation, clocks) — at least W steps; it also tells how long the run is: the timed passes below each
    #      start a fresh, identically seeded network at t=0 and cover the run to completion (every live node has
    #      reached the threshold: GSFSignature.newContIf, GSFSignature.java:670-682) in exactly K steps ----
    p, _ = make_gsf(n, seed)
    t_done = 0
    warm_steps = 0
    while warm_steps < W or (p.continue_if() and t_done < 60000):
        p.network().run_ms(50)
        t_done += 50
        warm_steps += 1
    p.network().msgs_size()
    del p
    t_done = int(max_over_ranks(t_done))
    S = args.step_ms if args.step_ms > 0 else max(10, -(-t_done // K))  # K steps of runMs(S) cover [0, t_done]

    # ---- pass 1: device-timed (value) ----
    p, init_s = make_gsf(n, seed)
    net = p.network()
    st0 = net.stats()
    sampler = ClockSampler(local)
    barrier()
    torch.cuda.synchronize()
    sampler.start()
    net.timer_start()
    for _ in range(K):
        net.run_ms(S)
    dev_ms = net.timer_stop_ms()
    torch.cuda.synchronize()
    barrier()
    sampler.stop_flag = True
    st1 = net.stats()
    ev = event_counts(st0, st1)
    launches = st1["kernel_launches"] - st0["kernel_launches"]
    card_end = p.scalars()["card"]
    done = not p.continue_if()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, gsf_outputs(p))
    dev_ms = max_over_ranks(dev_ms)
    ev_all = {k: int(total(v)) for k, v in ev.items()} if sharded else ev
    launches_all = int(total(launches)) if sharded else launches
    del p, net

    # ---- pass 2: end to end through the public API with host read-backs every step ----
    p, _ = make_gsf(n, seed)
    net = p.network()
    barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    d2h = 0
    for _ in range(K):
        net.run_ms(S)
        card = p.scalars()["card"]          # StatsGetter: verifiedSignatures.cardinality() of every node
        cnt = net.counters()                # msgReceived / msgSent / bytesSent / bytesReceived / doneAt
        d2h = card.nbytes * 5 + cnt.nbytes
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    assert (card == card_end).all(), "e2e pass diverged from the device-timed pass"
    ctl_bytes = 6000
    del p, net

    # ---- pass 2b: the reference arm's window, end to end: [0, K*ref_step_ms] with runMs(ref_step_ms) slicing and the
    #      same read-backs (what `bench.py --impl reference --steps K` times on the CPU) ----
    R = args.ref_step_ms
    p, _ = make_gsf(n, seed)
    net = p.network()
    barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(K):
        net.run_ms(R)
        p.scalars()["card"]
        net.counters()
    torch.cuda.synchronize()
    same_s = max_over_ranks(time.perf_counter() - t0)
    del p, net

    # ---- pass 3: per-kernel CUDA-event timing of the same window (roofline of the dominant kernel) ----
    prof = {}
    if not args.no_profile:
        p, _ = make_gsf(n, seed)
        net = p.network()
        net.profile_enable(True)
        for _ in range(K):
            net.run_ms(S)
        prof = net.profile_read()
        net.profile_enable(False)
        del p, net

    # ---- CPU baseline on a bounded sample (prefix of the same run), the GPU over the same prefix, and the bit-exact
    #      comparison of the two end states at the metric size (BASELINE.md §3) ----
    cpu = None
    parity = None
    if rank == 0 and not args.no_cpu:
        cpu, parity = cpu_baseline_and_parity(n, args)
    elif sharded and not args.no_cpu:
        cpu_baseline_and_parity(n, args)  # the other shards run their part of the same window and report their digests
    if rank == 0 and parity is not None and parity.get("status") != "bit-exact":
        print(json.dumps({"error": "GPU and oracle states differ", "parity": parity}))
        sys.stdout.flush()
        os._exit(3)

    value = jobs * K * S / (dev_ms / 1000.0)
    e2e = jobs * K * S / e2e_s
    msgs = ev["deliveries"] + ev["tasks"] + ev["cond_runs"]

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    roof = None
    if prof:
        ab = algorithmic_bytes(ev)
        top = max(prof.items(), key=lambda kv: kv[1][0])
        kname, (kms, kcnt) = top
        total_ms = sum(v[0] for v in prof.values())
        if kname in ab and kcnt:
            achieved = ab[kname] / (kms / 1000.0) / 1e9
            roof = {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": ncu_traffic(kname), "peak_source": "measured" if peaks else "fallback",
                    "avg_launch_us": 1000.0 * kms / kcnt, "algorithmic_bytes_per_launch": ab[kname] / kcnt,
                    "share_of_step": kms / total_ms,
                    "kernel_ms": {k: round(v[0], 3) for k, v in prof.items()},
                    "kernel_gbs": {k: round(ab[k] / (v[0] / 1000.0) / 1e9, 1) for k, v in prof.items() if k in ab and v[0] > 0}}

    line = {"metric": metric_name(n), "value": value, "unit": "simulated-ms/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": dev_ms / K, "higher_is_better": True,
            "scaling": "strong" if (sharded and mode == "sharded") else "weak", "vs_baseline": None,
            "dtype": "u64 bitmaps / int32", "data": "synthetic",
            "config": {"workload": workload_name(n),
                       "window": f"step = runMs({S}) of one run; timed window [0,{K*S}] ms = the whole run of a fresh network (every live "
                                 f"node reaches the threshold by {t_done} ms); warm-up = the same run on a throw-away network ({warm_steps} x runMs(50))",
                       "parallelism": "1 GPU" if world == 1 else (
                           f"node-sharded: ONE simulation, node ids split over {world} GPUs ({n // world} nodes each); per pass two "
                           "device-side exchanges through peer stores over NVLink (items -> global creation / draw offsets; envelopes "
                           "and pooled payloads into the destination shard), no host call or collective per tick"
                           if sharded else f"{world} independent seeded replicas (no data-path collective)"),
                       "mode": mode,
                       "l2": "per-step working set (node rows + queues + ring) exceeds L2 at this size",
                       "all_nodes_done_at_end": bool(done), "host": host_info()},
            "msgs_per_s": sum_over_ranks(msgs) / (dev_ms / 1000.0),
            "e2e": {"value": e2e, "unit": "simulated-ms/s", "h2d_bytes_per_step": ctl_bytes, "d2h_bytes_per_step": int(d2h + ctl_bytes * 3)},
            "e2e_same_window_as_reference": {"value": jobs * K * R / same_s, "unit": "simulated-ms/s",
                                             "window": f"[0,{K*R}] ms, {K} x runMs({R}) with the per-step read-backs, wall clock"},
            "gpu_launches": int(launches_all), "init_s": init_s, "events": ev_all, "clocks": sampler.summary()}
    if roof:
        line["roofline"] = roof
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if parity is not None:
        line["parity"] = parity
        line[f"parity_{n}"] = f"{parity['status']}@{parity['t']}"
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
