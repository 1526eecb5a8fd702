#!/usr/bin/env python
"""bench.py -- allocations/sec of one scheduling cycle on the BASELINE.json config
"10k nodes / 50k pending pods, 4 resource dims, no affinity" (configs[1]).

A step = one full scheduling cycle over the 50 000 pending asks of a fresh snapshot (node availability reset, all asks
pending).  ONE JSON line:
  value        allocations/s with the node and ask tables already resident in HBM when the timed region starts (the timed
               region is yk_cycle alone: device sort + sweeps, bitmap read-back, ordered commit, bindings out)
  e2e          the same metric through the C ABI from HOST buffers: yk_nodes_upsert + yk_asks_upsert (H2D inside) +
               yk_cycle (bindings D2H inside) per step
  roofline     the sweep kernel of the timed region: algorithmic bytes (64 B per (row,node) evaluation + 64 B per row,
               SURVEY 8d) / its CUDA-event time against MEASURED_PEAKS.json hbm_gbs, plus what ncu says actually bounds
               it (ALU pipe, L2 and DRAM bytes per launch: profiles/sweep_metrics.json)
  cpu_baseline the C++ restatement of the reference algorithm (oracle/, kind "port", 1 thread: the reference's scheduling
               loop is a single goroutine) on the same snapshot on this box's host cores
  cpu_engine   THIS engine without a GPU: the same ordering engine and ordered commit, the sweep done by the host cores
               (AVX-512, all threads; tests/host/engine_shim.cpp) -- isolates what the B200 contributes: gpu_over_cpu_engine
  workloads    the same measurement, shorter, on config 3 (taints + nodeAffinity masks: every ask its own row) and on the
               reference's own benchmark shape (every pod identical, pkg/shim/scheduler_perf_test.go:283-288), with the
               engine's default commit choice (commit_ran_on: the reference shape is one uniform run -> decided on the device
               by a grid-wide sort, csrc/yk_uniform.cuh; config 3 -> sweep + host commit)
  host_commit / device_commit  the same workloads with the ordered commit forced onto the host / the device
  scale_up     the reference shape x 10 (50k nodes / 500k pods), default commit choice and forced host commit
With --gpus N > 1 (torchrun): `value` = N YuniKorn partitions (disjoint node sets with their own queues: the core
schedules partitions independently), one per GPU, no data-path exchange -- weak scaling; `multi` = one partition with the
sweep of every batch split across the N GPUs and exchanged peer-to-peer (strong scaling of config 3), every rank checked
against the oracle and against each other.
`--impl reference` times the CPU port alone, same metric / config.
`--dump-outputs DIR` writes the bindings of the headline arm's last timed step as DIR/ask.npy and DIR/node.npy (float64, in
commit order; rank 0's partition at N > 1): the inputs are seeded, so two builds run with the same arguments can be compared
output for output.
The benchmark writes nothing into the source tree, which may be read-only: what it compiles goes to a temporary directory.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True     # no __pycache__ next to the modules imported from the tree
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

METRIC = "allocations/sec (10k nodes, 50k pending pods)"
UNIT = "allocations/s"
N_NODES, N_APPS, TASKS = 10_000, 400, 125
B_NODE, B_ASK = 64, 64   # SURVEY 8(d): bytes per (ask,node) evaluation at D=4; per ask 56 in + 8 out

WORKLOADS = {
    "config2": "config2: 10k nodes / 50k pending pods, D=4, no affinity, fair node sort, 1 leaf queue, 400 apps x 125",
    "config3": "config3: 10k nodes / 50k pods + taints + nodeAffinity bitmasks (64-bit sets), fair node sort, 400 apps x 125",
    "reference_shape": "reference benchmark shape: 5k identical nodes / 50k identical pods 10 mCPU + 1 MB (scheduler_perf_test.go:62-63,283-288)",
    "reference_shape_x10": "reference benchmark shape x 10: 50k identical nodes / 500k identical pods (4000 apps x 125)",
    "config4": "config4: 50k nodes / 200k pods, 73 queues (DRF parents, quotas), fifo leaves",
    "config5": "config5: 10k nodes / 2000 gangs x 10, all-or-nothing",
}


def make_snapshot(name, seed_shift=0):
    from yunikorn_k8shim_b200 import synth
    if name == "config2":
        return synth.perf(N_NODES, N_APPS, TASKS, seed=2 + seed_shift)
    if name == "config3":
        return synth.perf(N_NODES, N_APPS, TASKS, masks=True, seed=2 + seed_shift)
    if name == "reference_shape":
        return synth.reference_shape()
    if name == "reference_shape_x10":
        return synth.reference_shape(50_000, 4_000, 125)
    if name == "config4":
        return synth.hier()
    if name == "config5":
        return synth.gangs()
    raise ValueError(name)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu=0):
        self.gpu, self.rows, self._stop, self._t = gpu, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows if len(r) > 2 + i)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def _ref_worker(wl, seed_shift, warmup, steps, barrier, q):
    from oracle import oracle_ctypes as oc
    snap = make_snapshot(wl, seed_shift)
    r = None
    for _ in range(max(warmup, 1)):
        r = oc.run(snap)
    barrier.wait()
    t0 = time.perf_counter()      # CLOCK_MONOTONIC: comparable across the worker processes
    n = 0
    for _ in range(steps):
        r = oc.run(snap)
        n += len(r["ask"])
    t1 = time.perf_counter()
    q.put((seed_shift, t0, t1, n, oc.bindings_hash(r["ask"], r["node"]), snap.n_asks, snap.n_nodes))


def run_reference(args, rank, world):
    """CPU arm: the oracle port on the host cores (the Go reference cannot be built in this image).  --gpus N: N
    partitions at once, one host process each (the core schedules partitions independently), like the GPU arm's N GPUs."""
    if rank != 0:
        return
    import multiprocessing as mp
    wl = args.workload
    G = max(1, args.gpus)
    ctx = mp.get_context("fork")
    barrier, q = ctx.Barrier(G), ctx.Queue()
    procs = [ctx.Process(target=_ref_worker, args=(wl, 100 * r if G > 1 else 0, args.warmup, args.steps, barrier, q)) for r in range(G)]
    for p in procs:
        p.start()
    res = sorted(q.get() for _ in range(G))
    for p in procs:
        p.join()
    dt = max(r[2] for r in res) - min(r[1] for r in res)
    n = sum(r[3] for r in res)
    v = n / dt
    sample = f"full workload ({res[0][5]} asks x {res[0][6]} nodes per partition, {G} partition(s) on {G} host core(s)) per step, {args.steps} steps"
    emit({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64+f64", "data": "synthetic",
        "config": {"workload": WORKLOADS[wl], "parallelism": f"{G} YuniKorn partition(s), one host core each",
                   "note": "C++ restatement of the reference algorithm (oracle/), not the Go binary: no Go toolchain, hot loop lives in un-vendored yunikorn-core; parity unpinned vs the Go core"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": G, "kind": "port", "sample": sample,
                         "host_cores_available": os.cpu_count()},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "bindings_hash": f"{res[0][4]:#x}",
    })


class Arm:
    """one engine on one snapshot, host buffers in the ABI's layout prepared outside the timed region"""

    def __init__(self, snap, torch, dist, device, batch=0, share_rows=True, commit="host", rank=0, world=1, attach=False):
        from yunikorn_k8shim_b200 import Engine
        self.snap, self.torch, self.dist, self.world = snap, torch, dist, world
        N, A, D = snap.n_nodes, snap.n_asks, snap.D
        self.eng = Engine(D=D, policy=snap.policy, weights=snap.weights, max_nodes=N, max_asks=A, max_apps=snap.n_apps,
                          max_queues=snap.n_queues, batch=batch, device=device, rank=rank, world=world, share_rows=share_rows,
                          commit=commit)
        self.exchange = None
        if attach:
            from yunikorn_k8shim_b200 import multigpu
            self.exchange = multigpu.attach(self.eng, dist)
        e = self.eng
        e.queues_set(snap.q_parent, snap.q_guaranteed, snap.q_max, snap.q_alloc, snap.q_sort)
        e.apps_upsert(np.arange(snap.n_apps), snap.app_queue, snap.app_submit)
        self.idxN, self.idxA = np.arange(N, dtype=np.uint32), np.arange(A, dtype=np.uint32)
        self.totalT, self.availT = np.ascontiguousarray(snap.node_total.T), np.ascontiguousarray(snap.node_avail.T)
        self.reqT = np.ascontiguousarray(snap.ask_req.T)
        self.rank_arr = snap.node_rank()

        def u32(x):   # -1 -> YK_NONE, as the ABI encodes "no node" / "no gang"
            a = np.asarray(x, dtype=np.int64).copy()
            a[a < 0] = 0xFFFFFFFF
            return a.astype(np.uint32)
        self.a_app, self.a_node, self.a_gang, self.a_flags = u32(snap.ask_app), u32(snap.ask_node), u32(snap.ask_gang), u32(snap.ask_flags)
        self.a_prio = np.ascontiguousarray(snap.ask_prio, dtype=np.int32)
        self.n_flags = np.ascontiguousarray(snap.node_flags, dtype=np.uint32)
        self.h2d_payload = N * (16 * D + 8 + 8 + 4 + 4) + A * (8 * D + 8 * 3 + 4)
        self.d2h_payload = A * 8
        self.alloc = None
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")   # > 126 MB L2

    def upsert_all(self):
        s, e = self.snap, self.eng
        e.nodes_upsert(self.idxN, self.totalT, self.availT, s.node_taint, s.node_label, self.rank_arr, self.n_flags)
        e.asks_upsert(self.idxA, self.reqT, self.a_app, s.ask_create, s.ask_tol, s.ask_need, s.ask_deny,
                      self.a_prio, self.a_node, self.a_flags, self.a_gang)

    def barrier(self, sync_ranks):
        self.torch.cuda.synchronize()
        if sync_ranks and self.dist is not None:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def step(self, e2e, sync_ranks=False):
        e = self.eng
        if self.alloc is not None:
            e.release(self.alloc)
        if not e2e:
            self.upsert_all()
            e.evaluate(0, 0)              # forces the table upload: inputs resident in HBM before timing
        self.flush.add_(1)                # L2 flush between timed iterations
        self.barrier(sync_ranks)
        t0 = time.perf_counter()
        if e2e:
            self.upsert_all()
        ask, node, _ = e.cycle(self.snap.n_asks)
        self.torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        self.alloc = ask
        return dt, ask, node

    def measure(self, steps, warmup, e2e, sync_ranks=False):
        for _ in range(warmup):
            self.step(e2e, sync_ranks)
        self.eng.stats_reset()
        tot, n = 0.0, 0
        for _ in range(steps):
            dt, ask, node = self.step(e2e, sync_ranks)
            tot += dt
            n += len(ask)
        return {"seconds": tot, "allocations": n, "ask": ask, "node": node, "stats": self.eng.stats(), "steps": steps}

    def close(self):
        self.eng.close()


_CPU_ENGINE = None


def cpu_engine_lib():
    """tests/host/engine_shim.cpp, compiled once per run from the current sources into a temporary directory"""
    global _CPU_ENGINE
    if _CPU_ENGINE is None:
        tmp = tempfile.mkdtemp(prefix="yk_bench_")
        try:
            so = os.path.join(tmp, "engine_shim.so")
            subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", "-pthread", "-w", "-o", so,
                                   os.path.join(ROOT, "tests", "host", "engine_shim.cpp")])
            _CPU_ENGINE = C.CDLL(so)      # stays mapped once its file is gone
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    return _CPU_ENGINE


def cpu_engine_time(snap, threads, reps=2, batch=4096):
    """the same ordering engine + ordered commit with the sweep on the host cores (tests/host/engine_shim.cpp)"""
    from test_engine_host import run_engine_host
    lib = cpu_engine_lib()
    lib.host_set_bench_mode(C.c_int(threads), C.c_int(1))
    best, ask, node = 1e18, None, None
    # epoch length: the engine's general rule (5/8 of the nodes) and its few-signature rule (one epoch): the better of the two
    for epoch_limit in (None, 2 * snap.n_nodes):
        for _ in range(reps):
            t0 = time.perf_counter()
            rc, ask, node, _, _ = run_engine_host(lib, snap, batch=batch, epoch_limit=epoch_limit)
            best = min(best, time.perf_counter() - t0)
            assert rc == 0, rc
    lib.host_set_bench_mode(C.c_int(0), C.c_int(0))
    return best, ask, node


def sweep_metrics():
    p = os.path.join(ROOT, "profiles", "sweep_metrics.json")
    return json.load(open(p)) if os.path.exists(p) else {}


def sweep_roofline(st, steps, n_nodes, hbm, hbm_src):
    launches = max(st["sweep_launches"], 1)
    pairs_per_launch = st["evaluations"] / launches
    rows_per_launch = pairs_per_launch / n_nodes
    alg_bytes = pairs_per_launch * B_NODE + rows_per_launch * B_ASK
    ms_launch = st["sweep_ms"] / launches
    achieved = alg_bytes / max(ms_launch * 1e-3, 1e-12) / 1e9
    out = {"bound": "hbm", "achieved": achieved, "peak": hbm, "unit": "GB/s", "frac": achieved / hbm, "traffic": None,
           "peak_source": hbm_src, "kernel": "yk_sweep_kernel", "ms_per_launch": ms_launch, "pairs_per_launch": pairs_per_launch,
           "rows_per_launch": rows_per_launch, "launches_per_step": st["sweep_launches"] / steps}
    m = sweep_metrics()
    best = None
    for shape in m.get("shapes", []):   # the ncu capture whose launch shape is closest to this one
        d = abs(shape.get("rows_per_launch", 0) - rows_per_launch) / max(rows_per_launch, 1)
        if d < 0.5 and (best is None or d < best[0]):
            best = (d, shape)
    if best:
        sh = best[1]
        out["traffic"] = sh.get("dram_bytes_per_launch")
        out["ncu"] = {k: sh.get(k) for k in ("alu_pipe_pct", "issue_active_pct", "lts_bytes_per_launch", "dram_bytes_per_launch",
                                               "shared_wavefronts_per_launch", "source")}
    return out


_REAL_STDOUT = None


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--masks", action="store_true", help="config 3 (taints + nodeAffinity bitmasks) instead of config 2")
    ap.add_argument("--config", default="0", help="workload of the headline arm: 2 (default), 3, 4, 5 or 'reference'")
    ap.add_argument("--commit", default="auto", choices=["host", "device", "auto"],
                    help="ordered commit of the headline arm (auto = the engine's default: device for cycles made of long uniform runs, host otherwise)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline arm only (no side workloads, no CPU arms)")
    ap.add_argument("--no-row-sharing", action="store_true",
                    help="sweep one row per ask even when asks have identical predicate inputs (YK_FLAG_NO_ROW_SHARING)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the bindings of the headline arm's last timed step to DIR/ask.npy and DIR/node.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the engine computed: it needs --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    args.workload = {"0": "config2", "2": "config2", "3": "config3", "4": "config4", "5": "config5", "reference": "reference_shape"}[str(args.config)]
    if args.masks:
        args.workload = "config3"
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # ONE JSON line on stdout is the contract, and libraries write banners to descriptor 1 behind Python's back (NCCL's
    # version line at N > 1): descriptor 1 becomes stderr for the whole run, and emit() writes the line to the real stdout.
    sys.stdout.flush()
    global _REAL_STDOUT
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    D = dist if world > 1 else None
    from oracle import oracle_ctypes as oc
    hbm, hbm_src = peaks()

    # ---------------- headline arm: one partition per GPU ----------------
    # world == 1: the BASELINE config.  world > 1: rank r schedules its own partition (same shape, its own seed): YuniKorn
    # partitions are disjoint node sets with their own queue trees, scheduled independently -- no data-path exchange.
    wl = args.workload
    snap = make_snapshot(wl, seed_shift=100 * rank if world > 1 else 0)
    arm = Arm(snap, torch, D, local_rank, batch=args.batch, share_rows=not args.no_row_sharing, commit=args.commit)
    with ClockSampler(local_rank) as cs:
        res = arm.measure(args.steps, args.warmup, e2e=False, sync_ranks=True)
        res_e = arm.measure(args.steps, 1, e2e=True, sync_ranks=True)
    clocks = cs.summary()
    want = oc.run(snap)
    ok_local = bool(np.array_equal(res["ask"], want["ask"]) and np.array_equal(res["node"], want["node"])
                    and np.array_equal(res_e["ask"], want["ask"]) and np.array_equal(res_e["node"], want["node"]))
    if args.dump_outputs and rank == 0:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name in ("ask", "node"):      # uint32 ids: exact in float64
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), res[name].astype(np.float64))

    def agg(seconds, allocations, ok):
        """whole-job numbers: allocations of all ranks / max time over ranks; every rank identical to its oracle"""
        if world == 1:
            return seconds, allocations, ok
        t = torch.tensor([seconds], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        a = torch.tensor([allocations, int(ok)], dtype=torch.int64, device="cuda")
        dist.all_reduce(a[:1], op=dist.ReduceOp.SUM)
        dist.all_reduce(a[1:], op=dist.ReduceOp.MIN)
        return float(t.item()), int(a[0].item()), bool(a[1].item())

    tot, n, ok_all = agg(res["seconds"], res["allocations"], ok_local)
    tot_e, n_e, _ = agg(res_e["seconds"], res_e["allocations"], True)
    st, st_e = res["stats"], res_e["stats"]

    # ---------------- world > 1: the sweep of ONE partition split across the GPUs (strong scaling of config 3) ----------------
    multi = None
    if world > 1:
        from yunikorn_k8shim_b200 import multigpu
        s3 = make_snapshot("config3")
        arm.close()
        m_arm = Arm(s3, torch, D, local_rank, batch=args.batch, commit="host", rank=rank, world=world, attach=True)
        r3 = m_arm.measure(max(3, min(args.steps, 5)), 2, e2e=False, sync_ranks=True)
        w3 = oc.run(s3)
        ok3 = bool(np.array_equal(r3["ask"], w3["ask"]) and np.array_equal(r3["node"], w3["node"]))
        agree = multigpu.check_agreement(dist, r3["ask"], r3["node"], device="cuda")
        t3, _, ok3_all = agg(r3["seconds"], r3["allocations"], ok3 and agree)
        st3 = r3["stats"]
        multi = {"workload": WORKLOADS["config3"], "mode": "one partition, sweep rows of every batch split across the GPUs, ordered commit replicated",
                 "exchange": m_arm.exchange, "rows_split": bool(st3["evaluations"] < 0.9 * st3["rows_swept"] * s3.n_nodes),
                 "evaluations_per_rank_per_step": st3["evaluations"] / r3["steps"], "pairs_per_step": float(s3.n_asks) * s3.n_nodes,
                 "identical_all_ranks_and_oracle": ok3_all, "agreement_allreduce": bool(agree),
                 "value": r3["allocations"] / t3, "unit": UNIT, "ms_per_step": t3 / r3["steps"] * 1e3, "steps": r3["steps"],
                 "scaling": "strong"}
        m_arm.close()

    out = None
    if rank == 0:
        roof = sweep_roofline(st, args.steps, snap.n_nodes, hbm, hbm_src) if st["sweep_launches"] else None
        out = {
            "metric": METRIC, "value": n / tot, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": tot / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64+u64 (fit, masks), f64 (node score)", "data": "synthetic",
            "config": {"workload": WORKLOADS[wl], "batch": int(st["asks_swept"] // max(st["batches"], 1)) if st["asks_swept"] else None,
                       "row_sharing": (not args.no_row_sharing), "commit": args.commit, "l2": "flushed between steps (256 MiB write)",
                       "parallelism": (f"{world} YuniKorn partitions (disjoint node sets, own queue trees), one per GPU, no data-path exchange"
                                       if world > 1 else "single GPU, one partition")},
            "e2e": {"value": n_e / tot_e, "unit": UNIT, "ms_per_step": tot_e / args.steps * 1e3,
                    "h2d_bytes_per_step": int(st_e["h2d_bytes"] // args.steps), "d2h_bytes_per_step": int(st_e["d2h_bytes"] // args.steps),
                    "abi_h2d_payload": arm.h2d_payload, "abi_d2h_payload": arm.d2h_payload},
            "gpu_launches": int(st["sweep_launches"] + st["other_launches"] + st["lattice_launches"]),
            "evaluations_per_s": st["evaluations"] / res["seconds"],                       # (row,node) pairs the kernel really evaluated
            "evaluations_represented_per_s": st["asks_swept"] * snap.n_nodes / res["seconds"],   # (ask,node) pairs those rows stand for
            "rows_swept_per_step": st["rows_swept"] / args.steps, "asks_swept_per_step": st["asks_swept"] / args.steps,
            "phase_ms_per_step": {"sweep": st["sweep_ms"] / args.steps, "key_sort_gather": st["sort_ms"] / args.steps,
                                  "ordered_commit": st["commit_ms"] / args.steps, "lattice_kernel": st["lattice_ms"] / args.steps,
                                  "cycle_total": st["total_ms"] / args.steps,
                                  "host_split": dict(zip(("upload+device_order", "orderer_begin+ids", "orderer_fill", "wait_device", "commit",
                                                          "epoch_end", "launch", "hidden_on_helper"), [x / args.steps for x in st["host_ms"]]))},
            "clocks": clocks,
            "bindings_identical_to_oracle": ok_all,
            "bindings_hash": f"{oc.bindings_hash(res['ask'], res['node']):#x}",
            "parity_note": "oracle = C++ restatement of the reference algorithm; parity unpinned vs the Go core (no Go toolchain)",
        }
        if roof:
            out["roofline"] = dict(roof, note=(
                "algorithmic bytes follow SURVEY 8(d)'s streaming model (64 B per evaluation); the kernel keeps the node tile in "
                "registers and the ask chunk in shared memory, so DRAM traffic is far below the model: what bounds it is the "
                "integer-ALU pipe (roofline.ncu, profiles/), not HBM"))
        if multi:
            out["multi"] = multi
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()      # peers may still be signalling into an engine's sync block
        if rank == 0:
            emit(out)
        dist.destroy_process_group()
        return
    arm.close()

    # ---------------- single GPU: side arms (short) ----------------
    if not args.quick:
        threads = max(1, min(os.cpu_count() or 1, 64))
        side_steps = max(3, min(args.steps, 5))

        snaps, wants = {wl: snap}, {wl: want}

        def run_arm(name, commit, share=True, cpu_engine=True):
            if name not in snaps:
                snaps[name] = make_snapshot(name)
                wants[name] = oc.run(snaps[name])
            s = snaps[name]
            a = Arm(s, torch, None, local_rank, batch=args.batch, share_rows=share, commit=commit)
            r = a.measure(side_steps, 2, e2e=False)
            re_ = a.measure(side_steps, 1, e2e=True)
            a.close()
            w = wants[name]
            stx = r["stats"]
            o = {"workload": WORKLOADS[name], "commit": commit,
                 "commit_ran_on": "device" if stx["lattice_cycles"] else "host", "value": r["allocations"] / r["seconds"], "unit": UNIT,
                 "ms_per_step": r["seconds"] / side_steps * 1e3, "e2e_value": re_["allocations"] / re_["seconds"],
                 "e2e_ms_per_step": re_["seconds"] / side_steps * 1e3, "steps": side_steps,
                 "identical_to_oracle": bool(np.array_equal(r["ask"], w["ask"]) and np.array_equal(r["node"], w["node"])),
                 "d2h_bytes_per_step": int(stx["d2h_bytes"] // side_steps), "h2d_bytes_per_step": int(re_["stats"]["h2d_bytes"] // side_steps),
                 "rows_swept_per_step": stx["rows_swept"] / side_steps,
                 "phase_ms_per_step": {"sweep": stx["sweep_ms"] / side_steps, "ordered_commit": stx["commit_ms"] / side_steps,
                                       "lattice_kernel": stx["lattice_ms"] / side_steps, "cycle_total": stx["total_ms"] / side_steps}}
            if stx["sweep_launches"]:
                o["roofline"] = sweep_roofline(stx, side_steps, s.n_nodes, hbm, hbm_src)
            if stx["lattice_launches"]:
                o["lattice"] = {k: stx[k] / side_steps for k in ("lattice_subruns", "lattice_asks", "lattice_elements", "lattice_sorts",
                                                                  "lattice_fullscans", "lattice_handoffs", "uniform_runs", "uniform_asks",
                                                                  "uniform_elements", "uniform_retries")}
            if cpu_engine:
                dt, ask_c, node_c = cpu_engine_time(s, threads)
                o["cpu_engine"] = {"ms_per_step": dt * 1e3, "value": len(ask_c) / dt, "unit": UNIT, "threads": threads,
                                   "identical_to_oracle": bool(np.array_equal(ask_c, w["ask"]) and np.array_equal(node_c, w["node"])),
                                   "what": "same ordering engine + ordered commit, sweep on the host cores (AVX-512 when present)"}
                o["gpu_over_cpu_engine"] = o["value"] / o["cpu_engine"]["value"]
            return o

        # what the B200 contributes on the headline workload: the same engine with the sweep on the host cores
        dt, ask_c, node_c = cpu_engine_time(snap, threads)
        out["cpu_engine"] = {"ms_per_step": dt * 1e3, "value": len(ask_c) / dt, "unit": UNIT, "threads": threads,
                             "identical_to_oracle": bool(np.array_equal(ask_c, want["ask"]) and np.array_equal(node_c, want["node"])),
                             "what": "same ordering engine + ordered commit, sweep on the host cores (AVX-512 when present)"}
        out["gpu_over_cpu_engine"] = out["value"] / out["cpu_engine"]["value"]
        # the sweep kernel at full load on the headline workload: one row per ask
        if not args.no_row_sharing and st["rows_swept"] * 2 < st["asks_swept"]:
            o = run_arm(wl, "host", share=False, cpu_engine=False)
            out["one_row_per_ask"] = o
            if "roofline" in o:
                out["roofline_one_row_per_ask"] = o["roofline"]
        out["workloads"] = {name: run_arm(name, "auto") for name in ("config3", "reference_shape") if name != wl}
        out["host_commit"] = {name: run_arm(name, "host", cpu_engine=False) for name in ("reference_shape",) if name != wl}
        # the same shape ten times larger: the device's share of the cycle grows with the cluster, the host commit's does not shrink
        out["scale_up"] = {"auto": run_arm("reference_shape_x10", "auto"), "host": run_arm("reference_shape_x10", "host", cpu_engine=False)}
        out["device_commit"] = {name: run_arm(name, "device", cpu_engine=False) for name in ("config2", "config3", "reference_shape")}
    if not args.no_cpu_baseline and not args.quick:
        oc.run(snap)
        t0 = time.perf_counter()
        reps = 0
        while True:
            r = oc.run(snap)
            reps += 1
            if time.perf_counter() - t0 > 10.0 or reps >= 100:
                break
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": reps * len(r["ask"]) / dt, "unit": UNIT, "cores": 1, "kind": "port",
                               "sample": f"{reps} full cycles of the same snapshot ({dt:.1f} s)",
                               "host_cores_available": os.cpu_count()}
    emit(out)


if __name__ == "__main__":
    main()
