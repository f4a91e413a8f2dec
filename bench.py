#!/usr/bin/env python
"""bench.py -- simulated events per wall-second of the hot path on B200 (BASELINE.json metric).

Workload at N=1 (--config 1, the default): BASELINE.json configs[1], "65 536 independent M/M/1
replicas, 1e6 sim seconds, 1xB200" (Source.poisson(8) -> Server(Exponential(0.1)) -> Sink).  One STEP
advances every replica by one window of simulated time (default 1e4 s of the 1e6 s horizon, about
3.96e10 events at 65 536 replicas): consecutive steps are consecutive windows of ONE continuing run
(state resident in HBM, resumed by the kernel), exactly the reference's Simulation._run_window slicing;
--steps 100 --window-s 1e4 covers the whole horizon.  At N>1 (torchrun, one rank per GPU) every rank runs
its own 65 536 replicas (weak scaling, global replica ids keep the Philox streams disjoint); the only
collective is the end-of-run NCCL all-reduce of the fixed-layout summary vector (SURVEY.md 8(e)).

--config 3 / --config 4 run the two multi-GPU configurations of BASELINE.json where it puts them:
  3  examples/distributed chash: 1 024-node consistent-hash ring, 4 096 replicas over 4 GPUs (1 024 per GPU),
     10 sim-s horizon, one step = 1 sim-s window;
  4  M/M/c sweep, c in 1..32 x 8 arrival-rate levels = 256 cells, 262 144 replicas over 8 GPUs (32 768 per GPU,
     128 seeds per cell and GPU), 1 000 sim-s horizon, one step = 100 sim-s window; after the run the per-cell
     totals and latency histograms are all-reduced (one collective) and checked against the numpy reduction of
     the per-replica outputs gathered from every rank.
They print the same JSON line (kept under profiles/); the driver's headline stays --config 1.

Modes (--mode, config 1):
  record   (default, the headline) flight-recorder ON: every processed event writes its 16 B record, every
           Sink sample 16 B and every service start 8 B to per-replica rings in HBM (19.2 B per event for
           M/M/1, SURVEY.md 8(d)).  This is the mode the event-record HBM roofline of BASELINE.json refers to.
  summary  per-replica statistics only (negligible HBM traffic; issue-bound).

After the timed region `parity_sample` re-runs a few replicas of the SAME run (same seeds, same windows) on the
CPU oracle and compares their summaries, entity statistics and -- in record mode -- the raw recorder rings
byte for byte: the number printed is for a run whose results are the reference's.

--steps K times exactly K windows; when --warmup + --steps windows do not fit the horizon, the run continues past it
(the JSON line reports the horizon used).  --dump-outputs DIR writes what the last timed step left for a caller of
Engine.read_outputs (see dump_outputs) as float64 .npy files, at most 64 MB in all; the inputs depend only on the
arguments (--seed), so two builds run with the same arguments can be compared output for output.

--impl reference times the reference's own CPU path on the host cores: the UNMODIFIED Python reference
(installed by the recipe in DESIGN.md section 8 into baseline/_ref, which travels to the GPU box) through its
own ParallelRunner(max_workers=cores).run_replicas, kind "reference"; if that install is missing, the C
restatement (oracle port) on all cores, kind "port".  The port's figure is reported next to it either way.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
sys.dont_write_bytecode = True          # the bench runs from a built tree and leaves it as it found it

METRIC = "simulated_events_per_second"
UNIT = "events/s"
RATE, MEAN = 8.0, 0.1
BYTES_EVENT, BYTES_SAMPLE, BYTES_SERVICE = 16, 16, 8
REF_DIR = os.path.join(ROOT, "baseline", "_ref")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=1, choices=[1, 3, 4])
    ap.add_argument("--mode", default="record", choices=["record", "summary"])
    ap.add_argument("--replicas", type=int, default=0, help="replicas per GPU (default: the configuration's)")
    ap.add_argument("--window-s", type=float, default=0.0, help="simulated seconds per step (default: the configuration's)")
    ap.add_argument("--horizon-s", type=float, default=0.0)
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--parity-replicas", type=int, default=8)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-other-mode", action="store_true")
    ap.add_argument("--no-other-configs", action="store_true")
    ap.add_argument("--no-e2e-records", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step to DIR/<name>.npy (float64) for comparing builds")
    a = ap.parse_args()
    if a.steps < 1 or a.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return a


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def host_cores():
    """Threads this process may really use: the scheduler affinity, capped by the cgroup CPU quota."""
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            q, p = f.read().split()
            if q != "max":
                quota = float(q) / float(p)
    except Exception:
        try:
            with open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us") as f, open("/sys/fs/cgroup/cpu/cpu.cfs_period_us") as g:
                q, p = int(f.read()), int(g.read())
                if q > 0:
                    quota = q / p
        except Exception:
            pass
    cores = aff if quota is None else max(1, min(aff, int(math.floor(quota + 1e-9))))
    return cores, {"affinity": aff, "cgroup_quota_cpus": quota, "os_cpu_count": os.cpu_count()}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.p, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.p:
            self.p.terminate()
            try:
                self.p.wait(timeout=2)
            except Exception:
                self.p.kill()
        sm = sorted(int(r[1]) for r in self.rows if len(r) > 8 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) > 8 and r[2].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) > 8 for n, v in zip(names, r[5:9]) if v.lower().startswith("active")})
        pw = sorted(float(r[3]) for r in self.rows if len(r) > 8 and r[3].replace(".", "", 1).isdigit())
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm), "power_w_median": pw[len(pw) // 2] if pw else None}


# --------------------------------------------------------------------------- workloads

def make_config(a):
    """The model, sizes and recorder capacities of --config; everything bench-specific about a configuration."""
    import happysim_b200 as hs
    if a.config == 1:
        replicas, window_s, horizon_s = a.replicas or 65536, a.window_s or 1.0e4, a.horizon_s or 1.0e6
        caps = dict(record_cap=1024, sample_cap=128, service_cap=128) if a.mode == "record" else {}
        return dict(model=hs.mm1(RATE, MEAN), replicas=replicas, window_s=window_s, horizon_s=horizon_s, caps=caps,
                    extra={}, kernel="hs_lane_kernel", mode=a.mode, cells=0, replicas_per_cell=1,
                    workload="BASELINE configs[1]: 65 536 independent M/M/1 replicas (Source.poisson(8) -> "
                             "Server(ExponentialLatency(0.1)) -> Sink), 1e6 sim-s horizon, per GPU",
                    oracle_window_cap_s=None)
    if a.config == 3:
        replicas, window_s, horizon_s = a.replicas or 1024, a.window_s or 1.0, a.horizon_s or 10.0
        tab = hs.consistent_hash_table([f"S{i}" for i in range(1024)], 100, 10000)
        return dict(model=hs.lb_key_table(tab, 1024, rate=8192.0), replicas=replicas, window_s=window_s,
                    horizon_s=horizon_s, caps={}, extra={}, kernel="hs_thread_kernel", mode="summary", cells=0,
                    replicas_per_cell=1,
                    workload="BASELINE configs[3]: 1 024-node consistent-hash ring (Source(8192/s, 10 000 client ids) -> "
                             "LoadBalancer(ConsistentHash, 100 vnodes) -> 1 024 x Server(Exp 0.1) -> Sink), 4 096 replicas "
                             "over 4 GPUs = 1 024 per GPU, 10 sim-s horizon", oracle_window_cap_s=None)
    replicas, window_s, horizon_s = a.replicas or 32768, a.window_s or 100.0, a.horizon_s or 1000.0
    m = hs.mmc_sweep()
    return dict(model=m, replicas=replicas, window_s=window_s, horizon_s=horizon_s, caps={},
                extra=dict(queue_ring=4096), kernel="hs_lane_kernel", mode="summary", cells=m.n_cells,
                replicas_per_cell=max(1, replicas // m.n_cells), histogram=True,
                workload="BASELINE configs[4]: M/M/c sweep, c in 1..32 x 8 utilisation levels = 256 cells, 262 144 replicas "
                         "over 8 GPUs = 32 768 per GPU (128 seeds per cell and GPU), 1 000 sim-s horizon",
                oracle_window_cap_s=None)


def workload_config(a, cfg, world):
    return {"workload": cfg["workload"], "baseline_config": a.config,
            "replicas_per_gpu": cfg["replicas"], "replicas_total": cfg["replicas"] * world, "window_s": cfg["window_s"],
            "horizon_s": cfg["horizon_s"], "step": "one window of simulated time for every replica (resumed state)",
            "mode": cfg["mode"], "parallelism": f"replicas sharded over {world} GPU(s), no data-path collective",
            "l2": "working set (replica state + queue rings + recorder rings) > 126 MB L2; no explicit flush"
                  if a.config == 1 else "working set (per-replica state blocks) read and written once per window"}


# --------------------------------------------------------------------------- CPU legs

def cpu_port_throughput(budget_s, window_s, seed, threads):
    """The oracle port (oracle/hs_oracle.c) on `threads` POSIX threads, all inside C (hs_oracle_bench): M/M/1
    replicas of BASELINE configs[1], each simulated for `window_s` s, pulled from a shared counter until the
    time budget is spent."""
    import happysim_b200 as hs
    import oracle_lib as O
    L = O.lib()
    L.hs_oracle_bench.argtypes = [C.POINTER(O.A.ModelDesc), C.POINTER(O.A.RunParams), C.c_int, C.c_double, C.c_uint32,
                                  C.POINTER(C.c_int64), C.POINTER(C.c_uint32), C.POINTER(C.c_double)]
    L.hs_oracle_bench.restype = C.c_int
    model = hs.mm1(RATE, MEAN)
    d = model.desc()
    p = O.make_params(seed=seed, end_ns=int(window_s * 1e9), n_replicas=1, flags=0)
    ev, rp, wall = C.c_int64(), C.c_uint32(), C.c_double()
    rc = L.hs_oracle_bench(C.byref(d), C.byref(p), threads, budget_s, 1 << 30, C.byref(ev), C.byref(rp), C.byref(wall))
    assert rc == 0, rc
    v = ev.value / wall.value
    return {"value": v, "unit": UNIT, "cores": threads, "kind": "port", "per_core": v / threads,
            "sample": f"{rp.value} M/M/1 replicas x {window_s:g} sim-s ({ev.value:.3e} events, {wall.value:.1f} s wall) on "
                      f"the oracle port (oracle/hs_oracle.c, hs_oracle_bench), {threads} POSIX threads"}, ev.value, wall.value


def _ref_build_mm1(sim_s=2000.0):
    """build_fn for the reference's ParallelRunner: the README quick-start model.  _run_one has already seeded
    `random` with the replica's seed (parallel/runner.py:73-79); numpy's global generator, which the Poisson
    arrival provider draws from, is seeded here from it so that forked workers do not share one arrival stream."""
    import random
    import numpy as np
    np.random.seed(random.getrandbits(32))
    from happysimulator import Instant, Simulation, Sink, Source
    from happysimulator.components.server.server import Server
    from happysimulator.distributions.exponential import ExponentialLatency
    sink = Sink()
    server = Server("Server", service_time=ExponentialLatency(MEAN), downstream=sink)
    source = Source.poisson(rate=RATE, target=server)
    return Simulation(sources=[source], entities=[server, sink], end_time=Instant.from_seconds(sim_s))


def reference_available():
    return os.path.isdir(os.path.join(REF_DIR, "happysimulator"))


def cpu_reference_throughput(budget_s, cores, seed):
    """The unmodified Python reference through its own ParallelRunner(max_workers=cores).run_replicas
    (parallel/runner.py:115-142): cores x k replicas of 2 000 sim-s each, k chosen for ~budget_s of work
    (~1.5e5 events/s per core).  Wall time includes the process pool start-up, as it does for a user."""
    if REF_DIR not in sys.path:
        sys.path.insert(0, REF_DIR)
    from happysimulator.parallel.runner import ParallelRunner
    sim_s = 2000.0
    per_replica_s = sim_s * 59.6 / 1.5e5
    k = max(1, int(round(budget_s / per_replica_s)))
    n = cores * k
    t0 = time.perf_counter()
    res = ParallelRunner(max_workers=cores).run_replicas(_ref_build_mm1, n_replicas=n, base_seed=seed)
    dt = time.perf_counter() - t0
    ev = sum(r.summary.total_events_processed for r in res)
    v = ev / dt
    return {"value": v, "unit": UNIT, "cores": cores, "kind": "reference", "per_core": v / cores,
            "sample": f"{n} M/M/1 replicas x {sim_s:g} sim-s ({ev:.3e} events, {dt:.1f} s wall incl. pool start-up) on the "
                      f"unmodified Python reference (baseline/_ref), ParallelRunner(max_workers={cores}).run_replicas"}, ev, dt


def run_reference_arm(a, rank, world):
    if rank != 0:
        return
    cores, core_info = host_cores()
    n_runs = a.steps + a.warmup
    budget = max(2.0, min(8.0, 90.0 / max(1, n_runs)))
    use_ref = reference_available()
    cfg = make_config(a) if a.config == 1 else None

    def one(b):
        if use_ref:
            return cpu_reference_throughput(b, cores, a.seed)
        return cpu_port_throughput(b, 500.0, a.seed, cores)

    for _ in range(a.warmup):
        one(min(budget, 2.0))
    tot_ev, tot_t, last = 0, 0.0, None
    for _ in range(a.steps):
        last, ev, dt = one(budget)
        tot_ev += ev
        tot_t += dt
    value = tot_ev / tot_t
    cb = dict(last)
    cb["value"], cb["per_core"], cb["core_accounting"] = value, value / cores, core_info
    port, _, _ = cpu_port_throughput(6.0, 500.0, a.seed, cores)
    if cfg is None:
        a.config = 1
        cfg = make_config(a)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": 1e3 * tot_t / a.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": workload_config(a, cfg, 1),
            "cpu_baseline": cb, "cpu_baseline_port": port,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": ("the unmodified Python reference (baseline/_ref) through its own ParallelRunner on all usable host "
                     "cores, each step a bounded sample of configs[1]'s workload" if use_ref else
                     "baseline/_ref is not installed on this box: the reference arm is its C restatement (oracle port, "
                     "pinned event-by-event against the reference) on all usable host cores") +
                    "; cpu_baseline_port is the C port on the same cores for comparison"}
    print(json.dumps(line), flush=True)


DUMP_BYTES = 64 << 20
DUMP_KEYS = ("summaries", "entity_stats", "records", "sink_samples", "service_samples", "histograms", "sketches")


def dump_outputs(out_dir, outs, prefix, budget):
    """The per-replica outputs a caller of Engine.read_outputs receives, as float64 .npy files: one file per field of a
    structured array (<key>.<field>.npy; 64-bit unsigned fields, e.g. the order hash, split exactly into .hi / .lo
    32-bit halves).  Every key gets an equal share of `budget` bytes; a key whose replicas do not all fit keeps a
    fixed, seeded sample of them, and <key>.replica.npy names the replicas kept, in order."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    keys = [k for k in DUMP_KEYS if outs.get(k) is not None]
    order = np.random.default_rng(20240601).permutation(len(outs["summaries"]))
    for k in keys:
        arr = outs[k]
        cols = {}
        for f in (arr.dtype.names or [None]):
            if f == "pad":
                continue
            v = arr if f is None else arr[f]
            name = k if f is None else f"{k}.{f}"
            if v.dtype == np.uint64:
                cols[name + ".hi"], cols[name + ".lo"] = v >> np.uint64(32), v & np.uint64(0xFFFFFFFF)
            else:
                cols[name] = v
        per_replica = 8 * (1 + sum(int(np.prod(c.shape[1:])) for c in cols.values()))
        keep = min(len(arr), budget // len(keys) // max(1, per_replica))
        rows = np.arange(len(arr)) if keep == len(arr) else np.sort(order[:keep])
        np.save(os.path.join(out_dir, f"{prefix}{k}.replica.npy"), rows.astype(np.float64))
        for name, c in cols.items():
            np.save(os.path.join(out_dir, f"{prefix}{name}.npy"), np.ascontiguousarray(c[rows], dtype=np.float64))


# --------------------------------------------------------------------------- GPU arm

def main():
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference_arm(a, rank, world)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import happysim_b200 as hs
    from happysim_b200 import engine, _abi as A
    from happysim_b200 import distributed as D
    import oracle_lib as O

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cfg = make_config(a)
    model, n = cfg["model"], cfg["replicas"]
    end_ns = int(cfg["horizon_s"] * 1e9)
    win_ns = int(cfg["window_s"] * 1e9)
    if (a.warmup + a.steps) * win_ns > end_ns:      # every step asked for is timed: the run continues past the horizon
        end_ns = (a.warmup + a.steps) * win_ns
        cfg["horizon_s"] = end_ns / 1e9
    stream = torch.cuda.Stream()
    eng = engine.Engine(local, stream=stream.cuda_stream)
    eng.upload(model)
    flags = A.HS_RUN_HISTOGRAM if cfg.get("histogram") else 0
    caps_by_mode = {"record": dict(record_cap=1024, sample_cap=128, service_cap=128), "summary": {}}
    caps_by_mode[cfg["mode"]] = cfg["caps"]

    def window_end(k):
        we = min((k + 1) * win_ns, end_ns)
        return we if we < end_ns else -1

    def params(mode, k, resume, mk=engine.make_params):
        return mk(seed=a.seed, end_ns=end_ns, window_end_ns=window_end(k), n_replicas=n, replica_index_base=rank * n,
                  replicas_per_cell=cfg["replicas_per_cell"], resume=resume, flags=flags, **caps_by_mode[mode], **cfg["extra"])

    def counters():
        o = eng.read_outputs()
        s = o["summaries"]
        return int(s["events_processed"].sum()), int(s["n_sink_samples"].sum()), int(s["n_service_samples"].sum()), \
            int((s["status"] != 0).sum())

    def timed_run(mode, steps, warmup):
        """W untimed + K timed consecutive windows of one continuing run, device-timed."""
        k = 0
        for _ in range(warmup):
            eng.run(params(mode, k, resume=int(k > 0))); k += 1
        eng.sync()
        c0 = counters()
        l0 = eng.launch_count()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(steps):
            eng.run(params(mode, k, resume=int(k > 0))); k += 1
        e1.record(stream)
        barrier()
        wall = time.perf_counter() - t0
        ms = e0.elapsed_time(e1)
        l1 = eng.launch_count()
        c1 = counters()
        return {"ms": ms, "wall_s": wall, "events": c1[0] - c0[0], "sink": c1[1] - c0[1], "service": c1[2] - c0[2],
                "flagged": c1[3], "launches": l1 - l0, "last_launch_ms": eng.last_run_ms(), "windows_done": k}

    # ---- headline mode, device-timed ---------------------------------------
    clk = ClockSampler(local)
    if rank == 0:
        clk.start()
    res = timed_run(cfg["mode"], a.steps, a.warmup)
    clocks = clk.stop() if rank == 0 else None
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, eng.read_outputs(), f"rank{rank}." if world > 1 else "", DUMP_BYTES // world)

    def reduce_max(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MAX); return float(t)

    def reduce_sum(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.SUM); return float(t)

    ms = reduce_max(res["ms"])
    events = reduce_sum(float(res["events"]))
    value = events / (ms * 1e-3)

    # ---- parity sample: the run just timed, re-run on the CPU oracle for a few replicas ----------
    def parity_sample(mode, windows_done, k_rep):
        """Replicas spread over this rank's range, oracle-run with the same seeds up to the last window executed
        (the oracle pauses at the same window end), compared with the device state of the timed run."""
        got = eng.read_outputs()
        idx = sorted({int(i) for i in np.linspace(0, n - 1, k_rep)})
        p = params(mode, windows_done - 1, resume=0, mk=O.make_params)
        d = model.desc()
        bufs, o = O.alloc_outputs(model.n_entities, p, model.sketch_layout()[2])
        from concurrent.futures import ThreadPoolExecutor
        t0 = time.perf_counter()
        with ThreadPoolExecutor(min(len(idx), host_cores()[0])) as ex:
            list(ex.map(lambda r: O.lib().hs_oracle_run_range(C.byref(d), C.byref(p), C.byref(o), r, r + 1), idx))
        keys = ["summaries", "entity_stats"] + (["records", "sink_samples", "service_samples"] if caps_by_mode[mode] else [])
        if cfg.get("histogram"):
            keys.append("histograms")
        bad = [f"{k}[{r}]" for k in keys for r in idx if bufs[k] is not None and got[k][r].tobytes() != bufs[k][r].tobytes()]
        return {"replicas": len(idx), "ok": not bad, "compared": keys, "windows": windows_done,
                "sim_seconds_each": windows_done * cfg["window_s"], "oracle_s": round(time.perf_counter() - t0, 2),
                "events_checked": int(bufs["summaries"]["events_processed"][idx].sum()), "mismatches": bad[:8],
                "what": "same seeds and window ends on the CPU oracle (oracle/hs_oracle.c); raw rings, summaries and "
                        "entity statistics compared byte for byte with the device state of the timed run"}

    parity = parity_sample(cfg["mode"], res["windows_done"], a.parity_replicas) if a.parity_replicas > 0 else None
    parity_ok_all = reduce_sum(0.0 if (parity is None or parity["ok"]) else 1.0) == 0.0

    # ---- end-of-run aggregation: the NCCL all-reduce of the summary vector (+ per-cell vectors for the sweep)
    t = engine.totals_to_dict(D.allreduce_totals(eng.read_totals(), device="cuda"))
    agg = {"events_processed": t["events_processed"], "sink_events": t["sink_events"], "replicas": t["replicas"],
           "replicas_flagged": t["replicas_flagged"],
           "mean_latency_s": t["sum_latency"] / max(1, t["sink_events"]), "min_latency_s": t["min_latency"],
           "max_latency_s": t["max_latency"]}
    cell_check = None
    if cfg["cells"]:
        nc = cfg["cells"]
        local_cells = eng.read_cell_totals(nc)
        t0 = time.perf_counter()
        reduced = D.allreduce_cell_totals(local_cells, device="cuda")
        torch.cuda.synchronize()
        ar_ms = 1e3 * (time.perf_counter() - t0)
        # single-process numpy reduction of the per-replica outputs of every rank, gathered on rank 0
        out = eng.read_outputs()
        mine = D.cell_totals_from_outputs(model, out, nc, cfg["replicas_per_cell"], index_base=rank * n)
        mine = [(engine.totals_to_dict(tt), h) for tt, h in mine]
        gathered = [None] * world
        if world > 1:
            dist.all_gather_object(gathered, mine)
        else:
            gathered = [mine]
        if rank == 0:
            ints = ["events_processed", "sink_events", "server_completions", "source_ticks", "dropped", "replicas", "replicas_flagged"]
            ok, worst = True, 0.0
            for c in range(nc):
                for k in ints:
                    ok &= reduced[c][0][k] == sum(g[c][0][k] for g in gathered)
                ok &= bool((reduced[c][1] == sum(g[c][1].astype(np.uint64) for g in gathered)).all())
                ref = sum(g[c][0]["sum_latency"] for g in gathered)
                worst = max(worst, abs(reduced[c][0]["sum_latency"] - ref) / max(1e-300, abs(ref)))
                ok &= reduced[c][0]["min_latency"] == min(g[c][0]["min_latency"] for g in gathered)
                ok &= reduced[c][0]["max_latency"] == max(g[c][0]["max_latency"] for g in gathered)
            c_hi = max(range(nc), key=lambda c: reduced[c][0]["sum_latency"] / max(1, reduced[c][0]["sink_events"]))
            cell_check = {"cells": nc, "nccl_calls": D.CELL_ALLREDUCE_CALLS, "allreduce_ms_host": round(ar_ms, 3),
                          "equals_numpy_reduction": bool(ok and worst < 1e-12), "float_sum_rel_diff_max": worst,
                          "replicas_per_cell_total": int(reduced[0][0]["replicas"]),
                          "slowest_cell": {"cell": c_hi, "c_rho": list(model.cells[c_hi]) if hasattr(model, "cells") else None,
                                           "mean_latency_s": reduced[c_hi][0]["sum_latency"] / max(1, reduced[c_hi][0]["sink_events"]),
                                           "p99_latency_s": D.histogram_percentile(reduced[c_hi][1], 0.99)}}

    # ---- roofline of the dominant kernel (this rank's launches) -------------
    peak, peak_src = peaks()
    per_launch_ms = res["ms"] / a.steps
    if a.config == 1:
        state_bytes = n * (2 * 512 + 56 + 3 * 64)
    else:
        state_bytes = n * (56 + model.n_entities * (2 * 96 + 64))
    if cfg["mode"] == "record":
        algo_bytes = (res["events"] * BYTES_EVENT + res["sink"] * BYTES_SAMPLE + res["service"] * BYTES_SERVICE) / a.steps + state_bytes
    else:
        algo_bytes = state_bytes
    achieved = algo_bytes / (per_launch_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    try:        # DRAM bytes per event measured by one `ncu --set full` capture of this kernel (profiles/)
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)[cfg["mode"] if a.config == 1 else f"config{a.config}"]
        traffic = tj["dram_bytes"] / tj["events"] * res["events"] / a.steps
        traffic_src = tj["source"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "kernel": cfg["kernel"], "peak_source": peak_src,
                "algorithmic_bytes_per_launch": algo_bytes,
                "bytes_per_event": algo_bytes * a.steps / max(1, res["events"]),
                "note": ("record mode: 16 B/event + 16 B/Sink sample + 8 B/service start (SURVEY.md 8(d)) + replica "
                         "state load/store" if cfg["mode"] == "record" else
                         "summary mode moves only per-replica state/statistics: the kernel is issue-bound, "
                         "not HBM-bound, so this fraction is small by construction")}

    # ---- the other mode, for context ------------------------------------------
    other = None
    if a.config == 1 and not a.no_other_mode:
        om = "summary" if a.mode == "record" else "record"
        eng.upload(model)
        r2 = timed_run(om, max(2, min(a.steps, 5)), 3)
        ms2 = reduce_max(r2["ms"]); ev2 = reduce_sum(float(r2["events"]))
        other = {"mode": om, "value": ev2 / (ms2 * 1e-3), "unit": UNIT, "ms_per_step": ms2 / max(2, min(a.steps, 5))}

    # ---- end to end through the public API with host buffers -------------------
    # One continuing run again, cut into the same windows; every timed step is a RESUMED window (like the timed
    # region above) and includes: the model table H2D (hs_model_upload), hs_run, and the D2H read of the per-replica
    # summaries + entity statistics into pinned host memory.  config 1 goes through the modelling API
    # (Simulation.run_ensemble, lowering included once); configs 3/4 through the engine API (FlatModel).
    e2e_steps = max(2, min(a.steps, 5))
    e2e_warm = 2
    sim = None
    if a.config == 1:
        sink = hs.Sink()
        server = hs.Server("Server", service_time=hs.ExponentialLatency(MEAN), downstream=sink)
        source = hs.Source.poisson(rate=RATE, target=server)
        sim = hs.Simulation(sources=[source], entities=[server, sink], end_time=hs.Instant.from_seconds(cfg["horizon_s"]),
                            seed=a.seed, device=local)
        assert sim.model.entities.tobytes() == model.entities.tobytes()
        hs.api._engines[local] = eng            # the API's per-device engine = the one bound to this stream

    def e2e_run(with_rings):
        p0 = params(cfg["mode"], 0, 0)
        host = eng.alloc_host_outputs(p0, pinned=True)
        if not with_rings:
            host["records"] = host["sink_samples"] = host["service_samples"] = None    # rings stay on the device
        ev_prev, ev_e2e, t0 = 0, 0, 0.0
        for it in range(e2e_warm + e2e_steps):
            if it == e2e_warm:
                barrier(); t0 = time.perf_counter(); ev_e2e = 0
            if sim is not None:
                sim.run_ensemble(n, seed=a.seed, replica_index_base=rank * n, flags=flags,
                                 window_end_s=(it + 1) * cfg["window_s"], resume=it > 0, host=host, upload=True,
                                 totals=False, on_overflow="ignore", **caps_by_mode[cfg["mode"]])
            else:
                eng.upload(model) if it == 0 else None
                eng.run(params(cfg["mode"], it, resume=int(it > 0)))
                eng.read_outputs(host)
            tot = int(host["summaries"]["events_processed"].sum())
            if it >= e2e_warm:
                ev_e2e += tot - ev_prev
            ev_prev = tot
        barrier()
        dt = reduce_max(time.perf_counter() - t0)
        ev = reduce_sum(float(ev_e2e))
        d2h = sum(host[k].nbytes for k in ("summaries", "entity_stats", "records", "sink_samples", "service_samples", "histograms")
                  if host.get(k) is not None)
        return ev / dt, int(d2h), dt

    h2d = model.entities.nbytes + model.backends.nbytes + model.key_table.nbytes + \
        (model.cell_d0.nbytes + model.cell_i0.nbytes if model.cell_d0 is not None else 0)
    v_e2e, d2h, _ = e2e_run(False)
    e2e = {"value": v_e2e, "unit": UNIT, "h2d_bytes_per_step": int(h2d if a.config == 1 else 0), "d2h_bytes_per_step": d2h,
           "steps": e2e_steps,
           "what": ("Simulation.run_ensemble(window_end_s=..., resume=True, host=pinned buffers): hs_model_upload + hs_run "
                    "(resumed window) + hs_read_outputs(summaries, entity stats -> pinned host) per step, wall clock"
                    if a.config == 1 else
                    "Engine.run(resumed window) + Engine.read_outputs(summaries, entity stats -> pinned host) per step, wall clock")}
    e2e_records = None
    if cfg["mode"] == "record" and not a.no_e2e_records:
        v_r, d2h_r, _ = e2e_run(True)
        e2e_records = {"value": v_r, "unit": UNIT, "d2h_bytes_per_step": d2h_r, "steps": e2e_steps,
                       "what": "as e2e, but every step also copies the three recorder rings of every replica to pinned "
                               "host memory (the last 1024 events / 128 samples of each replica): PCIe-bound by construction"}

    # ---- the other BASELINE configs (parity-test cases, not bench lines): device throughput for context
    others = None
    if a.config == 1 and world == 1 and not a.no_other_configs:
        others = {}

        def ctx(name, mdl, replicas, sim_s, what, **kw):
            e2 = engine.Engine(local, stream=stream.cuda_stream)
            e2.upload(mdl)
            best = None
            for _ in range(2):
                e2.run(engine.make_params(seed=a.seed, end_ns=int(sim_s * 1e9), n_replicas=replicas, flags=0, **kw))
                e2.sync()
                best = e2.last_run_ms() if best is None else min(best, e2.last_run_ms())
            o = e2.read_outputs()
            ev = int(o["summaries"]["events_processed"].sum())
            others[name] = {"value": ev / (best * 1e-3), "unit": UNIT, "replicas": replicas, "sim_seconds": sim_s,
                            "device_ms": best, "replicas_flagged": int((o["summaries"]["status"] != 0).sum()),
                            "what": what}
            e2.close()
        ctx("configs[2]", hs.lb_round_robin(64, 512.0), 16384, 10.0,
            "Source(512/s) -> LoadBalancer(RoundRobin) -> 64 x Server -> Sink; thread engine; 10 s slice of the 100 s run")
        tab = hs.consistent_hash_table([f"S{i}" for i in range(1024)], 100, 10000)
        ctx("configs[3]", hs.lb_key_table(tab, 1024, rate=8192.0), 1024, 2.0,
            "Source(8192/s, 10000 client ids) -> LoadBalancer(ConsistentHash, 100 vnodes) -> 1024 x Server -> Sink; "
            "thread engine; one GPU's 1024 replicas, 2 s slice of the 10 s run (bench.py --config 3 --gpus 4 runs it whole)")
        ctx("configs[4]", hs.mmc_sweep(), 32768, 100.0,
            "M/M/c sweep, 256 (c, rho) cells x 128 seeds on one GPU; lane engine; 100 s slice of the 1000 s run "
            "(bench.py --config 4 --gpus 8 runs it whole)", replicas_per_cell=128, queue_ring=4096)

    if world > 1:
        dist.barrier()
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic", "config": workload_config(a, cfg, world),
                "roofline": roofline, "e2e": e2e, "e2e_records": e2e_records, "gpu_launches": res["launches"], "clocks": clocks,
                "events_timed": events, "per_gpu_events_per_s": value / world,
                "replicas_flagged": agg["replicas_flagged"], "aggregate": agg,
                "parity_sample": dict(parity, ok_all_ranks=parity_ok_all) if parity else None, "cell_allreduce": cell_check,
                "other_mode": other, "other_configs": others, "wall_s_timed_region": res["wall_s"]}
        if world == 1 and not a.no_cpu_baseline:
            cores, core_info = host_cores()
            port, _, _ = cpu_port_throughput(10.0, 500.0, a.seed, cores)
            port["core_accounting"] = core_info
            if reference_available():
                refl, _, _ = cpu_reference_throughput(12.0, cores, a.seed)
                refl["core_accounting"] = core_info
                line["cpu_baseline"] = refl
                line["cpu_baseline_port"] = port
            else:
                line["cpu_baseline"] = port
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
