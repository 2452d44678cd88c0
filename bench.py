#!/usr/bin/env python
"""
bench.py -- anomaly windows/sec of gordo's per-machine autoencoder anomaly path on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c2|c3|c4|c5]
                  [--dump-outputs DIR]

Workloads (BASELINE.json `configs`; SURVEY.md §8d fixes the synthetic inputs: Machine m draws from
default_rng(20260921 + m)):

  c2 (default, the headline): 128 Machines/GPU x 50 tags x 100 000 rows, feed-forward hourglass AE
      50-42-33-25-25-33-42-50 tanh, bf16 tensor-core inference fused with every DiffBasedAnomalyDetector
      .anomaly() column (thresholds / confidences included).  Weak scaling: Machines are dealt round-robin.
  c5: 1 250 Machines/GPU (10 000 on 8 GPUs) x 5 tags x 100 000 rows, same path (HBM-roofline stress).
  c4: 8 Machines x 200 tags x 100 000 rows, KerasLSTMAutoEncoder lookback 128 (167-133-100-100-133-167),
      tensor-core LSTM inference + scoring; STRONG scaling: the 798 984 windows are cut into N contiguous
      window ranges, a Machine's rows are split across ranks with lookback-1 rows of overlap.
  c3: 128 Machines/GPU (1 024 on 8) mixed FF / LSTM(lookback 16), 20-100 tags, 100 000 rows: the builder's
      full build (3 CV folds + final fit + fold scoring + thresholds + CV metrics) + offset inference.

A "step" = one pass of the workload's hot path over every row of every Machine of the rank.
`value` : whole-job windows/s, inputs resident in HBM, CUDA events around K steps, max over ranks.
`e2e`   : the same metric through the plugin surface with HOST buffers -- FleetAnomalyServer.anomaly(X):
          pinned host samples in, every host column out (H2D + kernel + D2H + host expansion timed).
`--impl reference` : the CPU arm = the oracle port of the reference path (Keras cannot be installed
          offline): persistent pool, one pinned process per host CPU, data / weights / scalers prepared
          outside the timed region exactly as the GPU arm prepares them, bounded sample per step.
"""
import os
import sys

if "--impl=reference" in sys.argv or any(a == "--impl" and sys.argv[i + 1:i + 2] == ["reference"]
                                          for i, a in enumerate(sys.argv)):
    # BEFORE numpy is imported: one BLAS / OpenMP thread per worker process (the pool supplies the parallelism)
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS", "NUMEXPR_NUM_THREADS", "VECLIB_MAXIMUM_THREADS"):
        os.environ[_v] = "1"

import argparse
import json
import math
import subprocess
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED0 = 20260921          # SURVEY.md §8d: Machine m uses default_rng(20260921 + m)
METRIC = "anomaly_windows_per_sec"
UNIT = "windows/s"

CONFIGS = {
    "c2": dict(kind="ff", tags=50, rows=100_000, machines_per_gpu=128, scaling="weak"),
    "c5": dict(kind="ff", tags=5, rows=100_000, machines_per_gpu=1250, scaling="weak"),
    "c4": dict(kind="lstm", tags=200, rows=100_000, lookback=128, machines_total=8, scaling="strong"),
    "c3": dict(kind="build", rows=100_000, machines_per_gpu=128, lstm_lookback=16, scaling="weak"),
}


def hourglass_widths(T, encoding_layers=3, cf=0.5):
    smallest = max(min(math.ceil(cf * T), T), 1)
    slope = (T - smallest) / encoding_layers
    dims = [round(T - i * slope) for i in range(1, encoding_layers + 1)]
    return [T] + dims + dims[::-1] + [T]


def machine_data(m, n_rows=100_000, T=50):
    rng = np.random.default_rng(SEED0 + m)
    return rng, rng.random((n_rows, T), dtype=np.float32)


def machine_params(rng, widths):
    parts = []
    for a, b in zip(widths[:-1], widths[1:]):
        lim = np.sqrt(6.0 / (a + b))
        parts += [rng.uniform(-lim, lim, size=(a, b)).astype(np.float32).ravel(), np.zeros(b, np.float32)]
    return np.concatenate(parts)


def machine_thresholds(rng, T):
    return rng.uniform(0.1, 0.5, T), float(rng.uniform(0.01, 0.1))


def c3_machine_shape(m, cfg):
    """SURVEY.md §8d: T_m = 20 + (m*37 mod 81); every 4th Machine is an LSTM autoencoder (lookback 16)."""
    return 20 + (m * 37) % 81, (m % 4 == 3)


DUMP_BYTES = 60 << 20     # --dump-outputs: at most this many bytes of array data (+ one .npy header per array)
DUMP_SEED = 0


def dump_outputs(dump_dir, columns):
    """
    --dump-outputs: write the output arrays of the timed path's last step as DIR/<name>.npy (float32 / float64).
    When they hold more than DUMP_BYTES (counted at 8 bytes a value), they must share their first axis (rows), and
    the same fixed, seeded sample of rows (sorted, default_rng(DUMP_SEED)) is taken from every one of them, so two
    builds of the project can be compared array by array.
    """
    import torch
    os.makedirs(dump_dir, exist_ok=True)
    shapes = [tuple(t.shape) for t in columns.values()]
    rows = shapes[0][0]
    idx = None
    if sum(8 * int(np.prod(s, dtype=np.int64)) for s in shapes) > DUMP_BYTES:
        if any(s[0] != rows for s in shapes):
            raise ValueError("dump_outputs: arrays to be sampled must share their first axis")
        per_row = sum(8 * int(np.prod(s[1:], dtype=np.int64)) for s in shapes)
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(rows, size=DUMP_BYTES // per_row, replace=False))
    for name, t in columns.items():
        if torch.is_tensor(t):
            arr = (t if idx is None else t.index_select(0, torch.as_tensor(idx, device=t.device))).detach().cpu().numpy()
        else:
            arr = np.asarray(t) if idx is None else np.asarray(t)[idx]
        arr = arr.astype(np.float64 if arr.dtype == np.float64 else np.float32, copy=False)
        np.save(os.path.join(dump_dir, f"{name}.npy"), arr)
    what = f"{rows} rows" if idx is None else f"{len(idx)} of {rows} rows, seed {DUMP_SEED}"
    print(f"bench: wrote {len(columns)} output arrays ({what}) to {dump_dir}", file=sys.stderr)


def ff_bytes_per_window(T, conf=True):
    return 4 * T + 4 * (3 * T + 2) + (4 * (T + 1) if conf else 0)


def lstm_flops_per_window(T, L, units):
    return L * sum(8 * u * (i + u) for i, u in zip([T] + list(units[:-1]), units)) + 2 * units[-1] * T


def workload_config(name, n_gpus):
    cfg = CONFIGS[name]
    if cfg["kind"] == "ff":
        T = cfg["tags"]
        w = "-".join(str(v) for v in hourglass_widths(T))
        return {"workload": f"{name}: {cfg['machines_per_gpu']} Machines/GPU x {T} tags x {cfg['rows']} timesteps, "
                            f"feedforward_hourglass AE {w} tanh, fused predict + DiffBasedAnomalyDetector.anomaly "
                            f"columns (with thresholds/confidences)",
                "machines": cfg["machines_per_gpu"] * n_gpus, "tags": T, "rows_per_machine": cfg["rows"],
                "partition": f"machines round-robin over {n_gpus} GPU(s), no collective", "io_dtype": "f32",
                "l2_policy": "inputs+outputs per pass far exceed the 126 MB L2"}
    if cfg["kind"] == "lstm":
        return {"workload": f"{name}: {cfg['machines_total']} Machines x {cfg['tags']} tags x {cfg['rows']} timesteps, "
                            f"KerasLSTMAutoEncoder lstm_hourglass lookback {cfg['lookback']}, predict + "
                            f"DiffBasedAnomalyDetector columns on the offset output",
                "machines": cfg["machines_total"], "tags": cfg["tags"], "rows_per_machine": cfg["rows"],
                "partition": f"windows cut into {n_gpus} contiguous ranges (a Machine's rows split across ranks "
                             f"with lookback-1 rows of overlap), no collective", "io_dtype": "f32",
                "l2_policy": "weights (3.8 MB bf16) L2-resident by design; activations per pass exceed L2"}
    return {"workload": f"{name}: {cfg['machines_per_gpu']} Machines/GPU, every 4th an LSTM AE (lookback "
                        f"{cfg['lstm_lookback']}), T_m = 20 + (37 m mod 81) tags x {cfg['rows']} timesteps, full build "
                        f"(TimeSeriesSplit(3) CV fits + final fit + fold scoring + thresholds + CV metrics, epochs 1, batch 32)",
            "machines": cfg["machines_per_gpu"] * n_gpus, "rows_per_machine": cfg["rows"],
            "partition": f"machines dealt by cost (LPT) over {n_gpus} GPU(s), no collective", "io_dtype": "f32",
            "l2_policy": "training sets (>= 3 GB per rank) exceed L2"}


# ============================================================================= CPU arm (oracle port)
def _prep_ff_case(m, T, rows):
    """Everything the reference holds BEFORE a request arrives: data, fitted weights / scalers / thresholds."""
    from oracle import dense, factories
    from oracle.scaler import MinMaxScaler
    spec = factories.feedforward_hourglass(T)
    rng, X = machine_data(m, rows, T)
    params = dense.ff_unflatten(machine_params(rng, spec["widths"]), spec["widths"])
    ft, at = machine_thresholds(rng, T)
    return dict(kind="ff", spec=spec, X=X, params=params, sx=MinMaxScaler().fit(X), sy=MinMaxScaler().fit(X),
                ft=ft, at=at, windows=rows)


def _run_ff_case(c):
    """The reference path for ONE Machine as the reference runs it: MinMax transform, Keras-style predict in
    batches of 32, float64 pandas-equivalent scoring (diff.py:336-444)."""
    from oracle import dense
    X = c["X"]
    yhat = dense.ff_predict(c["spec"], c["params"], c["sx"].transform(X).astype(np.float32), batch_size=32)
    d_s = np.abs(c["sy"].transform(yhat) - c["sy"].transform(X))
    tot_s = np.square(d_s).mean(axis=1)
    d_u = np.abs(yhat.astype(np.float64) - X)
    tot_u = np.square(d_u).mean(axis=1)
    conf = d_u / c["ft"]; tconf = tot_s / c["at"]
    return float(tot_s.sum() + tot_u.sum() + conf[0, 0] + tconf[0])


def _prep_lstm_case(m, T, L, windows):
    from oracle import factories, lstm as olstm
    from oracle.scaler import MinMaxScaler
    spec = factories.lstm_hourglass(T, lookback_window=L)
    rng, X = machine_data(m, windows + L - 1, T)
    params = olstm.lstm_init(spec, rng)
    return dict(kind="lstm", spec=spec, X=X, params=params, L=L, sx=MinMaxScaler().fit(X), sy=MinMaxScaler().fit(X),
                windows=windows)


def _run_lstm_case(c):
    from oracle import lstm as olstm
    X = c["X"]
    out = olstm.lstm_predict(c["spec"], c["params"], c["sx"].transform(X).astype(np.float32), c["L"], 0)
    y = X[-len(out):]
    d_s = np.abs(c["sy"].transform(out) - c["sy"].transform(y))
    d_u = np.abs(out.astype(np.float64) - y)
    return float(np.square(d_s).mean(axis=1).sum() + np.square(d_u).mean(axis=1).sum())


def _prep_build_case(m, rows):
    from oracle import factories
    T, is_lstm = c3_machine_shape(m, CONFIGS["c3"])
    L = CONFIGS["c3"]["lstm_lookback"]
    spec = factories.lstm_hourglass(T, lookback_window=L) if is_lstm else factories.feedforward_hourglass(T)
    rng, X = machine_data(m, rows, T)
    return dict(kind="build", spec=spec, X=X, rng_seed=SEED0 + m, windows=5 * rows, lstm=is_lstm, L=L)


def _run_build_case(c):
    """ModelBuilder._build's model section for one c3 Machine (feed-forward, or LSTM for every 4th) on a bounded
    row sample: TimeSeriesSplit(3) CV (fit + predict + thresholds per fold) then the final fit + predict."""
    from oracle import dense, lstm as olstm
    from oracle.anomaly import DiffDetector, FFBase, LSTMBase
    X = c["X"]
    rng = np.random.default_rng(c["rng_seed"])
    if c["lstm"]:
        det = DiffDetector(lambda tag: LSTMBase(c["spec"], olstm.lstm_init(c["spec"], rng), lookback_window=c["L"],
                                                epochs=1, batch_size=32))
    else:
        det = DiffDetector(lambda tag: FFBase(c["spec"], dense.ff_init(c["spec"], rng), epochs=1, batch_size=32))
    det.cross_validate(X, X, n_splits=3)
    det.fit(X, X)
    return float(np.asarray(det.predict(X)).sum())


_RUNNERS = {"ff": _run_ff_case, "lstm": _run_lstm_case, "build": _run_build_case}


def _ref_worker(conn, cpu):
    try:
        os.sched_setaffinity(0, {cpu})
    except Exception:
        pass
    cases = []
    while True:
        cmd = conn.recv()
        if cmd[0] == "prep":
            _, name, machines, arg = cmd
            cfg = CONFIGS[name]
            if cfg["kind"] == "ff":
                cases = [_prep_ff_case(m, cfg["tags"], cfg["rows"]) for m in machines]
            elif cfg["kind"] == "lstm":
                cases = [_prep_lstm_case(m, cfg["tags"], cfg["lookback"], arg) for m in machines]
            else:
                cases = [_prep_build_case(m, arg) for m in machines]
            conn.send(sum(c["windows"] for c in cases))
        elif cmd[0] == "run":
            t0 = time.perf_counter()
            chk = sum(_RUNNERS[c["kind"]](c) for c in cases)
            conn.send((time.perf_counter() - t0, chk))
        else:
            return


class ReferencePool:
    """Persistent fork pool, one worker pinned to each host CPU of the affinity mask."""

    def __init__(self, cpus):
        import multiprocessing as mp
        ctx = mp.get_context("fork")
        self.workers = []
        for cpu in cpus:
            a, b = ctx.Pipe()
            p = ctx.Process(target=_ref_worker, args=(b, cpu), daemon=True)
            p.start()
            self.workers.append((p, a))

    def prep(self, name, per_worker, arg=None):
        for w, (_, conn) in enumerate(self.workers):
            conn.send(("prep", name, per_worker[w], arg))
        return sum(conn.recv() for _, conn in self.workers)

    def run(self, only=None):
        ws = self.workers if only is None else [self.workers[i] for i in only]
        t0 = time.perf_counter()
        for _, conn in ws:
            conn.send(("run",))
        res = [conn.recv() for _, conn in ws]
        return time.perf_counter() - t0, res

    def close(self):
        for p, conn in self.workers:
            try:
                conn.send(("quit",))
            except Exception:
                pass
        for p, _ in self.workers:
            p.join(timeout=5)


def reference_sample(name):
    """(machines per worker, per-worker prep argument, description): ~1-3 s of work per worker per step."""
    cfg = CONFIGS[name]
    if cfg["kind"] == "ff":
        k = 4 if cfg["tags"] >= 20 else 8
        return k, None, f"{k} Machine(s) per host CPU ({cfg['tags']} tags x {cfg['rows']} rows each)"
    if cfg["kind"] == "lstm":
        return 1, 192, f"192 windows of one {cfg['tags']}-tag lookback-{cfg['lookback']} Machine per host CPU"
    return 4, 800, ("four consecutive c3 Machines per host CPU (three feed-forward + one LSTM lookback 16, T_m = 20 + (37 m mod 81)) "
                    "on an 800-row sample each (CV + final fit + predict)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    name = args.config
    from gordo_b200.hostbind import cpu_quota, effective_cpus
    cpus = sorted(os.sched_getaffinity(0))
    # one worker per CPU the container may actually use: a GPU lease can SEE every CPU of the host while its
    # cgroup grants the time of a few (round 1: 128 processes delivered 5x one core) -- oversubscribing the quota
    # only adds context switches.  Workers are spread over physical cores (stride over the sorted list).
    q = cpu_quota()                                     # the whole quota: the other ranks of a torchrun launch exit at once
    n_workers = args.ref_procs or (max(1, min(len(cpus), int(q + 0.5))) if q else len(cpus))
    stride = max(1, len(cpus) // n_workers)
    cpus = cpus[::stride][:n_workers]
    k, arg, what = reference_sample(name)
    pool = ReferencePool(cpus)
    try:
        per_worker = [[w * k + i for i in range(k)] for w in range(len(cpus))]
        windows = pool.prep(name, per_worker, arg)
        win_one = windows // len(cpus)
        # one core alone (the reference's builder / server pod is a 1-CPU container), then all of them
        pool.run(only=[0])
        dt1, _ = pool.run(only=[0])
        one_core = win_one / dt1
        for _ in range(args.warmup):
            pool.run()
        tot = 0.0
        for _ in range(args.steps):
            dt, _ = pool.run()
            tot += dt
    finally:
        pool.close()
    value = windows * args.steps / tot
    sample = (f"{what}; {len(cpus)} pinned worker processes, data / weights / scalers prepared outside the timed "
              f"region, oracle port (predict batch_size 32, float64 scoring), OMP/BLAS threads = 1 per worker")
    cpu = {"value": value, "unit": UNIT, "cores": len(cpus), "kind": "port", "sample": sample,
           "one_core_value": one_core, "parallel_efficiency": value / (one_core * len(cpus)),
           "host_cpus_visible": len(os.sched_getaffinity(0)), "cgroup_cpu_quota": cpu_quota()}
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / args.steps,
            "higher_is_better": True, "scaling": CONFIGS[name]["scaling"], "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(name, args.gpus),
            "cpu_baseline": cpu,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))
    return 0


def cpu_baseline_one_core(name, seconds=10.0):
    """cpu_baseline of the main line: the oracle on ONE host core, prepared outside the timed region."""
    cfg = CONFIGS[name]
    if cfg["kind"] == "ff":
        cases = [_prep_ff_case(0, cfg["tags"], cfg["rows"])]
        what = f"Machines of the same workload ({cfg['tags']} tags x {cfg['rows']} rows)"
    elif cfg["kind"] == "lstm":
        cases = [_prep_lstm_case(0, cfg["tags"], cfg["lookback"], 192)]
        what = "192-window slices of one Machine"
    else:
        cases = [_prep_build_case(m, 800) for m in range(4)]
        what = "800-row builds of c3 Machines 0-3 (three feed-forward + one LSTM)"
    run = _RUNNERS[cases[0]["kind"]]
    run(cases[0])
    n, t0 = 0, time.perf_counter()
    while True:
        for c in cases:
            run(c)
        n += 1
        dt = time.perf_counter() - t0
        if dt >= seconds or n >= 64:
            break
    return {"value": n * sum(c["windows"] for c in cases) / dt, "unit": UNIT, "cores": 1, "kind": "port",
            "sample": f"{n} x {what}, {dt:.1f} s, oracle port run as the reference runs it (one Machine at a time, "
                      f"predict batch 32), data / weights / scalers prepared outside the timed region"}


# ============================================================================= clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True); self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = float(r[1])
                for nme, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nme)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ============================================================================= GPU arm
class Ctx:
    """Rank / device / collectives of this process."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(self.world)))
        if self.world != args.gpus and self.world > 1:
            raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={self.world}")
        torch.cuda.set_device(self.local)
        self.dev = torch.device(f"cuda:{self.local}")
        # host side of the rank lives next to its GPU: CPU affinity + preferred NUMA node BEFORE any pinned allocation
        from gordo_b200 import hostbind
        self.bind = hostbind.bind_to_gpu(self.local, self.local, self.local_world) if not args.no_bind else {"source": "off"}
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.peaks = {}
        try:
            self.peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        # collective = False: the side measurements of the default run.  Every rank measures its own shard with
        # NO collective inside (a rank that fails must not strand the others in a barrier and take the headline
        # down); the per-rank results meet in ONE all_gather afterwards.
        self.collective = True

    @property
    def reports(self):
        """Does this rank assemble a result line?  (rank 0, or every rank while collectives are off.)"""
        return self.rank == 0 or not self.collective

    def barrier(self):
        if self.world > 1 and self.collective:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor(list(values), device=self.dev, dtype=self.torch.float64)
        if self.world > 1 and self.collective:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def sum_over_ranks(self, values):
        t = self.torch.tensor(list(values), device=self.dev, dtype=self.torch.float64)
        if self.world > 1 and self.collective:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(v) for v in t]

    def timed(self, fn, steps):
        """K calls of fn between two events on the launching stream, barrier + synchronize on both sides."""
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        return e0.elapsed_time(e1) / steps


def build_ff_fleet(ctx, name, machines=None):
    """This rank's Machines of an ff config: fleet (weights, scalers, thresholds) + pinned host samples."""
    torch = ctx.torch
    from gordo_b200.fleet import FFFleet, FFTopology, Schedule
    from gordo_b200.partition import round_robin
    cfg = CONFIGS[name]
    T, rows = cfg["tags"], cfg["rows"]
    M = machines or cfg["machines_per_gpu"]
    widths = hourglass_widths(T)
    acts = ["tanh"] * (len(widths) - 2) + ["linear"]
    l1 = [0.0] + [1e-4] * 2 + [0.0] * 4
    topo = FFTopology(widths, acts, l1)
    fleet = FFFleet(topo, M, ctx.dev)
    R = M * rows
    x_host = torch.empty((R, T), dtype=torch.float32, pin_memory=True)
    xh = x_host.numpy()
    params = np.empty((M, topo.n_params), np.float32)
    ft = np.empty((M, T), np.float32); at = np.empty((M,), np.float32)
    for i, gid in enumerate(round_robin(M * ctx.world, ctx.world, ctx.rank)):      # global ids rank, rank + world, ...
        rng, X = machine_data(gid, rows, T)
        xh[i * rows:(i + 1) * rows] = X
        params[i] = machine_params(rng, widths)
        f, a = machine_thresholds(rng, T)
        ft[i] = f; at[i] = a
    fleet.set_params(torch.from_numpy(params))
    x_dev = x_host.to(ctx.dev, non_blocking=True)
    lo = torch.arange(M, device=ctx.dev, dtype=torch.int64) * rows
    fleet.in_scale, fleet.in_min = FFFleet.minmax_fit(x_dev, lo, lo + rows)
    fleet.err_scale = fleet.in_scale.clone()
    fleet.feat_thr = torch.from_numpy(ft).to(ctx.dev); fleet.agg_thr = torch.from_numpy(at).to(ctx.dev)
    torch.cuda.synchronize()
    return fleet, Schedule([rows] * M), x_host, x_dev


def run_ff(ctx, args, name, steps, warmup, with_cpu=True, with_other=True, dump_dir=None):
    torch = ctx.torch
    cfg = CONFIGS[name]
    T, rows = cfg["tags"], cfg["rows"]
    fleet, sched, x_host, x_dev = build_ff_fleet(ctx, name, args.machines or None)
    M, R = fleet.M, fleet.M * rows
    prec = fleet.auto_precision(args.precision)
    out = fleet.score(sched, x_dev, precision=prec)                 # allocates the result columns once
    torch.cuda.synchronize()
    step = lambda: fleet.score(sched, x_dev, precision=prec, out=out)
    for _ in range(warmup):
        step()
    sampler = ClockSampler(ctx.local); sampler.start()
    ms_step = ctx.timed(step, steps)
    if dump_dir and ctx.rank == 0:
        dump_outputs(dump_dir, out)                                 # before the other precisions overwrite `out`
    other = []
    if with_other:
        for oprec in ("f16x3", "bf16", "f32"):
            if oprec == prec or (oprec != "f32" and not fleet.tc_eligible(oprec)):
                continue
            ofn = lambda: fleet.score(sched, x_dev, precision=oprec, out=out)
            ofn(); ms_o = ctx.timed(ofn, 3)
            other.append({"precision": oprec, "ms_per_step": ms_o, "value": R / (ms_o * 1e-3),
                          "hbm_frac": R * ff_bytes_per_window(T, True) / (ms_o * 1e-3) / 1e9 / float(ctx.peaks.get("hbm_gbs", 6650.0))})
        step()

    # ---- end to end through the plugin surface: pinned HOST samples in, every HOST column out
    from gordo_b200.serving import FleetAnomalyServer
    del out
    torch.cuda.empty_cache()
    srv = FleetAnomalyServer(fleet, [rows] * M, precision=prec, n_chunks=16, plan=args.plan)
    ctx.barrier()
    srv.anomaly(x_host)                        # first call: all ranks time their transfer plans together
    ctx.barrier()
    e2e_steps = max(1, min(steps, 3))
    res_holder = {}

    def e2e_step():
        res_holder["r"] = srv.anomaly(x_host)
    e2e_step()
    ms_e2e = ctx.timed(e2e_step, e2e_steps)
    clocks = sampler.stop()
    res = res_holder["r"]
    # the host columns of Machine 0 against the device-resident launch (same kernel, same inputs)
    chk = fleet.score(sched, x_dev, precision=prec)
    host_ok = all(bool(torch.allclose(res.columns[k][:rows], chk[k][:rows].cpu(), rtol=1e-5, atol=1e-6))
                  for k in res.columns)
    checksum = float(res.columns["total-anomaly-scaled"][:1000].double().sum())
    plan, by = srv.plan, srv.bytes_per_call()
    host_gbs = None
    try:
        import ctypes as C
        from gordo_b200 import _native as N
        n = 1 << 27
        src = res.columns["model-output"].view(-1)[:n]; dst = res.columns["tag-anomaly-scaled"].view(-1)[:n]
        ctx.barrier()
        s = N.lib().gb200_host_stream_seconds(C.c_void_p(dst.data_ptr()), C.c_void_p(src.data_ptr()), n, srv.n_threads, 3)
        host_gbs = 8 * n / s / 1e9
        ctx.barrier()
    except Exception:
        pass
    ms_step, ms_e2e = ctx.max_over_ranks([ms_step, ms_e2e])
    (all_ok,) = ctx.sum_over_ranks([0.0 if host_ok else 1.0])
    n_w = ctx.world if ctx.collective else 1            # collectives off: this rank's own numbers, combined later
    windows = R * n_w
    line = None
    if ctx.reports:
        peak = float(ctx.peaks.get("hbm_gbs", 6650.0))
        bpw = ff_bytes_per_window(T, conf=True)
        achieved = R * bpw / (ms_step * 1e-3) / 1e9                     # one rank's kernel
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(
                "ff_score_tc_bytes_per_launch" if (prec == "bf16" and name == "c2") else f"{name}_bytes_per_launch")
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": windows / (ms_step * 1e-3), "unit": UNIT, "n_gpus": ctx.world, "steps": steps,
            "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16" if prec == "bf16" else "f32", "data": "synthetic",
            "config": workload_config(name, ctx.world),
            "_raw": {"windows": R, "ms_step": ms_step, "e2e_rows": srv.rows, "ms_e2e": ms_e2e},
            "e2e": {"value": srv.rows * n_w / (ms_e2e * 1e-3), "unit": UNIT,
                    "h2d_bytes_per_step": by["h2d"] * n_w, "d2h_bytes_per_step": by["d2h"] * n_w,
                    "host_derived_bytes_per_step": by["host_derived_bytes"] * n_w,
                    "ms_per_step": ms_e2e, "steps": e2e_steps, "machines_per_gpu": srv.M,
                    "launches_per_step": srv.kernel_launches_per_call(),
                    "api": "gordo_b200.serving.FleetAnomalyServer.anomaly(pinned host X) -> every host column "
                           "(fleet twin of model.anomaly(X, y), server/blueprints/anomaly.py:50)",
                    "transfer_plan": {"host_derived_matrices": plan, "candidates_s": srv.plan_timings,
                                      "host_threads": srv.n_threads, "host_stream_gbs_rank0": host_gbs},
                    "host_columns_match_device": all_ok == 0.0, "numa_bind": {k: v for k, v in ctx.bind.items() if k != "cpus"}},
            "gpu_launches": steps,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if ctx.peaks else "fallback 6650 GB/s",
                         "kernel": "ff_score_tc_kernel" if prec == "bf16" else "ff_score_f32_kernel",
                         "algorithmic_bytes_per_window": bpw},
            "clocks": clocks, "checksum": checksum,
        }
        if other:
            line["other_precisions"] = other
        if with_cpu and ctx.world == 1:          # rank 0 at N = 1 only (the contract); --impl reference is the N-way CPU arm
            line["cpu_baseline"] = cpu_baseline_one_core(name, args.cpu_seconds)
    srv.close()
    del srv, fleet, x_dev, x_host, res, chk
    torch.cuda.empty_cache()
    return line


def lstm_shards(n_machines, rows, L, world):
    """Cut the concatenated window range of all Machines into `world` contiguous pieces ->
    per rank a list of (machine, first window, last window + 1)."""
    per = rows - L + 1
    total = n_machines * per
    cuts = [total * r // world for r in range(world + 1)]
    out = []
    for r in range(world):
        a, b, parts = cuts[r], cuts[r + 1], []
        while a < b:
            m = a // per
            e = min(b, (m + 1) * per)
            parts.append((m, a - m * per, e - m * per))
            a = e
        out.append(parts)
    return out


def run_lstm(ctx, args, name, steps, warmup, with_cpu=True, dump_dir=None):
    torch = ctx.torch
    from gordo_b200.fleet import FFFleet, Schedule
    from gordo_b200.lstm import LSTMFleet
    from gordo_b200.machine.model.factories.lstm_autoencoder import lstm_hourglass
    cfg = CONFIGS[name]
    T, rows, L, Mtot = cfg["tags"], cfg["rows"], cfg["lookback"], cfg["machines_total"]
    topo = lstm_hourglass(T, lookback_window=L)
    mine = lstm_shards(Mtot, rows, L, ctx.world)[ctx.rank]       # (machine, w0, w1): rows [w0, w1 + L - 1)
    J = len(mine)
    counts = [w1 - w0 + L - 1 for _, w0, w1 in mine]
    R = int(sum(counts))
    x_host = torch.empty((R, T), dtype=torch.float32, pin_memory=True)
    gen = torch.Generator(device=ctx.dev)
    params = torch.empty((J, topo.n_params), dtype=torch.float32, device=ctx.dev)
    in_scale = torch.empty((J, T), dtype=torch.float32, device=ctx.dev); in_min = torch.empty_like(in_scale)
    o = 0
    for j, (m, w0, w1) in enumerate(mine):
        rng, X = machine_data(m, rows, T)
        x_host[o:o + counts[j]] = torch.from_numpy(X[w0:w1 + L - 1]); o += counts[j]
        gen.manual_seed(SEED0 + m)                               # a Machine's weights do not depend on the sharding
        params[j] = topo.init_params(1, gen, ctx.dev)[0]
        mn, mx = X.min(axis=0), X.max(axis=0)                    # the Machine's fitted scaler (full rows)
        sc = 1.0 / np.where(mx > mn, mx - mn, 1.0)
        in_scale[j] = torch.from_numpy(sc.astype(np.float32)); in_min[j] = torch.from_numpy((-mn * sc).astype(np.float32))
    fleet = LSTMFleet(topo, J, 0, ctx.dev)
    fleet.set_params(params); fleet.in_scale, fleet.in_min = in_scale, in_min
    err_scale = in_scale.clone()
    x_dev = x_host.to(ctx.dev)
    sched = Schedule(counts)
    prec = "bf16" if fleet.tc_eligible() else "f32"
    y_off = np.concatenate([[0], np.cumsum(counts)])[:-1] + (L - 1)
    n_win = int(sum(w1 - w0 for _, w0, w1 in mine))

    last = {}                                                    # --dump-outputs: the columns of the latest step

    def step():
        out, off = fleet.predict(sched, x_dev, max_windows=18944, precision=prec)
        res = FFFleet.score_outputs(out, x_dev, off, y_off, err_scale=err_scale)
        if dump_dir:
            last.clear(); last["model-output"] = out; last.update(res)
        return out, res
    for _ in range(max(1, warmup)):
        step()
    sampler = ClockSampler(ctx.local); sampler.start()
    ms_step = ctx.timed(step, steps)
    if dump_dir and ctx.rank == 0:
        dump_outputs(dump_dir, last)
    last.clear()
    # e2e: pinned host samples in, host columns out
    host_cols = {}

    def e2e_step():
        xd = x_host.to(ctx.dev, non_blocking=True)
        out, off = fleet.predict(sched, xd, max_windows=18944, precision=prec)
        res = FFFleet.score_outputs(out, xd, off, y_off, err_scale=err_scale)
        res["model-output"] = out
        for k, v in res.items():
            if k not in host_cols:
                host_cols[k] = torch.empty(v.shape, dtype=v.dtype, pin_memory=True)
            host_cols[k].copy_(v, non_blocking=True)
    e2e_step()
    ms_e2e = ctx.timed(e2e_step, max(1, min(steps, 3)))
    clocks = sampler.stop()
    ms_step, ms_e2e = ctx.max_over_ranks([ms_step, ms_e2e])
    (windows,) = ctx.sum_over_ranks([n_win])
    n_w = ctx.world if ctx.collective else 1
    line = None
    if ctx.reports:
        fpw = lstm_flops_per_window(T, L, topo.units)
        peak = float(ctx.peaks.get("bf16_tflops_sustained", 1400.0))
        achieved = n_win * fpw / (ms_step * 1e-3) / 1e12
        d2h = sum(int(v.numel()) * 4 for v in host_cols.values())
        line = {"metric": METRIC, "value": windows / (ms_step * 1e-3), "unit": UNIT, "n_gpus": ctx.world, "steps": steps,
                "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": prec, "data": "synthetic", "config": workload_config(name, ctx.world),
                "_raw": {"windows": n_win, "ms_step": ms_step, "e2e_rows": n_win, "ms_e2e": ms_e2e},
                "e2e": {"value": windows / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": R * T * 4 * n_w,
                        "d2h_bytes_per_step": d2h * n_w, "ms_per_step": ms_e2e,
                        "api": "LSTMFleet.predict + FFFleet.score_outputs on pinned host samples -> pinned host columns"},
                "gpu_launches": steps * 2,
                "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                             "traffic": None, "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if ctx.peaks else "fallback 1400",
                             "kernel": "lstm_persist_tc_kernel" if prec == "bf16" else "lstm_step_kernel",
                             "algorithmic_flops_per_window": fpw},
                "shards_rank0": mine, "clocks": clocks}
        if with_cpu and ctx.world == 1:          # rank 0 at N = 1 only (the contract); --impl reference is the N-way CPU arm
            line["cpu_baseline"] = cpu_baseline_one_core(name, args.cpu_seconds)
    del fleet, x_dev, x_host
    torch.cuda.empty_cache()
    return line


def c3_fleet_machines(ctx, name, machines_per_gpu=None, rows=None):
    """This rank's share of the c3 project as FleetMachine objects (LPT over the model cost)."""
    from gordo_b200.builder import FleetMachine
    from gordo_b200.partition import lpt, machine_cost
    cfg = CONFIGS[name]
    rows = rows or cfg["rows"]
    M_total = (machines_per_gpu or cfg["machines_per_gpu"]) * ctx.world
    shapes = [c3_machine_shape(m, cfg) for m in range(M_total)]
    costs = []
    for T, is_lstm in shapes:
        w = hourglass_widths(T)
        f = 2.0 * sum(a * b for a, b in zip(w[:-1], w[1:]))
        costs.append(machine_cost(rows, f * (4.0 if is_lstm else 1.0), 1, cfg["lstm_lookback"] if is_lstm else 1))
    mine = lpt(costs, ctx.world)[ctx.rank]
    out = []
    for m in mine:
        T, is_lstm = shapes[m]
        _, X = machine_data(m, rows, T)
        if is_lstm:
            est = {"gordo_b200.machine.model.models.KerasLSTMAutoEncoder": {
                "kind": "lstm_hourglass", "lookback_window": cfg["lstm_lookback"], "precision": "bf16"}}
        else:
            est = {"gordo_b200.machine.model.models.KerasAutoEncoder": {"kind": "feedforward_hourglass"}}
        model = {"gordo_b200.machine.model.anomaly.diff.DiffBasedAnomalyDetector": {
            "base_estimator": {"sklearn.pipeline.Pipeline": {"steps": ["sklearn.preprocessing.MinMaxScaler", est]}}}}
        out.append(FleetMachine(name=f"c3-machine-{m}", X=X, model=model, evaluation={"cv_mode": "full_build", "seed": m}))
    return out, shapes, mine


def run_build(ctx, args, name, steps, warmup, with_cpu=True, dump_dir=None):
    torch = ctx.torch
    from gordo_b200.builder import FleetBuild
    cfg = CONFIGS[name]
    rows = args.rows or cfg["rows"]
    machines, shapes, mine = c3_fleet_machines(ctx, name, args.machines or None, rows)
    n_lstm = sum(1 for m in mine if shapes[m][1])
    windows_rank = 5 * rows * len(machines)          # 2.5 N training rows + 2.5 N inference rows per Machine (§8d)
    builder = FleetBuild(machines, device=str(ctx.dev), streams=args.streams)
    for _ in range(min(warmup, 1)):
        builder.build()
    sampler = ClockSampler(ctx.local); sampler.start()
    ctx.barrier()
    t0 = time.perf_counter()
    launches = 0
    for _ in range(steps):
        res = builder.build()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    ctx.barrier()
    clocks = sampler.stop()
    (ms_step,) = ctx.max_over_ranks([dt * 1e3])
    (windows,) = ctx.sum_over_ranks([windows_rank])
    if dump_dir and ctx.rank == 0:
        # what the callers receive: each fitted detector's thresholds, in the order of this rank's Machines
        dump_outputs(dump_dir, {
            "aggregate-threshold": np.array([float(r[0].aggregate_threshold_) for r in res], np.float64),
            "feature-thresholds": np.concatenate([np.asarray(r[0].feature_thresholds_, np.float64) for r in res])})
    line = None
    if ctx.rank == 0:
        thr = [float(r[0].aggregate_threshold_) for r in res[:4]]
        line = {"metric": "build_rows_per_sec", "value": windows / (ms_step * 1e-3), "unit": "rows/s", "n_gpus": ctx.world,
                "steps": steps, "warmup": min(warmup, 1), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32 train, f32/bf16 infer", "data": "synthetic",
                "config": workload_config(name, ctx.world),
                "e2e": {"value": windows / (ms_step * 1e-3), "unit": "rows/s", "ms_per_step": ms_step,
                        "h2d_bytes_per_step": int(sum(np.asarray(m.X).nbytes for m in machines)) * ctx.world,
                        "d2h_bytes_per_step": None,
                        "api": "FleetModelBuilder(machines).build(): host arrays in, fitted host models + metadata out "
                               "(value IS the end-to-end number: the build has no device-resident variant)"},
                "gpu_launches": getattr(builder, "launch_count", None),
                "machines_rank0": {"total": len(machines), "lstm": n_lstm, "buckets": getattr(builder, "last_bucket_count", None),
                                   "bucket_seconds": {k: [round(sum(b[3] for b in builder.bucket_log if b[0] == k), 2),
                                                          round(max([b[3] for b in builder.bucket_log if b[0] == k] or [0]), 2)]
                                                      for k in ("ff", "lstm")},
                                   "slowest_buckets": sorted(((b[0], b[1], round(b[3], 2)) for b in builder.bucket_log), key=lambda b: -b[2])[:6]},
                "rows_per_machine": rows, "aggregate_thresholds_first4": thr, "clocks": clocks}
        if with_cpu and ctx.world == 1:          # rank 0 at N = 1 only (the contract); --impl reference is the N-way CPU arm
            line["cpu_baseline"] = cpu_baseline_one_core(name, args.cpu_seconds)
            if "cpu_baseline" in line:
                line["cpu_baseline"]["unit"] = "rows/s"
    return line


def run_request(ctx, rounds=100):
    """
    The reference's own benchmark shape (benchmarks/test_ml_server.py:21-44: 100 rounds of one POST of 100 rows x 4
    tags to /anomaly/prediction): a fitted Machine, `model.anomaly(X, y, frequency)` host frame in -> host frame out
    (server/blueprints/anomaly.py:50) plus the response body in both wire formats (server/utils.py:47-142), per request.
    """
    import pandas as pd
    from sklearn.pipeline import Pipeline
    from sklearn.preprocessing import MinMaxScaler
    from gordo_b200.machine.model.anomaly.diff import DiffBasedAnomalyDetector
    from gordo_b200.machine.model.models import KerasAutoEncoder
    from gordo_b200.server import utils as server_utils
    rng = np.random.default_rng(SEED0)
    tags = [f"tag-{i}" for i in range(4)]
    Xtrain = pd.DataFrame(rng.random((1000, 4)), columns=tags, index=pd.date_range("2019-01-01", periods=1000, freq="10min", tz="UTC"))
    det = DiffBasedAnomalyDetector(base_estimator=Pipeline([("s", MinMaxScaler()), ("m", KerasAutoEncoder(kind="feedforward_hourglass"))]))
    det.cross_validate(X=Xtrain, y=Xtrain)
    det.fit(Xtrain, Xtrain)
    X = Xtrain.iloc[:100]
    freq = pd.Timedelta("10min")
    out = {}
    for name, fn in (("anomaly_frame", lambda: det.anomaly(X, X, frequency=freq)),
                     ("anomaly_parquet", lambda: server_utils.dataframe_into_parquet_bytes(det.anomaly(X, X, frequency=freq))),
                     ("anomaly_json_dict", lambda: server_utils.dataframe_to_dict(det.anomaly(X, X, frequency=freq))),
                     # the same response bodies straight from the column groups (no DataFrame pivot)
                     ("response_parquet_from_columns", lambda: det.anomaly_response(X, X, frequency=freq, fmt="parquet")),
                     ("response_json_from_columns", lambda: det.anomaly_response(X, X, frequency=freq, fmt="json"))):
        for _ in range(10):
            fn()
        ctx.torch.cuda.synchronize()
        ts = []
        for _ in range(rounds):
            t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
        ts = np.array(ts) * 1e3
        out[name] = {"ms_median": float(np.median(ts)), "ms_p95": float(np.percentile(ts, 95))}
    out["shape"] = "100 rows x 4 tags, 100 rounds (benchmarks/test_ml_server.py:21-44); the reference documents 160-190 ms per request (docs/general/endpoints.rst:223)"
    return out


def run_upstream(ctx, machines=16, tags=50, seconds=86_400, resolution="10T"):
    """
    Upstream of X (SURVEY.md §8 f-4; build_model.py:208-213 -> gordo-core `TimeSeriesDataset.join_timeseries`): raw
    one-second tag series of a small fleet -> resampled, interpolated, joined grids.  `join_call`: host pandas Series in,
    device matrices out (staging + H2D + kernels); `resample_kernel`: the dominant kernel alone on resident samples,
    against the HBM roofline at 16 B per raw point; `cpu_baseline`: the pandas path of the oracle on one Machine.
    """
    import pandas as pd
    from gordo_b200 import dataset as gbd, _native as N
    from oracle import dataset as odataset
    torch = ctx.torch
    start = pd.Timestamp("2022-01-01 00:00:00+00:00"); end = start + pd.Timedelta(seconds=seconds)
    idx = pd.date_range(start, periods=seconds, freq="s")
    rng = np.random.default_rng(SEED0)
    fleet_in = [gbd.MachineSeries([pd.Series(rng.normal(j, 1, seconds), index=idx, name=f"m{m}-t{j}") for j in range(tags)], start, end)
                for m in range(machines)]
    n_points = machines * tags * seconds
    fleet = gbd.FleetTimeSeries(str(ctx.dev))
    walls = []
    for _ in range(4):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        joined = fleet.join(fleet_in, resolution)
        torch.cuda.synchronize(); walls.append(time.perf_counter() - t0)
    wall = float(np.median(walls[1:]))
    out = {"shape": f"{machines} Machines x {tags} tags x {seconds} one-second samples -> {resolution} bins",
           "join_call": {"value": n_points / wall, "unit": "points/s", "s": wall, "rows_out": int(sum(len(j) for j in joined)),
                         "api": "gordo_b200.dataset.FleetTimeSeries.join (host Series in, device grids out)",
                         "h2d_bytes": 16 * n_points}}
    dev = ctx.dev
    step = gbd._step_ns(resolution)
    S = machines * tags
    t = torch.as_tensor(np.tile(idx.as_unit("ns").asi8, S), device=dev)
    v = torch.randn(S * seconds, dtype=torch.float64, device=dev)
    poff = torch.arange(S + 1, device=dev, dtype=torch.int64) * seconds
    nb = seconds * 10 ** 9 // step + 1
    bin0 = torch.full((S,), int(start.value), dtype=torch.int64, device=dev)
    nbins = torch.full((S,), nb, dtype=torch.int64, device=dev)
    ar = torch.arange(S, device=dev, dtype=torch.int64)
    off = (ar // tags) * (nb * tags) + ar % tags
    stride = torch.full((S,), tags, dtype=torch.int64, device=dev)
    res = torch.empty(S * nb, dtype=torch.float64, device=dev)

    def launch():
        N.check(N.lib().gb200_resample(S, N.ptr(poff), N.ptr(t), N.ptr(v), N.ptr(bin0), N.ptr(nbins), N.ptr(off), N.ptr(stride),
                                       step, 0, nb, S * seconds, S * nb, N.ptr(res), torch.cuda.current_stream().cuda_stream),
                "gb200_resample")
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        launch()
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 10
    peak = float(ctx.peaks.get("hbm_gbs", 6650.0))
    ach = (16.0 * n_points + 8.0 * S * nb) / (ms * 1e-3) / 1e9
    out["resample_kernel"] = {"ms": ms, "value": n_points / (ms * 1e-3), "unit": "points/s",
                              "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                           "traffic": None, "bytes": "16 B per raw point (timestamp + value) + 8 B per bin",
                                           "note": "inputs (1.1 GB) exceed L2; 10 back-to-back launches"}}
    t0 = time.perf_counter()
    odataset.join_timeseries(fleet_in[0].series, start, end, resolution)
    out["cpu_baseline"] = {"value": tags * seconds / (time.perf_counter() - t0), "unit": "points/s", "cores": 1, "kind": "port",
                           "sample": "oracle/dataset.py join_timeseries (the pandas calls gordo-core makes) on Machine 0"}
    return out


def run_ours(args):
    ctx = Ctx(args)
    name = args.config
    kind = CONFIGS[name]["kind"]
    t_start = time.perf_counter()
    if kind == "ff":
        line = run_ff(ctx, args, name, args.steps, args.warmup, dump_dir=args.dump_outputs)
    elif kind == "lstm":
        line = run_lstm(ctx, args, name, args.steps, args.warmup, dump_dir=args.dump_outputs)
    else:
        line = run_build(ctx, args, name, args.steps, args.warmup, dump_dir=args.dump_outputs)
    # the default line also carries the other single-pass configurations, measured the same way in the same job.
    # Collective-free (see Ctx.collective): each rank measures its shard alone, one all_gather combines them.
    extras = {}
    if name == "c2" and not args.no_extras:
        (elapsed,) = ctx.max_over_ranks([time.perf_counter() - t_start])
        ctx.barrier()
        ctx.collective = False
        mine = {}
        for other, fn in (("c5", run_ff), ("c4", run_lstm)):
            if elapsed > args.extras_budget:
                mine[other] = {"skipped": "time budget of the default run spent"}
                continue
            t_x = time.perf_counter()
            try:
                kw = dict(with_cpu=False)
                if fn is run_ff:
                    kw["with_other"] = False
                sub = fn(ctx, args, other, max(3, min(args.steps, 5)), 3, **kw)
                mine[other] = {k: sub[k] for k in ("value", "unit", "ms_per_step", "scaling", "dtype", "roofline", "e2e", "config", "_raw")
                               if k in sub}
            except Exception as e:               # an extra must never take the headline down with it
                mine[other] = {"error": f"{type(e).__name__}: {e}"[:300]}
                try:
                    ctx.torch.cuda.synchronize(); ctx.torch.cuda.empty_cache()
                except Exception:
                    pass
            elapsed += time.perf_counter() - t_x
        if ctx.rank == 0 and elapsed <= args.extras_budget:
            try:
                mine["request"] = run_request(ctx)
            except Exception as e:
                mine["request"] = {"error": f"{type(e).__name__}: {e}"[:300]}
            try:
                mine["upstream"] = run_upstream(ctx)
            except Exception as e:
                mine["upstream"] = {"error": f"{type(e).__name__}: {e}"[:300]}
        ctx.collective = True
        gathered = [mine]
        if ctx.world > 1:
            gathered = [None] * ctx.world
            ctx.dist.all_gather_object(gathered, mine)
        if ctx.rank == 0:
            for other in ("c5", "c4"):
                parts = [g.get(other, {}) for g in gathered]
                bad = [p for p in parts if "_raw" not in p]
                if bad:
                    extras[other] = bad[0] if bad[0] else {"error": "missing"}
                    continue
                e = dict(parts[0])
                raws = [p["_raw"] for p in parts]
                ms, ms_e = max(r["ms_step"] for r in raws), max(r["ms_e2e"] for r in raws)
                e["ms_per_step"] = ms
                e["value"] = sum(r["windows"] for r in raws) / (ms * 1e-3)
                e["e2e"] = dict(e["e2e"], value=sum(r["e2e_rows"] for r in raws) / (ms_e * 1e-3), ms_per_step=ms_e,
                                h2d_bytes_per_step=sum(p["e2e"]["h2d_bytes_per_step"] for p in parts),
                                d2h_bytes_per_step=sum(p["e2e"]["d2h_bytes_per_step"] for p in parts))
                e["timing"] = "per-rank CUDA events, no barrier inside the side measurement; max over ranks"
                e.pop("_raw", None)
                extras[other] = e
            if "request" in gathered[0]:
                extras["request_latency"] = gathered[0]["request"]
            if "upstream" in gathered[0]:
                extras["upstream_of_x"] = gathered[0]["upstream"]
    if ctx.rank == 0:
        line.pop("_raw", None)
        if extras:
            line["other_configs"] = extras
        print(json.dumps(line))
    if ctx.world > 1:
        ctx.dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--machines", type=int, default=0, help="Machines per GPU (default: the config's)")
    ap.add_argument("--rows", type=int, default=0, help="c3 only: rows per Machine (default 100 000)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "f32"])
    ap.add_argument("--plan", default="auto", help="e2e transfer plan: auto | 0..3 matrices derived on the host")
    ap.add_argument("--streams", type=int, default=32, help="c3: topology buckets built concurrently (32 LSTM buckets per GPU: 16 -> 32 streams = 47.5 -> 39.2 s)")
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="cpu_baseline sample length (one core)")
    ap.add_argument("--ref-procs", type=int, default=0, help="reference arm: worker processes (default: every host CPU)")
    ap.add_argument("--no-bind", action="store_true", help="do not bind the rank to the GPU's NUMA node")
    ap.add_argument("--no-extras", action="store_true", help="default run: skip the c5 / c4 side measurements")
    ap.add_argument("--extras-budget", type=float, default=150.0, help="seconds after which extras are skipped")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the output columns of the last step (rank 0's Machines; a fixed, "
                         "seeded sample of rows when larger than 60 MB) as DIR/<column>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "ours" and args.warmup < 3:
        args.warmup = 3
    if args.config == "c3" and args.steps > 2 and "--steps" not in " ".join(sys.argv):
        args.steps = 1
    return run_reference(args) if args.impl == "reference" else run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
