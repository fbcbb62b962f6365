#!/usr/bin/env python
"""bench.py — Gibbs-sweep throughput of the hot path.

  python bench.py --gpus N --steps K --warmup W            (our CUDA engine, through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  (the CPU restatement of the reference path)
  python bench.py ... --dump-outputs DIR                   (also write the last step's outputs as DIR/*.npy)

One "step" = one `pgibbs_sweep!`-equivalent over the observation class: the K-particle row
moves of every row + the table-update pass (`--sweep all`: over EVERY class in class_order,
inference.jl:60-81).  Workloads (`--workload`, BASELINE.json configs):
  h1m     synthetic hospital-schema, 1,000,000 dirty rows, K = 20        (configs[3], the default:
          the configuration the north-star target is quoted on; it fits one GPU)
  rents   experiments/rents, 50,000 rows, particle Gibbs K = 20           (configs[1])
  flights experiments/flights, 2,376 rows, particle Gibbs K = 20          (configs[2])
  r10m    synthetic rents-schema, 5 AddTypos columns (--rows, default 10M) (configs[4])
With N > 1 the table is row-sharded across ranks (strong scaling) with the NCCL exchange of
DESIGN.md section 6 per sweep.

Prints ONE JSON line (rank 0).  The oracle (`oracle/`) is only used for the cpu_baseline leg
and for `--impl reference`; the measured product path never touches it.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "gibbs_sweep_rows_x_particles_per_sec"
UNIT = "rows*particles/s"
L2_NOTE = "inputs larger than L2 (126 MB): the distance matrices a sweep streams are GiBs (h1m: 41.9 GiB resident, ~45 KB of them per row)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="h1m", choices=["h1m", "rents", "flights", "r10m"])
    ap.add_argument("--sweep", default="obs", choices=["obs", "all"], help="obs: the observation class (what shards); all: every class in class_order")
    ap.add_argument("--rows", type=int, default=0, help="h1m / r10m: number of synthetic rows (default 1,000,000 / 10,000,000)")
    ap.add_argument("--particles", type=int, default=0, help="default: 20 (r10m: 50)")
    ap.add_argument("--hospitals", type=int, default=4096)
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="time budget of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-rows", type=int, default=0, help="--impl reference: rows each process sweeps per step (default per workload)")
    ap.add_argument("--seed", type=int, default=20260924)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the caller received in the last end-to-end step "
                         "(log-weights and reference slots of the observation rows; with several GPUs, the rows "
                         "rank 0 owns) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    if a.rows <= 0:
        a.rows = {"h1m": 1_000_000, "r10m": 10_000_000, "rents": 50_000, "flights": 2_376}[a.workload]
    if a.particles <= 0:
        a.particles = 50 if a.workload == "r10m" else 20
    return a


WORKLOAD_NAMES = {
    "h1m": "synthetic hospital-schema {rows} rows K={K} (BASELINE.json configs[3])",
    "rents": "experiments/rents {rows} rows, particle Gibbs K={K} (BASELINE.json configs[1])",
    "flights": "experiments/flights {rows} rows, particle Gibbs K={K} (BASELINE.json configs[2])",
    "r10m": "synthetic rents-schema {rows} rows, 5 AddTypos columns, K={K} (BASELINE.json configs[4])",
}


def make_config(a):
    """identical in both arms (the driver compares the dicts)"""
    c = {"workload": WORKLOAD_NAMES[a.workload].format(rows=a.rows, K=a.particles), "rows": a.rows, "particles": a.particles,
         "sweep": "observation class" if a.sweep == "obs" else "all classes (pgibbs_sweep!)", "seed": a.seed,
         "parallelism": f"row-shard x{a.gpus}" if a.gpus > 1 else "single GPU", "l2": L2_NOTE}
    if a.workload == "h1m":
        c.update(hospitals=a.hospitals, typo_rate=0.05)
    return c


def build_workload(a, log):
    """-> dict(model, query, dirty, clean, ir, obs, snap | None, cfg)"""
    from pclean_b200.host_fixture import model as M
    t0 = time.time()
    if a.workload == "h1m":
        from pclean_b200.host_fixture.synth import build_synthetic_hospital
        scale = {} if a.hospitals == 4096 else dict(H=a.hospitals, P=max(4, a.hospitals // 2), C=max(4, a.hospitals // 8))
        model, query, dirty, truth, ir, obs, snap = build_synthetic_hospital(a.rows, a.seed, **scale)
        w = dict(model=model, query=query, dirty=dirty, clean=truth["clean"], ir=ir, obs=obs, snap=snap)
    elif a.workload == "r10m":
        from pclean_b200.host_fixture.synth import build_synthetic_rents
        model, query, dirty, truth, ir, obs, snap = build_synthetic_rents(a.rows, a.seed + 1)
        w = dict(model=model, query=query, dirty=dirty, clean=truth["clean"], ir=ir, obs=obs, snap=snap)
    else:
        from pclean_b200.host_fixture.experiments import load_experiment
        model, query, dirty, clean, ir, obs = load_experiment(a.workload, max_rows=a.rows)
        w = dict(model=model, query=query, dirty=dirty, clean=clean, ir=ir, obs=obs, snap=None)
    rf = 500 if a.workload in ("rents", "r10m") else 50
    w["cfg"] = M.InferenceConfig(1, a.particles, rejuv_frequency=rf)
    log(f"workload {a.workload} built in {time.time() - t0:.1f}s: rows={w['obs'].n_rows} strings={len(w['ir'].strings)}")
    return w


# ------------------------------------------------------------------------------------------
# CPU arm: the oracle (the C++ restatement of the reference path; the reference is Julia and
# cannot run in this image)
# ------------------------------------------------------------------------------------------
_ORACLE = {}


def oracle_for(a, w, log):
    """one oracle per process holding the trace the sweeps start from: the generator's ground truth
    (synthetic workloads; only a prefix of the observation rows is installed, scored against the FULL
    latent tables) or the oracle's own initialize_trace (shipped datasets)"""
    from oracle import Oracle
    o = _ORACLE.get("o")              # forked workers inherit the parent's instance copy-on-write
    if o is not None:
        return o
    from pclean_b200.host_fixture import model as M
    t0 = time.time()
    o = Oracle(w["ir"], w["cfg"], seed=a.seed)
    o.load_observations(w["obs"])
    if w["snap"] is not None:
        cap = min(a.rows, 4096)
        o.install_snapshot(w["ir"], w["model"], w["query"].cls, w["snap"], n_obs_rows=cap, bump_to_full=True)
        o.prefix = cap
    else:
        init_cfg = M.InferenceConfig(1, 2, use_mh_instead_of_pg=True, rejuv_frequency=w["cfg"].rejuv_frequency)
        o.set_config(init_cfg)
        o.initialize_trace()
        o.set_config(w["cfg"])
        o.prefix = w["obs"].n_rows
    log(f"oracle trace ready in {time.time() - t0:.1f}s")
    _ORACLE["o"] = o
    return o


def oracle_sweep_rows(a, w, o, begin, count):
    """run_smc! over `count` observation rows starting at `begin` (wrapping inside the installed prefix)"""
    cls = w["ir"].class_index[w["query"].cls]
    begin %= o.prefix
    end = min(o.prefix, begin + count)
    o.sweep_class(cls, begin, end)
    if end - begin < count:
        o.sweep_class(cls, 0, count - (end - begin))


def cpu_baseline_leg(a, w, seconds, log):
    """single thread (the reference is single-threaded), rows in chunks until the time budget is spent"""
    o = oracle_for(a, w, log)
    o.begin_sweep()
    chunk = 2 if a.workload in ("h1m",) else 50
    done = 0
    t0 = time.perf_counter()
    while done < o.prefix and time.perf_counter() - t0 < seconds:
        oracle_sweep_rows(a, w, o, done, min(chunk, o.prefix - done))
        done += min(chunk, o.prefix - done)
    dt = time.perf_counter() - t0
    return dict(value=done * a.particles / dt, unit=UNIT, cores=1, kind="port",
                sample=f"{done} rows x {a.particles} particles of the same table (full latent tables and option lists) in {dt:.1f}s, "
                       f"single thread (the reference is single-threaded), oracle/pclean_oracle.cpp -O2; host has {os.cpu_count()} logical cores")


_REF = None


def _ref_worker(args):
    step, proc, rows_per_proc = args
    a, w = _REF
    o = oracle_for(a, w, lambda m: None)
    if rows_per_proc <= 0:
        return 0.0
    o.begin_sweep()
    t0 = time.perf_counter()
    oracle_sweep_rows(a, w, o, (step * 9973 + proc) * rows_per_proc, rows_per_proc)
    return time.perf_counter() - t0


def reference_arm(a, config, log):
    """The reference's CPU implementation of the path on the host cores.  The reference is
    single-threaded; rows of the observation class are independent given the table snapshot, so the
    port runs one process per host core (fork), each moving a FIXED number of rows per step (no
    time-boxed chunks: the step is as long as the slowest process), and the rows add up."""
    import multiprocessing as mp
    w = build_workload(a, log)
    ncpu = os.cpu_count() or 1
    procs = max(1, min(int(os.environ.get("PCLEAN_BENCH_PROCS", "0")) or ncpu, 64))
    rows_per_proc = a.ref_rows or {"h1m": 2, "r10m": 20, "rents": 100, "flights": 30}[a.workload]
    global _REF
    _REF = (a, w)
    oracle_for(a, w, log)                      # built once in the parent: the workers inherit it copy-on-write
    times = []
    with mp.get_context("fork").Pool(procs) as pool:
        pool.map(_ref_worker, [(0, p, 0) for p in range(procs)])          # start every worker
        for s in range(a.warmup + a.steps):
            ts = pool.map(_ref_worker, [(s, p, rows_per_proc) for p in range(procs)], chunksize=1)
            if s >= a.warmup:
                times.append(max(ts))
    rows = procs * rows_per_proc * a.steps
    secs = sum(times)
    value = rows * a.particles / secs
    cb = dict(value=value, unit=UNIT, cores=procs, kind="port", host_logical_cores=ncpu,
              sample=f"{procs} processes x 1 thread x {rows_per_proc} rows x {a.particles} particles per step, {a.steps} steps "
                     f"(rows of the same table against the full latent tables; oracle/pclean_oracle.cpp -O2; the reference itself is "
                     f"single-threaded Julia and cannot run in this image); step time = slowest process")
    return {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": 1000.0 * secs / max(1, a.steps), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic" if w["snap"] is not None else "shipped dataset",
            "config": config, "cpu_baseline": cb,
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}


class ClockSampler:
    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        q = "timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        atexit.register(self._close)      # an exception before stop() must not leave nvidia-smi running

    def _close(self):
        if self.p and self.p.poll() is None:
            self.p.terminate()
            try:
                self.p.wait(timeout=5)
            except Exception:
                self.p.kill()
        if os.path.exists(self.f.name):
            self.f.close()
            os.unlink(self.f.name)

    def stop(self, t_begin=None, t_end=None):
        """median SM clock / throttle reasons over the samples taken inside [t_begin, t_end] (time.time());
        nvidia-smi needs ~0.5 s to start, so it is launched long before the timed region"""
        import datetime
        if not self.p:
            self._close()
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        lines = self.f.read().strip().splitlines()
        self._close()
        sm, mx, reasons = [], [], set()
        rows = []
        for line in lines:
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(parts[1]), float(parts[2]), parts[5:9]))
            except ValueError:
                continue
        inside = [r for r in rows if t_begin is None or (t_begin - 0.05 <= r[0] <= t_end + 0.05)]
        if not inside and rows:           # timed region shorter than the sampling period: the samples closest to it (under the same load)
            inside = sorted(rows, key=lambda r: abs(r[0] - (t_end if t_end else r[0])))[:3]
        for ts, a, b, flags in inside:
            sm.append(a); mx.append(b)
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], flags):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def survey_bytes_per_row_particle(model, query, ir, e, nb):
    """SURVEY.md section 8(d): sum_b |C_b| * 4 (F_b + 1) + 4 F_total + 12 bytes per row x particle, with
    |C_b| = candidates of block b's reference table + the new-row branch, F_b = its likelihood terms"""
    tot, ftot = 0.0, 0
    for b in range(nb):
        bm = e.block_metrics(b)
        cands = bm["root_candidates"] + 1
        f = bm["root_terms"]
        tot += cands * 4.0 * (f + 1)
        ftot += f
    return tot + 4.0 * ftot + 12.0


DUMP_BYTES = 60_000_000      # under 64 MB with the .npy headers


def dump_outputs(out_dir, received, r0, r1, seed, log):
    """Write the arrays of `received` (one entry per row of [r0, r1)) as float64 .npy files, with
    `rows.npy` holding the global row indices.  When they do not fit DUMP_BYTES, the same sample of
    rows, drawn from `seed`, is taken from every array, so runs with the same arguments dump the
    same rows."""
    import numpy as np
    n = r1 - r0
    keep = max(1, DUMP_BYTES // (8 * (len(received) + 1)))
    idx = np.arange(n)
    if n > keep:
        idx = np.sort(np.random.default_rng(seed).choice(n, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "rows.npy"), (r0 + idx).astype(np.float64))
    for name, v in received.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), np.asarray(v)[idx].astype(np.float64))
    log(f"dumped {len(received) + 1} arrays of {len(idx)} of {n} rows to {out_dir}")


def main():
    a = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != a.gpus and world > 1:
        a.gpus = world

    def log(msg):
        print(f"[bench r{rank}] {msg}", file=sys.stderr, flush=True)

    config = make_config(a)

    # stdout carries exactly one line, the JSON: whatever libraries write there meanwhile (NCCL's version banner
    # under NCCL_DEBUG=VERSION, for one) goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(json_fd, 1)
        print(json.dumps(obj), flush=True)
        os.dup2(2, 1)

    # ------------------------------------------------------------------ reference arm (CPU)
    if a.impl == "reference":
        if rank != 0:
            return
        emit(reference_arm(a, config, log))
        return

    # ------------------------------------------------------------------ our arm (CUDA)
    import numpy as np
    import torch
    import torch.distributed as dist
    from pclean_b200.engine import Engine, load_trace_from_snapshot

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the engine has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    sampler = ClockSampler(local_rank) if rank == 0 else None      # samples are filtered to the timed region afterwards
    if world > 1:
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local_rank))
    w = build_workload(a, log)
    model, query, ir, obs = w["model"], w["query"], w["ir"], w["obs"]
    n_rows = obs.n_rows
    t0 = time.time()
    e = Engine(ir, w["cfg"], device=local_rank)
    e.load_observations(obs)
    cls = ir.class_index[query.cls]
    nb = len(model.classes[query.cls].blocks)
    fks = [v for v, nd in enumerate(model.classes[query.cls].nodes) if type(nd).__name__ == "ForeignKeyNode"]
    cold = None
    if w["snap"] is not None:
        load_trace_from_snapshot(e, ir, model, query.cls, w["snap"])       # the generator's ground-truth trace
    else:
        t1 = time.time()
        e.init_trace(a.seed)                                              # initialize_trace on the device (setup, untimed)
        cold = {"init_trace_s": time.time() - t1}
    from pclean_b200.parallel import attach_row_shard
    r0, r1 = attach_row_shard(e, cls, n_rows, rank, world)        # contiguous row range per rank + the engine's own NCCL communicator
    sweep_cls = cls if a.sweep == "obs" else -1
    t1 = time.time()
    st = e.sweep(sweep_cls, a.seed, 1)      # first sweep also builds every distance matrix (setup, untimed)
    torch.cuda.synchronize()
    first = {"first_sweep_s": time.time() - t1, "first_sweep_device_ms": st["total_ms"], "changed_rows": st["changed_rows"], "new_rows": st["new_rows"]}
    log(f"engine ready in {time.time() - t0:.1f}s; matrices {e.matrix_bytes() / 2**30:.2f} GiB; first sweep {st}")

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks are sampled from the warm-up steps on (nvidia-smi needs ~0.3 s before its first
    # sample; the GPU is under the same load during warm-up and the timed steps)
    sweep_idx = 2
    for _ in range(max(0, a.warmup - 1)):
        e.sweep(sweep_cls, a.seed, sweep_idx); sweep_idx += 1

    # ---- timed region: device-resident inputs ("value")
    barrier()
    t_begin = time.time()
    wall0 = time.perf_counter()
    kernel_ms = [0.0] * nb
    launches = 0
    tot_ms = 0.0
    stats = []
    for _ in range(a.steps):
        s = e.sweep(sweep_cls, a.seed, sweep_idx); sweep_idx += 1
        tot_ms += s["total_ms"]; launches += s["launches"]; stats.append(s)
        for b in range(nb):
            kernel_ms[b] += e.block_metrics(b)["kernel_ms"]
    barrier()
    wall = time.perf_counter() - wall0
    clocks = sampler.stop(t_begin, time.time()) if sampler else None
    # device time of the steps (engine CUDA events on its own stream), max over ranks
    t = torch.tensor([tot_ms / 1000.0, wall], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_s, wall_s = float(t[0]), float(t[1])
    value = n_rows * a.particles * a.steps / wall_s

    # ---- end-to-end through the C ABI with the CALLER's buffers: the encoded dataset columns a host keeps
    # (dictionary ids / doubles, pinned) go host -> device every step, the sweep runs, the rows' reference
    # slots and log-weights come back — each rank moves only the rows it owns
    from pclean_b200 import lowering as LW
    voc, cells = obs._keep
    cells2 = np.asarray(cells).reshape(obs.n_cols, n_rows)
    sid_cols, real_cols = [], []
    for c in range(obs.n_cols):
        tags = cells2[c]["tag"]
        if np.any((tags == LW.VAL_REAL) | (tags == LW.VAL_INT)):
            buf = torch.empty(n_rows, dtype=torch.float64, pin_memory=True).numpy()
            buf[:] = np.where(tags == LW.VAL_REAL, cells2[c]["d"], np.where(tags == LW.VAL_INT, cells2[c]["i"].astype(np.float64), np.nan))
            sid_cols.append(None); real_cols.append(buf)
        else:
            buf = torch.empty(n_rows, dtype=torch.int32, pin_memory=True).numpy()
            buf[:] = np.where(tags == LW.VAL_STR, cells2[c]["i"], -1)
            sid_cols.append(buf); real_cols.append(None)
    e.update_observations(sid_cols, real_cols, r0, r1)            # untimed first pass (builds the id -> unique-value maps)
    e.download_logweights_range(cls, r0, r1)
    barrier()
    w0 = time.perf_counter()
    h2d = d2h = 0
    received = {}
    for _ in range(a.steps):
        h2d = e.update_observations(sid_cols, real_cols, r0, r1)
        e.sweep(sweep_cls, a.seed, sweep_idx); sweep_idx += 1
        d2h = 0
        for f in fks:
            k = e.download_assignment_range(cls, f, r0, r1)
            d2h += k.nbytes // 2                                   # device side: int32 slots
            received[f"assignment_v{f}"] = k
        lw = e.download_logweights_range(cls, r0, r1)
        d2h += lw.nbytes
        received["logweights"] = lw
    barrier()
    t = torch.tensor([time.perf_counter() - w0, float(h2d), float(d2h)], dtype=torch.float64, device="cuda")
    tsum = t.clone()
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
    e2e_value = n_rows * a.particles * a.steps / float(t[0])
    h2d_total, d2h_total = int(tsum[1]), int(tsum[2])                 # whole job, all ranks

    if rank == 0 and a.dump_outputs:
        dump_outputs(a.dump_outputs, received, r0, r1, a.seed, log)
    if rank == 0:
        # roofline of the dominant kernel (the block kernel with the larger device time)
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
        dom = max(range(nb), key=lambda b: kernel_ms[b])
        bm = e.block_metrics(dom)
        rows_rank = r1 - r0
        k_ms = kernel_ms[dom] / a.steps
        # (1) what the kernel is built to read: 1 B per (enumerated element x likelihood term) per ROW
        #     (shared by the K particles, before pruning) + 12 B per row x particle written
        alg_engine = bm["distance_bytes_per_row"] * rows_rank + 12.0 * a.particles * rows_rank
        # (2) SURVEY 8(d)'s per row x particle figure (the reference re-enumerates per particle, int32 codes)
        alg_survey = survey_bytes_per_row_particle(model, query, ir, e, nb) * rows_rank * a.particles
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "kblock_traffic_r2.json")
        if world == 1 and a.workload == "h1m" and a.rows == 1000000 and a.particles == 20 and os.path.exists(tpath):
            traffic = json.load(open(tpath)).get(f"k_block(block={dom})")     # ncu dram__bytes_read+write of this exact workload, per launch
        secs = k_ms * 1e-3
        measured = traffic / secs / 1e9 if (traffic and secs > 0) else None
        eng_gbs = alg_engine / secs / 1e9 if secs > 0 else 0.0
        achieved = measured if measured is not None else eng_gbs
        roofline = {"bound": "hbm", "kernel": f"k_block(block={dom})", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src, "kernel_ms": k_ms,
                    "achieved_basis": "measured DRAM bytes (ncu dram__bytes_read.sum + dram__bytes_write.sum of this workload, profiles/) / live kernel time"
                                      if measured is not None else "engine-algorithmic bytes (no ncu capture of this configuration)",
                    "algorithmic": {"engine_bytes_per_launch": alg_engine, "engine_gbs": eng_gbs, "engine_frac": eng_gbs / peak,
                                    "survey_8d_bytes_per_launch": alg_survey, "survey_8d_gbs": alg_survey / secs / 1e9 if secs > 0 else 0.0,
                                    "note": "engine: 1 B per (enumerated element x likelihood term) per row, shared by the K particles of a row, + 12 B per "
                                            "row x particle written; survey 8(d): |C| x 4 (F + 1) B per row x PARTICLE (the reference re-enumerates per "
                                            "particle).  K-sharing, uint8 distances, pruning and the memo are why the kernel never reads the survey figure: "
                                            "it is an algorithmic credit, not a bandwidth."},
                    "all_blocks_ms": [x / a.steps for x in kernel_ms]}
        npath = os.path.join(ROOT, "profiles", "kblock_ncu_r2.json")
        if traffic is not None and os.path.exists(npath):
            # what the kernel is bound by instead (it moves 3 % of the HBM peak): the committed ncu capture of this workload
            roofline["ncu"] = json.load(open(npath)).get(f"k_block(block={dom})")
            roofline["limiter"] = "issue slots / dependent-load latency (32 resident warps per SM at the 64-register cap), not bytes: see DESIGN.md 5.1"
        cpu_baseline = None
        if not a.no_cpu_baseline and world == 1:
            cpu_baseline = cpu_baseline_leg(a, w, a.cpu_seconds, log)
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
               "ms_per_step": 1000.0 * wall_s / a.steps, "device_ms_per_step": 1000.0 * dev_s / a.steps,
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": "f64", "data": "synthetic" if w["snap"] is not None else "shipped dataset", "config": config,
               "roofline": roofline, "cpu_baseline": cpu_baseline, "clocks": clocks,
               "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_total, "d2h_bytes_per_step": d2h_total},
               "gpu_launches": int(launches), "matrices_gib": e.matrix_bytes() / 2**30,
               "setup": dict(first, **(cold or {})),
               "sweep": {"new_rows": sum(s["new_rows"] for s in stats), "changed_rows": sum(s["changed_rows"] for s in stats),
                         "dummy_draws": sum(s["dummy_draws"] for s in stats)}}
        if w["snap"] is None:
            # shipped datasets: the F1 of the trace the timed sweeps left behind (analysis.jl:36-88)
            from pclean_b200.host_fixture.analysis import evaluate_accuracy
            cols = list(query.cleanmap.keys())
            cells = e.download_cells(cls, [query.cleanmap[c] - 1 for c in cols], n_rows)
            ours = {c: [e.decode(cells[k, r]) for r in range(n_rows)] for k, c in enumerate(cols)}
            acc = evaluate_accuracy(w["dirty"], w["clean"], ours, cols)
            out["f1"] = {"f1": acc["f1"], "precision": acc["precision"], "recall": acc["recall"],
                         "after": f"initialize_trace + {1 + max(0, a.warmup - 1) + 2 * a.steps} sweeps ({config['sweep']})"}
        emit(out)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
