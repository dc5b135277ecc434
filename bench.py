#!/usr/bin/env python
"""bench.py — LM iterations/sec (linearize + damped multifrontal solve + retract + error)
on the BAL-style workloads of BASELINE.json, through the C-ABI library.

    python bench.py --gpus N --steps K --warmup W [--workload NAME] [--impl reference] [--dump-outputs DIR]

One "step" = one LevenbergMarquardtOptimizer::iterate() from the same initial
estimate (values restored, lambda reset), i.e. one linearize + >=1 damped
factor/solve/retract/error tries.  `value` times it with the inputs resident in
HBM; `e2e` times the same step through the public call with HOST buffers
(host->device copy of the Values, device->host read-back of the new Values and
the error inside the timed region).

Default workload (every N): BASELINE.json configs[4], the 10M-factor graph (5k cameras / 2M points, the
reference's METIS ordering, FP32 linearize output + FP64 solve) — the largest config, it fits one B200 — so the
driver's 1 -> 8 GPU curve is north_star's strong-scaling curve ("value" = iterations/s of THAT graph at every N; the
N ranks shard it).  At N = 1 the same line also carries north_star's 1M-factor graph (bal_1m, the >= 10x target) and
configs[2] (bal_c3) as `other_workloads`, each with its own phases, roofline and CPU baseline.  At N > 1 rank 0
also solves the same graph unsharded once and the line carries `parity` (sharded vs single-GPU delta / error).

`--impl reference` times the UNMODIFIED reference (oracle/_ref, built from /root/reference by oracle/Makefile;
falls back to the plain-C oracle port when that binary is absent) on the host cores, on the same workload.

`--dump-outputs DIR` writes, per workload, what the last timed step handed its caller: the packed Values after the
iterate() (`<workload>_values.npy`, float64; above DUMP_VALUES_MAX entries a fixed, seeded sample of them) and the LM
error and lambda (`<workload>_error.npy`, `<workload>_lambda.npy`).  The workloads are generated from fixed seeds, so
two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

PRIMARY = "bal_c5_metis"            # BASELINE configs[4]
SECONDARY = ("bal_1m", "bal_c3")    # north_star's 1M-factor target, BASELINE configs[2]
# seconds per reference iterate() measured in the build container (one thread): bounds the CPU legs
REF_EST = {"bal_c3": 2.0, "bal_1m": 9.0, "bal_c4": 40.0, "bal_c5": 200.0, "sphere2500": 0.3, "sphere2500_metis": 0.3,
           "bal_1m_metis": 9.0, "bal_c4_metis": 35.0, "bal_c5_metis": 140.0}


def int_at_least(lo):
    def parse_int(s):
        v = int(s)
        if v < lo:
            raise argparse.ArgumentTypeError(f"must be >= {lo}, got {v}")
        return v
    return parse_int


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int_at_least(1),
                    help="timed steps, one LM iterate() each (default 20; --impl reference: as many as fit about 150 s "
                         "of the reference's iterate())")
    ap.add_argument("--warmup", type=int_at_least(0),
                    help="untimed steps before them (default 3, and at least 3 on the GPU; --impl reference: 0 to 3 by "
                         "the reference's iterate() time)")
    ap.add_argument("--workload", default="auto", help=f"auto = {PRIMARY} (+ {', '.join(SECONDARY)} as other_workloads at N = 1)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-others", action="store_true", help="N = 1: skip the other_workloads records")
    ap.add_argument("--no-flush-l2", action="store_true", help="time the K steps back to back with L2 left warm")
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="N > 1: strong = the named graph sharded over the N ranks (default; BASELINE configs[3]/[4]); "
                         "weak = BAL graphs get N x the points (cameras fixed)")
    ap.add_argument("--jacobian", default="auto", choices=["auto", "fp64", "fp32"],
                    help="storage of the whitened Jacobians; auto = fp32 for the 10M-factor config (BASELINE configs[4]: "
                         "'FP32 linearize + FP64 solve'), fp64 otherwise")
    ap.add_argument("--jacobian-fp32", action="store_true", help="same as --jacobian fp32")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes what the library computed; --impl reference runs no library step")
    else:
        args.steps = 20 if args.steps is None else args.steps
        args.warmup = 3 if args.warmup is None else args.warmup
    return args


METRIC = "LM iterations/sec (linearize+solve) on BAL-style graph"
UNIT = "iterations/s"


def jac32_for(args, workload):
    if args.jacobian_fp32 or args.jacobian == "fp32":
        return True
    return args.jacobian == "auto" and workload.startswith("bal_c5")


def workload_config(prob, workload, jac32, world, scaling, flush=True):
    return {
        "workload": f"{workload}: {prob.name}", "factors": prob.nfactors, "variables": prob.nvars,
        "factor_types": sorted({int(g.type) for g in prob.groups}),
        "ordering": ("Schur (points, then cameras)" if prob.meta.get("ordering", "schur") == "schur" else
                     f"{prob.meta['ordering'].upper()} by the reference's Ordering::Create (shipped as data)") if prob.meta.get("kind") == "bal"
        else prob.meta.get("ordering", "natural"),
        "lm_params": "LevenbergMarquardtParams::LegacyDefaults (lambda0=1e-5, factor 10)",
        "jacobian_storage": "fp32 (b200_set_jacobian_precision: FP64 evaluation, float [A|b], FP64 solve)" if jac32 else "fp64",
        "cache": ("L2 flushed between timed iterations: 256 MiB memset on the stream, outside the per-iteration CUDA-event pairs" if flush
                  else "L2 left warm between iterations (--no-flush-l2)"),
        "parallelism": "single GPU" if world == 1 else
        f"{world} ranks, one per GPU, {scaling} scaling: junction-tree subtrees (BAL: the points and the lower camera supernodes) "
        f"+ their factors sharded by rank; the top of the tree is distributed: every top front has an owner, per top level one NCCL "
        f"all-reduce (FP64 sum over NVLink / NVSwitch) of that level's fronts, the owners factor them; back-substitution exchanges the "
        f"owners' solutions per level; one all-reduce of the LM scalars per try; value = iterations/s of the graph actually solved",
    }


# float64 entries of one workload's Values written by --dump-outputs (16 MiB): the three workloads of a default run
# stay under 64 MiB in all
DUMP_VALUES_MAX = 1 << 21


def dump_outputs(outdir, workload, values, error, lam):
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    if values.size > DUMP_VALUES_MAX:        # same indices at every run: the seed and the size fix them
        idx = np.sort(np.random.default_rng(0).choice(values.size, DUMP_VALUES_MAX, replace=False))
        values = values[idx]
    np.save(os.path.join(outdir, f"{workload}_values.npy"), np.ascontiguousarray(values, dtype=np.float64))
    np.save(os.path.join(outdir, f"{workload}_error.npy"), np.array([error], dtype=np.float64))
    np.save(os.path.join(outdir, f"{workload}_lambda.npy"), np.array([lam], dtype=np.float64))


# ------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,timestamp")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "20"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            # nvidia-smi needs a few hundred ms before its first row; the timed region of a 20-step run is shorter than that,
            # so the sampler is started before the one-time problem setup and the bench waits here for the first row
            t0 = time.time()
            while not self.rows and time.time() - t0 < 5.0 and self.proc.poll() is None:
                time.sleep(0.02)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    @staticmethod
    def _epoch(ts):
        import datetime
        try:
            return datetime.datetime.strptime(ts.strip(), "%Y/%m/%d %H:%M:%S.%f").timestamp()
        except Exception:
            return None

    def stop(self, region=None):
        """region = (epoch start, epoch end) of the timed loop: only samples taken inside it count (a short
        region may hold none: then all samples of the run, warm-up included, are used and `in_region` is 0)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = self.rows
        in_region = 0
        if region is not None:
            inside = [r for r in rows if len(r) > 7 and self._epoch(r[7]) is not None
                      and region[0] - 0.02 <= self._epoch(r[7]) <= region[1] + 0.02]
            in_region = len(inside)
            if inside:
                rows = inside
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "in_region": in_region, "reasons": sorted(reasons)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------
def reference_time(prob, steps, warmup):
    """Times LevenbergMarquardtOptimizer::iterate() of the reference on the host cores.
    Returns (seconds per iterate, dict describing the run)."""
    from oracle import refio
    ncores = os.cpu_count()
    if refio.have_ref():
        try:
            r = refio.time_lm(prob, steps, warmup)
            return r["mean_s"], {"kind": "reference", "cores": 1, "host_cores": ncores,
                                 "sample": f"{steps} x LevenbergMarquardtOptimizer::iterate() of the unmodified reference "
                                           f"(oracle/_ref, -O3, no TBB in this image => single thread) on the full workload, "
                                           f"{warmup} warm-up; linearize {r['linearize_s']:.3f}s, damped solve {r['solve_s']:.3f}s",
                                 "error_after": r["error_after"], "inner_iterations": r["inner_iterations"]}
        except Exception as e:  # binary present but not runnable on this box
            note = f"oracle/_ref not runnable here ({type(e).__name__}); "
    else:
        note = "oracle/_ref absent; "
    from gtsam_b200 import problem as P
    from oracle import oracle_py as O
    op = O.OracleProblem(prob)
    v0 = prob.values.copy()
    prm = P.CLMParams(100, 1e-5, 1e-5, 0.0, 1e-5, 10.0, 1e5, 0.0, 1e-3, 0, 1, 1e-6, 1e32)
    ts = []
    for s in range(warmup + steps):
        op.set_values(v0)
        lm = op.lm(prm)
        t0 = time.perf_counter()
        op.lm_iterate(lm)
        if s >= warmup:
            ts.append(time.perf_counter() - t0)
    return sum(ts) / len(ts), {"kind": "port", "cores": 1, "host_cores": ncores,
                               "sample": note + f"{steps} x LM iterate of the plain-C oracle port on the full workload"}


def make_problem(args, workload, world):
    """The graph the N ranks solve: the named workload itself (strong scaling, default), or N x its points (weak)."""
    from gtsam_b200 import datasets
    over = {}
    if world > 1 and args.scaling == "weak":
        base = datasets.WORKLOADS[workload][1]
        if "npoints" in base and base.get("ordering", "schur") == "schur":   # stored orderings fit one size
            over["npoints"] = base["npoints"] * world
    return datasets.make(workload, **over), bool(over)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    workload = PRIMARY if args.workload == "auto" else args.workload
    prob, weak = make_problem(args, workload, args.gpus)      # the same graph as the GPU arm at this N
    est = REF_EST.get(workload, 1.0) * (args.gpus if weak else 1)
    # unless given, steps and warm-up are bounded by the reference's iterate() time (bal_c5_metis: 140 s per step)
    steps = args.steps if args.steps is not None else max(1, min(20, int(150.0 / est)))
    warmup = args.warmup if args.warmup is not None else (0 if est > 30 else (1 if est > 1 else 3))
    sec, info = reference_time(prob, steps, warmup)
    val = 1.0 / sec
    line = {"metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak" if weak else "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "impl": "reference",
            "config": workload_config(prob, workload, False, args.gpus, "weak" if weak else "strong"),
            "cpu_baseline": dict(info, value=val, unit=UNIT),
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------
def schur_bytes(prob, jb=8):
    """Algorithmic bytes of leaf_point_schur_kernel: read [S' d'] (3 x DC per factor + 3 per point, FP64) and
    [A_c b] (2 x DC + 2 per factor, jb bytes each); the run's extend-add output is negligible."""
    from gtsam_b200 import problem as P
    total = 24 * int((prob.var_type == P.VAR_POINT3).sum())
    for g in prob.groups:
        if g.type in (P.FACTOR_PROJECTION_CAL3S2, P.FACTOR_SFM_BUNDLER):
            dc = P.factor_ncols(g.type) - 4       # camera dofs: ncols = DC + 3 + 1
            total += g.count * (8 * 3 * dc + jb * (2 * dc + 2))
    return total


def P_ncols(g):
    from gtsam_b200 import problem as P
    return P.FACTOR_DIM[g.type] * P.factor_ncols(g.type)


def dense_front_model(dev, prob):
    """Flops (f^3/3 + f^2 s + f s^2) and conditional bytes of the supernodes that go through the dense-front kernels,
    i.e. everything but the fused leaf cliques (level 0, <= 6 pivots, f x n <= 768: the BAL points / Pose3 leaves);
    plus the bytes of every conditional [R S d] (what back-substitution reads once)."""
    import numpy as np
    fp, fv, sp, sv, par = dev.supernodes()
    dims = prob.var_dims.astype(np.int64)
    cf = np.concatenate([[0], np.cumsum(dims[fv])])
    cs = np.concatenate([[0], np.cumsum(dims[sv])]) if len(sv) else np.zeros(1, dtype=np.int64)
    nf = (cf[fp[1:]] - cf[fp[:-1]]).astype(np.float64)
    ns = (cs[sp[1:]] - cs[sp[:-1]]).astype(np.float64)
    has_child = np.zeros(len(par), dtype=bool)
    has_child[par[par >= 0]] = True
    leaf = (~has_child) & (nf <= 6) & (nf * (nf + ns + 1) <= 768)
    fl = nf ** 3 / 3 + nf ** 2 * ns + nf * ns ** 2
    return {"dense_flops": float(fl[~leaf].sum()), "leaf_flops": float(fl[leaf].sum()), "dense_fronts": int((~leaf).sum()),
            "conditional_bytes": float((nf * (nf + ns + 1)).sum() * 8),
            "max_dense_front": [int(nf[~leaf].max()) if (~leaf).any() else 0, int(ns[~leaf].max()) if (~leaf).any() else 0]}


def measure(args, workload, ctx, dist, rank, local, world, primary):
    """One workload through the library: returns the record (rank 0) or None."""
    import numpy as np
    import torch
    from gtsam_b200 import capi, optimizer

    jac32 = jac32_for(args, workload)
    jb = 4 if jac32 else 8
    sampler = ClockSampler(local)
    if rank == 0 and primary:
        sampler.start()
    t0 = time.perf_counter()
    prob, weak = make_problem(args, workload, world)
    gen_s = time.perf_counter() - t0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    dev = capi.DeviceProblem(ctx, prob)       # one-time: pack + symbolic phase (host) + upload
    if jac32:
        dev.set_jacobian_precision(True)
    dev.synchronize()
    setup_ms = (time.perf_counter() - t0) * 1e3
    lm = optimizer.LevenbergMarquardtOptimizer(ctx, prob, device_problem=dev)
    stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", local))
    L = dev.L
    # the step's host buffers are page-locked (contract: inputs come from pinned host memory)
    host_values = torch.from_numpy(prob.values.copy()).pin_memory().numpy()
    host_out = torch.empty(host_values.size, dtype=torch.float64).pin_memory().numpy()
    dev.save_values()

    # One step = one iterate().  Putting the optimizer back on the initial estimate (values restored device-side, state <-
    # (values, lambda0, graph.error)) is the counterpart of CONSTRUCTING the optimizer, which the reference arm does before its
    # clock starts (oracle/ref_harness.cpp cmd_time: fresh LevenbergMarquardtOptimizer, then the timed lm.iterate()): untimed here too.
    def prepare_resident():
        dev.restore_values()                    # D2D: inputs already in HBM
        capi._check(L.b200_lm_reset(lm.h))      # state <- (values, lambda0); recomputes graph.error

    def step_resident():
        lm.iterate()

    # sharded: a rank moves only its share (b200_values_view): in = the variables its factors touch + its cliques' and the
    # top's frontal variables; out = the variables it owns (rank 0 reports the top); the caller stitches the N owned views
    if world > 1:
        idx_in, idx_own = dev.view_index(0), dev.view_index(1)
        host_in = torch.from_numpy(np.ascontiguousarray(prob.values[idx_in])).pin_memory().numpy()
        host_own = torch.empty(idx_own.size, dtype=torch.float64).pin_memory().numpy()
        h2d_bytes, d2h_bytes = int(host_in.nbytes), int(host_own.nbytes) + 64

        def step_e2e():
            dev.set_values_view(host_in)            # pinned host -> device, this rank's input view
            capi._check(L.b200_lm_reset(lm.h))
            lm.iterate()
            out = dev.get_values_view(host_own)     # device -> pinned host, the variables this rank owns
            return out, lm.error()
    else:
        h2d_bytes, d2h_bytes = int(host_values.nbytes), int(host_values.nbytes) + 64

        def step_e2e():
            dev.set_values(host_values)             # pinned host -> device
            capi._check(L.b200_lm_reset(lm.h))
            lm.iterate()
            out = dev.get_values(host_out)          # device -> pinned host
            return out, lm.error()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # L2 flush between timed iterations (the working set of bal_c3 is about the size of the 126 MB L2): each iteration
    # is timed on its own (event pair on the library's stream) and a 256 MiB memset on the same stream evicts L2 in
    # between, outside the event pairs.  (The 1M+ factor workloads stream more than L2 holds anyway.)
    flush_buf = None if args.no_flush_l2 else torch.empty(256 << 20, dtype=torch.uint8, device=torch.device("cuda", local))

    def flush_l2():
        with torch.cuda.stream(stream):
            flush_buf.zero_()

    def timed(fn, steps, warmup, flush=True, prepare=None):
        """Every step has its own CUDA-event pair on the library's stream; `prepare` (and the L2 flush) run between the pairs."""
        for _ in range(warmup):
            if prepare:
                prepare()
            fn()
        barrier()
        flush = flush and flush_buf is not None
        pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        nlaunch = 0
        t0 = time.perf_counter()
        timed.region = [time.time(), None]
        for a, b in pairs:
            if prepare:
                prepare()
            if flush:
                flush_l2()
            l0 = ctx.launch_count()
            a.record(stream)
            fn()
            b.record(stream)
            nlaunch += ctx.launch_count() - l0
        barrier()
        wall = time.perf_counter() - t0
        timed.region[1] = time.time()
        ms = sum(a.elapsed_time(b) for a, b in pairs)
        if dist is not None:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, wall, nlaunch

    steps = args.steps
    ms, wall, launches = timed(step_resident, steps, max(3, args.warmup), prepare=prepare_resident)
    clocks = sampler.stop(tuple(timed.region)) if (rank == 0 and primary) else None
    if args.dump_outputs:
        out_values = dev.get_values_all() if world > 1 else dev.get_values()    # (get_values_all is collective)
        if rank == 0:
            out_state = lm._state()
            dump_outputs(args.dump_outputs, workload, out_values, out_state.error, out_state.lambda_)
    ms_e2e, wall_e2e, _ = timed(step_e2e, steps, 1)
    ms_warm, _, _ = timed(step_resident, steps, 1, flush=False, prepare=prepare_resident)   # information only: L2 left warm between iterations

    # phase profile (separate pass; event records add ~1 us per phase)
    for it in range(steps):
        prepare_resident()
        dev.profile_enable(1 if it == 0 else 2)       # the phase timers see the timed part only (2 = resume)
        step_resident()
        dev.synchronize()
        dev.profile_enable(0)
    prof = dev.profile()
    st = lm._state()

    parity = None
    if world > 1:
        parity = sharded_parity(prob, dev, lm, ctx, dist, rank, local, world, jac32, st)
    if rank != 0:
        del lm
        dev.close()
        return None
    value = steps / (ms * 1e-3)          # iterations/s of the graph actually solved (at every N)
    e2e = steps / (ms_e2e * 1e-3)
    info = dev.symbolic_info()
    model = dense_front_model(dev, prob)
    peak, peak_src = measured_peaks()
    per_step = {k: (v[0] / steps, v[1] / steps) for k, v in prof.items()}
    tries = max(1.0, per_step["leaf_fused"][1] if per_step["leaf_fused"][1] else per_step["back_substitute"][1])
    jac_bytes = sum(g.count * jb * P_ncols(g) for g in prob.groups)
    # algorithmic bytes / flops per launch of every phase with a model (DESIGN.md 5); sharded: each rank does 1/world
    alg_bytes = {
        "linearize": prob.linearize_bytes(jb),                   # SURVEY 8(d): 184 B/projection factor + Values
        "memset_fronts": info.front_bytes,
        "leaf_fused": jac_bytes + info.front_bytes,              # read [A|b] of the leaf factors, write [R S d]
        "leaf_schur": schur_bytes(prob, jb),
        "back_substitute": model["conditional_bytes"],           # every conditional [R S d] read once
        "linear_error": jac_bytes, "error": prob.linearize_bytes(jb) - jac_bytes,
    }
    kernels = {"linearize": "linearize_kernel", "leaf_fused": "leaf_point_factor_kernel / leaf_fused_kernel",
               "leaf_schur": "leaf_point_schur_mma_kernel (per-run Schur complement of the point leaves: 8x8 DMMA tiles)", "memset_fronts": "memset", "linear_error": "linerr_kernel",
               "error": "error_kernel", "eliminate_large": "front_df_kernel (tile dataflow: Cholesky + TRSM + DMMA rank-32 updates + extend-add of every non-leaf front, one launch)",
               "back_substitute": "backsub_large_kernel / backsub_small_kernel / backsub_point_kernel"}
    fp64 = measure.fp64_peaks

    def roof(name):
        """achieved = algorithmic bytes (or flops) of the phase per lambda try / its duration (CUDA events on the launching
        stream, the library's phase timers); linearize runs once per step, the solve phases once per try."""
        ms_phase, _calls = per_step[name]
        if ms_phase <= 0:
            return None
        units = 1.0 if name == "linearize" else tries
        if name == "eliminate_large":
            fl = model["dense_flops"]                # supernodes that go through the dense-front kernels ONLY (no leaf flops)
            ach = fl * units / (ms_phase * 1e-3) / 1e12
            return {"kernel": kernels[name], "phase": name, "bound": "tensor", "achieved": ach, "peak": fp64[0], "unit": "TFLOP/s",
                    "frac": ach / fp64[0] if fp64[0] else None, "traffic": measure.traffic.get(workload, {}).get(name),
                    "peak_source": "measured live: b200_measure_fp64_peak (mma.sync.m8n8k4.f64 from registers, all SMs); MEASURED_PEAKS.json "
                                   f"has no FP64 figure; FMA pipe measured {fp64[1]:.1f} TFLOP/s",
                    "ms_per_launch": ms_phase / units, "algorithmic_flops_per_launch": fl,
                    "note": f"{model['dense_fronts']} supernodes, widest {model['max_dense_front']}; the phase is bound by the chain of "
                            f"dependent 32-pivot steps (Cholesky of the diagonal block -> TRSM -> update), not by flops"}
        if name not in alg_bytes:
            return None
        nbytes = alg_bytes[name] / world
        ach = nbytes * units / (ms_phase * 1e-3) / 1e9
        return {"kernel": kernels.get(name, name), "phase": name, "bound": "hbm", "achieved": ach, "peak": peak,
                "unit": "GB/s", "frac": ach / peak, "traffic": measure.traffic.get(workload, {}).get(name),
                "peak_source": peak_src, "ms_per_launch": ms_phase / units, "algorithmic_bytes_per_launch": nbytes}

    # the dominant phase = the largest entry of phases_ms_per_step, whatever it is
    dom = max(per_step, key=lambda k: per_step[k][0])
    rec = {
        "value": value, "unit": UNIT, "ms_per_step": ms / steps, "steps": steps,
        "dtype": "f32 Jacobians + f64 solve" if jac32 else "f64",
        "config": workload_config(prob, workload, jac32, world, "weak" if weak else "strong", flush_buf is not None),
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes, "ms_per_step": ms_e2e / steps,
                "note": "single GPU: the whole packed Values both ways" if world == 1 else
                "per rank (rank 0's counts): its input view up, its owned view down (b200_set_values_view / b200_get_values_view)"},
        "gpu_launches": int(launches),
        "warm_l2": {"ms_per_step": ms_warm / steps, "value": steps / (ms_warm * 1e-3),
                    "note": "same K steps back to back without the L2 flush (information only)"},
        "roofline": roof(dom) or {"phase": dom, "bound": "latency", "achieved": None, "peak": None, "unit": None, "frac": None, "traffic": None,
                                  "note": "no byte / flop model for this phase"},
        "roofline_linearize": roof("linearize"),
        "roofline_dense_fronts": roof("eliminate_large"),
        "roofline_back_substitute": roof("back_substitute"),
        "roofline_leaf_factor": roof("leaf_fused"), "roofline_leaf_schur": roof("leaf_schur"),
        "phases_ms_per_step": {k: round(v[0], 4) for k, v in per_step.items()},
        "lm": {"error_after": st.error, "lambda_after": st.lambda_, "tries_per_step": tries},
        "tree": {"cliques": info.ncliques, "levels": info.nlevels, "max_frontal": info.max_frontal_dim,
                 "max_separator": info.max_separator_dim, "factor_flops": info.factor_flops,
                 "supernodes": info.supernodes, "supernode_levels": info.supernode_levels, "supernode_flops": info.supernode_flops,
                 "dense_front_flops": model["dense_flops"], "leaf_flops": model["leaf_flops"], "front_bytes": info.front_bytes},
        "setup_ms": {"pack_symbolic_upload": setup_ms, "note": "one-time b200_problem_create (host pack + symbolic phase + upload), outside "
                     "value and e2e; amortised over the iterations of an optimize()", "synthetic_generation_s": gen_s},
        "wall_ms_per_step": wall * 1e3 / steps,
    }
    if clocks is not None:
        rec["clocks"] = clocks
    if parity is not None:
        rec["parity"] = parity
    if world == 1 and not args.no_cpu_baseline:
        rec["cpu_baseline"] = cpu_baseline(prob, workload)
    del lm
    dev.close()
    return rec


measure.fp64_peaks = (None, None)
measure.traffic = {}


def cpu_baseline(prob, workload):
    """The unmodified reference on the host cores, bounded to ~10-30 s: the full workload when one iterate() fits, else the
    same generator at 1/10 of the factors (bal_1m_metis stands in for bal_c5_metis), scaled linearly — which flatters the CPU
    (its solve grows faster than linearly)."""
    try:
        from gtsam_b200 import datasets
        est = REF_EST.get(workload, 1.0)
        if est <= 30.0:
            n = max(1, min(5, int(20.0 / est)))
            sec, cinfo = reference_time(prob, n, 1 if est <= 10.0 else 0)
            return dict(cinfo, value=1.0 / sec, unit=UNIT)
        small = {"bal_c5_metis": ("bal_1m_metis", 10.0), "bal_c5": ("bal_1m", 10.0), "bal_c4_metis": ("bal_1m_metis", 3.0),
                 "bal_c4": ("bal_1m", 3.0)}[workload]
        sp = datasets.make(small[0])
        sec, cinfo = reference_time(sp, 2, 0)
        scale = prob.nfactors / sp.nfactors
        cinfo["sample"] = (f"bounded sample: {small[0]} ({sp.nfactors} of the {prob.nfactors} factors, same generator and ordering kind), "
                           f"{sec:.2f} s per iterate() there, scaled x{scale:.1f} by factor count (linear: favours the CPU; the full "
                           f"iterate() measured {est:.0f} s in the build container; `--impl reference` times it in full). " + cinfo["sample"])
        return dict(cinfo, value=1.0 / (sec * scale), unit=UNIT, sample_value=1.0 / sec)
    except Exception as e:
        return {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"failed: {e}"}


def sharded_parity(prob, dev, lm, ctx, dist, rank, local, world, jac32, st):
    """Driver-visible parity of the sharded solve: after the timed region every rank's view of delta (its own subtrees +
    the replicated top, zeros elsewhere) is combined, and rank 0 solves the SAME graph unsharded on its GPU (a second,
    communicator-free context): delta of the damped solve, the linear error and the error after one LM iteration."""
    import numpy as np
    import torch
    from gtsam_b200 import capi, optimizer
    if os.environ.get("B200_BENCH_NO_PARITY"):
        return None
    lam = 1e-2          # diagonal damping (Ceres-style): well conditioned, so delta is comparable to ~1e-10; the LM iteration
    dev.restore_values()   # compared below runs the bench's own additive lambda0 = 1e-5
    dev.linearize()
    status, e0, e1, _ = dev.solve(lam, True)
    d = torch.from_numpy(dev.get_delta()).cuda()
    hi, lo = d.clone(), d.clone()
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    full = torch.where(hi.abs() >= lo.abs(), hi, lo).cpu().numpy()
    out = None
    if rank == 0:
        t0 = time.perf_counter()
        solo_ctx = capi.Context(local)
        solo = capi.DeviceProblem(solo_ctx, prob)
        if jac32:
            solo.set_jacobian_precision(True)
        solo.linearize()
        s1, f0, f1, _ = solo.solve(lam, True)
        d1 = solo.get_delta()
        slm = optimizer.LevenbergMarquardtOptimizer(solo_ctx, prob, device_problem=solo)
        # single-GPU time of the same graph: 3 warm + 5 timed iterations, CUDA events on the solo stream
        solo.save_values()
        sstream = torch.cuda.ExternalStream(solo_ctx.stream(), device=torch.device("cuda", local))
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        for it in range(8):
            if it == 3:
                ev[0].record(sstream)
            solo.restore_values()
            capi._check(solo.L.b200_lm_reset(slm.h))
            slm.iterate()
        ev[1].record(sstream)
        torch.cuda.synchronize()
        solo_ms = ev[0].elapsed_time(ev[1]) / 5
        out = {"delta_rel": float(np.linalg.norm(full - d1) / np.linalg.norm(d1)), "status": [int(status), int(s1)],
               "linear_error_rel": abs(e1 - f1) / abs(f1), "error_after_rel": abs(st.error - slm.error()) / abs(slm.error()),
               "single_gpu_same_graph_ms_per_step": solo_ms,
               "note": "rank 0 solved the same graph unsharded (second context, no communicator) after the timed region: delta of the "
                       "damped solve (lambda 1e-2, diagonal damping) combined over the ranks' views, linear error, error after one LM iteration; "
                       "single_gpu_same_graph_ms_per_step = that unsharded problem timed warm, L2 not flushed, 5 iterations",
               "check_s": time.perf_counter() - t0}
        del slm
        solo.close()
        solo_ctx.close()
    dist.barrier()
    return out


# ------------------------------------------------------------------------------------------
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    import torch
    from gtsam_b200 import capi

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — gtsam_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = capi.Context(local)
    if world > 1:
        ids = [capi.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        ctx.comm_init(ids[0], rank, world)
    measure.fp64_peaks = ctx.measure_fp64_peak()
    tpath = os.path.join(ROOT, "profiles", "r02_kernel_traffic.json")
    if os.path.exists(tpath):
        measure.traffic = {k: v for k, v in json.load(open(tpath)).items() if isinstance(v, dict)}

    workload = PRIMARY if args.workload == "auto" else args.workload
    rec = measure(args, workload, ctx, dist, rank, local, world, primary=True)
    others = {}
    if world == 1 and args.workload == "auto" and not args.no_others:
        for w in SECONDARY:
            others[w] = measure(args, w, ctx, dist, rank, local, world, primary=False)
    if rank == 0:
        line = {"metric": METRIC, "value": rec["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": rec["ms_per_step"], "higher_is_better": True,
                "scaling": "weak" if (world > 1 and args.scaling == "weak") else "strong",
                "vs_baseline": None, "data": "synthetic"}
        line.update({k: v for k, v in rec.items() if k not in ("value", "unit", "ms_per_step", "steps")})
        line["fp64_peaks_tflops"] = {"dmma": measure.fp64_peaks[0], "fma": measure.fp64_peaks[1],
                                     "how": "b200_measure_fp64_peak: register-resident loops, all SMs, best of 3"}
        if others:
            line["other_workloads"] = others
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
