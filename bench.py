#!/usr/bin/env python
"""bench.py -- grid-point Lyapunov checks/sec on the 2-D inverted pendulum (BASELINE.json).

One "step" = one complete ``Lyapunov.update_safe_set()`` over a 256x256 GridWorld per GPU with
two stacked RBF GPs (M=500, distinct hyper-parameters => two Cholesky factors): the decision for
EVERY grid point (no early exit; certified filter + full fp64 posterior where the outcome depends
on it) + first-fail reduction with the inter-rank key exchange + prefix application.  With N GPUs
the grid is (256 N) x 256 and each rank owns one contiguous 256x256 slab (weak scaling, SURVEY.md
section 8e); ``--scaling strong`` splits one 2048x2048 grid over the ranks instead.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scaling weak|strong]
                    [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  ``--impl reference`` times the reference algorithm's CPU path
(the numpy oracle, all host threads) on a bounded sample of the same workload.
``--dump-outputs DIR`` writes what the last timed step returned to its caller as DIR/<name>.npy:
``safe_set`` (float32 0/1 over the global grid) and ``c_max`` (float64, one element).  The inputs
are seeded, so two builds run with the same arguments can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "grid-point Lyapunov checks/sec (2D pendulum, M=500 GP)"
UNIT = "points/s"
GRID = 256
STRONG_GRID = 2048
M_TRAIN = 500


def algorithmic_flops_per_point(M, d_in, n_factors, n_outputs):
    """SURVEY.md section 8d: sum over distinct factors of [M^2 + M (3 d_in + 6)] + D M E_exp
    (E_exp = 1) + F_small (~100)."""
    return n_factors * (M * M + M * (3 * d_in + 6)) + n_outputs * M * 1 + 100


def algorithmic_bytes_per_point(d):
    """8 d (coordinates, charged although generated) + 1 (flag) + 8 (V written)."""
    return 8 * d + 1 + 8


# --------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.QUERY,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                smax = float(r[1])
            except (ValueError, IndexError):
                continue
            for name, val in zip(names, r[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        busy = [v for v in sm if smax and v > 0.4 * smax] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": smax,
                "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------- CPU reference
def _host_threads():
    # every host thread this process may use -- not the BLAS pools' current size, which torchrun
    # pins to 1 through OMP_NUM_THREADS (threadpool_limits / torch.set_num_threads raise it again)
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        return os.cpu_count() or 1


def cpu_reference_rate(par, seconds_budget, steps=1, warmup=0):
    """Reference algorithm on the host: the per-batch graph of lyapunov.py:433-441 over `sample`
    grid points in 10 000-point batches (early exit disabled), timed in two restatements
    (BASELINE.md section 3.4) -- the numpy/scipy oracle with its best BLAS thread count and a
    torch-CPU fp64 variant with every host thread -- the FASTER one is reported.
    Returns (points/s, cores, sample description, per-step seconds)."""
    import torch
    import bench_workloads as W
    import oracle as O
    from oracle.torch_path import TorchPendulumGraph
    threads = _host_threads()
    lyap = W.build_oracle(par)
    grid = lyap.discretization
    batch = O.config.gp_batch_size
    order = O.stable_value_order(lyap.values)
    first = grid.index_to_state(order[:batch])
    candidates = []            # (seconds per batch, label, threads, callable, context factory)
    try:
        from threadpoolctl import threadpool_limits
    except Exception:  # pragma: no cover
        threadpool_limits = None
    for nt in sorted({threads, 32, 16, 8}, reverse=True):
        if nt > threads or (threadpool_limits is None and nt != threads):
            continue
        ctx = (lambda n=nt: threadpool_limits(limits=n)) if threadpool_limits else None
        guard = ctx() if ctx else None
        lyap.negative(first)
        t0 = time.perf_counter()
        lyap.negative(first)
        dt = time.perf_counter() - t0
        if guard is not None:
            guard.restore_original_limits()
        candidates.append((dt, "numpy/scipy oracle, %d BLAS threads" % nt, nt, lyap.negative, ctx))
    try:
        graph = TorchPendulumGraph(lyap)
        old_threads = torch.get_num_threads()
        torch.set_num_threads(threads)
        ref = lyap.negative(first)
        assert np.array_equal(graph.negative(first), ref), "torch baseline disagrees with the oracle"
        t0 = time.perf_counter()
        graph.negative(first)
        dt = time.perf_counter() - t0
        candidates.append((dt, "torch-CPU fp64 variant, %d threads" % threads, threads,
                           graph.negative, None))
    except TypeError:
        old_threads = None
    t_batch, label, cores, fn, ctx = min(candidates, key=lambda c: c[0])
    guard = ctx() if ctx else None
    total_steps = max(1, steps + warmup)
    nb_max = -(-grid.nindex // batch)
    nb = int(max(1, min(nb_max, seconds_budget / total_steps / max(t_batch, 1e-6))))
    sample = order[:min(nb * batch, grid.nindex)]
    times = []
    for s in range(total_steps):
        t0 = time.perf_counter()
        for i, (idx,) in O.batchify((sample,), batch):
            fn(grid.index_to_state(idx))
        dt = time.perf_counter() - t0
        if s >= warmup:
            times.append(dt)
    if guard is not None:
        guard.restore_original_limits()
    if old_threads is not None:
        torch.set_num_threads(old_threads)
    rate = len(sample) / (sum(times) / len(times))
    others = "; ".join("%s: %.0f points/s" % (c[1], batch / c[0]) for c in candidates)
    desc = ("%d of %d grid points (V-sorted order, %d batches of %d, early exit disabled), %s "
            "(fastest of: %s)" % (len(sample), grid.nindex, nb, batch, label, others))
    return rate, cores, desc, times


# --------------------------------------------------------------------------- main arms
def run_reference(args, rank, world):
    if rank != 0:
        return
    import bench_workloads as W
    par = W.make_pendulum(num_points=GRID, M=M_TRAIN, shared_hypers=False)
    rate, cores, desc, times = cpu_reference_rate(par, seconds_budget=150.0, steps=args.steps,
                                                  warmup=args.warmup)
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * float(np.mean(times)),
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(world, args.scaling),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": desc},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def grid_shape(world, scaling):
    """Weak scaling: one 256 x 256 slab per GPU.  Strong scaling: one fixed 2048 x 2048 grid
    (64 slabs' worth) split over the ranks by contiguous index range."""
    if scaling == "strong":
        return [STRONG_GRID, STRONG_GRID]
    return [GRID * world, GRID]


def workload_config(world, scaling="weak"):
    rows, cols = grid_shape(world, scaling)
    return {"workload": "inverted pendulum 2D, %s GridWorld (global %dx%d), 2 stacked "
                        "RBF GPs on [x,u] (M=%d, distinct ARD hyper-parameters => 2 Cholesky "
                        "factors), linear prior mean, saturated LQR policy, quadratic V, "
                        "update_safe_set full-grid (every point decided, no early exit)"
                        % ("%dx%d per GPU" % (GRID, GRID) if scaling == "weak" else
                           "one %dx%d grid split over %d rank(s)" % (rows, cols, world),
                           rows, cols, M_TRAIN),
            "grid_points_per_gpu": rows * cols // world, "M": M_TRAIN, "gp_outputs": 2,
            "gp_factors": 2,
            "parallelism": "grid sharded by contiguous index range, %d rank(s)" % world,
            "l2": "L2 flushed (256 MiB write) before every timed step"}


def run_ours(args, rank, world, local_rank):
    import torch
    import __graft_entry__
    if rank == 0 or not os.path.exists(os.path.join(ROOT, "safe_learning_b200", "libslb200.so")):
        __graft_entry__.build()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (safe_learning_b200 has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        dist.barrier()
    import bench_workloads as W
    from safe_learning_b200 import _device as dev
    from safe_learning_b200 import _native as nat

    par = W.make_pendulum(num_points=grid_shape(world, args.scaling), M=M_TRAIN,
                          shared_hypers=False)
    lyap = W.build_product(par)
    n_local = lyap._end - lyap._begin
    n_total = lyap.discretization.nindex
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """Per-step CUDA-event times.  L2 is flushed (256 MiB write, outside the event pair)
        before each step; steps are enqueued without extra host synchronisation, so the GPU sees
        the same back-to-back cadence as a learning loop."""
        events = []
        for _ in range(steps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            events.append((e0, e1))
        torch.cuda.synchronize()
        per = [a.elapsed_time(b) for a, b in events]
        return float(sum(per)), per

    def max_over_ranks(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def spread(per):
        return {"min": float(np.min(per)), "median": float(np.median(per)),
                "max": float(np.max(per))}

    # ---- device-resident arm: whole update_safe_set per step (the product's default path)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    n_warm = max(args.warmup, 3)
    for _ in range(n_warm):
        lyap.update_safe_set()
    barrier()
    launches0 = nat.launch_count()
    ms_total, per_step = timed(lyap.update_safe_set, args.steps)
    launches = nat.launch_count() - launches0
    barrier()
    ms_total = max_over_ranks(ms_total)
    value = n_total * args.steps / (ms_total * 1e-3)
    safe_points = int(lyap.last_sweep.get("n_safe", -1))     # first host read-back of the run
    outputs = None
    if args.dump_outputs:
        # what the last timed step hands its caller (reading safe_set is collective over ranks)
        outputs = {"safe_set": lyap.safe_set.astype(np.float32),
                   "c_max": np.array([lyap.feed_dict[lyap.c_max]], dtype=np.float64)}

    # The timed region lasts K x ~0.3 ms, shorter than one nvidia-smi sample.  The SAME step is
    # therefore continued for ~1.5 s (a fixed count, identical on every rank) under the sampler;
    # the clock record covers the timed region and this continuation, whose rate is reported too.
    n_cont = int(min(20000, max(200, 1500.0 / max(ms_total / args.steps, 1e-3))))
    if dist is not None:
        t = torch.tensor([n_cont], dtype=torch.int64, device="cuda")
        dist.broadcast(t, 0)
        n_cont = int(t.item())
    c_total, _ = timed(lyap.update_safe_set, n_cont)
    c_total = max_over_ranks(c_total)
    barrier()

    # ---- what the filter decided (statistics of ONE sweep, summed over ranks)
    cfg = lyap.sweep_descriptor()
    filtered = lyap._filter_enabled(cfg)
    lyap.reset_filter_stats()
    lyap.compute_negative()
    fs = lyap.filter_stats
    if dist is not None:
        t = torch.tensor([fs["prior"], fs["head"], fs["refined"], fs["points"]],
                         dtype=torch.int64, device="cuda")
        dist.all_reduce(t)
        fs = dict(zip(("prior", "head", "refined", "points"), (int(v) for v in t.cpu())))
    k_total, _ = timed(lyap.compute_negative, args.steps)
    filter_ms = k_total / args.steps
    # stage times, live: the mean stage alone, then mean + head (diagnostic switch of the library;
    # the flags of these timing runs are incomplete and not used)
    lib = nat.load()
    stage_ms = {}
    if filtered:
        for label, mask in (("mean", 0), ("mean_head", 1)):
            lib.slb_debug_filter_stages(mask)
            for _ in range(3):
                lyap.compute_negative()
            t_total, _ = timed(lyap.compute_negative, args.steps)
            stage_ms[label] = t_total / args.steps
        lib.slb_debug_filter_stages(3)
        lyap.compute_negative()

    # ---- the full posterior for EVERY point (filter off): the round-1 step and the kernel the
    # algorithmic FLOP count of SURVEY.md section 8d describes
    lyap.filter = False
    for _ in range(3):
        lyap.update_safe_set()
    barrier()
    f_total, f_per = timed(lyap.update_safe_set, args.steps)
    f_total = max_over_ranks(f_total)
    barrier()
    for _ in range(3):
        lyap.compute_negative()
    torch.cuda.synchronize()
    k_total, k_per = timed(lyap.compute_negative, args.steps)
    kernel_ms = k_total / args.steps
    lyap.filter = "auto"

    # ---- end-to-end arm through the public API: host buffers in, host buffers out, every step.
    # In: the cached GP tables (FunctionStack.export_cache / import_cache: one page-locked host
    # buffer mirroring one device arena -- what add_data_point leaves in HBM -- copied H2D every
    # step) and the initial safe set as a numpy mask.  Out: the safe set as a numpy array
    # (lyapunov.safe_set) and c_max (lyapunov.feed_dict), read back with one synchronisation.
    tables = lyap.dynamics.export_cache(pinned=True)
    init_mask = np.zeros(n_total, dtype=bool)
    init_mask[par["initial"]] = True
    h2d_box = [0]

    def e2e_step():
        h2d_box[0] = lyap.dynamics.import_cache(tables)
        lyap.initial_safe_set = init_mask
        lyap.update_safe_set()
        safe = lyap.safe_set                      # numpy bool [N]: D2H (all-gathered over ranks)
        return safe, lyap.feed_dict[lyap.c_max]

    for _ in range(3):
        e2e_step()
    barrier()
    e_total, e_per = timed(e2e_step, args.steps)
    barrier()
    e_total = max_over_ranks(e_total)
    e2e_value = n_total * args.steps / (e_total * 1e-3)
    h2d = h2d_box[0]                             # GP tables (the mask is hashed on the host and
                                                 # re-uploaded only when its content changed)
    d2h = n_local + 64                           # this rank's slab of the safe set + key/stats
    clocks = sampler.stop() if rank == 0 else None

    # ---- parity of the timed configuration against the oracle, on the same global grid
    safe_gpu = lyap.safe_set                     # collective: every rank takes part
    c_max_gpu = lyap.feed_dict[lyap.c_max]
    parity = None
    if rank == 0 and (n_total <= (1 << 20) or args.parity):
        cpu = W.build_oracle(par)
        cpu.update_safe_set()
        parity = {"points": int(n_total),
                  "mismatches": int(np.count_nonzero(safe_gpu != cpu.safe_set)),
                  "c_max_equal": bool(c_max_gpu == cpu.c_max),
                  "safe_points_oracle": int(cpu.safe_set.sum()),
                  "checked": "safe_set and c_max of update_safe_set vs the numpy oracle running "
                             "the reference loop (lyapunov.py:497-606) on the global grid"}
    exchange = "none (1 rank)"
    if world > 1:
        exchange = ("peer-memory stores inside the reduction kernels (slb_exchange), no collective "
                    "call per sweep" if dev.get_exchange() is not None else
                    "NCCL all-gather of one 32-byte key per sweep (no peer mapping: %s)"
                    % dev._EXCHANGE.get("error"))

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- roofline of the full-posterior kernel
    flops_pt = algorithmic_flops_per_point(M_TRAIN, 3, 2, 2)
    achieved_tf = flops_pt * n_local / (kernel_ms * 1e-3) * 1e-12
    peak_tf, peak_src = 37.1, "fallback 37.1 (tools/fp64_peaks.cu on this pool, r01)"
    try:
        with open(os.path.join(ROOT, "profiles", "r01_fp64_peaks.json")) as fh:
            peak_tf = float(json.load(fh)["dmma_tflops_w8_acc8"])
            peak_src = "measured DMMA.8x8x4 peak, tools/fp64_peaks.cu (profiles/r01_fp64_peaks.json)"
    except Exception:
        pass
    hbm_peak = 6650.0
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            hbm_peak = float(json.load(fh)["hbm_gbs"])
    except Exception:
        pass
    traffic = None
    for name in ("r02b_gp_tile_kernel_ncu.json", "r02_gp_tile_kernel_ncu.json", "r01_gp_tile_kernel_ncu.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as fh:
                traffic = json.load(fh).get("dram_bytes_per_launch")
            break
        except Exception:
            pass
    hbm_gbs = algorithmic_bytes_per_point(2) * n_local / (kernel_ms * 1e-3) * 1e-9
    roofline = {"bound": "tensor",
                "kernel": "gp_tile_kernel<3> (fp64 DMMA.8x8x4): the full posterior for EVERY grid "
                          "point, timed with the decision filter switched off; the default step "
                          "runs it only on the points the filter cannot decide (see `filter`)",
                "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": achieved_tf / peak_tf, "traffic": traffic, "peak_source": peak_src,
                "kernel_ms": kernel_ms, "kernel_ms_spread": spread(k_per),
                "algorithmic_flops_per_point": flops_pt,
                "hbm": {"achieved": hbm_gbs, "peak": hbm_peak, "unit": "GB/s",
                        "frac": hbm_gbs / hbm_peak,
                        "note": "path is fp64-compute-bound (AI ~3e4 FLOP/B); HBM fraction "
                                "reported for completeness"}}
    # Rooflines of the three stages of the DEFAULT step (stage times measured live with the library's
    # stage switch, L2 flushed before each); `roofline` is the stage that takes the most time.
    #  * stage 1, fp32 screening kernel (filter_mean32_kernel): per point and training row d_in FFMA for the
    #    exponent, one MUFU.EX2, one FFMA per output for the dot product -> bound by the SFU (16 ex2 per
    #    clock and SM) and the fp32 issue rate; algorithmic flops F_B = D M (3 d_in + 4 + E_exp), E_exp = 1
    #    (SURVEY.md section 8d), against the fp32 FFMA peak 148 SMs x 128 lanes x 2 x 1.965 GHz.
    #  * stage 1, fp64 mean kernel (filter_mean_kernel, where screening does not apply): the same count on
    #    the fp64 pipe (DFMA shares the pipe and the peak of the DMMA tensor op: tools/fp64_peaks.cu).
    #  * head stage (filter_head_kernel): latency bound at C2 (one 8-point group per warp); reported as
    #    points per second only.
    #  * refine pass (gp_tile_kernel, 32-point row/factor-split tiles): the O(M^2) flops of the refined
    #    points against the DMMA peak.
    npts = max(fs["points"], 1)
    mean_ms = stage_ms.get("mean")
    roofline_filter = None
    stage_rooflines = None
    if mean_ms:
        stage1 = int(lib.slb_filter_stage1(cfg))

        def ncu_traffic(name):
            """dram__bytes_read.sum + dram__bytes_write.sum of one launch from the committed ncu summary"""
            try:
                with open(os.path.join(ROOT, "profiles", name)) as fh:
                    return json.load(fh).get("dram_bytes_per_launch")
            except Exception:
                return None
        head_ms = stage_ms["mean_head"] - mean_ms
        refine_ms = filter_ms - stage_ms["mean_head"]
        flops_mean = 2 * M_TRAIN * (3 * 3 + 4 + 1)
        ach = flops_mean * n_local / (mean_ms * 1e-3) * 1e-12
        exp_rate1 = 2 * M_TRAIN * n_local / (mean_ms * 1e-3)
        sm_ghz = 1.965
        if stage1 == 32:
            fp32_peak = 148 * 128 * 2 * sm_ghz * 1e-3
            mufu_peak = 148 * 16 * sm_ghz * 1e9
            r_mean = {
                "bound": "compute", "bound_detail": "neither HBM nor tensor cores: SFU (MUFU.EX2, 16 per "
                "clock and SM) and fp32 issue rate; `peak` is the fp32 FFMA peak 148 x 128 x 2 x 1.965 GHz",
                "kernel": "filter_mean32_kernel<3>: fp32 screening mean of every grid point (3 FFMA + "
                          "MUFU.EX2 + 1 FFMA per kernel value) with a certified error bound, decision "
                          "over the mean's error box and the prior variance",
                "achieved": ach, "peak": fp32_peak, "unit": "TFLOP/s", "frac": ach / fp32_peak,
                "kernel_ms": mean_ms, "algorithmic_flops_per_point": flops_mean,
                "exp_per_s": exp_rate1, "exp_peak_per_s": mufu_peak, "exp_frac": exp_rate1 / mufu_peak,
                "traffic": ncu_traffic("r02b_filter_mean_kernel_ncu.json")}
        else:
            r_mean = {
                "bound": "tensor", "kernel": "filter_mean_kernel<3> (fp64 pipe: DFMA, the pipe and peak "
                                             "of the DMMA tensor op): GP mean of every point, prior-variance decision",
                "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                "kernel_ms": mean_ms, "algorithmic_flops_per_point": flops_mean,
                "executed_fp64_ops_per_entry": 12,
                "exp_per_s": exp_rate1, "exp_peak_per_s": 8.4e11, "exp_frac": exp_rate1 / 8.4e11,
                "traffic": None}
        ach_ref = flops_pt * fs["refined"] / max(refine_ms * 1e-3, 1e-9) * 1e-12
        r_refine = {
            "bound": "tensor", "kernel": "gp_tile_kernel<3, 32> on the refine list (fp64 DMMA.8x8x4; rows "
                                         "and factors of every 32-point tile split over spare CTAs)",
            "achieved": ach_ref, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_ref / peak_tf,
            "kernel_ms": refine_ms, "points": fs["refined"], "algorithmic_flops_per_point": flops_pt,
            "traffic": ncu_traffic("r02b_refine_tile_kernel_ncu.json"),
            "note": "a few hundred points cannot fill 148 SMs: the pass is bound by the latency of one "
                    "tile's serial chain (generation -> contraction -> reduction), not by the pipe"}
        r_head = {"kernel": "filter_head_kernel<3>", "kernel_ms": head_ms,
                  "points": fs["head"] + fs["refined"],
                  "note": "one 8-point group per warp: latency bound at this list length"}
        stage_rooflines = {"mean": r_mean, "head": r_head, "refine": r_refine}
        roofline_filter = dict(r_refine if refine_ms > mean_ms else r_mean)
        roofline_filter["stage_ms"] = {"mean": mean_ms, "head": head_ms, "refine": refine_ms}
        roofline_filter["stage1"] = "fp32 screening" if stage1 == 32 else "fp64 mean"
        roofline_filter["note"] = (
            "dominant stage of the default step by time; stage times measured live with the library's "
            "stage switch (L2 flushed before each); E_exp = 1 charges one flop per exp; all three stages: "
            "`stage_rooflines`; the kernel carrying the O(M^2) cost over the whole grid: "
            "`roofline_full_posterior`")
    exp_rate = 2 * M_TRAIN * n_local / (filter_ms * 1e-3)
    filter_info = {
        "enabled": bool(filtered),
        "decided_by_mean_and_prior_bound": fs["prior"] / npts,
        "decided_by_head_rank_bound": fs["head"] / npts,
        "refined_by_full_posterior": fs["refined"] / npts, "points": fs["points"],
        "head_rank": nat.SLB_HEAD_RANK,
        "decision_kernels_ms": filter_ms,
        "exp_per_s": exp_rate, "exp_peak_per_s": 8.4e11, "exp_frac": exp_rate / 8.4e11,
        "note": "flags identical to the full posterior (tests/test_gpu_bench_shapes.py, `parity`); "
                "the fractions depend on the workload: a point is decided early only when "
                "`decrease < threshold` has the same outcome for every sigma between 0 and a "
                "certified upper bound",
    }

    # ---- CPU baseline, bounded sample, same run (rank 0 at N = 1 only: the N > 1 lines of a scaling
    # run refer to the N = 1 line's baseline)
    cpu_baseline = None
    if world == 1:
        cpu_par = W.make_pendulum(num_points=GRID, M=M_TRAIN, shared_hypers=False)
        rate, cores, desc, _ = cpu_reference_rate(cpu_par, seconds_budget=20.0, steps=1, warmup=0)
        cpu_baseline = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": desc}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": n_warm, "ms_per_step": ms_total / args.steps,
        "ms_per_step_spread": spread(per_step),
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
        "data": "synthetic", "config": workload_config(world, args.scaling), "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h), "ms_per_step": e_total / args.steps,
                "ms_per_step_spread": spread(e_per),
                "api": "FunctionStack.import_cache(page-locked host mirror of the GP tables -> device "
                       "arena in one library call: small tables on the sweep's stream, the packed "
                       "factors on a second stream behind an event the factor-reading launches wait "
                       "for), lyapunov.initial_safe_set = numpy mask (hashed, re-uploaded when it "
                       "changes), update_safe_set(), lyapunov.safe_set (numpy), feed_dict[c_max]"},
        "gpu_launches": int(launches),
        # `roofline`: the dominant kernel of the timed (default, filtered) step; the kernel that carries
        # the O(M^2) algorithmic cost of SURVEY.md section 8d is reported next to it
        "roofline": roofline_filter if roofline_filter is not None else roofline,
        "roofline_full_posterior": roofline,
        "stage_rooflines": stage_rooflines,
        "filter": filter_info,
        "full_posterior": {"value": n_total * args.steps / (f_total * 1e-3), "unit": UNIT,
                           "ms_per_step": f_total / args.steps,
                           "ms_per_step_spread": spread(f_per),
                           "note": "same step with the filter off: every point through the O(M^2) "
                                   "posterior (the round-1 path)"},
        "sustained": {"steps": n_cont, "ms_per_step": c_total / n_cont,
                      "value": n_total * n_cont / (c_total * 1e-3),
                      "note": "the timed step continued for ~1.5 s so that nvidia-smi samples "
                              "exist under load; `clocks` covers the timed region and this"},
        "cpu_baseline": cpu_baseline,
        "safe_points": safe_points, "parity": parity, "exchange": exchange,
    }
    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, array in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), array)
    print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: 256x256 per GPU (default); strong: one 2048x2048 grid split over N")
    ap.add_argument("--parity", action="store_true",
                    help="run the oracle parity check even on grids above 2^20 points")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
