"""GPU parity at the BASELINE.json sizes -- the launch shapes ``bench.py`` and ``tools/bench_extra.py``
time (VERDICT r01 item 1): C2 exactly as ``bench.py`` builds it (256 x 256, M=500, two Cholesky
factors: 7 row panels per factor, 1024 tiles, first-wave L2 prefetch), C3 at 512 x 512 and a C4
slab (64^4 grid descriptor, M=2000, the first and last 4096 flat indices through the C ABI's index
ranges).  The oracle needs a second or two for each.
"""
import numpy as np
import pytest
from numpy.testing import assert_allclose, assert_array_equal

import bench_workloads as W
import oracle as O
from test_gpu_parity import RTOL, _assert_negative_parity, _rl_objects, _sweep_details, sl  # noqa: F401

pytestmark = pytest.mark.gpu


def test_c2_bench_shape_vs_oracle(sl):
    """The workload of bench.py's N=1 line: reference loop of lyapunov.py:497-606 on the full grid."""
    import bench
    par = W.make_pendulum(num_points=[bench.GRID, bench.GRID], M=bench.M_TRAIN, shared_hypers=False)
    gpu, cpu = W.build_product(par), W.build_oracle(par)
    assert gpu.discretization.nindex == 65536 and gpu.dynamics.functions[0].X.shape[0] == 500
    assert_array_equal(gpu.values, cpu.values)
    det = _sweep_details(gpu)
    _assert_negative_parity(gpu, cpu, det)
    states = cpu.discretization.all_points
    m_cpu, e_cpu = cpu.dynamics(states, cpu.policy(states))
    assert_allclose(det["mean"], m_cpu, rtol=RTOL, atol=1e-12)
    assert_allclose(det["err"], e_cpu, rtol=RTOL, atol=1e-12)
    for _ in range(2):                       # the second call replays cached descriptors
        gpu.update_safe_set()
    cpu.update_safe_set()
    # (with tau = sum(unit_maxes) / 2 the first point outside the initial set fails: the safe set
    # stays the initial one -- the benchmark still decides every grid point)
    assert par["initial"].sum() <= cpu.safe_set.sum() < cpu.safe_set.size
    assert_array_equal(gpu.safe_set, cpu.safe_set)
    assert gpu.feed_dict[gpu.c_max] == cpu.c_max
    assert gpu.last_sweep["n_safe"] == int(cpu.safe_set.sum())
    # the flags of the default (filtered) sweep equal the full-posterior flags everywhere
    assert_array_equal(gpu.compute_negative().cpu().numpy().astype(bool), det["negative"])


def test_bench_dump_outputs_vs_oracle(sl, tmp_path):
    """`bench.py --dump-outputs DIR` writes what the last timed step handed its caller -- the safe
    set (float32 0/1) and c_max (float64) -- equal to the oracle's.  Run on the strong-scaling grid
    (2048 x 2048), where the safe set grows past the initial set, so a dump of the initial mask or
    of a state before any step would not match.  The launches counted in the timed region are
    exactly `--steps` sweeps."""
    import json
    import os
    import subprocess
    import sys
    import bench
    from safe_learning_b200 import _native as nat
    steps = 3
    out = tmp_path / "outputs"
    proc = subprocess.run([sys.executable, os.path.join(bench.ROOT, "bench.py"), "--gpus", "1",
                           "--scaling", "strong", "--steps", str(steps), "--warmup", "0",
                           "--dump-outputs", str(out)],
                          stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert proc.returncode == 0, proc.stderr[-4000:]
    line = json.loads(proc.stdout.strip().splitlines()[-1])
    assert sorted(os.listdir(out)) == ["c_max.npy", "safe_set.npy"]
    safe, c_max = np.load(out / "safe_set.npy"), np.load(out / "c_max.npy")
    assert safe.dtype == np.float32 and c_max.dtype == np.float64 and c_max.shape == (1,)
    par = W.make_pendulum(num_points=bench.grid_shape(1, "strong"), M=bench.M_TRAIN,
                          shared_hypers=False)
    cpu = W.build_oracle(par)
    cpu.update_safe_set()                   # stops at the first failing batch: a few seconds
    assert cpu.safe_set.sum() > par["initial"].sum()
    assert_array_equal(safe, cpu.safe_set.astype(np.float32))
    assert c_max[0] == cpu.c_max
    # launches of one warmed-up sweep (a CUDA-graph replay, like every timed step)
    gpu = W.build_product(par)
    for _ in range(3):
        gpu.update_safe_set()
    before = nat.launch_count()
    gpu.update_safe_set()
    per_sweep = nat.launch_count() - before
    assert per_sweep > 0 and line["gpu_launches"] == steps * per_sweep


def test_c2_bench_shape_growing_safe_set_vs_oracle(sl):
    """Same shape with a finer discretisation constant (tau / 64): 59% of the points satisfy the
    decrease condition, the safe set grows far beyond the initial one and the filter has to hand
    ~6% of the grid to the full posterior."""
    par = W.make_pendulum(num_points=[256, 256], M=500, shared_hypers=False, tau_scale=1 / 64.)
    gpu, cpu = W.build_product(par), W.build_oracle(par)
    det = _sweep_details(gpu)
    _assert_negative_parity(gpu, cpu, det)
    assert_array_equal(gpu.compute_negative().cpu().numpy().astype(bool), det["negative"])
    gpu.update_safe_set()
    cpu.update_safe_set()
    assert 4 * par["initial"].sum() < cpu.safe_set.sum() < cpu.safe_set.size
    assert_array_equal(gpu.safe_set, cpu.safe_set)
    assert gpu.feed_dict[gpu.c_max] == cpu.c_max


def test_c2_shared_factor_bench_shape_vs_oracle(sl):
    """Same grid with one shared Cholesky factor (the 8.9e7 points/s variant of DESIGN section 6)."""
    par = W.make_pendulum(num_points=[256, 256], M=500, shared_hypers=True)
    gpu, cpu = W.build_product(par), W.build_oracle(par)
    det = _sweep_details(gpu)
    _assert_negative_parity(gpu, cpu, det)
    gpu.update_safe_set()
    cpu.update_safe_set()
    assert_array_equal(gpu.safe_set, cpu.safe_set)
    assert gpu.feed_dict[gpu.c_max] == cpu.c_max


def test_c3_value_iteration_512_vs_oracle(sl):
    """C3: 512 x 512 value grid, GP-mean dynamics with M=500, three Jacobi sweeps
    (reinforcement_learning.py:65-114, 135-140)."""
    par = W.make_pendulum(num_points=8, M=500)
    rl_gpu, _ = _rl_objects(sl, par, "product", num=512)
    rl_cpu, _ = _rl_objects(O, par, "oracle", num=512)
    states = rl_cpu.state_space
    for sweep in range(3):
        res = rl_gpu.value_iteration()
        old = rl_cpu.value_function.parameters.copy()
        new = np.concatenate([rl_cpu.future_values(states[i:i + 32768])
                              for i in range(0, len(states), 32768)])
        rl_cpu.value_function.parameters = new
        assert_allclose(rl_gpu.value_function.parameters[0], new, rtol=1e-9, atol=1e-12)
        assert_allclose(res, np.max(np.abs(new - old)), rtol=1e-9)


def test_c4_slab_64pow4_m2000_vs_oracle(sl):
    """C4 at its stated size: 64^4 GridWorld descriptor, four GPs with M=2000 on 5-D inputs (four
    Cholesky factors, 8 row panels each), V = LyapunovNetwork; the first and the last 4096 flat
    indices through ``slb_lyapunov_sweep``'s index range, as a sharded rank would sweep them."""
    import torch
    from safe_learning_b200 import _device as dev
    from safe_learning_b200 import _native as nat
    par = W.make_cartpole(num_points=64, M=2000, tau_scale=0.01, with_initial=False)
    gpu = W.build_product(par)
    n = gpu.discretization.nindex
    assert n == 64 ** 4
    # oracle objects on a tiny grid (its negative() only needs the functions and tau); the states
    # come from the 64^4 grid's own index arithmetic (functions.py:714-731)
    small = dict(par)
    small["num_points"] = np.array([3, 3, 3, 3])
    cpu = W.build_oracle(small)
    cpu.tau = par["tau"]
    big = O.GridWorld(par["limits"], par["num_points"])
    lib = nat.load()
    cfg = gpu.sweep_descriptor()
    slab = 4096
    for begin in (0, n - slab, n // 2 + 17):
        neg = dev.empty((slab,), torch.uint8)
        val, dec, thr = dev.empty((slab,)), dev.empty((slab,)), dev.empty((slab,))
        mean, err = dev.empty((slab, 4)), dev.empty((slab, 4))
        nat.check(lib.slb_lyapunov_sweep(dev.stream(), cfg, begin, begin + slab, neg.data_ptr(),
                                         val.data_ptr(), dec.data_ptr(), thr.data_ptr(),
                                         mean.data_ptr(), err.data_ptr()), "slb_lyapunov_sweep")
        states = big.index_to_state(np.arange(begin, begin + slab))
        actions = cpu.policy(states)
        m_cpu, e_cpu = cpu.dynamics(states, actions)
        assert_allclose(mean.cpu().numpy(), m_cpu, rtol=RTOL, atol=1e-12)
        assert_allclose(err.cpu().numpy(), e_cpu, rtol=RTOL, atol=1e-12)
        d_cpu = cpu.v_decrease_bound(states, (m_cpu, e_cpu)).ravel()
        t_cpu = np.broadcast_to(cpu.threshold(states), (slab, 1)).ravel()
        assert_allclose(val.cpu().numpy(), cpu.lyapunov_function(states).ravel(), rtol=1e-12,
                        atol=1e-14)
        assert_allclose(dec.cpu().numpy(), d_cpu, rtol=RTOL, atol=1e-10)
        assert_array_equal(thr.cpu().numpy(), t_cpu)
        margin = np.abs(d_cpu - t_cpu)
        assert (margin > 1e-7 * np.maximum(np.abs(d_cpu), np.abs(t_cpu))).all(), \
            "slab has a point within rounding distance of the threshold"
        assert_array_equal(neg.cpu().numpy().astype(bool), d_cpu < t_cpu)
        # the default (filtered) decision on the same range
        neg2 = dev.empty((slab,), torch.uint8)
        gpu_flags = gpu.compute_negative_range(begin, begin + slab, out=neg2)
        assert_array_equal(gpu_flags.cpu().numpy(), neg.cpu().numpy())
