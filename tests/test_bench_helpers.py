"""bench.py host logic that runs without a GPU: the JSON config block, the clock-sample summary, the scenario
chunking used for the synthetic CDU workload."""
import argparse

import numpy as np

import bench


def test_clock_sampler_summary_parses_nvidia_smi_rows():
    cs = bench.ClockSampler(0)
    cs.rows = [["1965", "1965", "700.1", "Not Active", "Not Active", "Not Active", "Active"],
               ["1700", "1965", "990.0", "Not Active", "Not Active", "Not Active", "Active"],
               ["[N/A]", "1965", "1", "Not Active", "Not Active", "Not Active", "Not Active"],
               ["1800", "1965", "800.0", "Not Active", "Active", "Not Active", "Not Active"]]
    s = cs.summary()
    assert s["sm_mhz"] == 1800.0 and s["sm_max_mhz"] == 1965.0 and s["samples"] == 3
    assert s["reasons"] == ["hw_thermal_slowdown", "sw_power_cap"]
    assert bench.ClockSampler(0).summary()["samples"] == 0


def _args(**kw):
    base = dict(workload="cdu_closed_loop", horizon=140, gpus=2, precision="mixed", slots=16384, unique_slabs=6, traj=65536,
                slab=16, steps=5, warmup=3, samples=10e6, batch=None, gain_norm=None, r_weight=None)
    base.update(kw)
    return argparse.Namespace(**base)


def test_config_block_names_the_workload_and_is_the_same_for_both_arms():
    c = bench._config(_args())
    assert c["qp_vars"] == 4480 and c["trajectories_per_gpu"] == 65536 and c["concurrent_slots_per_gpu"] == 16384
    assert "configs[2]" in c["workload"] and "model" not in c and c["sim_steps_per_step"] == 16
    # a function of the command line only: the reference arm prints the identical block
    assert c == bench._config(_args(), world=2)
    for wl, tag in (("horizon_sweep", "configs[4]"), ("cstr_qp_1m", "configs[1]"), ("nn_10m", "configs[3]")):
        cw = bench._config(_args(workload=wl, traj=16384))
        assert tag in cw["workload"] and "model" not in cw
        assert wl in bench.WORKLOADS and len(bench.WORKLOADS[wl]) == 2


def test_horizon_sweep_slab_covers_the_requested_samples():
    a = _args(workload="horizon_sweep", traj=16384, steps=5, samples=10e6)
    slab = bench._sweep_slab(a, 8)
    assert slab == 16 and 8 * 16384 * 5 * slab >= 10e6 > 8 * 16384 * 5 * (slab - 1)
    assert bench._sweep_slab(_args(workload="horizon_sweep", traj=16384, steps=1, samples=1e6), 1) == 62


def test_cpu_pool_steps_are_timed_closed_loop_steps():
    """The reference arm's worker pool on a short horizon: persistent workers, one closed-loop step per worker and
    step, dense-G and diagonal-G interior point reach the same trajectory."""
    pool = bench.CduCpuPool(horizon=4)
    try:
        r1, s1, it1 = pool.step(1)
        r2, s2, it2 = pool.step(2, strong=True)
        assert r1 > 0 and r2 > 0 and len(it1) == pool.workers and len(it2) == 2 * pool.workers
        assert "dense-G" in pool.sample(1, it1) and "diagonal-G" in pool.sample(2, it2, strong=True)
    finally:
        pool.close()


def test_dump_outputs_writes_float64_within_budget_and_samples_the_same_rows(tmp_path, monkeypatch):
    rng = np.random.default_rng(5)
    small = {"u": rng.standard_normal((7, 3)), "iters": np.arange(7, dtype=np.int32)}
    bench.dump_outputs(str(tmp_path / "small"), small)
    for k, v in small.items():
        back = np.load(tmp_path / "small" / f"{k}.npy")
        assert back.dtype == np.float64 and np.array_equal(back, v)
    monkeypatch.setattr(bench, "DUMP_BYTES", 64_000)
    big = {"x": np.arange(5000 * 4 * 3, dtype=np.float64).reshape(5000, 4, 3), "kkt": np.arange(5000.0)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), big)
    files = sorted((tmp_path / "a").iterdir())
    assert sum(f.stat().st_size for f in files) <= 64_000
    x, kkt = np.load(tmp_path / "a" / "x.npy"), np.load(tmp_path / "a" / "kkt.npy")
    rows = kkt.astype(int)
    assert 0 < len(rows) < 5000 and np.all(np.diff(rows) > 0) and np.array_equal(x, big["x"][rows])
    assert all(np.array_equal(np.load(f), np.load(tmp_path / "b" / f.name)) for f in files)


def test_scenarios_are_contiguous_chunks_of_one_prbs_signal():
    p, sp, ds = bench._scenarios(5, 400, seed=3)
    assert sp.shape == (5, 400, p.Ny) and ds.shape == (5, 400, p.Nd)
    assert np.array_equal(sp.reshape(2000, p.Ny), p.setpoints) and np.array_equal(ds.reshape(2000, p.Nd), p.disturbances)
    # piecewise constant with the reference's hold statistics (mean 400 / 200 steps): few distinct rows
    assert len(np.unique(p.setpoints, axis=0)) < 20 and len(np.unique(p.disturbances, axis=0)) < 40
