#!/usr/bin/env python
"""bench.py — trajectory-steps/sec of the batched propagation hot path (BASELINE.json metric).

A "step" of this benchmark is ONE pass of the hot path over one ensemble: every trajectory of the
workload is propagated from t0 to the end epoch (MonteCarlo::run_until_epoch).  Workload at N=1 is
BASELINE.json configs[1]: 10 000-trajectory LEO Monte Carlo, two-body + JGM-3 21x21 harmonics,
adaptive RK89 (IntegratorOptions::default), 3-day span.  Multi-GPU is weak scaling: every rank
integrates its own 10 000-trajectory shard (contiguous run indices) and the final states are
exchanged with one all-gather inside the timed region.

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--dump-outputs DIR]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

S = 10**9
DAY = 86400 * S

# Algorithmic FP64 work per accepted RK89 step (SURVEY.md §8d / BASELINE.md §4; mul/add/div/sqrt = 1 flop):
#   F_step = 16 * F_rhs + F_rk,  F_rk = 1308,
#   F_rhs(two-body) = 12,  F_rhs(harmonics NxN) = 24*N(N+3)/2 + 4*N(N+1)/2 + 16*N + 60
def flops_per_step(degree: int, stages: int = 16) -> float:
    n = degree
    f_rhs = 12.0 + (24.0 * n * (n + 3) / 2 + 4.0 * n * (n + 1) / 2 + 16.0 * n + 60.0 if n > 0 else 0.0)
    return stages * f_rhs + 1308.0


BYTES_PER_TRAJ = 13 * 8 + 8 + 9 * 8 + 24  # in: state+consts+epoch; out: state + details (SURVEY.md §8d: 208 B)

DUMP_BYTES = 64 * 10**6   # --dump-outputs: all files of one dump together stay below 64 MB


def dump_outputs(out_dir, arrays, first_index=0):
    """--dump-outputs: every array of `arrays` (trajectories on the last axis) goes to <out_dir>/<name>.npy as float64, and the
    ensemble index of each column to trajectory_index.npy.  An output larger than DUMP_BYTES keeps the same seeded sample of
    trajectories in every array, so two builds run with the same arguments can be compared file by file."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    n = next(iter(arrays.values())).shape[-1]
    assert all(a.shape[-1] == n for a in arrays.values())
    rows = 1 + sum(a.size // max(n, 1) for a in arrays.values())
    keep = min(n, (DUMP_BYTES - 128 * (len(arrays) + 1)) // (8 * rows))   # 128: .npy header
    cols = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    for name, a in arrays.items():
        np.save(out_dir / f"{name}.npy", np.ascontiguousarray(a[..., cols]))
    np.save(out_dir / "trajectory_index.npy", (first_index + cols).astype(np.float64))


def details_arrays(det):
    """The fields of nyxb_details (one record per trajectory) as separate arrays for dump_outputs."""
    return {f"details_{f}": det[f] for f in ("step_ns", "error", "attempts", "n_steps", "n_rejected", "n_rhs")}


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="nyxb", choices=["nyxb", "reference"])
    p.add_argument("--n-traj", type=int, default=10_000, help="trajectories per GPU")
    p.add_argument("--span-days", type=float, default=None, help="default: 3 days (c2-c4), 2 days (c5)")
    p.add_argument("--degree", type=int, default=21)
    p.add_argument("--mode", default="fast", choices=["fast", "strict"])
    p.add_argument("--lanes", type=int, default=0)
    p.add_argument("--kernel", default="auto", choices=["auto", "thread", "coop", "transposed"],
                   help="kernel family (nyxb_engine_set_kernel); auto = the library's own dispatch")
    p.add_argument("--tx-positions", type=int, default=0, help="transposed kernel: walker warps per set (0 = library default)")
    p.add_argument("--tx-slice", type=int, default=0, help="transposed kernel: step attempts per time slice (0 = library default)")
    p.add_argument("--cpu-sample", type=int, default=0,
                   help="trajectories in the bounded CPU-baseline sample (0: 32 per host core, ~10 s of CPU work)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-strict", action="store_true", help="skip the extra bit-parity (STRICT mode) pass at N=1")
    p.add_argument("--record", type=int, default=0, metavar="CAP",
                   help="also time one pass with trajectory recording (CAP records per trajectory, device-resident sink)")
    p.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                   help="weak: --n-traj trajectories PER GPU (the driver's scaling run); strong: --n-traj in total, sharded over the GPUs")
    p.add_argument("--workload", default="c2", choices=["c2", "c3", "c4", "c5"],
                   help="c2 = BASELINE configs[1] (the metric's workload); c3/c4/c5 = configs[2]/[3]/[4], reported for context only")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="after the timed steps, write what the last timed step returned (final states, epochs in ns, details, status; "
                        "trajectories on the last axis) as DIR/<name>.npy in float64, at most 64 MB (a seeded sample of trajectories "
                        "above that, indices in trajectory_index.npy); with several GPUs each rank writes its shard to DIR/rank<r>/")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.span_days is None:
        a.span_days = 2.0 if a.workload == "c5" else 3.0
    if a.workload == "c5" and a.n_traj == 10_000:
        a.n_traj = 1000
    return a


def build_workload(args, n_total, nb):
    """Synthetic inputs of SURVEY.md §8(d); returns (frame, dynamics, almanac, state[9][n], consts[4][n], epoch0[n])."""
    rng = np.random.Generator(np.random.PCG64(0))
    almanac = None
    if args.workload == "c2":
        # C2: example-01 orbit (examples/01_orbit_prop/main.rs:52-53) + N(0, diag(1 km, 1 m/s)), JGM-3 NxN
        frame = nb.EARTH_J2000
        gd = nb.GravityFieldData.from_fixture("jgm3_70x70", args.degree, args.degree, nb.IAU_EARTH_FRAME)
        dyn = nb.SpacecraftDynamics.new(nb.OrbitalDynamics.from_model(nb.GravityField.new(gd)))
        orbit = nb.Orbit.keplerian(6378.1363 + 300.0, 0.015, 68.5, 65.2, 75.0, 0.0, 0, frame)
        template = nb.Spacecraft(orbit=orbit, mass=nb.Mass(1000.0, 0.0, 0.0))
        mvn = nb.MvnSpacecraft.from_cartesian_std(template, 1.0, 1e-3)
    elif args.workload == "c3":
        # C3: JWST-like (examples/02_jwst_covar_monte_carlo/main.rs:63-86, README.md:52): Sun+Moon point masses + SRP
        frame = nb.EARTH_J2000
        almanac = nb.Almanac.synthetic(frame, 0, args.span_days + 2.0)
        srp = nb.SolarPressure.new([nb.EARTH_J2000, nb.MOON_J2000], almanac)
        dyn = nb.SpacecraftDynamics.from_model(nb.OrbitalDynamics.point_masses([nb.MOON, nb.SUN]), srp)
        orbit = nb.Orbit.cartesian(119901.070276, -1389299.665421, -1041369.150539, 0.045956, -0.013168, 0.034535, 0, frame)
        template = nb.Spacecraft(orbit=orbit, mass=nb.Mass(6200.0, 0.0, 0.0), srp=nb.SRPData(21.197 * 14.162, 1.56))
        mvn = nb.MvnSpacecraft.from_cartesian_std(template, 0.5, 1e-4)
    else:
        # C4: low lunar orbit, GRAIL 70x70 + Earth/Sun point masses, Moon-centred
        from nyx_b200.frames import EARTH

        frame = nb.MOON_J2000
        almanac = nb.Almanac.synthetic(frame, 0, args.span_days + 2.0, bodies=(EARTH, nb.SUN))
        gd = nb.GravityFieldData.from_fixture("luna_jggrx_80x80", 70, 70, nb.IAU_MOON_FRAME)
        dyn = nb.SpacecraftDynamics.new(nb.OrbitalDynamics.new([nb.PointMasses.new([EARTH, nb.SUN]), nb.GravityField.new(gd)]))
        orbit = nb.Orbit.keplerian(1737.4 + 100.0, 0.001, 90.0, 10.0, 0.0, 0.0, 0, frame)
        template = nb.Spacecraft(orbit=orbit, mass=nb.Mass(1000.0, 0.0, 0.0))
        mvn = nb.MvnSpacecraft.from_cartesian_std(template, 0.1, 1e-4)
    x = mvn.sample_vectors(rng, n_total)  # serial host stream, run index == draw order (montecarlo.rs:290-295)
    st = np.ascontiguousarray((template.to_vector()[None, :] + x).T)  # [9][n]
    cs = np.zeros((4, n_total))
    cs[0] = template.mass.dry_mass_kg
    cs[2] = template.srp.area_m2
    ep = np.zeros(n_total, dtype=np.int64)
    return frame, dyn, almanac, st, cs, ep


def c5_scenario(args, nb, n, n_msr, device, truth_on_cpu, fixed_step_s=None):
    """LRO-like orbit determination ensemble (BASELINE configs[4]): dynamics, DSN stations, tracking arc, dispersed initial estimates."""
    from nyx_b200.frames import EARTH

    S_ = 10**9
    frame = nb.MOON_J2000
    deg = args.degree if args.degree != 21 else 70
    alm = nb.Almanac.synthetic(frame, 0, args.span_days + 2.0, bodies=(EARTH, nb.SUN))
    gd = nb.GravityFieldData.from_fixture("luna_jggrx_80x80", deg, deg, nb.IAU_MOON_FRAME)
    srp = nb.SolarPressure.new([nb.EARTH_J2000, nb.MOON_J2000], alm)
    dyn = nb.SpacecraftDynamics.from_model(nb.OrbitalDynamics.new([nb.PointMasses.new([EARTH, nb.SUN]), nb.GravityField.new(gd)]), srp)
    mode = nb.MODE_FAST if args.mode == "fast" else nb.MODE_STRICT
    prop = nb.Propagator.default_dp78(dyn, mode=mode, device=device)   # examples/04_lro_od/main.rs:163
    if fixed_step_s is not None:   # parity tests: no controller feedback, so the arithmetic itself is compared
        prop = nb.Propagator.dp78(dyn, nb.IntegratorOptions.with_fixed_step_s(fixed_step_s), mode=mode, device=device)
    orbit = nb.Orbit.keplerian(1737.4 + 100.0, 0.002, 88.0, 20.0, 10.0, 0.0, 0, frame)
    truth0 = nb.Spacecraft(orbit=orbit, mass=nb.Mass(1018.0, 900.0, 0.0), srp=nb.SRPData(3.9 * 2.7, 0.96))
    rn, dn = nb.StochasticNoise(5e-3), nb.StochasticNoise(5e-6)
    devices = {"Madrid": nb.GroundStation.dss65_madrid(5.0, rn, dn), "Canberra": nb.GroundStation.dss34_canberra(5.0, rn, dn),
               "Goldstone": nb.GroundStation.dss13_goldstone(5.0, rn, dn)}
    names = list(devices)
    epochs = (np.arange(1, n_msr + 1) * 60 * S_).astype(np.int64)
    schedule = [names[(k // 240) % 3] for k in range(n_msr)]   # 4-hour passes
    # truth trajectory: one spacecraft, fixed 60 s steps, recorded (the product's recording path, or the CPU oracle in the reference arm)
    topts = nb.IntegratorOptions.with_fixed_step_s(60.0)
    st1, cs1, ep1 = nb.pack_spacecraft([truth0])
    if truth_on_cpu:
        from oracle import pyoracle

        _, _, _, tstat, (t_ep, t_st, t_cnt) = pyoracle.propagate_batch(dyn.pack(frame, alm).c, topts.to_c(nb.IntegratorMethod.RungeKutta89), st1, cs1, ep1,
                                                                       int(epochs[-1]), traj_capacity=n_msr + 2)
    else:
        tprop = nb.Propagator.new(dyn, nb.IntegratorMethod.RungeKutta89, topts, mode=nb.MODE_FAST, device=device)
        _, _, _, tstat, (t_ep, t_st, t_cnt) = tprop.engine(frame, alm).propagate_batch(st1, cs1, ep1, int(epochs[-1]), traj_capacity=n_msr + 2)
    assert tstat[0] == 0 and np.array_equal(t_ep[1: n_msr + 1, 0], epochs)
    truth = np.repeat(t_st[:, 1: n_msr + 1, 0].T[:, :, None], n, axis=2)
    rng = np.random.default_rng(0)
    arc = nb.simulate_tracking(epochs, truth, devices, schedule, frame, alm, rng)
    ests = []
    for i in range(n):   # examples/04_lro_od/main.rs:268-282: 0.5 km / 5 m/s RIC sigmas; smaller velocity dispersion here
        v = truth0.to_vector()
        v[:6] += np.concatenate([rng.normal(0, 0.3, 3), rng.normal(0, 3e-4, 3)])
        ests.append(nb.KfEstimate.from_diag(truth0.with_vector(0, v), [0.25, 0.25, 0.25, 2.5e-7, 2.5e-7, 2.5e-7, 0.04, 0.0, 0.0]))
    odp = nb.SpacecraftKalmanOD(prop, nb.KalmanVariant.ReferenceUpdate, nb.SigmaRejection(3.0), devices, alm)
    odp.with_process_noise(nb.ProcessNoise3D.from_velocity_km_s([1e-10, 1e-10, 1e-10], 1 * nb.Unit.Hour, 10 * nb.Unit.Minute, None))
    return dict(frame=frame, alm=alm, dyn=dyn, prop=prop, devices=devices, arc=arc, ests=ests, odp=odp, truth=truth, deg=deg, mode=mode)


def _c5_ref_worker(job):
    """One filter of the reference arm: numpy + C oracle (od/process/mod.rs restated), run in a worker process."""
    import nyx_b200 as nb
    from oracle import pyoracle_od

    args, i, m_s = job
    sc = _C5_SC
    odp, arc, est = sc["odp"], sc["arc"], sc["ests"][i]
    names_c, st_c = odp.stations_c(sc["frame"])
    tracker = np.array([names_c.index(t) for t in arc.tracker[:m_s]], dtype=np.int32)
    msc = est.nominal_state.mass
    cs0 = np.array([msc.dry_mass_kg, msc.extra_mass_kg, est.nominal_state.srp.area_m2, 0.0])
    ref = pyoracle_od.process_arc(sc["dyn"].pack(sc["frame"], sc["alm"]).c, sc["prop"].opts.to_c(sc["prop"].method), odp.config_c(), st_c,
                                  arc.epoch_ns[:m_s], tracker, np.ascontiguousarray(arc.obs[:m_s, :, i]), est.nominal_state.to_vector(), cs0, 0, est.covar)
    return ref["n_steps"]


def _c5_ref_full(i):
    """Filter i of the scenario in _C5_SC over its WHOLE arc on the numpy + C oracle (parity tests at the BASELINE span)."""
    from oracle import pyoracle_od

    sc = _C5_SC
    odp, arc, est = sc["odp"], sc["arc"], sc["ests"][i]
    names_c, st_c = odp.stations_c(sc["frame"])
    tracker = np.array([names_c.index(t) for t in arc.tracker], dtype=np.int32)
    msc = est.nominal_state.mass
    cs0 = np.array([msc.dry_mass_kg, msc.extra_mass_kg, est.nominal_state.srp.area_m2, 0.0])
    ref = pyoracle_od.process_arc(sc["dyn"].pack(sc["frame"], sc["alm"]).c, sc["prop"].opts.to_c(sc["prop"].method), odp.config_c(), st_c,
                                  arc.epoch_ns, tracker, np.ascontiguousarray(arc.obs[:, :, i]), est.nominal_state.to_vector(), cs0, 0, est.covar)
    return {k: ref[k] for k in ("est_state", "msr_flags", "state", "n_steps", "status", "covar")}


_C5_SC = None


def bench_c5_reference(args, nb):
    """`--impl reference --workload c5`: the CPU restatement of the filter on all host cores (one filter per process), each step a
    bounded sample: `cores` filters over the first 60 measurement epochs."""
    import multiprocessing as mp

    global _C5_SC
    host = host_cores()
    cores = host["usable"]
    m_s = 60
    args_small = argparse.Namespace(**vars(args))
    args_small.span_days = max(m_s * 60 / 86400.0 + 0.01, 0.05)
    _C5_SC = c5_scenario(args_small, nb, cores, m_s, 0, truth_on_cpu=True)
    ctx = mp.get_context("fork")
    times, steps = [], 0
    with ctx.Pool(cores) as pool:
        for it in range(max(0, min(args.warmup, 1)) + args.steps):
            t0 = time.perf_counter()
            res = pool.map(_c5_ref_worker, [(None, i, m_s) for i in range(cores)])
            if it >= max(0, min(args.warmup, 1)):
                times.append(time.perf_counter() - t0)
                steps = int(sum(res))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"details_n_steps": np.array(res)})
    value = steps * len(times) / sum(times)
    line = {"impl": "reference", "metric": "trajectory-steps/sec (ensemble)", "value": value, "unit": "trajectory-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"C5 sample: {cores} LRO-like EKFs (GRAIL {_C5_SC['deg']}x{_C5_SC['deg']} + Earth/Sun + SRP), first {m_s} measurement epochs"},
            "cpu_baseline": {"value": value, "unit": "trajectory-steps/s", "cores": cores, "host": host, "kind": "port",
                             "sample": f"{cores} filters x {m_s} measurement epochs per step, one process per filter (numpy + C oracle)"},
            "e2e": {"value": value, "unit": "trajectory-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


def bench_c5(args, nb, local_rank):
    """BASELINE configs[4] (context only, N=1): LRO-like ensemble, every trajectory runs its own EKF over the same tracking
    schedule — `nyxb_od_ekf_batch`, ONE launch for the whole arc (propagation with STM + time/measurement updates)."""
    n = args.n_traj
    n_msr = int(args.span_days * 86400 // 60)
    sc = c5_scenario(args, nb, n, n_msr, local_rank, truth_on_cpu=False)
    frame, alm, dyn, prop, devices, arc, ests, odp, truth, deg, mode = (sc[k] for k in ("frame", "alm", "dyn", "prop", "devices", "arc", "ests", "odp", "truth", "deg", "mode"))
    eng = prop.engine(frame, alm)
    # warm-up: a short arc
    warm = nb.TrackingDataArc(arc.epoch_ns[:4], arc.tracker[:4], arc.obs[:4, :, :min(n, 64)])
    odp.process_arcs(ests[:min(n, 64)], warm)
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = eng.launch_count()
    walls, kern = [], []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        sol = odp.process_arcs(ests, arc)
        walls.append(time.perf_counter() - t0)
        kern.append(eng.last_kernel_ms())
    wall, kern_ms = float(np.mean(walls)), float(np.mean(kern))
    clocks = sampler.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"final_state": sol.final_state_soa, "final_epoch_ns": sol.final_epoch_ns,
                                         "covar": sol.covar.transpose(1, 2, 0), "state_deviation": sol.state_deviation,
                                         "resid_ratio": sol.resid_ratio, "prefit": sol.prefit, "postfit": sol.postfit,
                                         "msr_flags": sol.msr_flags, "status": sol.status, **details_arrays(sol.details)})
    steps = int(sol.details["n_steps"].sum())
    ok = int((sol.status == 0).sum())
    acc = int(sol.accepted().sum())
    err = np.linalg.norm(sol.final_state_soa[:3] - truth[-1, :3, :], axis=0)
    last_vis = np.where(~np.isnan(arc.obs[:, 0, 0]))[0]
    line = {"metric": "trajectory-steps/sec (ensemble)", "value": steps / (kern_ms * 1e-3), "unit": "trajectory-steps/s", "n_gpus": 1,
            "steps": args.steps, "warmup": 1, "ms_per_step": kern_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"C5: {n} LRO-like filters (Moon-centred, GRAIL {deg}x{deg} + Earth/Sun point masses + SRP with Cr estimated), "
                                   f"EKF over {n_msr} range+Doppler measurement epochs at 60 s from 3 DSN stations, {args.span_days:g}-day span, DP78",
                       "ok_trajectories": ok, "measurement_updates_accepted": acc, "mode": args.mode,
                       "kernel": "nyxb_k_od_coop (1 warp = 1 filter, harmonic gradient split by columns over the lanes)"
                                 if (mode == nb.MODE_FAST and deg >= 8) else "nyxb_k_od (1 thread = 1 filter)",
                       "median_final_position_error_km": float(np.median(err)) if last_vis.size and last_vis[-1] == n_msr - 1 else None},
            "e2e": {"value": steps / wall, "unit": "trajectory-steps/s", "h2d_bytes_per_step": int(arc.obs.nbytes + n * (13 + 81) * 8),
                    "d2h_bytes_per_step": int(n * (9 + 81 + 9) * 8 + 3 * arc.obs.nbytes + n_msr * n * 4), "ms_per_step": wall * 1e3},
            "gpu_launches": eng.launch_count() - launches0, "clocks": clocks,
            "measurement_updates_per_s": acc / (kern_ms * 1e-3)}
    # FP64 roofline of the filter kernel: algorithmic work of the dual-number harmonic gradient (gravity_field.rs:273-431 with 3
    # partials): ~150 flop per (n, m) entry (two column recursions, three products with rr_n, six accumulations; FMA = 2), entries =
    # N + N(N+1)/2, 13 DP78 stages per step; everything else (point masses, SRP, 9x9 filter algebra) is < 3 % and not counted.
    entries = deg + deg * (deg + 1) // 2
    fps5 = 13 * 150.0 * entries
    fp64_peak = eng._lib.nyxb_measure_fp64_tflops(local_rank, 4096)
    ach = steps * fps5 / (kern_ms * 1e-3) / 1e12
    line["roofline"] = {"bound": "fp64", "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s", "frac": ach / fp64_peak if fp64_peak > 0 else None,
                        "traffic": None, "kernel_ms": kern_ms,
                        "note": f"algorithmic {fps5:.3g} flop per accepted step (dual-number {deg}x{deg} gradient x 13 stages); peak = live DFMA probe"}
    if not args.no_cpu_baseline:
        # numpy + C oracle filter (tests' checker) on ONE filter over the first measurements: a bounded sample
        from oracle import pyoracle_od

        m_s = min(n_msr, 90)
        names_c, st_c = odp.stations_c(frame)
        tracker = np.array([names_c.index(t) for t in arc.tracker[:m_s]], dtype=np.int32)
        e0 = ests[0]
        msc = e0.nominal_state.mass
        cs0 = np.array([msc.dry_mass_kg, msc.extra_mass_kg, e0.nominal_state.srp.area_m2, 0.0])
        packed = dyn.pack(frame, alm)
        t0 = time.perf_counter()
        ref = pyoracle_od.process_arc(packed.c, prop.opts.to_c(prop.method), odp.config_c(), st_c, arc.epoch_ns[:m_s], tracker,
                                      np.ascontiguousarray(arc.obs[:m_s, :, 0]), e0.nominal_state.to_vector(), cs0, 0, e0.covar)
        ct = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": ref["n_steps"] / ct, "unit": "trajectory-steps/s", "cores": 1, "kind": "port",
                                "sample": f"filter 0 over the first {m_s} measurement epochs ({ref['n_steps']} steps, {ct:.1f} s), numpy + C oracle"}
        k_last = int(np.where(~np.isnan(ref["est_state"][:, 0]))[0][-1])
        sub = odp.process_arcs(ests[:1], nb.TrackingDataArc(arc.epoch_ns[:m_s], arc.tracker[:m_s], arc.obs[:m_s, :, :1]), record_estimates=True)
        line["max_dr_km"] = float(np.abs(sub.est_state[k_last, :3, 0] - ref["est_state"][k_last, :3]).max())
    print(json.dumps(line))
    return 0


# bounded CPU samples of the reference arm (trajectories over the FULL span): fixed, so that runs are comparable
REF_SAMPLE = {"c2": 1024, "c3": 8192, "c4": 64}
PARITY_BOUND_KM = 1e-6   # north-star: sub-mm position over the benchmark span

WORKLOAD_TEXT = {
    "c2": "C2: {n} LEO trajectories/GPU (alt 300 km, e 0.015, i 68.5 deg; N(0, 1 km / 1 m/s) dispersions), two-body + JGM-3 {deg}x{deg}, "
          "adaptive RK89 (IntegratorOptions::default), {span:g}-day span",
    "c3": "C3: {n} JWST-like trajectories/GPU, Sun+Moon point masses + SRP (Earth & Moon shadows), adaptive RK89 defaults, {span:g}-day span",
    "c4": "C4: {n} low-lunar-orbit trajectories/GPU, GRAIL 70x70 + Earth/Sun point masses, adaptive RK89 defaults, {span:g}-day span",
}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self._halt = threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def host_cores():
    """What the CPU arm really gets: logical CPUs the process may run on (affinity mask), the cgroup CPU quota if any, and the
    machine's nominal count.  os.cpu_count() alone said 128 on two boxes whose CPU arms differed 5.6x (VERDICT r01)."""
    info = {"logical": os.cpu_count()}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        info["affinity"] = info["logical"]
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = Path(path).read_text().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
            break
        except Exception:
            continue
    info["cgroup_quota_cpus"] = quota
    usable = info["affinity"] if quota is None else max(1, min(info["affinity"], int(quota)))
    info["usable"] = usable
    try:
        info["loadavg_1m"] = os.getloadavg()[0]
    except Exception:
        pass
    return info


def cpu_reference_leg(args, nb, sample_n, repeats=1, speed_build=False):
    """The reference's CPU path for the same workload: the C restatement of the reference algorithm
    (oracle/, OpenMP over trajectories == the rayon par_iter of mc/montecarlo.rs:233-253), all host cores,
    on a bounded sample of the same ensemble."""
    from oracle import pyoracle

    frame, dyn, almanac, st, cs, ep = build_workload(args, sample_n, nb)
    prop = nb.Propagator.default(dyn)
    packed = dyn.pack(frame, almanac)
    end = int(args.span_days * DAY)
    host = host_cores()
    cores = host["usable"]  # explicit thread count: torchrun exports OMP_NUM_THREADS=1
    times, steps = [], 0
    out = oep = det = status = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        out, oep, det, status = pyoracle.propagate_batch(packed.c, prop.opts.to_c(prop.method), st, cs, ep, end, n_threads=cores,
                                                         speed_build=speed_build)
        times.append(time.perf_counter() - t0)
        steps = int(det["n_steps"].sum())
    return {"steps": steps, "times": times, "cores": cores, "host": host, "final": out, "inputs": (st, cs, ep),
            "outputs": {"final_state": out, "final_epoch_ns": oep, "status": status, **details_arrays(det)}}


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    import nyx_b200 as nb

    if args.cpu_sample <= 0:
        args.cpu_sample = 32 * host_cores()["usable"]
    if args.workload == "c5":
        if rank != 0:
            return 0
        return bench_c5_reference(args, nb) if args.impl == "reference" else bench_c5(args, nb, local_rank)
    workload = WORKLOAD_TEXT[args.workload].format(n=args.n_traj, deg=args.degree, span=args.span_days)
    # algorithmic flop per accepted step (BASELINE.md §4): C2 from the degree; C3 ~ 9 k (two ephemeris bodies + SRP); C4 = 70x70
    fps = {"c2": flops_per_step(args.degree), "c3": 9.0e3, "c4": flops_per_step(70) + 16 * 200.0}[args.workload]

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return 0
        # FIXED bounded sample: the first REF_SAMPLE trajectories of the same ensemble over the full span, every step; one untimed
        # warm-up pass (page-in of the library, thread pool).  Both oracle builds are timed: the parity build (-O2, no FMA
        # contraction: rustc never contracts) is the line's value, the speed build (-O3, AVX2 + FMA) is reported beside it.
        sample_n = REF_SAMPLE[args.workload]
        cpu_reference_leg(args, nb, min(sample_n, 64))
        leg = cpu_reference_leg(args, nb, sample_n, repeats=args.steps)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, leg["outputs"])
        total_t = sum(leg["times"])
        value = leg["steps"] * args.steps / total_t
        fast = cpu_reference_leg(args, nb, sample_n, repeats=1, speed_build=True)
        line = {
            "impl": "reference", "metric": "trajectory-steps/sec (ensemble)", "value": value, "unit": "trajectory-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_t / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload, "sample": f"first {sample_n} trajectories of the same ensemble, full span"},
            "cpu_baseline": {"value": value, "unit": "trajectory-steps/s", "cores": leg["cores"], "host": leg["host"], "kind": "port",
                             "build": "-O2 -ffp-contract=off (parity build, the checker)",
                             "speed_build": {"value": fast["steps"] / fast["times"][0], "build": "-O3 -march=x86-64-v3 -ffp-contract=fast"},
                             "sample": f"{sample_n} trajectories x {args.span_days:g} days per step, OpenMP schedule(dynamic) over trajectories, "
                                       f"{leg['cores']} threads"},
            "e2e": {"value": value, "unit": "trajectory-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ nyxb arm (GPU)
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl nyxb needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from nyx_b200.dist import all_gather_final_states, shard_bounds

    n_total = args.n_traj * world if args.scaling == "weak" else args.n_traj  # weak: per-GPU work fixed; strong: total fixed
    frame, dyn, almanac, st, cs, ep = build_workload(args, n_total, nb)
    lo, hi = shard_bounds(n_total, world, rank)
    n = hi - lo
    mode = nb.MODE_FAST if args.mode == "fast" else nb.MODE_STRICT
    prop = nb.Propagator.default(dyn, mode=mode, device=local_rank)
    eng = prop.engine(frame, almanac)
    if args.lanes:
        eng.set_lanes(args.lanes)
    if args.kernel != "auto":
        eng.set_kernel({"thread": nb.KERNEL_THREAD, "coop": nb.KERNEL_COOP, "transposed": nb.KERNEL_TRANSPOSED}[args.kernel])
    if args.tx_slice:
        eng.set_tx_tuning(args.tx_slice, 0)
    if args.tx_positions:
        eng.set_tx_positions(args.tx_positions)
    end = int(args.span_days * DAY)

    # pinned host inputs of this rank's shard (e2e leg) and HBM-resident copies (value leg)
    h_st = torch.from_numpy(np.ascontiguousarray(st[:, lo:hi])).pin_memory()
    h_cs = torch.from_numpy(np.ascontiguousarray(cs[:, lo:hi])).pin_memory()
    h_ep = torch.from_numpy(np.ascontiguousarray(ep[lo:hi])).pin_memory()
    d_st, d_cs, d_ep = h_st.to(dev), h_cs.to(dev), h_ep.to(dev)
    d_out = torch.empty((9, n), dtype=torch.float64, device=dev)
    d_oep = torch.empty(n, dtype=torch.int64, device=dev)
    d_det = torch.empty(n * 48, dtype=torch.uint8, device=dev)
    d_status = torch.empty(n, dtype=torch.int32, device=dev)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def one_pass():
        stream = torch.cuda.current_stream(dev)
        eng.propagate_batch_dev(n, d_st.data_ptr(), d_cs.data_ptr(), d_ep.data_ptr(), end, None, d_out.data_ptr(),
                                d_oep.data_ptr(), d_det.data_ptr(), d_status.data_ptr(), stream.cuda_stream)
        if world > 1:
            return all_gather_final_states(d_out, n_total)
        return d_out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    for _ in range(args.warmup):
        one_pass()
    barrier()

    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = eng.launch_count()
    total_ms = 0.0
    kernel_ms = []
    barrier()
    for _ in range(args.steps):
        flush.fill_(1)  # L2 flush between timed iterations (not timed)
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        barrier()
        e0.record()
        stream = torch.cuda.current_stream(dev)
        eng.propagate_batch_dev(n, d_st.data_ptr(), d_cs.data_ptr(), d_ep.data_ptr(), end, None, d_out.data_ptr(),
                                d_oep.data_ptr(), d_det.data_ptr(), d_status.data_ptr(), stream.cuda_stream)
        e1.record()
        if world > 1:
            all_gather_final_states(d_out, n_total)
        e2.record()
        barrier()
        kernel_ms.append(e0.elapsed_time(e1))
        total_ms += e0.elapsed_time(e2)
    launches = eng.launch_count() - launches0
    clocks = sampler.stop()

    det = np.frombuffer(d_det.cpu().numpy().tobytes(), dtype=nb.abi.DETAILS_DTYPE)
    local_steps = int(det["n_steps"].sum())
    local_rej = int(det["n_rejected"].sum())
    status = d_status.cpu().numpy()
    ok = int((status == 0).sum())
    if args.dump_outputs:
        # the device buffers still hold the last timed step's results (this rank's shard)
        dump_outputs(Path(args.dump_outputs) / f"rank{rank}" if world > 1 else args.dump_outputs,
                     {"final_state": d_out.cpu().numpy(), "final_epoch_ns": d_oep.cpu().numpy(), "status": status, **details_arrays(det)},
                     first_index=lo)

    # ---- e2e: the public host-buffer call (H2D of the inputs + kernel + D2H of results inside the timed region)
    e2e_t = []
    for it in range(2 + args.steps):
        barrier()
        t0 = time.perf_counter()
        out_h, oep_h, det_h, st_h = eng.propagate_batch(h_st.numpy(), h_cs.numpy(), h_ep.numpy(), end)
        barrier()
        if it >= 2:
            e2e_t.append(time.perf_counter() - t0)
    e2e_s = float(np.mean(e2e_t))

    # max over ranks / sums over ranks
    t_dev = torch.tensor([total_ms, e2e_s, float(np.mean(kernel_ms))], dtype=torch.float64, device=dev)
    cnt = torch.tensor([local_steps, local_rej, ok, launches], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
        dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
    total_ms, e2e_s, kern_ms = (float(v) for v in t_dev.cpu())
    all_steps, all_rej, all_ok, all_launches = (int(v) for v in cnt.cpu())

    parity_failed = False
    if rank == 0:
        value = all_steps * args.steps / (total_ms * 1e-3)
        e2e_value = all_steps / e2e_s
        # FP64 roofline of the dominant (only) kernel, measured live
        fp64_peak = eng._lib.nyxb_measure_fp64_tflops(local_rank, 4096)
        achieved_tf = local_steps * fps / (kern_ms * 1e-3) / 1e12
        peaks = {}
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        # dram__bytes_read + dram__bytes_write of ONE launch of this workload by the kernel used here, from the ncu capture committed
        # with the kernel (profiles/r02_traffic.json, written by scripts/make_traffic_json.py from the same gpurun call as the bench)
        traffic = None
        try:
            tj = json.loads((ROOT / "profiles" / "r02_traffic.json").read_text())
            kname = {nb.KERNEL_THREAD: "nyxb_k_thread", nb.KERNEL_COOP: "nyxb_k_coop", nb.KERNEL_TRANSPOSED: "nyxb_k_tx"}.get(eng.last_kernel())
            if (args.workload == tj.get("workload") and n == tj.get("n_traj") and args.span_days == tj.get("span_days")
                    and args.degree == tj.get("degree") and kname and kname in tj.get("kernel", "")):
                traffic = tj["dram_bytes_per_launch"]
        except Exception:
            pass
        hbm_achieved = n * BYTES_PER_TRAJ / (kern_ms * 1e-3) / 1e9
        line = {
            "metric": "trajectory-steps/sec (ensemble)", "value": value, "unit": "trajectory-steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload, "trajectories_total": n_total, "accepted_steps_per_pass": all_steps,
                       "rejected_attempts_per_pass": all_rej, "ok_trajectories": all_ok, "mode": args.mode,
                       "kernel": {nb.KERNEL_THREAD: "nyxb_k_thread (1 thread = 1 trajectory)", nb.KERNEL_COOP: f"nyxb_k_coop ({eng.lanes()} lanes = 1 trajectory)",
                                  nb.KERNEL_TRANSPOSED: "nyxb_k_tx (1 CTA = 32 trajectories, lane = trajectory, warp = column position)"}.get(eng.last_kernel(), "?"),
                       "l2": "flushed between timed iterations (256 MiB write)",
                       "parallelism": f"ensemble-sharded x{world}, one all-gather of final states"},
            "e2e": {"value": e2e_value, "unit": "trajectory-steps/s", "h2d_bytes_per_step": n * (13 * 8 + 8) * world,
                    "d2h_bytes_per_step": n * (9 * 8 + 8 + 48 + 4) * world, "ms_per_step": e2e_s * 1e3},
            "gpu_launches": all_launches,
            "clocks": clocks,
            "roofline": {"bound": "fp64", "achieved": achieved_tf, "peak": fp64_peak, "unit": "TFLOP/s",
                         "frac": achieved_tf / fp64_peak if fp64_peak > 0 else None, "traffic": traffic,
                         "algorithmic_bytes": n * BYTES_PER_TRAJ,
                         "note": "FP64-pipe bound (no tensor-core or HBM-bound work on this path); peak = live DFMA probe "
                                 f"(nyxb_measure_fp64_tflops); algorithmic {fps:.0f} flop per accepted step",
                         "kernel_ms": kern_ms},
            "roofline_hbm": {"bound": "hbm", "achieved": hbm_achieved, "peak": hbm_peak, "unit": "GB/s",
                             "frac": hbm_achieved / hbm_peak, "of": "measured" if peaks else "fallback",
                             "note": f"{BYTES_PER_TRAJ} algorithmic bytes per trajectory, independent of step count"},
        }
        if world == 1 and args.record > 0:
            # trajectory recording (SURVEY §8 f-1): 56 B per accepted step streamed to HBM, step-major SoA
            cap = args.record
            t_ep = torch.empty((cap, n), dtype=torch.int64, device=dev)
            t_st = torch.empty((6, cap, n), dtype=torch.float64, device=dev)
            t_cnt = torch.empty(n, dtype=torch.int64, device=dev)
            sink = nb.abi.TrajSink(cap, t_ep.data_ptr(), t_st.data_ptr(), t_cnt.data_ptr())
            import ctypes as C

            def rec_pass():
                rc = eng._lib.nyxb_propagate_batch_traj_dev(eng.handle, n, d_st.data_ptr(), d_cs.data_ptr(), d_ep.data_ptr(), end, None,
                                                            d_out.data_ptr(), d_oep.data_ptr(), d_det.data_ptr(), d_status.data_ptr(),
                                                            C.byref(sink), torch.cuda.current_stream(dev).cuda_stream)
                assert rc == 0
            rec_pass()
            torch.cuda.synchronize(dev)
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record(); rec_pass(); r1.record(); torch.cuda.synchronize(dev)
            rec_ms = r0.elapsed_time(r1)
            recs = int(t_cnt.sum().item())
            line["recording"] = {"value": local_steps / (rec_ms * 1e-3), "unit": "trajectory-steps/s", "ms": rec_ms, "records": recs,
                                 "bytes_written": recs * 56, "write_gbs": recs * 56 / (rec_ms * 1e-3) / 1e9,
                                 "note": "same pass with the start state + every accepted step recorded (instance.rs:297-326)"}
            # batched resampling of that recording on a 5-minute grid (Traj::every, traj.rs:148-162): one launch, device buffers
            grid = torch.arange(0, end + 1, 300 * 10**9, dtype=torch.int64, device=dev)
            m = int(grid.numel())
            r_out = torch.empty((6, m, n), dtype=torch.float64, device=dev)
            r_status = torch.empty((m, n), dtype=torch.int32, device=dev)

            def resample_pass():
                rc = eng._lib.nyxb_traj_resample_dev(eng.handle, n, C.byref(sink), m, grid.data_ptr(), r_out.data_ptr(), r_status.data_ptr(),
                                                     torch.cuda.current_stream(dev).cuda_stream)
                assert rc == 0
            resample_pass()
            torch.cuda.synchronize(dev)
            flush.fill_(1)
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record(); resample_pass(); r1.record(); torch.cuda.synchronize(dev)
            rs_ms = r0.elapsed_time(r1)
            n_ok = int((r_status == 0).sum().item())
            rs_bytes = recs * 56 + m * n * 52   # every record read once (neighbouring queries share windows through L2) + the outputs
            line["resample"] = {"value": m * n / (rs_ms * 1e-3), "unit": "interpolated states/s", "ms": rs_ms, "queries": m, "ok": n_ok,
                                "algorithmic_bytes": rs_bytes, "gbs": rs_bytes / (rs_ms * 1e-3) / 1e9,
                                "hbm_frac": rs_bytes / (rs_ms * 1e-3) / 1e9 / hbm_peak,
                                "note": "nyxb_k_traj_resample: Traj::at (13-record Hermite window) for every trajectory at every grid epoch; "
                                        "975 FP64 divisions per interpolated state (divided differences, no FMA: bit-identical to the host "
                                        "restatement) make it division-bound, not HBM-bound"}
        if world == 1 and not args.no_cpu_baseline:
            leg = cpu_reference_leg(args, nb, min(args.cpu_sample, n))
            sample_n = min(args.cpu_sample, n)
            cpu_value = leg["steps"] / leg["times"][0]
            dr = np.sqrt(((out_h[:3, :sample_n] - leg["final"][:3]) ** 2).sum(0))
            dv = np.sqrt(((out_h[3:6, :sample_n] - leg["final"][3:6]) ** 2).sum(0))
            fast = cpu_reference_leg(args, nb, min(sample_n, 1024), speed_build=True)
            line["cpu_baseline"] = {"value": cpu_value, "unit": "trajectory-steps/s", "cores": leg["cores"], "host": leg["host"], "kind": "port",
                                    "build": "-O2 -ffp-contract=off (parity build, the checker)",
                                    "speed_build": {"value": fast["steps"] / fast["times"][0], "build": "-O3 -march=x86-64-v3 -ffp-contract=fast",
                                                    "sample": min(sample_n, 1024)},
                                    "sample": f"first {sample_n} trajectories of the same ensemble, full {args.span_days:g}-day span, "
                                              f"{leg['times'][0]:.1f} s, {leg['cores']} OpenMP threads"}
            q = np.percentile(dr, [50, 99])
            line["parity"] = {"max_dr_km": float(dr.max()), "median_dr_km": float(q[0]), "p99_dr_km": float(q[1]), "max_dv_km_s": float(dv.max()),
                              "bound_km": PARITY_BOUND_KM, "pass": bool(dr.max() < PARITY_BOUND_KM), "sample": sample_n,
                              "against": "CPU oracle (parity build), same inputs, full span; the oracle against its own one-ulp-perturbed "
                                         "error norm moves by up to 7.3e-7 km on this workload (profiles/r02_oracle_sensitivity_c2.json)"}
            line["max_dr_km"] = float(dr.max())
            line["max_dv_km_s"] = float(dv.max())
            line["parity_sample"] = sample_n
            if not args.no_strict:
                # bit-parity pass: the STRICT kernel over the SAME full ensemble, compared bit for bit with the oracle sample
                sprop = nb.Propagator.default(dyn, mode=nb.MODE_STRICT, device=local_rank)
                seng = sprop.engine(frame, almanac)
                seng.propagate_batch(h_st.numpy()[:, :256].copy(), h_cs.numpy()[:, :256].copy(), h_ep.numpy()[:256].copy(), end)  # warm-up
                t0 = time.perf_counter()
                s_out, _, s_det, s_status = seng.propagate_batch(h_st.numpy(), h_cs.numpy(), h_ep.numpy(), end)
                s_t = time.perf_counter() - t0
                same = (s_out[:, :sample_n] == leg["final"]).all(axis=0)
                sdr = np.sqrt(((s_out[:3, :sample_n] - leg["final"][:3]) ** 2).sum(0))
                line["strict"] = {"value": float(s_det["n_steps"].sum() / s_t), "unit": "trajectory-steps/s (host buffers, e2e)",
                                  "bit_identical_trajectories": int(same.sum()), "of": int(sample_n), "max_dr_km": float(sdr.max()),
                                  "lanes_per_trajectory": seng.lanes(),
                                  "note": "NYXB_MODE_STRICT kernel (no FMA, reference operation order) over the full ensemble vs the CPU oracle sample"}
        print(json.dumps(line))
        if "parity" in line and not line["parity"]["pass"]:
            parity_failed = True
    if world > 1:
        dist.destroy_process_group()
    return 3 if parity_failed else 0


if __name__ == "__main__":
    sys.exit(main())
