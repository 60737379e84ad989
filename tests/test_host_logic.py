"""Host-side logic (CPU only): gravity-file loaders, packing, Monte Carlo state generation, option builders."""
import gzip

import numpy as np
import pytest

import nyx_b200 as nb
from nyx_b200 import abi
from nyx_b200.gravity import _split_cof_pair


def test_cof_pair_splitting_quirk():
    """io/gravity.rs:236-312: C and S are glued together when S is negative."""
    assert _split_cof_pair("2.43926074865630e-06-1.40026639758800e-06") == (2.4392607486563e-06, -1.400266397588e-06)
    assert _split_cof_pair("-5.36243554298510e-07-4.73772370615970e-07") == (-5.3624355429851e-07, -4.7377237061597e-07)
    assert _split_cof_pair("-4.84165374886470e-04") == (-4.8416537488647e-04, None)
    assert _split_cof_pair("9.57170590888000e-07") == (9.57170590888e-07, None)


def test_from_cof_and_fixture_agree_with_reference_values(tmp_path):
    """JGM-3 values quoted in SURVEY.md a13; from_cof on a synthetic file mirrors degree/order truncation semantics."""
    gd = nb.GravityFieldData.from_fixture("jgm3_70x70", 21, 21, nb.IAU_EARTH_FRAME)
    assert (gd.degree, gd.order) == (21, 21)
    assert gd.cs_nm(2, 0) == (-4.8416537488647e-4, 0.0)
    assert gd.cs_nm(2, 2) == (2.4392607486563e-6, -1.400266397588e-6)
    assert np.count_nonzero(gd.c_nm) == 250
    text = ("COMMENT\nPOTFIELD 3 3 1 3.986e14 6.378e6 1.0\nRECOEF    2  0   -4.84165374886470e-04\n"
            "RECOEF    2  1   -1.86987640000000e-10 1.19528010000000e-09\nRECOEF    2  2    2.43926074865630e-06-1.40026639758800e-06\n"
            "RECOEF    3  0    9.57170590888000e-07\nRECOEF    3  3    7.21144939823090e-07 1.41420398473540e-06\nEND\n")
    p = tmp_path / "t.cof.gz"
    with gzip.open(p, "wt") as fh:
        fh.write(text)
    g = nb.GravityFieldData.from_cof(p, 2, 1, True, nb.IAU_EARTH_FRAME)
    assert (g.degree, g.order) == (2, 2)      # maxima SEEN within the requested degree (io/gravity.rs:345-367)
    assert g.cs_nm(2, 1) == (-1.8698764e-10, 1.1952801e-09) and g.cs_nm(2, 2) == (0.0, 0.0)  # order 2 > requested 1: skipped
    j2 = nb.GravityFieldData.from_j2(-4.84e-4, nb.IAU_EARTH_FRAME)
    assert (j2.degree, j2.order, j2.c_nm[2, 0]) == (2, 0, -4.84e-4)


def test_from_shadr_skips_header(tmp_path):
    p = tmp_path / "m.tab"
    p.write_text(" 0.1738E+04, 0.49028E+04, 0.1, 3, 3, 1, 0.0, 0.0\n    1,    0, 0.0, 0.0, 0.0, 0.0\n"
                 "    2,    0,-0.9088017496403000E-04, 0.0, 0.7D-11, 0.0\n    2,    1, 0.1729508721878000D-09, 0.1041216830058000E-08, 0, 0\n"
                 "    3,    0, 1.0, 2.0, 0, 0\n")
    g = nb.GravityFieldData.from_shadr(p, 2, 2, False, nb.IAU_MOON_FRAME)
    assert g.degree == 2 and g.cs_nm(2, 0)[0] == -0.9088017496403e-04 and g.cs_nm(2, 1) == (0.1729508721878e-09, 0.1041216830058e-08)


def test_integrator_option_builders_follow_reference():
    d = nb.IntegratorOptions.default()
    assert (d.init_step, d.min_step, d.max_step, d.tolerance, d.attempts, d.fixed_step) == (60 * 10**9, 10**6, 2700 * 10**9, 1e-12, 50, False)
    a = nb.IntegratorOptions.with_adaptive_step_s(0.1, 30.0, 1e-12, nb.ErrorControl.RSSCartesianState)
    assert a.init_step == a.max_step == 30 * 10**9 and a.min_step == 10**8            # options.rs:66-82
    f = nb.IntegratorOptions.with_fixed_step_s(10.0)
    assert f.fixed_step and f.tolerance == 0.0 and f.attempts == 0 and f.min_step == f.max_step == f.init_step == 10**10
    m = nb.IntegratorOptions.with_max_step(30 * nb.Unit.Second)
    assert m.init_step == 30 * 10**9                                                  # options.rs:127-131
    c = a.to_c(nb.IntegratorMethod.DormandPrince78)
    assert (c.method, c.error_ctrl, c.init_step_ns) == (abi.DP78, abi.RSS_CARTESIAN_STATE, 30 * 10**9)
    assert nb.IntegratorMethod.from_str("rungekutta89") is nb.IntegratorMethod.RungeKutta89
    with pytest.raises(nb.PropagationError):
        nb.IntegratorMethod.from_str("blah")
    assert [m.stages() for m in nb.IntegratorMethod] == [16, 13, 7, 4, 6, 8]


def test_monte_carlo_generation_is_a_single_serial_stream():
    """mc/montecarlo.rs:277-296: run index == draw order; `skip` discards the head of the same stream."""
    frame = nb.EARTH_J2000
    tmpl = nb.Spacecraft(orbit=nb.Orbit.keplerian(7000.0, 0.01, 30.0, 10.0, 20.0, 30.0, 0, frame), mass=nb.Mass(100.0, 5.0, 1.0),
                         srp=nb.SRPData(4.0, 1.5), drag=nb.DragData(3.0, 2.1))
    cov = np.diag([1.0, 1.0, 1.0, 1e-6, 1e-6, 1e-6, 1e-4, 0.0, 0.0])
    cov[0, 1] = cov[1, 0] = 0.5
    mc = nb.MonteCarlo(tmpl, nb.MvnSpacecraft.from_spacecraft_cov(tmpl, cov), "t", seed=7)
    a = mc.generate_states(0, 50)
    b = mc.generate_states(40, 10)
    assert [i for i, _ in a] == list(range(50))
    assert all(a[40 + k][1].state == b[k][1].state for k in range(10))
    x = np.array([ds.state.to_vector() - tmpl.to_vector() for _, ds in mc.generate_states(0, 4000)])
    assert np.abs(np.cov(x.T)[:2, :2] - cov[:2, :2]).max() < 0.08 and np.abs(x[:, 7:]).max() == 0.0
    st, cs, ep = nb.pack_spacecraft(ds.state for _, ds in a)
    assert st.shape == (9, 50) and cs.shape == (4, 50) and np.array_equal(cs[:, 0], [100.0, 1.0, 4.0, 3.0])
    with pytest.raises(ValueError):
        nb.MvnSpacecraft.from_spacecraft_cov(tmpl, -np.eye(9))


def test_dynamics_lowering_to_the_c_abi():
    frame = nb.EARTH_J2000
    alm = nb.Almanac.synthetic(frame, 0, 5.0)
    gd = nb.GravityFieldData.from_fixture("jgm3_70x70", 8, 8, nb.IAU_EARTH_FRAME)
    dyn = nb.SpacecraftDynamics.from_models(nb.OrbitalDynamics.new([nb.PointMasses.new([nb.EARTH, nb.MOON, nb.SUN]), nb.GravityField.new(gd)]),
                                            [nb.SolarPressure.new([nb.EARTH_J2000, nb.MOON_J2000], alm), nb.Drag.earth_exp(alm)])
    p = dyn.pack(frame, alm).c
    assert p.n_bodies == 2 and p.point_mass_mask == 0b11            # the central body is skipped (orbital.rs:219-222)
    assert p.gravity.contents.degree == 8 and p.gravity.contents.rot.kind == 1 and p.gravity.contents.r_eq_km == 6378.14
    assert p.srp.contents.n_shadow == 2 and p.srp.contents.shadow_body[0] == abi.NYXB_CENTRAL_BODY
    assert p.drag.contents.density == abi.DENSITY_EXPONENTIAL and p.drag.contents.r0 == 700_000.0
    with pytest.raises(nb.DynamicsError):
        nb.SpacecraftDynamics.new(nb.OrbitalDynamics.new([object()])).pack(frame, alm)
    with pytest.raises(nb.DynamicsError):
        nb.SpacecraftDynamics.new(nb.OrbitalDynamics.point_masses([nb.SUN])).pack(frame, None)
    kep = nb.Orbit.keplerian(7000.0, 0.01, 30.0, 10.0, 20.0, 30.0, 0, frame)
    assert abs(kep.rmag_km() - 7000.0 * (1 - 0.01**2) / (1 + 0.01 * np.cos(np.radians(30.0)))) < 1e-9


def test_od_host_objects():
    """Host-side OD mirror (nyx_b200/od.py): RIC DCM, SpacecraftUncertainty::to_estimate (sc_uncertainty.rs:70-138, D^T C D as coded),
    KfEstimate::state (Spacecraft + OVector<9> clamps Cr, cosmic/spacecraft.rs:713-728), SNC from a velocity noise (snc.rs:288-311),
    geodetic -> body-fixed station coordinates."""
    import numpy as np

    import nyx_b200 as nb
    from nyx_b200.od import dcm_ric_to_inertial

    orbit = nb.Orbit.keplerian(7000.0, 0.01, 51.6, 30.0, 40.0, 10.0, 0, nb.EARTH_J2000)
    D = dcm_ric_to_inertial(orbit)
    assert np.allclose(D @ D.T, np.eye(3), atol=1e-14) and abs(np.linalg.det(D) - 1.0) < 1e-14
    r, v = orbit.radius_km, orbit.velocity_km_s
    assert np.allclose(D[:, 0], r / np.linalg.norm(r)) and np.allclose(D[:, 2], np.cross(r, v) / np.linalg.norm(np.cross(r, v)))
    sc = nb.Spacecraft(orbit=orbit, srp=nb.SRPData(2.0, 1.9))
    unc = nb.SpacecraftUncertainty(sc, nb.LocalFrame.RIC, 0.5, 0.3, 1.5, 1e-4, 6e-4, 3e-3, coeff_reflectivity=0.2)
    est = unc.to_estimate()
    P = est.covar
    assert np.allclose(P, P.T) and (np.linalg.eigvalsh(P[:6, :6]) > 0).all()
    assert abs(np.trace(P[:3, :3]) - (0.5**2 + 0.3**2 + 1.5**2)) < 1e-12 and abs(P[6, 6] - 0.04) < 1e-15 and P[7, 7] == 0.0
    d6 = np.zeros((6, 6)); d6[:3, :3] = D; d6[3:, 3:] = D
    assert np.allclose(P[:6, :6], d6.T @ np.diag([0.25, 0.09, 2.25, 1e-8, 3.6e-7, 9e-6]) @ d6)
    inertial = nb.SpacecraftUncertainty(sc).to_estimate().covar
    assert np.allclose(np.diag(inertial)[:6], [0.25, 0.25, 0.25, 2.5e-7, 2.5e-7, 2.5e-7])
    with pytest.raises(nb.ODError):
        nb.SpacecraftUncertainty(sc, x_km=-1.0).to_estimate()
    est.state_deviation = np.array([1, 0, 0, 0, 0, 0, 0.5, 0.1, 2.0])
    st = est.state()
    assert st.srp.coeff_reflectivity == 2.0 and abs(st.orbit.radius_km[0] - (r[0] + 1.0)) < 1e-12 and st.mass.prop_mass_kg == 2.0
    snc = nb.ProcessNoise3D.from_velocity_km_s([1e-10, 2e-10, 3e-10], 1 * nb.Unit.Hour, 10 * nb.Unit.Minute)
    assert np.allclose(snc.diag, np.array([1e-10, 2e-10, 3e-10]) / 3600.0) and snc.disable_time == 600 * 10**9
    gs = nb.GroundStation("pole", 90.0, 0.0, 0.0, nb.IAU_EARTH_FRAME)
    pos, up = gs.body_fixed()
    assert abs(pos[2] - 6356.75) < 1e-9 and abs(pos[0]) < 1e-9 and np.allclose(up, [0, 0, 1], atol=1e-15)
    eq = nb.GroundStation("equator", 0.0, 90.0, 1.0, nb.IAU_EARTH_FRAME).body_fixed()[0]
    assert np.allclose(eq, [0.0, 6379.14, 0.0], atol=1e-9)


def test_bench_reference_arm_for_c5_runs_on_cpu(tmp_path):
    """`bench.py --workload c5 --impl reference` is the CPU restatement of the filter (no GPU, none of the product's kernels):
    it must print one JSON result line with the benchmark's keys, and --dump-outputs writes the last step's per-filter step counts."""
    import json
    import subprocess
    import sys
    from pathlib import Path

    root = Path(__file__).resolve().parent.parent
    out = subprocess.run([sys.executable, str(root / "bench.py"), "--workload", "c5", "--impl", "reference", "--degree", "8", "--steps", "1", "--warmup", "0",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=300, cwd=root)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["kind"] == "port"
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["cpu_baseline"]["cores"] >= 1
    steps = np.load(tmp_path / "details_n_steps.npy")
    assert steps.dtype == np.float64 and steps.shape == (line["cpu_baseline"]["cores"],) and (steps > 0).all()
    assert np.array_equal(np.load(tmp_path / "trajectory_index.npy"), np.arange(steps.size))


def test_bench_dump_outputs_keeps_a_fixed_sample_under_the_size_limit(tmp_path, monkeypatch):
    """bench.py --dump-outputs: float64 files, trajectories on the last axis; above the size limit every array keeps the same
    seeded sample of trajectories, so two runs with the same arguments write the same files."""
    import bench

    n = 5000
    rng = np.random.default_rng(5)
    arrays = {"final_state": rng.normal(size=(9, n)), "final_epoch_ns": np.arange(n, dtype=np.int64) * 10**9 + 7,
              "status": np.zeros(n, dtype=np.int32)}
    bench.dump_outputs(tmp_path / "all", arrays, first_index=100)
    assert np.array_equal(np.load(tmp_path / "all" / "final_state.npy"), arrays["final_state"])
    assert np.array_equal(np.load(tmp_path / "all" / "final_epoch_ns.npy"), arrays["final_epoch_ns"].astype(np.float64))
    assert np.array_equal(np.load(tmp_path / "all" / "trajectory_index.npy"), 100 + np.arange(n))
    monkeypatch.setattr(bench, "DUMP_BYTES", 100_000)
    for run in ("a", "b"):
        bench.dump_outputs(tmp_path / run, arrays)
    files = sorted((tmp_path / "a").glob("*.npy"))
    assert sum(f.stat().st_size for f in files) <= 100_000
    idx = np.load(tmp_path / "a" / "trajectory_index.npy").astype(np.int64)
    assert 1000 < idx.size < n and (np.diff(idx) > 0).all()
    for f in files:
        a = np.load(f)
        assert a.dtype == np.float64 and np.array_equal(a, np.load(tmp_path / "b" / f.name))
    assert np.array_equal(np.load(tmp_path / "a" / "final_state.npy"), arrays["final_state"][:, idx])
    assert np.array_equal(np.load(tmp_path / "a" / "status.npy"), arrays["status"][idx])


def test_utc_iso_round_trip_across_leap_seconds():
    from nyx_b200.cosmic import epochs_to_utc_iso, utc_iso_to_epochs
    S = 10**9
    ep = np.array([0, 1, -86400 * 366 * S, 5 * 365 * 86400 * S + 123_456_789, 17 * 365 * 86400 * S, 25 * 365 * 86400 * S + 5], dtype=np.int64)
    assert np.array_equal(utc_iso_to_epochs(epochs_to_utc_iso(ep)), ep)
    assert utc_iso_to_epochs(["2000-01-01T11:58:55.816"])[0] == 0 and utc_iso_to_epochs("2000-01-01T11:58:55.816 UTC")[0] == 0
    # one UTC second apart on either side of the 2006-01-01 leap second = two TAI seconds
    a, b = utc_iso_to_epochs(["2005-12-31T23:59:59", "2006-01-01T00:00:00"])
    assert b - a == 2 * S


def test_tracking_arc_parquet_round_trip(tmp_path):
    """od/msr/trackingdata/io_parquet.rs layout: one arc per file; absent measurements are not written, a type absent from a
    measurement is null; `stack` rebuilds the batched arc `process_arcs` takes."""
    import pyarrow.parquet as pq
    S = 10**9
    epochs = np.array([60, 120, 180, 240, 300], dtype=np.int64) * S + 7
    tracker = ["Madrid", "Madrid", "Goldstone", "Goldstone", "Canberra"]
    obs = np.full((5, 2, 3), np.nan)
    rng = np.random.default_rng(0)
    obs[:, 0, :] = rng.uniform(4e5, 5e5, (5, 3))
    obs[:, 1, :] = rng.uniform(-1, 1, (5, 3))
    obs[2, :, 1] = np.nan          # arc 1 misses measurement 2 altogether
    obs[3, 1, 1] = np.nan          # ... and has no Doppler in measurement 3
    obs[:, 1, 2] = np.nan          # arc 2 is range-only
    arc = nb.TrackingDataArc(epochs, tracker, obs)
    paths = [arc.to_parquet(tmp_path / f"arc{i}.parquet", index=i, metadata={"who": "test"}) for i in range(3)]
    t1 = pq.read_table(str(paths[1]))
    assert t1.column_names == ["Epoch (UTC)", "Tracking device", "Range (km)", "Doppler (km/s)"] and t1.num_rows == 4
    assert t1["Doppler (km/s)"].null_count == 1 and t1.schema.metadata[b"Purpose"] == b"Tracking Arc Data" and t1.schema.metadata[b"who"] == b"test"
    assert t1["Epoch (UTC)"][0].as_py() == nb.epochs_to_utc_iso(epochs[:1])[0]
    assert pq.read_table(str(paths[2])).column_names == ["Epoch (UTC)", "Tracking device", "Range (km)"]
    back = [nb.TrackingDataArc.from_parquet(p) for p in paths]
    assert back[0].n == 1 and np.array_equal(back[0].epoch_ns, epochs) and back[0].tracker == tracker
    assert np.array_equal(back[0].obs[:, :, 0], obs[:, :, 0])
    assert len(back[1]) == 4 and np.array_equal(back[1].epoch_ns, epochs[[0, 1, 3, 4]])
    again = nb.TrackingDataArc.stack(back)
    assert again.n == 3 and np.array_equal(again.epoch_ns, epochs) and again.tracker == tracker
    assert np.array_equal(again.obs, obs, equal_nan=True)
    with pytest.raises(nb.ODError, match="EmptyDataset"):
        nb.TrackingDataArc(epochs, tracker, np.full((5, 2, 1), np.nan)).to_parquet(tmp_path / "none.parquet")
    import pyarrow as pa
    pq.write_table(pa.table({"Epoch (UTC)": ["2020-01-01T00:00:00"], "Range (km)": [1.0]}), str(tmp_path / "bad.parquet"))
    with pytest.raises(nb.ODError, match="Tracking device"):
        nb.TrackingDataArc.from_parquet(tmp_path / "bad.parquet")
    pq.write_table(pa.table({"Epoch (UTC)": ["2020-01-01T00:00:00"], "Tracking device": ["X"], "Azimuth (deg)": [1.0]}), str(tmp_path / "bad2.parquet"))
    with pytest.raises(nb.ODError, match="Range"):
        nb.TrackingDataArc.from_parquet(tmp_path / "bad2.parquet")


def test_od_solution_parquet_export(tmp_path):
    """od/process/solution/export.rs columns this path records, from a hand-built solution (no device needed)."""
    import pyarrow.parquet as pq
    from nyx_b200.od import ODSolution
    S = 10**9
    m, n = 4, 2
    frame = nb.EARTH_J2000
    sc = nb.Spacecraft(orbit=nb.Orbit.keplerian(7000.0, 0.01, 30.0, 10.0, 20.0, 40.0, 0, frame), mass=nb.Mass(100.0, 5.0, 0.0))
    rn, dn = nb.StochasticNoise(1e-3), nb.StochasticNoise(1e-6)
    dop_first = nb.GroundStation("DopFirst", 0.0, 0.0, 0.0, measurement_types=[nb.MeasurementType.Doppler, nb.MeasurementType.Range],
                                 stochastic_noises={nb.MeasurementType.Range: rn, nb.MeasurementType.Doppler: dn})
    devices = {"Madrid": nb.GroundStation.dss65_madrid(0.0, rn, dn), "DopFirst": dop_first}
    arc = nb.TrackingDataArc(np.arange(1, m + 1, dtype=np.int64) * 60 * S, ["Madrid", "Madrid", "DopFirst", "Madrid"], np.ones((m, 2, n)))
    est = np.zeros((m, 9, n))
    est[:, :, :] = sc.to_vector()[None, :, None]
    est[:, 0, 1] += np.arange(m)
    cov = np.tile(np.array([4.0, 4.0, 4.0, 1e-6, 1e-6, 1e-6, 0.25, 0.0, 0.0])[None, :, None], (m, 1, n))
    prefit = np.arange(m * 2 * n, dtype=float).reshape(m, 2, n)
    postfit = -prefit
    ratio = np.full((m, 2, n), np.nan)
    ratio[:, 0, :] = 1.5
    flags = np.full((m, n), 1, dtype=np.int32)
    flags[1, 1] = 1 | 2        # processed and rejected
    flags[3, 1] = 4            # not visible: no row
    sol = ODSolution(np.zeros((9, n)), np.zeros(n, dtype=np.int64), np.zeros((n, 9, 9)), np.zeros((9, n)), ratio, prefit, postfit, flags,
                     est, cov, None, np.zeros(n, dtype=np.int32), templates=[sc, sc], arc=arc, devices=devices)
    tab = pq.read_table(str(sol.to_parquet(tmp_path / "od.parquet", index=1, metadata={"run": "7"})))
    assert tab.num_rows == 3 and tab.column_names[0] == "Epoch (UTC)" and "SemiMajorAxis (km)" in tab.column_names
    assert tab["X (km)"].to_pylist() == (sc.orbit.x_km + np.arange(3)).tolist()
    sig_cols = [c for c in tab.column_names if c.startswith("Sigma ")]
    assert len(sig_cols) == 9 and tab[sig_cols[0]].to_pylist() == [2.0] * 3 and tab[sig_cols[6]].to_pylist() == [0.5] * 3
    # slot order follows the tracker's type list: row 2 (DopFirst) has Doppler in slot 0
    assert tab["Prefit residual: Range (km)"].to_pylist() == [prefit[0, 0, 1], prefit[1, 0, 1], prefit[2, 1, 1]]
    assert tab["Prefit residual: Doppler (km/s)"].to_pylist() == [prefit[0, 1, 1], prefit[1, 1, 1], prefit[2, 0, 1]]
    assert tab["Postfit residual: Range (km)"].to_pylist()[2] == postfit[2, 1, 1]
    assert tab["Residual ratio"].to_pylist() == [1.5] * 3 and tab["Residual Rejected"].to_pylist() == [False, True, False]
    assert tab["Tracker"].to_pylist() == ["Madrid", "Madrid", "DopFirst"] and tab.schema.metadata[b"run"] == b"7"
    bare = ODSolution(np.zeros((9, n)), np.zeros(n, dtype=np.int64), np.zeros((n, 9, 9)), np.zeros((9, n)), ratio, prefit, postfit, flags,
                      None, None, None, np.zeros(n, dtype=np.int32), templates=[sc, sc], arc=arc)
    with pytest.raises(nb.ODError, match="record_estimates"):
        bare.to_parquet(tmp_path / "x.parquet")
