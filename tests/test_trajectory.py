"""Trajectory recording + interpolation (SURVEY.md §8 (f)-1): `for_duration_with_traj` / `Traj::at`."""
from pathlib import Path

import numpy as np
import pytest

import nyx_b200 as nb
from nyx_b200.trajectory import Traj, hermite_eval
from tests.util import (S, hermite_shim, leo_ensemble, leo_state, max_dr_dv, oracle_run, resample_queries,
                        resample_reference)


def _dyn(degree=8):
    gd = nb.GravityFieldData.from_fixture("jgm3_70x70", degree, degree, nb.IAU_EARTH_FRAME)
    return nb.SpacecraftDynamics.new(nb.OrbitalDynamics.from_model(nb.GravityField.new(gd)))


def _oracle_traj(oracle, prop, frame, st, cs, ep, end, cap):
    packed = prop.dynamics.pack(frame, None)
    return oracle.propagate_batch(packed.c, prop.opts.to_c(prop.method), st, cs, ep, end, traj_capacity=cap)


def test_hermite_eval_reproduces_polynomials_and_derivatives():
    xs = np.array([0.0, 0.7, 1.1, 2.0, 3.5])
    f = lambda x: 3 * x**5 - x**3 + 2 * x - 1
    df = lambda x: 15 * x**4 - 3 * x**2 + 2
    y, yd = hermite_eval(xs, f(xs), df(xs), 1.7)  # degree 9 interpolant of a quintic: exact
    assert abs(y - f(1.7)) < 1e-11 and abs(yd - df(1.7)) < 1e-10


def test_oracle_recording_matches_channel_semantics(oracle):
    """instance.rs:297-326: start state + every accepted step incl. the final partial one; overflow drops the tail."""
    frame = nb.EARTH_J2000
    mc, (st, cs, ep) = leo_ensemble(5, seed=41)
    prop = nb.Propagator.default(_dyn())
    end = 2 * 3600 * S
    out, out_ep, det, status, (t_ep, t_st, t_cnt) = _oracle_traj(oracle, prop, frame, st, cs, ep, end, 256)
    assert np.array_equal(t_cnt, det["n_steps"] + 1)
    for i in range(5):
        k = t_cnt[i]
        assert t_ep[0, i] == 0 and np.array_equal(t_st[:, 0, i], st[:6, i])          # start state
        assert t_ep[k - 1, i] == end and np.array_equal(t_st[:, k - 1, i], out[:6, i])  # final state
        assert (np.diff(t_ep[:k, i]) > 0).all()
    small = _oracle_traj(oracle, prop, frame, st, cs, ep, end, 10)
    assert (small[4][2] == 10).all() and np.array_equal(small[4][0], t_ep[:10]) and np.array_equal(small[0], out)


def test_traj_at_exact_hit_window_and_accuracy(oracle):
    """Traj::at (traj.rs:83-126): exact epochs return the stored state; in between, the 13-sample Hermite window
    reproduces an independent fine propagation to well below a millimetre."""
    frame = nb.EARTH_J2000
    sc = leo_state(frame)
    st, cs, ep = nb.pack_spacecraft([sc])
    prop = nb.Propagator.default(_dyn())
    end = 3 * 3600 * S
    out, _, det, _, (t_ep, t_st, t_cnt) = _oracle_traj(oracle, prop, frame, st, cs, ep, end, 512)
    k = int(t_cnt[0])
    tr = Traj(sc, t_ep[:k, 0].copy(), np.ascontiguousarray(t_st[:, :k, 0].T)).finalize()
    assert len(tr) == k and tr.first().epoch() == 0 and tr.last().epoch() == end
    mid = tr.at(int(tr.epochs_ns[7]))
    assert np.array_equal(mid.orbit.to_cartesian_pos_vel(), tr.states[7])
    for probe in (12_345_678_901, 5_000 * S + 17, end - 3):
        direct, *_ = oracle_run(oracle, prop, frame, None, st, cs, ep, probe)
        got = tr.at(probe).orbit.to_cartesian_pos_vel()
        assert np.linalg.norm(got[:3] - direct[:3, 0]) < 2e-7 and np.linalg.norm(got[3:] - direct[3:6, 0]) < 1e-9
    with pytest.raises(nb.TrajError):
        tr.at(end + 1)
    with pytest.raises(nb.TrajError):
        tr.at(-1)


def test_traj_finalize_sorts_back_propagation(oracle):
    frame = nb.EARTH_J2000
    sc = leo_state(frame, epoch_ns=3600 * S)
    st, cs, ep = nb.pack_spacecraft([sc])
    prop = nb.Propagator.default(nb.SpacecraftDynamics.new(nb.OrbitalDynamics.two_body()))
    out, out_ep, det, _, (t_ep, t_st, t_cnt) = _oracle_traj(oracle, prop, frame.with_mu_km3_s2(nb.GMAT_EARTH_GM), st, cs, ep, 0, 256)
    k = int(t_cnt[0])
    assert out_ep[0] == 0 and (np.diff(t_ep[:k, 0]) < 0).all()  # recorded in propagation order (descending epochs)
    tr = Traj(sc, t_ep[:k, 0].copy(), np.ascontiguousarray(t_st[:, :k, 0].T)).finalize()
    assert (np.diff(tr.epochs_ns) > 0).all() and tr.first().epoch() == 0 and tr.last().epoch() == 3600 * S


@pytest.mark.gpu
@pytest.mark.parametrize("mode,lanes", [(nb.MODE_STRICT, 1), (nb.MODE_STRICT, 8), (nb.MODE_FAST, 1), (nb.MODE_FAST, 8), (nb.MODE_FAST, 16)])
def test_gpu_recording_matches_oracle(oracle, mode, lanes):
    """Every kernel writes the same step-major SoA stream the oracle records: bit-identical in STRICT mode."""
    frame = nb.EARTH_J2000
    mc, (st, cs, ep) = leo_ensemble(40, seed=42)
    ep = ep + (np.arange(40, dtype=np.int64) % 3) * 900 * S
    prop = nb.Propagator.default(_dyn(21), mode=mode)
    eng = prop.engine(frame, None)
    eng.set_lanes(lanes)
    end = 2 * 3600 * S
    out, out_ep, det, status, (g_ep, g_st, g_cnt) = eng.propagate_batch(st, cs, ep, end, traj_capacity=128)
    ref, ref_ep, ref_det, ref_status, (o_ep, o_st, o_cnt) = _oracle_traj(oracle, prop, frame, st, cs, ep, end, 128)
    assert (status == 0).all() and np.array_equal(g_cnt, det["n_steps"] + 1)
    if mode == nb.MODE_STRICT:
        assert np.array_equal(g_cnt, o_cnt) and np.array_equal(g_ep, o_ep) and np.array_equal(g_st, o_st)
    else:
        assert np.abs(g_cnt - o_cnt).max() <= 1
        for i in range(40):
            k = int(min(g_cnt[i], o_cnt[i])) - 1
            assert np.abs(g_ep[:k, i] - o_ep[:k, i]).max() < 1_000_000_000  # step epochs drift by the controller's noise only (< 1 s over 2 h)
            assert np.array_equal(g_st[:, 0, i], st[:6, i])
        assert max_dr_dv(out, ref)[0] < 5e-7
    # capacity overflow keeps the head of the stream and still returns the right final state
    o2, _, d2, _, (e2, s2, c2) = eng.propagate_batch(st, cs, ep, end, traj_capacity=7)
    assert (c2 == 7).all() and np.array_equal(e2, g_ep[:7]) and np.array_equal(o2, out)


@pytest.mark.gpu
def test_prop_instance_with_traj_api(oracle):
    """`PropInstance::for_duration_with_traj` (instance.rs:297-326) + `Traj::at` through the public API."""
    frame = nb.EARTH_J2000
    sc = leo_state(frame)
    prop = nb.Propagator.default(_dyn(21), mode=nb.MODE_STRICT)
    inst = prop.with_(sc)
    final, tr = inst.for_duration_with_traj(6 * 3600 * S)
    assert final.epoch() == 6 * 3600 * S and tr.last().epoch() == final.epoch() and tr.first().epoch() == 0
    assert len(tr) == inst.latest_details().n_steps + 1
    assert np.array_equal(tr.last().orbit.to_cartesian_pos_vel(), final.orbit.to_cartesian_pos_vel())
    st, cs, ep = nb.pack_spacecraft([sc])
    direct, *_ = oracle_run(oracle, prop, frame, None, st, cs, ep, 10_000 * S)
    assert np.linalg.norm(tr.at(10_000 * S).orbit.radius_km - direct[:3, 0]) < 2e-7
    # explicit capacity that the run overflows: an error, never a silently truncated Traj (the reference's Traj holds every step)
    with pytest.raises(nb.PropagationError, match="capacity 16 too small"):
        prop.with_(sc).for_duration_with_traj(6 * 3600 * S, capacity=16)
    f2, tr2 = prop.with_(sc).for_duration_with_traj(6 * 3600 * S, capacity=len(tr))
    assert len(tr2) == len(tr) and np.array_equal(f2.orbit.to_cartesian_pos_vel(), final.orbit.to_cartesian_pos_vel())


# ---- batched resampling (nyxb_traj_resample): the kernel's per-(query, trajectory) function on the CPU
def test_resample_core_matches_traj_at(oracle, tmp_path):
    """The function the CUDA kernel runs per (query, trajectory), compiled for the host: bit-identical to Traj.at on ragged
    recordings (different step counts per trajectory, capacity overflow, empty), forward and backward."""
    frame = nb.EARTH_J2000
    mc, (st, cs, ep) = leo_ensemble(7, seed=77)
    prop = nb.Propagator.default(_dyn())
    run = hermite_shim(tmp_path)
    sc = leo_state(frame)
    for end, cap in ((3 * 3600 * S, 256), (3 * 3600 * S, 40), (-2 * 3600 * S, 256)):
        ep_b = ep.copy()
        _, _, det, status, (t_ep, t_st, t_cnt) = _oracle_traj(oracle, prop, frame, st, cs, ep_b, end, cap)
        assert (status == 0).all()
        t_cnt = t_cnt.copy()
        t_cnt -= 5 * np.arange(7)   # ragged: every trajectory keeps a different prefix of its records
        t_cnt[6] = 0                # a run that recorded nothing
        t_cnt[5] = 9                # fewer records than one interpolation window
        lo, hi = min(0, end), max(0, end)
        queries = resample_queries(t_ep if end > 0 else t_ep[::-1], t_cnt, hi) if end > 0 else \
            np.concatenate([np.array([lo - 1, lo, lo + 1, -1, 0, 1, int(t_ep[2, 1])], dtype=np.int64),
                            np.arange(lo, 0, 450 * S, dtype=np.int64) + 987_654_321])
        want, want_status = resample_reference(sc, t_ep, t_st, t_cnt, queries)
        got, got_status = run(t_ep, t_st, t_cnt, queries)
        assert np.array_equal(got_status, want_status)
        assert (want_status == 0).any() and (want_status == 1).any()
        assert np.array_equal(np.isnan(got), np.isnan(want))
        ok = want_status == 0
        assert np.array_equal(got[:, ok], want[:, ok])   # same operations in the same order, no FMA: bit-identical


def test_traj_iteration_filter_and_parquet(oracle, tmp_path):
    """traj.rs:148-193, 226-360: `every`, `every_between` (clamped to the span), `filter_by_epoch`, `to_parquet`."""
    import pyarrow.parquet as pq
    from nyx_b200.param import EXPORT_PARAMS, StateParameter as P
    frame = nb.EARTH_J2000
    sc = leo_state(frame)
    st, cs, ep = nb.pack_spacecraft([sc])
    prop = nb.Propagator.default(_dyn())
    end = 2 * 3600 * S
    _, _, _, _, (t_ep, t_st, t_cnt) = _oracle_traj(oracle, prop, frame, st, cs, ep, end, 256)
    k = int(t_cnt[0])
    tr = Traj(sc, t_ep[:k, 0].copy(), np.ascontiguousarray(t_st[:, :k, 0].T)).finalize()
    step = 7 * 60 * S
    every = list(tr.every(step))
    assert [s.epoch() for s in every] == list(range(0, end + 1, step))
    assert np.array_equal(every[3].orbit.to_cartesian_pos_vel(), tr.at(3 * step).orbit.to_cartesian_pos_vel())
    clamped = list(tr.every_between(step, -5 * S, end + 5 * S))
    assert [s.epoch() for s in clamped] == [s.epoch() for s in every]
    inner = list(tr.every_between(step, 1000 * S, 5000 * S))
    assert inner[0].epoch() == 1000 * S and inner[-1].epoch() <= 5000 * S and len(inner) == (4000 * S) // step + 1
    assert list(tr.every_between(step, end + 1, end + 2)) == []
    with pytest.raises(ValueError):
        list(tr.every(0))
    sub = tr.filter_by_epoch(int(tr.epochs_ns[5]), int(tr.epochs_ns[20]))
    assert len(sub) == 16 and sub.first().epoch() == tr.epochs_ns[5] and np.array_equal(sub.states, tr.states[5:21])
    raw = pq.read_table(str(tr.to_parquet(tmp_path / "traj.parquet")))
    assert raw.num_rows == k and raw.column_names == ["Epoch (UTC)"] + [str(p) for p in EXPORT_PARAMS]
    assert np.array_equal(np.array(raw["VZ (km/s)"].to_pylist()), tr.states[:, 5])
    assert raw.schema.metadata[b"Purpose"] == b"Trajectory data"
    grid = pq.read_table(str(tr.to_parquet(tmp_path / "traj_grid.parquet", fields=[P.X, P.Thrust, P.Rmag], step_ns=step, metadata={"k": "v"})))
    assert grid.column_names == ["Epoch (UTC)", "X (km)", "Rmag (km)"] and grid.num_rows == len(every)
    assert grid["X (km)"].to_pylist() == [s.orbit.x_km for s in every] and grid.schema.metadata[b"k"] == b"v"
    assert grid["Epoch (UTC)"][1].as_py() == nb.epochs_to_utc_iso([step])[0]
    # sc_traj.rs:212-440: read back
    back = Traj.from_parquet(tmp_path / "traj.parquet", sc)
    assert np.array_equal(back.epochs_ns, tr.epochs_ns) and np.array_equal(back.states, tr.states)
    with pytest.raises(nb.TrajError, match="MissingData"):
        Traj.from_parquet(tmp_path / "traj_grid.parquet", sc)          # no velocity columns
    moon_sc = nb.Spacecraft.from_orbit(nb.Orbit.cartesian(1800.0, 0, 0, 0, 1.6, 0, 0, nb.MOON_J2000))
    with pytest.raises(nb.TrajError, match="frame"):
        Traj.from_parquet(tmp_path / "traj.parquet", moon_sc)


OEM_DIR = Path(__file__).parent / "golden" / "oem"


def test_reference_oem_samples(tmp_path):
    """The reference's own OEM tests (md/trajectory/sc_traj.rs:450-585) on its sample files, stored unchanged under
    tests/golden/oem: state counts after removing the duplicate epochs (361 / 61 / 181), the name taken from OBJECT_ID, an
    export / reload round trip, and the trimmed, re-interpolated export (one state fewer, first + 1 s, last - 19 s)."""
    for name, count in (("LEO_10s", 361), ("MEO_60s", 61), ("GEO_20s", 181)):
        tr = Traj.from_oem_file(f"{OEM_DIR}/{name}.oem")
        assert len(tr) == count and tr.name == "0000-000A" and (np.diff(tr.epochs_ns) > 0).all()
    geo = Traj.from_oem_file(f"{OEM_DIR}/GEO_20s.oem")
    assert nb.epochs_to_utc_iso(geo.epochs_ns[:1])[0].startswith("2020-06-01T12:00:00")
    out = tmp_path / "GEO_20s_rebuilt.oem"
    geo.to_oem_file(out, "0000-000A", "Test Suite", "TEST_OBJ")
    again = Traj.from_oem_file(out)
    assert again.name == geo.name and np.array_equal(again.epochs_ns, geo.epochs_ns) and np.array_equal(again.states, geo.states)
    S_ = 10**9
    geo.to_oem_file(out, "TEST-OBJ-ID", "Test Suite", "TEST_OBJ", start_ns=int(geo.epochs_ns[0]) + S_, end_ns=int(geo.epochs_ns[-1]) - S_,
                    step_ns=20 * S_)
    trimmed = Traj.from_oem_file(out)
    assert trimmed.name == "TEST-OBJ-ID" and len(trimmed) == len(geo) - 1
    assert trimmed.epochs_ns[0] == geo.epochs_ns[0] + S_ and trimmed.epochs_ns[-1] == geo.epochs_ns[-1] - 19 * S_
    # the interpolated states sit on the sampled orbit: compare with the neighbouring samples' chord to GEO accuracy
    mid = trimmed.states[10, :3]
    assert np.linalg.norm(mid - geo.states[10, :3]) < 3.2 and np.linalg.norm(mid - geo.states[11, :3]) > 50.0


def test_oem_round_trip_and_errors(oracle, tmp_path):
    frame = nb.EARTH_J2000
    sc = leo_state(frame)
    st, cs, ep = nb.pack_spacecraft([sc])
    _, _, _, _, (t_ep, t_st, t_cnt) = _oracle_traj(oracle, nb.Propagator.default(_dyn()), frame, st, cs, ep, 1800 * S, 64)
    k = int(t_cnt[0])
    tr = Traj(sc, t_ep[:k, 0].copy(), np.ascontiguousarray(t_st[:, :k, 0].T)).finalize()
    path = tr.to_oem_file(tmp_path / "leo.oem", "2024-001A", object_name="LEO")
    back = Traj.from_oem_file(path, sc)
    assert back.name == "2024-001A" and np.array_equal(back.epochs_ns, tr.epochs_ns) and np.array_equal(back.states, tr.states)
    assert Traj.from_oem_file(path).template.orbit.frame.ephemeris_id == frame.ephemeris_id     # frame from CENTER_NAME
    text = open(path).read()
    (tmp_path / "tai.oem").write_text(text.replace("TIME_SYSTEM = UTC", "TIME_SYSTEM = TAI"))
    tai = Traj.from_oem_file(tmp_path / "tai.oem")
    assert tai.epochs_ns[0] - tr.epochs_ns[0] == -32 * S         # the same stamp read as TAI is 32 s earlier than read as UTC (2000)
    (tmp_path / "bad.oem").write_text("META_START\nMETA_STOP\n")
    with pytest.raises(nb.TrajError):
        Traj.from_oem_file(tmp_path / "bad.oem")
    (tmp_path / "mars.oem").write_text(text.replace("CENTER_NAME = EARTH", "CENTER_NAME = MARS"))
    with pytest.raises(nb.TrajError, match="CENTER_NAME"):
        Traj.from_oem_file(tmp_path / "mars.oem")
