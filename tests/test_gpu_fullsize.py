"""Size-independent properties at BASELINE.json's FULL sizes (the oracle cannot cover these in seconds): shard / permutation
invariance (trajectories are independent, so any split of the ensemble must give bit-identical results), forward-backward round
trips, span splitting, and bit-parity of the STRICT kernel against the oracle on a sample drawn from the full ensemble.
Tolerances: round trip over 3 days (two adaptive passes, FAST) < 1e-4 km; split span < 1e-5 km (different step sequence after
the restart); everything that only regroups trajectories: bit-exact."""
import numpy as np
import pytest

import nyx_b200 as nb

from .util import S

pytestmark = pytest.mark.gpu
DAY = 86400 * S


def _c2(n, degree=21):
    rng = np.random.Generator(np.random.PCG64(0))
    frame = nb.EARTH_J2000
    gd = nb.GravityFieldData.from_fixture("jgm3_70x70", degree, degree, nb.IAU_EARTH_FRAME)
    dyn = nb.SpacecraftDynamics.new(nb.OrbitalDynamics.from_model(nb.GravityField.new(gd)))
    orbit = nb.Orbit.keplerian(6378.1363 + 300.0, 0.015, 68.5, 65.2, 75.0, 0.0, 0, frame)
    template = nb.Spacecraft(orbit=orbit, mass=nb.Mass(1000.0, 0.0, 0.0))
    mvn = nb.MvnSpacecraft.from_cartesian_std(template, 1.0, 1e-3)
    st = np.ascontiguousarray((template.to_vector()[None, :] + mvn.sample_vectors(rng, n)).T)
    cs = np.zeros((4, n)); cs[0] = 1000.0
    return frame, dyn, st, cs, np.zeros(n, dtype=np.int64)


def test_c2_full_size_invariances_fast():
    n = 10_000
    frame, dyn, st, cs, ep = _c2(n)
    eng = nb.Propagator.default(dyn, mode=nb.MODE_FAST).engine(frame, None)
    out, oep, det, status = eng.propagate_batch(st, cs, ep, 3 * DAY)
    assert (status == 0).all() and (oep == 3 * DAY).all()
    assert 3.5e7 < det["n_steps"].sum() < 4.5e7                       # ~3.9e7 accepted steps (SURVEY.md §8d)
    # The automatic dispatch picks the kernel family by ensemble size (transposed kernel from 1 024 trajectories, the lane-
    # cooperative one below): FAST results are bit-reproducible per family, tolerance-equal across families.
    assert eng.last_kernel() == nb.KERNEL_TRANSPOSED
    eng.set_kernel(nb.KERNEL_COOP)
    a_coop = eng.propagate_batch(st[:, :2000].copy(), cs[:, :2000].copy(), ep[:2000].copy(), 3 * DAY)[0]
    assert eng.last_kernel() == nb.KERNEL_COOP
    assert np.sqrt(((a_coop[:3] - out[:3, :2000]) ** 2).sum(0)).max() < 3e-6   # each within 1e-6 km of the reference
    # shards: whatever family the dispatch picks, the two halves on their own reproduce the full batch bit for bit when it is the same one
    eng.set_kernel(nb.KERNEL_AUTO)
    a = eng.propagate_batch(st[:, :5000].copy(), cs[:, :5000].copy(), ep[:5000].copy(), 3 * DAY)[0]
    b = eng.propagate_batch(st[:, 5000:].copy(), cs[:, 5000:].copy(), ep[5000:].copy(), 3 * DAY)[0]
    assert np.array_equal(np.concatenate([a, b], axis=1), out)
    # permutation of the run order permutes the results
    perm = np.random.default_rng(1).permutation(n)
    p = eng.propagate_batch(np.ascontiguousarray(st[:, perm]), cs[:, perm].copy(), ep[perm].copy(), 3 * DAY)[0]
    assert np.array_equal(p, out[:, perm])
    # forward then backward returns to the start
    back, bep, _, bst = eng.propagate_batch(out, cs, oep, 0)
    assert (bst == 0).all() and (bep == 0).all()
    assert np.sqrt(((back[:3] - st[:3]) ** 2).sum(0)).max() < 1e-4
    # split span (the adapted step is carried like a PropInstance would): same end state to the truncation level
    step = np.full(n, 60 * S, dtype=np.int64)
    mid, mep, _, _ = eng.propagate_batch(st, cs, ep, 3 * DAY // 2, step_ns=step)
    fin, fep, _, _ = eng.propagate_batch(mid, cs, mep, 3 * DAY, step_ns=step)
    assert np.sqrt(((fin[:3] - out[:3]) ** 2).sum(0)).max() < 1e-5


def test_c2_full_size_strict_bit_parity_sample(oracle):
    n = 10_000
    frame, dyn, st, cs, ep = _c2(n)
    prop = nb.Propagator.default(dyn, mode=nb.MODE_STRICT)
    out, oep, det, status = prop.engine(frame, None).propagate_batch(st, cs, ep, 3 * DAY)
    assert (status == 0).all()
    idx = np.random.default_rng(2).choice(n, 256, replace=False)
    packed = dyn.pack(frame, None)
    ref, _, rdet, _ = oracle.propagate_batch(packed.c, prop.opts.to_c(prop.method), np.ascontiguousarray(st[:, idx]), cs[:, idx].copy(), ep[idx].copy(), 3 * DAY)
    assert np.array_equal(out[:, idx], ref) and np.array_equal(det["n_steps"][idx], rdet["n_steps"])


def test_c3_full_size_invariances():
    """100 000 JWST-like trajectories, Sun + Moon point masses + SRP with Earth / Moon shadows, 30 days (BASELINE configs[2])."""
    n = 100_000
    frame = nb.EARTH_J2000
    alm = nb.Almanac.synthetic(frame, 0, 32.0)
    srp = nb.SolarPressure.new([nb.EARTH_J2000, nb.MOON_J2000], alm)
    dyn = nb.SpacecraftDynamics.from_model(nb.OrbitalDynamics.point_masses([nb.MOON, nb.SUN]), srp)
    orbit = nb.Orbit.cartesian(119901.070276, -1389299.665421, -1041369.150539, 0.045956, -0.013168, 0.034535, 0, frame)
    template = nb.Spacecraft(orbit=orbit, mass=nb.Mass(6200.0, 0.0, 0.0), srp=nb.SRPData(21.197 * 14.162, 1.56))
    mvn = nb.MvnSpacecraft.from_cartesian_std(template, 0.5, 1e-4)
    st = np.ascontiguousarray((template.to_vector()[None, :] + mvn.sample_vectors(np.random.default_rng(0), n)).T)
    cs = np.zeros((4, n)); cs[0] = 6200.0; cs[2] = template.srp.area_m2
    ep = np.zeros(n, dtype=np.int64)
    eng = nb.Propagator.default(dyn, mode=nb.MODE_FAST).engine(frame, alm)
    out, oep, det, status = eng.propagate_batch(st, cs, ep, 30 * DAY)
    assert (status == 0).all() and det["n_steps"].min() > 900          # steps saturate near max_step = 2700 s
    k = 37_123
    a = eng.propagate_batch(st[:, :k].copy(), cs[:, :k].copy(), ep[:k].copy(), 30 * DAY)[0]
    b = eng.propagate_batch(st[:, k:].copy(), cs[:, k:].copy(), ep[k:].copy(), 30 * DAY)[0]
    assert np.array_equal(np.concatenate([a, b], axis=1), out)
    back, bep, _, bst = eng.propagate_batch(out, cs, oep, 0)
    assert (bst == 0).all() and np.sqrt(((back[:3] - st[:3]) ** 2).sum(0)).max() < 1e-3   # 1.7e6 km from the Earth, 2 x 30 days


def test_c4_size_shard_invariance_and_round_trip():
    """2 000 low-lunar-orbit trajectories, GRAIL 70x70 + Earth/Sun point masses (BASELINE configs[3]; 1 of the 7 days)."""
    from nyx_b200.frames import EARTH

    n = 2000
    frame = nb.MOON_J2000
    alm = nb.Almanac.synthetic(frame, 0, 3.0, bodies=(EARTH, nb.SUN))
    gd = nb.GravityFieldData.from_fixture("luna_jggrx_80x80", 70, 70, nb.IAU_MOON_FRAME)
    dyn = nb.SpacecraftDynamics.new(nb.OrbitalDynamics.new([nb.PointMasses.new([EARTH, nb.SUN]), nb.GravityField.new(gd)]))
    orbit = nb.Orbit.keplerian(1737.4 + 100.0, 0.001, 90.0, 10.0, 0.0, 0.0, 0, frame)
    template = nb.Spacecraft(orbit=orbit, mass=nb.Mass(1000.0, 0.0, 0.0))
    mvn = nb.MvnSpacecraft.from_cartesian_std(template, 0.1, 1e-4)
    st = np.ascontiguousarray((template.to_vector()[None, :] + mvn.sample_vectors(np.random.default_rng(0), n)).T)
    cs = np.zeros((4, n)); cs[0] = 1000.0
    ep = np.zeros(n, dtype=np.int64)
    eng = nb.Propagator.default(dyn, mode=nb.MODE_FAST).engine(frame, alm)
    out, oep, det, status = eng.propagate_batch(st, cs, ep, DAY)
    assert (status == 0).all() and eng.lanes() == 32
    # the automatic dispatch sends 2 000 trajectories to the transposed kernel and a shard of 777 to the lane-cooperative one;
    # FAST results are bit-reproducible per family, so each family is pinned for the whole batch and both of its shards
    assert eng.last_kernel() == nb.KERNEL_TRANSPOSED
    for family in (nb.KERNEL_TRANSPOSED, nb.KERNEL_COOP):
        eng.set_kernel(family)
        whole = out if family == nb.KERNEL_TRANSPOSED else eng.propagate_batch(st, cs, ep, DAY)[0]
        a = eng.propagate_batch(st[:, :777].copy(), cs[:, :777].copy(), ep[:777].copy(), DAY)[0]
        assert eng.last_kernel() == family
        b = eng.propagate_batch(st[:, 777:].copy(), cs[:, 777:].copy(), ep[777:].copy(), DAY)[0]
        assert np.array_equal(np.concatenate([a, b], axis=1), whole)
    eng.set_kernel(nb.KERNEL_AUTO)
    back, _, _, bst = eng.propagate_batch(out, cs, oep, 0)
    assert (bst == 0).all() and np.sqrt(((back[:3] - st[:3]) ** 2).sum(0)).max() < 1e-5


def test_large_ensemble_dispatches_to_per_thread_column_walk_and_matches_cooperative_kernel(oracle):
    """FAST, 21x21, >= 65 536 trajectories: the engine picks the per-thread column-walk kernel.  Same ensemble through the
    cooperative kernel (lanes = 8): both are FAST regroupings of the same sums -> agreement at the step-sequence level, and
    both agree with the oracle on a sample."""
    n = 70_000
    frame, dyn, st, cs, ep = _c2(n)
    end = 3600 * S
    auto = nb.Propagator.default(dyn, mode=nb.MODE_FAST).engine(frame, None)
    out_a, _, det_a, status_a = auto.propagate_batch(st, cs, ep, end)
    coop = nb.Propagator.default(dyn, mode=nb.MODE_FAST).engine(frame, None)
    coop.set_lanes(8)
    out_c, _, det_c, status_c = coop.propagate_batch(st, cs, ep, end)
    assert (status_a == 0).all() and (status_c == 0).all()
    assert np.sqrt(((out_a[:3] - out_c[:3]) ** 2).sum(0)).max() < 5e-7   # measured 1.5e-7 km over 70 000 (step-sequence sensitivity)
    assert np.abs(det_a["n_steps"] - det_c["n_steps"]).max() <= 1
    idx = np.random.default_rng(3).choice(n, 128, replace=False)
    prop = nb.Propagator.default(dyn)
    ref, _, _, _ = oracle.propagate_batch(dyn.pack(frame, None).c, prop.opts.to_c(prop.method), np.ascontiguousarray(st[:, idx]), cs[:, idx].copy(), ep[idx].copy(), end)
    assert np.sqrt(((out_a[:3, idx] - ref[:3]) ** 2).sum(0)).max() < 3e-7


def test_c2_full_size_resampling_properties():
    """nyxb_traj_resample over the full C2 ensemble (10 000 recorded trajectories, adaptive steps, 6 h): queries on a regular
    grid reproduce an independent propagation to the same epochs (Hermite window of 13 records, < 1e-6 km / 1e-9 km/s — the
    window spans ~1000 s of a 90-minute orbit); every trajectory's own record epochs come back bit for bit (exact hits);
    shards reproduce the whole; epochs outside a trajectory's span are flagged, never extrapolated."""
    n = 10_000
    frame, dyn, st, cs, ep = _c2(n)
    eng = nb.Propagator.default(dyn, mode=nb.MODE_FAST).engine(frame, None)
    end = 6 * 3600 * S
    out, oep, det, status, (t_ep, t_st, t_cnt) = eng.propagate_batch(st, cs, ep, end, traj_capacity=400)
    assert (status == 0).all() and np.array_equal(t_cnt, det["n_steps"] + 1) and t_cnt.max() <= 400
    grid = np.arange(0, end + 1, 1800 * S, dtype=np.int64) + 777
    grid[-1] = end
    rs, rstat = eng.resample(np.concatenate([grid, [end + 1, -1]]), n=n)          # resident recording
    assert (rstat[:-2] == 0).all() and (rstat[-2:] == 1).all() and np.isnan(rs[:, -2:, :]).all()
    assert np.array_equal(rs[:, len(grid) - 1, :], out[:6])                       # the final record is the final state
    for j in (1, 5, 9):
        direct = eng.propagate_batch(st, cs, ep, int(grid[j]))[0]
        assert np.sqrt(((rs[:3, j] - direct[:3]) ** 2).sum(0)).max() < 1e-6
        assert np.sqrt(((rs[3:, j] - direct[3:6]) ** 2).sum(0)).max() < 1e-9
    # exact hits: each trajectory's 7th and last-but-one record epochs (different per trajectory) queried for everyone;
    # the owner must get its record back bit for bit
    for i in (0, 4999, 9999):
        q = np.array([t_ep[7, i], t_ep[t_cnt[i] - 2, i]], dtype=np.int64)
        r2, s2 = eng.resample(q, (t_ep, t_st, t_cnt))
        assert (s2 == 0).all()
        assert np.array_equal(r2[:, 0, i], t_st[:, 7, i]) and np.array_equal(r2[:, 1, i], t_st[:, t_cnt[i] - 2, i])
    # shards
    lo = slice(0, 3000)
    r3, s3 = eng.resample(grid, (np.ascontiguousarray(t_ep[:, lo]), np.ascontiguousarray(t_st[:, :, lo]), t_cnt[lo].copy()))
    assert np.array_equal(r3, rs[:, :len(grid), lo]) and (s3 == 0).all()
