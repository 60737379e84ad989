"""Config / wire formats (SURVEY.md §8 f-4): the reference's serde layouts build the same host objects as the constructors."""
from pathlib import Path

import numpy as np
import pytest

import nyx_b200 as nb

FIX = Path(__file__).parent / "fixtures"


def test_parse_duration_forms():
    assert nb.parse_duration("1 min") == 60 * 10**9
    assert nb.parse_duration("2 h 30 min") == 9000 * 10**9
    assert nb.parse_duration("0.5 s") == 5 * 10**8
    assert nb.parse_duration("1 ms") == 10**6
    assert nb.parse_duration(42) == 42
    with pytest.raises(ValueError):
        nb.parse_duration("3 fortnights")


def test_ground_stations_from_yaml():
    st = nb.load_ground_stations(FIX / "stations.yaml")
    assert list(st) == ["Station A", "Station B"]
    a, b = st["Station A"], st["Station B"]
    ref = nb.GroundStation.dss65_madrid(5.0, nb.StochasticNoise(5e-3), nb.StochasticNoise(50e-6, 1e-7))
    assert (a.latitude_deg, a.longitude_deg, a.height_km, a.elevation_mask_deg) == (ref.latitude_deg, ref.longitude_deg, ref.height_km, 5.0)
    assert a.stochastic_noises == ref.stochastic_noises and list(a.measurement_types) == [nb.MeasurementType.Range, nb.MeasurementType.Doppler]
    assert b.elevation_mask_deg == 7.5 and list(b.measurement_types) == [nb.MeasurementType.Doppler]
    ca = a.to_c(nb.EARTH_J2000, None)
    assert ca.n_types == 2 and abs(ca.noise_var[0] - 25e-6) < 1e-18 and ca.bias[1] == 1e-7 and ca.body == -1
    cb = b.to_c(nb.EARTH_J2000, None)
    assert cb.n_types == 1 and cb.types[0] == nb.abi.MSR_DOPPLER and abs(cb.noise_var[0] - 9e-12) < 1e-24


def test_propagator_config_builds_the_closed_model_set():
    cfg = nb.PropagatorConfig.load({
        "method": "DormandPrince78",
        "options": {"init_step": "30 s", "min_step": "1 ms", "max_step": "10 min", "tolerance": 1e-10, "attempts": 20, "error_ctrl": "RSSCartesianState"},
        "dynamics": {"accel_models": {"point_masses": {"celestial_objects": [301, 10], "correction": None}},
                     "force_models": {"solar_pressure": {"phi": 1367.0, "shadow_bodies": [399, 301], "estimate": False}}}})
    alm = nb.Almanac.synthetic(nb.EARTH_J2000, 0, 3.0)
    prop = cfg.build(alm)
    assert prop.method == nb.IntegratorMethod.DormandPrince78
    assert (prop.opts.init_step, prop.opts.min_step, prop.opts.max_step) == (30 * 10**9, 10**6, 600 * 10**9)
    assert prop.opts.tolerance == 1e-10 and prop.opts.attempts == 20 and prop.opts.error_ctrl == nb.ErrorControl.RSSCartesianState
    packed = prop.dynamics.pack(nb.EARTH_J2000, alm)
    assert packed.c.point_mass_mask != 0 and packed.c.srp.contents.n_shadow == 2 and packed.c.srp.contents.estimate == 0
    # same descriptor as the constructor route
    ref = nb.SpacecraftDynamics.from_model(nb.OrbitalDynamics.point_masses([nb.MOON, nb.SUN]),
                                           nb.SolarPressure.default_no_estimation([nb.EARTH_J2000, nb.MOON_J2000], alm)).pack(nb.EARTH_J2000, alm)
    assert packed.c.point_mass_mask == ref.c.point_mass_mask and packed.c.mu_central_km3_s2 == ref.c.mu_central_km3_s2
    with pytest.raises(nb.DynamicsError, match="SolidTides"):
        nb.PropagatorConfig.load({"dynamics": {"accel_models": {"solid_tides": {"k2": 0.3}}}}).build(alm)
    assert nb.PropagatorConfig.load({}).build().opts.init_step == 60 * 10**9


# ---- Dhall (the format the reference ships its configurations in)
def test_dhall_data_subset_reader():
    from nyx_b200 import dhall
    v = dhall.loads('''
      -- comment
      { a = +3, b = -2.5e-3, c = [ 1, 2 ], d = [] : List { x : Double }, e = Some "t\\"x\\n", f = None (Optional Text), g = True
      , u = < A | B : { k : Natural } | C : Double >.B { k = 7 }, w = < A | B : Text >.A, `odd key` = {=}, n = { z = 12 }
      {- block
         comment -} , big = 1.0e-12, nat = 50, t = { _1 = "k", _2 = 2 } }''')
    assert v == {"a": 3, "b": -2.5e-3, "c": [1, 2], "d": [], "e": 't"x\n', "f": None, "g": True, "u": {"B": {"k": 7}}, "w": "A",
                 "odd key": {}, "n": {"z": 12}, "big": 1e-12, "nat": 50, "t": {"_1": "k", "_2": 2}}
    assert isinstance(v["a"], int) and isinstance(v["big"], float)
    assert dhall.pairs_to_dict([{"_1": "x", "_2": 1}, {"_1": "y", "_2": 2}]) == {"x": 1, "y": 2}
    assert dhall.pairs_to_dict([{"mapKey": "x", "mapValue": 1}]) == {"x": 1} and dhall.pairs_to_dict([1, 2]) == [1, 2]
    for bad in ("let x = 1 in x", "{ a = 1 } // { b = 2 }", "./other.dhall", '{ a = "${x}" }', "< A | B >.C", "{ a = 1", "[ 1, 2 ] 3",
                "\\(x : Natural) -> x"):
        with pytest.raises(dhall.DhallError):
            dhall.loads(bad)


def test_propagator_config_from_dhall(tmp_path):
    """data/02_config/prop_config.dhall layout -> PropagatorConfig -> engine descriptor, identical to the constructor route."""
    import shutil
    from pathlib import Path
    src = Path(__file__).parent / "fixtures" / "prop_config.dhall"
    shutil.copy(src, tmp_path / "prop_config.dhall")
    # the gravity file the config names: JGM-3 written in the SHADR text layout (header line + "n, m, C, S" records)
    z = np.load(Path(__file__).parent.parent / "data" / "jgm3_70x70.npz")
    with open(tmp_path / "jgm3_12x12.sha.tab", "w") as fh:
        fh.write("0.6378136300E+04, 0.3986004415E+06, 70, 70\n")
        for n, m, c, s in zip(z["n"], z["m"], z["c"], z["s"]):
            if n <= 14:
                fh.write(f"{int(n):5d},{int(m):5d}, {float(c)!r}, {float(s)!r}\n")
    cfg = nb.PropagatorConfig.load(tmp_path / "prop_config.dhall")
    assert cfg.method == nb.IntegratorMethod.DormandPrince78
    o = cfg.options
    assert (o.init_step, o.min_step, o.max_step, o.tolerance, o.attempts, o.fixed_step) == (30 * 10**9, 10**6, 600 * 10**9, 1e-11, 30, False)
    assert o.error_ctrl == nb.ErrorControl.RSSCartesianState
    g = cfg.dynamics["accel_models"]["gravity_field"]
    assert g["_1"]["degree"] == 12 and g["_2"] == {"ephemeris_id": 399, "orientation_id": 399}
    assert cfg.dynamics["force_models"]["solar_pressure"] is None
    assert cfg.dynamics["force_models"]["drag"]["density"] == {"Exponential": {"r0": 700000.0, "ref_alt_m": 88667.0, "rho0": 3.614e-13}}
    g["_1"]["filepath"] = str(tmp_path / g["_1"]["filepath"])
    alm = nb.Almanac.synthetic(nb.EARTH_J2000, 0, 3.0)
    prop = cfg.build(alm)
    packed = prop.dynamics.pack(nb.EARTH_J2000, alm)
    gd = nb.GravityFieldData.from_fixture("jgm3_70x70", 12, 10, nb.IAU_EARTH_FRAME)
    ref = nb.SpacecraftDynamics.from_models(
        nb.OrbitalDynamics.new([nb.PointMasses.new([nb.MOON]), nb.GravityField.new(gd)]),
        [nb.Drag(nb.AtmDensity.Exponential(3.614e-13, 700000.0, 88667.0), nb.IAU_EARTH_FRAME, False)]).pack(nb.EARTH_J2000, alm)
    gc, rc = packed.c.gravity.contents, ref.c.gravity.contents
    assert (gc.degree, gc.order) == (rc.degree, rc.order) == (12, 12)   # io/gravity.rs:335-363: the order kept is the largest seen;
    nn = (gc.degree + 1) ** 2                                          # the coefficients beyond the requested order stay zero
    assert np.ctypeslib.as_array(gc.c_nm, (nn,)).reshape(13, 13)[12, 11] == 0.0 and np.ctypeslib.as_array(gc.c_nm, (nn,)).reshape(13, 13)[12, 10] != 0.0
    assert np.array_equal(np.ctypeslib.as_array(gc.c_nm, (nn,)), np.ctypeslib.as_array(rc.c_nm, (nn,)))
    assert np.array_equal(np.ctypeslib.as_array(gc.s_nm, (nn,)), np.ctypeslib.as_array(rc.s_nm, (nn,)))
    assert packed.c.point_mass_mask == ref.c.point_mass_mask != 0
    dc, dr_ = packed.c.drag.contents, ref.c.drag.contents
    assert (dc.density, dc.rho0, dc.r0, dc.ref_alt_m) == (dr_.density, dr_.rho0, dr_.r0, dr_.ref_alt_m)
    # a sequence's `propagators` map: list of { _1 = name, _2 = config }
    named = nb.PropagatorConfig.load_named({"propagators": [{"_1": "Near Earth", "_2": {"method": "RungeKutta4", "options": {"fixed_step": True, "init_step": "10 s"}}},
                                                            {"_1": "Deep space", "_2": {}}]})
    assert set(named) == {"Near Earth", "Deep space"} and named["Near Earth"].method == nb.IntegratorMethod.RungeKutta4
    assert named["Near Earth"].options.fixed_step and named["Deep space"].options.init_step == 60 * 10**9


def test_reference_dhall_files_parse():
    """The reference's own configuration files (data/02_config, stored unchanged under tests/golden/dhall) go through the reader
    and the config mirror."""
    from nyx_b200 import dhall
    ref = Path(__file__).parent / "golden" / "dhall"
    cfg = nb.PropagatorConfig.load(ref / "prop_config.dhall")
    assert cfg.method == nb.IntegratorMethod.RungeKutta89 and cfg.options.max_step == 45 * 60 * 10**9 and cfg.options.min_step == 10**6
    assert cfg.options.error_ctrl == nb.ErrorControl.RSSCartesianStep and cfg.options.tolerance == 1e-12 and cfg.options.attempts == 50
    am = cfg.dynamics["accel_models"]
    assert am["point_masses"]["celestial_objects"] == [399, 301] and am["gravity_field"]["_1"]["degree"] == 21
    assert cfg.dynamics["force_models"]["drag"]["density"] == {"StdAtm": {"max_alt_m": 1000000.0}}
    named = nb.PropagatorConfig.load_named(ref / "full_seq.dhall")
    assert len(named) >= 1 and all(isinstance(c, nb.PropagatorConfig) for c in named.values())
    assert len(dhall.load(ref / "ci_almanac.dhall")["files"]) == 3
