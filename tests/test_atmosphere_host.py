"""fit_atmosphere (the host side of the altitude-dependent atmosphere) and the option checks that reject an atmosphere
before any device work -- no GPU, no library."""
import numpy as np
import pytest

import mpconstellation_b200 as M
from mpconstellation_b200 import _lib, batch


def power_law(h):
    return 8e26 * h ** -6.828          # simulator.py:110


def test_power_law_is_fitted_to_round_off():
    a = M.fit_atmosphere(power_law, 300e3, 1000e3)
    assert a.max_rel_err <= 1e-12
    h = np.linspace(300e3, 1000e3, 777)
    assert np.max(np.abs(a.density(h) / power_law(h) - 1)) <= 1e-12
    assert len(a.coef) <= 32


def test_exponential_atmosphere_from_200_to_20000_km():
    rho0, h0, H = 3.7e-12, 400e3, 58e3
    a = M.fit_atmosphere(lambda h: rho0 * np.exp(-(h - h0) / H), 200e3, 20000e3)
    assert a.max_rel_err <= 1e-9 and len(a.coef) <= 32
    assert abs(a.density(h0) / rho0 - 1) <= 1e-9


def test_kinked_model_is_rejected():
    def kinked(h):
        return max(1e-12 * np.exp(-(h - 500e3) / 60e3), 1e-14 * np.exp(-(h - 500e3) / 300e3))
    with pytest.raises(NotImplementedError, match="no CPU fallback"):
        M.fit_atmosphere(kinked, 200e3, 2000e3)


@pytest.mark.parametrize("rho", [lambda h: 0.0, lambda h: -1e-12, lambda h: np.nan, lambda h: np.inf,
                                 lambda h: 1e-12 if h < 900e3 else 0.0])
def test_non_positive_or_non_finite_density_is_rejected(rho):
    with pytest.raises(ValueError):
        M.fit_atmosphere(rho, 300e3, 1000e3)


@pytest.mark.parametrize("lo, hi", [(0.0, 1e6), (-1e5, 1e6), (1e6, 1e6), (1e6, 5e5), (np.nan, 1e6), (3e5, np.inf)])
def test_bad_ranges_are_rejected(lo, hi):
    with pytest.raises(ValueError):
        M.fit_atmosphere(power_law, lo, hi)


def test_atmosphere_is_immutable():
    a = M.fit_atmosphere(power_law, 300e3, 1000e3)
    with pytest.raises(AttributeError):
        a.h_min = 1.0
    with pytest.raises(ValueError):
        a.coef[0] = 0.0
    s = a.struct()
    assert (s.h_min, s.h_max, s.n) == (300e3, 1000e3, len(a.coef)) and s.r_earth == M.model.R_EARTH


@pytest.fixture
def no_device(monkeypatch):
    """any use of the library or of a device context fails the test"""
    def boom(*a, **k):
        raise AssertionError("the library was loaded")
    monkeypatch.setattr(_lib, "lib", boom)
    monkeypatch.setattr(batch, "_ctx", boom)
    monkeypatch.setattr(batch, "_torch", boom)


def _inputs():
    scale = M.SatelliteScale()
    return np.tile(scale.normalize_state(np.array([6.771e6, 0, 0, 0, 7.67e3, 0, 1000.0])), (2, 1)), \
        scale.get_normalized_constants()


def test_rejected_combinations_raise_before_the_library_is_loaded(no_device):
    a = M.fit_atmosphere(power_law, 300e3, 1000e3)
    y0, const = _inputs()
    ctrl = M.Controller()
    with pytest.raises(ValueError, match="include_drag"):
        M.propagate_batch(y0, 0.1, ctrl, const, include_drag=False, atmosphere=a)
    with pytest.raises(ValueError, match="reference integrator"):
        M.propagate_batch(y0, 0.1, ctrl, const, n_sub=4, atmosphere=a)
    with pytest.raises(ValueError, match="Atmosphere"):
        M.propagate_batch(y0, 0.1, ctrl, const, atmosphere=lambda h: 1e-12)
    with pytest.raises(ValueError, match="include_drag"):
        M.propagate_batch_device(y0, 0.1, ctrl, const, include_drag=False, atmosphere=a)
    with pytest.raises(ValueError, match="reference integrator"):
        M.propagate_batch_device(y0, 0.1, ctrl, const, n_sub=4, atmosphere=a)
    with pytest.raises(ValueError, match="constant density"):
        M.propagate_discretize(y0, 0.1, ctrl, const, T=5, atmosphere=a)
    with pytest.raises(ValueError, match="constant density"):
        M.propagate_discretize_device(y0, 0.1, ctrl, const, T=5, atmosphere=a)
    sim = M.Simulator(sats=[M.Satellite(np.array([6.771e6, 0, 0]), np.array([0, 7.67e3, 0]), 1000.0)])
    sim.atmosphere = a
    sim.integrator = "rk4"
    with pytest.raises(ValueError, match="reference integrator"):
        sim.run(tf=0.1)
    from mpconstellation_b200.scp import BatchedSCP
    scp = BatchedSCP.__new__(BatchedSCP)
    scp.const = const
    with pytest.raises(ValueError, match="include_drag"):
        scp.run_segments(y0, 1, include_drag=False, atmosphere=a)


def test_atmosphere_status_names_the_satellite_and_the_range():
    a = M.fit_atmosphere(power_law, 300e3, 1000e3)
    with pytest.raises(ValueError, match=r"satellite 2: .*\[300000, 1e\+06\] m"):
        batch.raise_on_status(np.array([0, 0, _lib.ST_ATMO], np.int32), a)
