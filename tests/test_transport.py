"""Sampler surface (SURVEY.md section 8f-2): zigma_b200.transport against golden vectors produced by the
UNMODIFIED reference transport/ package (oracle/gen_golden_transport.py), and the restated
torchdiffeq solvers against closed forms / scipy's RK45 (same Dormand-Prince tableau)."""
import math
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

import gen_golden_transport as gg          # noqa: E402  (test infrastructure: the shared toy problem)
from zigma_b200 import transport as tp     # noqa: E402
from zigma_b200.transport import odeint    # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden", "transport.npz")


def test_reference_golden_replay():
    """check_interval table, plan algebra, drift/score closures, training losses (all 9 path x
    prediction x weighting combos) and 24 seeded SDE runs: bit-exact on the finite entries, and
    non-finite exactly where the reference is (SBDM diffusion from t0 = 0)."""
    gold = np.load(GOLD)
    got = gg.run_all(tp)
    assert set(got) == set(gold.files)
    for k in gold.files:
        a, b = got[k], gold[k]
        assert a.shape == b.shape, k
        assert np.array_equal(np.isfinite(a), np.isfinite(b)), k
        assert np.allclose(a, b, rtol=1e-6, atol=1e-7, equal_nan=True), (k, np.nanmax(np.abs(a - b)))


def test_create_transport_eps_quirk_and_errors():
    tr = tp.create_transport("Linear", "noise")
    assert tr.train_eps == 1e-3 and tr.sample_eps is None      # transport/__init__.py:52-57 as written
    tr = tp.create_transport("Linear", "velocity", None, 0.5, 0.5)
    assert (tr.train_eps, tr.sample_eps) == (0, 0)
    with pytest.raises(ValueError):
        tp.create_transport(prediction="x0")
    with pytest.raises(ValueError):
        tp.create_transport(loss_weight="snr")
    with pytest.raises(KeyError):
        tp.create_transport(path_type="cosine")
    with pytest.raises(NotImplementedError):
        tp.path.ICPlan().compute_diffusion(torch.zeros(2, 3), torch.ones(2) * 0.5, form="nope")
    s = tp.Sampler(tp.create_transport())
    with pytest.raises(NotImplementedError):
        s.sample_sde(last_step="Magic")
    with pytest.raises(NotImplementedError):
        s.sample_sde(sampling_method="Milstein", num_steps=4)(torch.zeros(2, 3), lambda x, t: x)
    with pytest.raises(ValueError):
        s.sample_ode(sampling_method="rk45", num_steps=4)(torch.zeros(2, 3), lambda x, t: x)


def test_sde_constant_diffusion_runs():
    """The reference raises on the python-float 'constant' form (integrators.py:39); here it runs."""
    fn = tp.Sampler(tp.create_transport()).sample_sde(diffusion_form="constant", diffusion_norm=0.3, num_steps=10)
    torch.manual_seed(0)
    xs = fn(gg.toy_x(), gg.toy_model())
    assert len(xs) == 10 and all(torch.isfinite(v).all() for v in xs)


# ---- odeint ---------------------------------------------------------------------------------------------
def _lin(t, y):          # y' = -2 y + sin(3 t)
    return -2 * y + torch.sin(3 * t)


def _lin_exact(t, y0):
    # y = C e^{-2t} + (2 sin 3t - 3 cos 3t) / 13
    return (y0 + 3 / 13) * math.exp(-2 * t) + (2 * math.sin(3 * t) - 3 * math.cos(3 * t)) / 13


@pytest.mark.parametrize("method,order", [("euler", 1), ("midpoint", 2), ("heun2", 2), ("heun3", 3), ("rk4", 4)])
def test_fixed_grid_convergence_order(method, order):
    y0 = torch.tensor([1.0, -0.5], dtype=torch.float64)
    errs = []
    for n in (20, 40, 80):
        t = torch.linspace(0, 1.5, n + 1, dtype=torch.float64)
        y = odeint(_lin, y0, t, method=method)
        assert y.shape == (n + 1, 2)
        errs.append(max(abs(float(y[-1, i]) - _lin_exact(1.5, float(y0[i]))) for i in range(2)))
    for e0, e1 in zip(errs, errs[1:]):
        assert abs(math.log2(e0 / e1) - order) < 0.35, (method, errs)


def test_euler_is_the_plain_recurrence():
    W = torch.randn(4, 4)
    f = lambda t, y: torch.tanh(y @ W) * (1 + t)
    y0 = torch.randn(3, 4)
    t = torch.linspace(0, 1, 9)
    got = odeint(f, y0, t, method="euler")
    y = y0
    for i in range(8):
        y = y + (float(t[i + 1]) - float(t[i])) * f(t[i], y)
    assert torch.allclose(got[-1], y, rtol=1e-6, atol=1e-7)


@pytest.mark.parametrize("method,tol,rtol", [("dopri5", 2e-6, 1e-6), ("bosh3", 2e-4, 1e-6), ("adaptive_heun", 3e-3, 1e-5)])
def test_adaptive_solvers_dense_output(method, tol, rtol):
    y0 = torch.tensor([1.0, -0.5, 0.25], dtype=torch.float64)
    t = torch.linspace(0, 2.0, 17, dtype=torch.float64)
    calls = []
    f = lambda tt, y: (calls.append(float(tt)), _lin(tt, y))[1]
    y = odeint(f, y0, t, method=method, rtol=rtol, atol=rtol * 1e-2)
    exact = np.array([[_lin_exact(float(tt), float(v)) for v in y0] for tt in t])
    assert np.abs(y.numpy() - exact).max() < tol
    assert y[0].equal(y0)
    # tighter tolerance -> more work, smaller error
    n_loose = len(calls); calls.clear()
    y2 = odeint(f, y0, t, method=method, rtol=rtol * 1e-2, atol=rtol * 1e-4)
    assert len(calls) > n_loose and np.abs(y2.numpy() - exact).max() < np.abs(y.numpy() - exact).max()


def test_dopri5_against_scipy_rk45():
    scipy_integrate = pytest.importorskip("scipy.integrate")
    rs = np.random.RandomState(0)
    A = rs.randn(5, 5) * 0.7
    f_np = lambda t, y: np.tanh(A @ y) * (1 + t) - 0.3 * y
    At = torch.from_numpy(A)
    f_t = lambda t, y: torch.tanh(At @ y) * (1 + t) - 0.3 * y
    y0 = rs.randn(5)
    ts = np.linspace(0, 1, 11)
    ref = scipy_integrate.solve_ivp(f_np, (0, 1), y0, method="RK45", t_eval=ts, rtol=1e-10, atol=1e-12).y.T
    got = odeint(f_t, torch.from_numpy(y0), torch.from_numpy(ts), method="dopri5", rtol=1e-8, atol=1e-10).numpy()
    assert np.abs(got - ref).max() < 1e-7
    # and at the sampler's default tolerance the end point is within that tolerance's reach
    got = odeint(f_t, torch.from_numpy(y0), torch.from_numpy(ts), method="dopri5", rtol=1e-3, atol=1e-6).numpy()
    assert np.abs(got[-1] - ref[-1]).max() < 1e-2


def test_dopri5_single_step_matches_tableau_by_hand():
    """One accepted step of size h reproduces the 5th-order Dormand-Prince update written out longhand."""
    f = lambda t, y: torch.cos(y) + t
    y0 = torch.tensor([0.3], dtype=torch.float64)
    h = 0.05
    k1 = f(0.0, y0)
    k2 = f(h / 5, y0 + h * k1 / 5)
    k3 = f(3 * h / 10, y0 + h * (3 * k1 / 40 + 9 * k2 / 40))
    k4 = f(4 * h / 5, y0 + h * (44 * k1 / 45 - 56 * k2 / 15 + 32 * k3 / 9))
    k5 = f(8 * h / 9, y0 + h * (19372 * k1 / 6561 - 25360 * k2 / 2187 + 64448 * k3 / 6561 - 212 * k4 / 729))
    k6 = f(h, y0 + h * (9017 * k1 / 3168 - 355 * k2 / 33 + 46732 * k3 / 5247 + 49 * k4 / 176 - 5103 * k5 / 18656))
    y1 = y0 + h * (35 * k1 / 384 + 500 * k3 / 1113 + 125 * k4 / 192 - 2187 * k5 / 6784 + 11 * k6 / 84)
    got = odeint(f, y0, torch.tensor([0.0, h], dtype=torch.float64), method="dopri5", rtol=1e-3, atol=1e-6,
                 options={"first_step": h})
    assert torch.allclose(got[-1], y1, rtol=0, atol=1e-15)


def test_reverse_time_and_tuple_state():
    y0 = torch.tensor([0.7], dtype=torch.float64)
    fwd = odeint(_lin, y0, torch.tensor([0.0, 1.0], dtype=torch.float64), method="dopri5", rtol=1e-9, atol=1e-11)
    back = odeint(_lin, fwd[-1], torch.tensor([1.0, 0.5, 0.0], dtype=torch.float64), method="dopri5", rtol=1e-9, atol=1e-11)
    assert abs(float(back[-1]) - 0.7) < 1e-7
    assert abs(float(back[1]) - _lin_exact(0.5, 0.7)) < 1e-7
    # tuple state: (y, integral of y) with per-tensor tolerances in lists, like the reference passes them
    f = lambda t, s: (-s[0], s[0].sum(1))
    ya, yb = odeint(f, (torch.ones(2, 3), torch.zeros(2)), torch.linspace(0, 1, 5), method="dopri5", rtol=[1e-6], atol=[1e-8])
    assert ya.shape == (5, 2, 3) and yb.shape == (5, 2)
    assert torch.allclose(ya[-1], torch.full((2, 3), math.exp(-1)), atol=1e-5)
    assert torch.allclose(yb[-1], torch.full((2,), 3 * (1 - math.exp(-1))), atol=1e-5)
    for m in tp._odeint.FIXED_METHODS:
        ya, yb = odeint(f, (torch.ones(2, 3), torch.zeros(2)), torch.linspace(0, 1, 65), method=m)
        assert torch.allclose(ya[-1], torch.full((2, 3), math.exp(-1)), atol=2e-2)


# ---- Sampler over odeint ----------------------------------------------------------------------------------
def test_sample_ode_default_dopri5_and_fixed_methods_agree():
    model, x = gg.toy_model(), gg.toy_x()
    s = tp.Sampler(tp.create_transport())
    ref = s.sample_ode(sampling_method="dopri5", num_steps=20, atol=1e-9, rtol=1e-8)(x, model)
    assert ref.shape == (20, *x.shape)
    default = s.sample_ode()(x, model)                 # dopri5, 50 saved points (train_acc.py:531 uses this)
    assert default.shape == (50, *x.shape)
    assert torch.allclose(default[-1], ref[-1], atol=5e-3)
    for m, n, tol in (("euler", 400, 5e-3), ("heun2", 60, 1e-3), ("midpoint", 60, 1e-3), ("rk4", 20, 1e-4), ("heun3", 30, 1e-4)):
        out = s.sample_ode(sampling_method=m, num_steps=n)(x, model)
        assert out.shape[0] == n and torch.allclose(out[-1], ref[-1], atol=tol), m
    # reverse=True as the reference defines it (transport.py:391-396 + check_interval's swap): t runs 1 -> 0
    # and the model is queried at 1 - t, i.e. dx/ds = -v(x, s) for s = 0 -> 1
    z = s.sample_ode(sampling_method="dopri5", num_steps=5, atol=1e-9, rtol=1e-8, reverse=True)(x, model)[-1]
    want = odeint(lambda tt, y: -model(y, torch.ones(y.size(0)) * tt), x, torch.tensor([0.0, 1.0]), method="dopri5",
                  atol=1e-9, rtol=1e-8)[-1]
    assert torch.allclose(z, want, atol=1e-5)


def test_sample_ode_likelihood_on_gaussian_flow():
    """Velocity field of the linear path between N(0, I) and N(0, s^2 I): v(x, t) = x d/dt log std_t with
    std_t^2 = (1-t)^2 + t^2 s^2.  Its divergence is exact under the Rademacher estimator (the Jacobian
    is a multiple of I), so logp must equal the N(0, s^2 I) log density."""
    s_data, dim = 0.5, 4
    def model(x, t, **kw):
        tb = t.view(-1, 1)
        var = (1 - tb) ** 2 + (tb * s_data) ** 2
        return x * (-(1 - tb) + tb * s_data ** 2) / var
    x = torch.randn(6, dim, dtype=torch.float64) * s_data
    fn = tp.Sampler(tp.create_transport()).sample_ode_likelihood(sampling_method="dopri5", num_steps=4, atol=1e-9, rtol=1e-8)
    logp, z = fn(x, model)
    want = -0.5 * dim * math.log(2 * math.pi * s_data ** 2) - x.pow(2).sum(1) / (2 * s_data ** 2)
    assert torch.allclose(logp, want, atol=1e-5)
    assert torch.allclose(z, x / s_data, atol=1e-5)    # the flow is the linear rescaling
