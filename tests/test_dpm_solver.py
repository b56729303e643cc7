"""DPM-Solver++(2M) host side, CPU only: evaluation indices, the fp32 coefficient table against the oracle, the tie of
the first-order update to the reference's DDIM step, convergence on Gaussian data with its exact denoiser, and the
--sampler flag."""
import numpy as np
import pytest

import dpm_solver_oracle as DO
import musediff_oracle as O
from musediffusion_b200.diffusion import (GaussianDiffusion, SpacedDiffusion, dpm_solver_coefficients, dpm_solver_indices,
                                          get_named_beta_schedule, space_timesteps)

SCHEDULES = {"sqrt-2000": ("sqrt", 2000, ""), "cosine-500": ("cosine", 500, ""), "sqrt-2000-ddim50": ("sqrt", 2000, "ddim50")}


def _diffusion(name):
    sched, T, resp = SCHEDULES[name]
    return SpacedDiffusion(use_timesteps=space_timesteps(T, resp or [T]), betas=get_named_beta_schedule(sched, T),
                           rescale_timesteps=True, predict_xstart=True)


def _oracle_schedule(name):
    sched, T, resp = SCHEDULES[name]
    return O.make_schedule(sched, T, resp)


@pytest.mark.parametrize("name", list(SCHEDULES))
def test_indices_distinct_descending_from_t_start_to_zero(name):
    """exactly N distinct descending indices, the first t_start and the last 0, for every N in 1..t_start + 1 (N = 1 is the
    single evaluation at t_start), from the last index and from one inside the table; equal to the oracle's."""
    d, s = _diffusion(name), _oracle_schedule(name)
    T = d.num_timesteps
    for t_start in (T - 1, (2 * T) // 3):
        for N in range(1, t_start + 2):
            idx = dpm_solver_indices(d.alphas_cumprod, t_start, N)
            assert len(idx) == N and idx[0] == t_start, (t_start, N)
            assert all(a > b for a, b in zip(idx, idx[1:])), (t_start, N)
            if N > 1:
                assert idx[-1] == 0, (t_start, N)
            if N in (1, 2, 10, 20, 50, t_start + 1):
                assert idx == DO.dpm_solver_indices(s, t_start, N), (t_start, N)
        assert dpm_solver_indices(d.alphas_cumprod, t_start, t_start + 1) == list(range(t_start, -1, -1))


def test_indices_are_uniform_in_log_snr():
    """away from the rounding and distinctness clips the indices sit where lambda is evenly spaced: at N = 20 on the
    2000-step sqrt table every free index is the nearest integer to its lambda target."""
    d = _diffusion("sqrt-2000")
    ab = d.alphas_cumprod
    lam = 0.5 * np.log(ab) - 0.5 * np.log1p(-ab)
    N = 20
    idx = dpm_solver_indices(ab, 1999, N)
    targets = np.linspace(lam[1999], lam[0], N)
    for k in range(1, N - 1):
        g = np.interp(targets[k], lam[::-1], np.arange(2000)[::-1].astype(np.float64))
        if N - 1 - k < round(g) < idx[k - 1] - 1:
            assert idx[k] == round(g), (k, g)
            assert lam[idx[k] + 1] <= targets[k] <= lam[idx[k] - 1]


def test_bad_arguments_raise():
    d = _diffusion("cosine-500")
    ab = d.alphas_cumprod
    for t_start, N in ((499, 0), (499, 501), (10, 12), (-1, 1), (500, 3)):
        with pytest.raises(ValueError):
            dpm_solver_indices(ab, t_start, N)
    for order in (0, 3, 1.5):
        with pytest.raises(ValueError):
            dpm_solver_coefficients(ab, [499, 200, 0], order)
    with pytest.raises(ValueError):
        d.dpm_solver_sample_loop(None, (1, 4, 8), steps=0)
    with pytest.raises(ValueError):
        d.dpm_solver_sample_loop(None, (1, 4, 8), steps=5, order=3)


@pytest.mark.parametrize("name", list(SCHEDULES))
@pytest.mark.parametrize("order", [1, 2])
def test_fp32_coefficient_table_equals_oracle(name, order):
    """the table the kernel receives (float64 rows cast to fp32 once) equals the oracle's bit for bit; the last row is
    (0, 1, 1, 0), the first row and every order-1 row are first order (c0 = 1, c1 = 0)."""
    d, s = _diffusion(name), _oracle_schedule(name)
    T = d.num_timesteps
    for t_start in (T - 1, T // 2):
        for N in sorted({n for n in (1, 2, 3, 10, 20, 50) if n <= t_start + 1} | {t_start + 1}):
            idx = dpm_solver_indices(d.alphas_cumprod, t_start, N)
            got = dpm_solver_coefficients(d.alphas_cumprod, idx, order).astype(np.float32)
            want = DO.dpm_solver_coefficients(s, idx, order).astype(np.float32)
            assert got.shape == (N, 4)
            assert np.array_equal(got.view(np.int32), want.view(np.int32)), (t_start, N)
            assert tuple(got[-1]) == (0.0, 1.0, 1.0, 0.0)
            first_order = got[:-1] if order == 1 else got[:1]
            if N > 1:
                assert (first_order[:, 2] == 1.0).all() and (first_order[:, 3] == 0.0).all()
            if order == 2 and N > 2:
                assert (got[1:-1, 3] != 0.0).all() and np.allclose(got[1:-1, 2] + got[1:-1, 3], 1.0)


@pytest.mark.parametrize("name", list(SCHEDULES))
def test_order1_every_index_is_the_ddim_eta0_step(name):
    """order 1 with N = t_start + 1 (every index) is the reference's DDIM eta = 0 step at gap 1, written in float64 from the
    same Schedule tables: x' = sqrt(abar_prev) x0 + sqrt(1 - abar_prev) (sqrt_recip x - x0) / sqrt_recipm1 =
    sigma'/sigma x + (alpha' - sigma' alpha / sigma) x0 at every index, and at t = 0 (abar_prev = 1) x' = x0 (the last row)."""
    s = _oracle_schedule(name)
    T = s.num_timesteps
    idx = dpm_solver_indices(s.alphas_cumprod, T - 1, T)
    coef = dpm_solver_coefficients(s.alphas_cumprod, idx, 1)
    abp = s.alphas_cumprod_prev[idx]
    sr, srm1 = s.sqrt_recip_alphas_cumprod[idx], s.sqrt_recipm1_alphas_cumprod[idx]
    # x' = sqrt(abp) x0 + sqrt(1 - abp) (sr x - x0) / srm1  ->  coefficient of x and of x0
    a_ddim = np.sqrt(1.0 - abp) * sr / srm1
    b_ddim = np.sqrt(abp) - np.sqrt(1.0 - abp) / srm1
    assert np.abs(coef[:, 0] - a_ddim).max() <= 1e-12
    assert np.abs(coef[:, 1] - b_ddim).max() <= 1e-12
    assert (coef[:, 2] == 1.0).all() and (coef[:, 3] == 0.0).all()


def _gaussian_chain(ab, N, order, t_start=1999, mu=0.3, sd=0.7):
    """float64 run of the sampler on data N(mu, sd^2) with its exact denoiser E[x0 | x_t], from a grid of states at t_start;
    max error at index 0 against the probability-flow ODE, which keeps (x - alpha mu) / sqrt(alpha^2 sd^2 + sigma^2)."""
    def x0_hat(x, i):
        a, s = np.sqrt(ab[i]), np.sqrt(1.0 - ab[i])
        return mu + a * sd * sd / (a * a * sd * sd + s * s) * (x - a * mu)

    idx = dpm_solver_indices(ab, t_start, N)
    coef = dpm_solver_coefficients(ab, idx, order)
    z = np.linspace(-3.0, 3.0, 61)
    a0 = np.sqrt(ab[t_start])
    x = a0 * mu + np.sqrt(ab[t_start] * sd * sd + 1.0 - ab[t_start]) * z
    prev = None
    for k, i in enumerate(idx[:-1]):             # the state at idx[-1] = 0, before the last row returns its x0
        p = x0_hat(x, i)
        a, b, c0, c1 = coef[k]
        x = a * x + b * (c0 * p + (c1 * prev if c1 != 0 else 0.0))
        prev = p
    exact = np.sqrt(ab[0]) * mu + np.sqrt(ab[0] * sd * sd + 1.0 - ab[0]) * z
    return float(np.abs(x - exact).max())


def test_second_order_converges_on_gaussian_data():
    """sqrt schedule, T = 2000, from index 1999: the 2M error is below a fifth of the first-order error at N = 10, 20, 40,
    and both decrease with N."""
    ab = _diffusion("sqrt-2000").alphas_cumprod
    e1 = [_gaussian_chain(ab, N, 1) for N in (10, 20, 40)]
    e2 = [_gaussian_chain(ab, N, 2) for N in (10, 20, 40)]
    print("order 1:", e1, "2M:", e2)
    assert all(b < a / 5 for a, b in zip(e1, e2)), (e1, e2)
    assert e1[0] > e1[1] > e1[2] and e2[0] > e2[1] > e2[2], (e1, e2)


def test_cli_sampler_flag():
    from musediffusion_b200.sample import SAMPLERS, create_parser
    p = create_parser()
    for mode in ("generation", "modification"):
        assert p.parse_args([mode, "--model_path", "m.pt"]).sampler == "reference"
        assert p.parse_args([mode, "--model_path", "m.pt", "--sampler", "dpm_solver++", "--step", "20"]).sampler == "dpm_solver++"
        with pytest.raises(SystemExit):
            p.parse_args([mode, "--model_path", "m.pt", "--sampler", "ddim"])
    assert SAMPLERS == ("reference", "dpm_solver++")


def test_sample_batch_rejects_unknown_sampler():
    from musediffusion_b200.sample import sample_batch
    with pytest.raises(ValueError):
        sample_batch(None, GaussianDiffusion(betas=get_named_beta_schedule("sqrt", 10), predict_xstart=True), None, {},
                     "generation", 5, 10, sampler="dpm")
