"""DDIM sampler, host side: the default timestep sequences, argument validation, and the fp64 oracle pinned by two identities
(the reference has no DDIM, so there is no golden file): eta = 1 over consecutive steps is the reference's posterior step, and
eta = 0 maps an exactly-noised field to the same field noised at t'.  The library's coefficient function is checked against the
oracle through its Python mirror."""
import numpy as np
import pytest
import torch

from diffusionmodelscustom_b200 import DiffusionUtils, DiffusionUtilsV2
from diffusionmodelscustom_b200.diffusion import ddim_coefficients
from oracle import ddpm_oracle as O
from tests import ddim_oracle as DO

SCHEDULES = [("linear", 1), ("cosine", 1), ("cosine", 2)]


def _tables(T, scheduler, version):
    """fp64 tables from the schedule's betas: alpha_hat_t = alpha_hat_{t-1} alpha_t holds to fp64 rounding, which the identities
    need (the fp32 cumprod of the reference breaks it at the 1e-7 level)."""
    betas = O.beta_schedule(T, 1e-4, 0.02, scheduler, version).double()
    alphas = 1 - betas
    return betas, alphas, torch.cumprod(alphas, dim=0)


@pytest.mark.parametrize("T", [12, 1000])
@pytest.mark.parametrize("S", [1, 2, 7, 50, "T-1"])
def test_default_sequence_is_strictly_decreasing_from_T_minus_1_to_1(T, S):
    S = T - 1 if S == "T-1" else S
    if S > T - 1:
        pytest.skip("more steps than the schedule has")
    ts = DiffusionUtils(T, 1e-4, 0.02).ddim_timesteps(S)
    assert len(ts) == S and all(isinstance(t, int) for t in ts)
    assert ts[0] == T - 1
    if S >= 2:
        assert ts[-1] == 1
    assert all(b < a for a, b in zip(ts, ts[1:]))
    assert all(1 <= t <= T - 1 for t in ts)
    if S == T - 1:
        assert ts == list(range(T - 1, 0, -1))


def test_invalid_sequences_and_eta_raise_value_error():
    du = DiffusionUtils(12, 1e-4, 0.02)
    for S in (0, -3, 12, 13):
        with pytest.raises(ValueError):
            du.ddim_timesteps(S)
    for ts in ([5, 5, 1], [3, 7, 1], [11, 12], [11, 0], [], [12]):
        with pytest.raises(ValueError):
            du._ddim_plan(None, 0.0, ts)
    for eta in (-0.1, 1.5, float("nan")):
        with pytest.raises(ValueError):
            du._ddim_plan(5, eta, None)
    assert du._ddim_plan(3, 0.5, torch.tensor([9, 4, 2])) == ([9, 4, 2], 0.5)
    assert du._ddim_plan(3, 1, None) == (du.ddim_timesteps(3), 1.0)
    # the sampler entry validates before touching the model or the device
    with pytest.raises(ValueError):
        du.sample_ddim(torch.zeros(1, 1, 8, 8), None, steps=20)
    assert DiffusionUtilsV2(1000).ddim_timesteps(50) == DiffusionUtils(1000, 1e-4, 0.02).ddim_timesteps(50)


@pytest.mark.parametrize("scheduler,version", SCHEDULES)
def test_oracle_eta1_consecutive_steps_is_the_reference_posterior(scheduler, version):
    T = 1000
    betas, alphas, ahat = _tables(T, scheduler, version)
    g = torch.Generator().manual_seed(1)
    x = torch.randn(2, 1, 8, 8, generator=g, dtype=torch.float64) * 3
    eps = torch.randn(2, 1, 8, 8, generator=g, dtype=torch.float64)
    z = torch.randn(2, 1, 8, 8, generator=g, dtype=torch.float64)
    for t in (2, 3, 10, 250, 500, 998, 999):
        mean = DO.ddim_step(x, eps, None, t, t - 1, 1.0, ahat)
        ref_mean = O.posterior_update(x, eps, torch.zeros_like(x), t, betas, alphas, ahat)
        assert float((mean - ref_mean).norm() / ref_mean.norm()) <= 1e-10, (t, scheduler, version)
        _, _, sigma = DO.ddim_coefficients(t, t - 1, 1.0, ahat)
        beta_tilde = float((1 - ahat[t - 1]) / (1 - ahat[t]) * betas[t])
        assert abs(sigma ** 2 - beta_tilde) <= 1e-10 * beta_tilde, (t, scheduler, version)
        # and the noise enters with exactly that sigma
        full = DO.ddim_step(x, eps, z, t, t - 1, 1.0, ahat)
        assert float((full - mean - sigma * z).norm()) <= 1e-10 * float(full.norm())


@pytest.mark.parametrize("scheduler,version", SCHEDULES)
def test_oracle_eta0_maps_exact_noise_to_the_same_noise_at_t_prev(scheduler, version):
    _, _, ahat = _tables(1000, scheduler, version)
    g = torch.Generator().manual_seed(2)
    x0 = torch.randn(3, 1, 8, 8, generator=g, dtype=torch.float64)
    e = torch.randn(3, 1, 8, 8, generator=g, dtype=torch.float64)
    for t, tp in ((999, 899), (999, 1), (500, 499), (37, 5), (2, 1), (999, -1), (17, -1)):
        xt = torch.sqrt(ahat[t]) * x0 + torch.sqrt(1 - ahat[t]) * e
        out = DO.ddim_step(xt, e, torch.randn(xt.shape, generator=g, dtype=torch.float64), t, tp, 0.0, ahat)
        want = x0 if tp < 0 else torch.sqrt(ahat[tp]) * x0 + torch.sqrt(1 - ahat[tp]) * e
        assert float((out - want).norm() / want.norm()) <= 1e-10, (t, tp)
    # the whole sampler with the exact-noise model lands on x0
    ts = DiffusionUtils(1000, 1e-4, 0.02).ddim_timesteps(10)
    xT = torch.sqrt(ahat[ts[0]]) * x0 + torch.sqrt(1 - ahat[ts[0]]) * e
    out = DO.ddim_sample(lambda x, t: e, xT, ts, 0.0, ahat)
    assert float((out - x0).norm() / x0.norm()) <= 1e-10


@pytest.mark.parametrize("scheduler,version", SCHEDULES)
def test_library_coefficients_match_the_oracle_to_fp32_rounding(scheduler, version):
    T = 1000
    _, _, ahat32 = O.schedule_tables(T, 1e-4, 0.02, scheduler, version)
    ahat = ahat32.double()        # the library computes from the fp32 table: the oracle gets the same values
    steps = [(999, 998), (999, 899), (500, 499), (500, 1), (2, 1), (999, -1), (1, -1), (40, 20)]
    for eta in (0.0, 0.3, 1.0):
        for t, tp in steps:
            ours = ddim_coefficients(ahat32, t, tp, eta)
            ref = DO.ddim_coefficients(t, tp, eta, ahat)
            for name, a, b in zip(("cx", "ce", "sigma"), ours, ref):
                assert a == np.float32(b) or abs(a - b) <= 2 ** -23 * abs(b), (name, t, tp, eta, a, b)
            if eta == 0.0 or tp < 0:
                assert ours[2] == 0.0
