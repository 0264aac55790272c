"""Host maths of the fewer-step samplers (models/diffusion_models/samplers.py): timestep selection, the folded DDIM and
DPM-Solver++(2M) tables against the DDPM posterior and the paper-form chains of sampler_oracle.py, convergence to the exact
probability-flow endpoint on an analytic Gaussian denoiser, argument validation and the sample.py flags."""
import numpy as np
import pytest
import torch

import wsr
from oracle import schedule
from oracle.cases import LINEAR_1000, short_schedule
from sampler_oracle import alphas_cumprod, ddim_chain, dpmpp2m_chain

sm = wsr.sub("models.diffusion_models.samplers")
ABAR = alphas_cumprod(LINEAR_1000)


def test_timesteps():
    for T, S in ((1000, 1), (1000, 2), (1000, 20), (1000, 999), (1000, 1000), (8, 4), (8, 8), (3, 2)):
        ts = sm.timesteps(T, S)
        assert len(ts) == S and len(set(ts.tolist())) == S
        assert np.all(np.diff(ts) < 0)
        assert ts[0] == T - 1
        if S > 1:
            assert ts[-1] == 0
    assert sm.timesteps(1000, 1000).tolist() == list(range(999, -1, -1))
    assert sm.timesteps(1000, 5).tolist() == [999, 749, 500, 250, 0]
    for S in (0, 1001):
        with pytest.raises(ValueError):
            sm.timesteps(1000, S)


def test_ddim_eta1_all_steps_is_the_ddpm_posterior():
    tab, levels = sm.ddim_tables(ABAR, 1000, eta=1.0)
    b = schedule.betas_for("linear", 1000, 1e-6, 1e-2)
    ap = np.append(1.0, ABAR[:-1])
    coef1 = b * np.sqrt(ap) / (1.0 - ABAR)
    coef2 = (1.0 - ap) * np.sqrt(1.0 - b) / (1.0 - ABAR)
    var = b * (1.0 - ap) / (1.0 - ABAR)
    np.testing.assert_allclose(tab[0], np.sqrt(1.0 / ABAR), rtol=1e-12)
    np.testing.assert_allclose(tab[1], np.sqrt(1.0 / ABAR - 1.0), rtol=1e-12)
    np.testing.assert_allclose(tab[2], coef1, rtol=1e-9)
    np.testing.assert_allclose(tab[3][1:], coef2[1:], rtol=1e-9)
    np.testing.assert_allclose(np.exp(tab[4][1:]), var[1:], rtol=1e-9)
    _, sap = schedule.ddpm_tables(LINEAR_1000)
    np.testing.assert_allclose(levels, sap[1:], rtol=1e-12)        # the level DDPM feeds at each timestep


@pytest.mark.parametrize("S", [1, 2, 3, 20, 1000])
def test_final_and_first_rows(S):
    for eta in (0.0, 0.5, 1.0):
        tab, _ = sm.ddim_tables(ABAR, S, eta)
        assert (tab[2, 0], tab[3, 0]) == (1.0, 0.0) and tab[4, 0] == -np.inf          # x' = x0, no noise
        if eta == 0.0:
            assert np.all(tab[4] == -np.inf)
    tab, levels = sm.dpmpp2m_tables(ABAR, S)
    assert (tab[2, 0], tab[3, 0], tab[4, 0]) == (1.0, 0.0, 0.0)
    assert tab[4, S - 1] == 0.0                                   # first step: first order
    if S > 1:
        assert tab[4, 1] == 0.0                                   # step into tau = 0: first order (lower order final)
    if S > 3:
        assert np.all(tab[4, 2:S - 1] != 0.0)
    np.testing.assert_allclose(levels, np.sqrt(ABAR[sm.timesteps(1000, S)[::-1]]), rtol=1e-15)


def _gaussian(mu=0.0, s=0.5):
    """eps_hat of data N(mu, s^2): E[eps | x_t] at level sqrt(abar)."""
    def den(x, level):
        a = level.double().view(-1, *([1] * (x.dim() - 1))) ** 2
        return torch.sqrt(1 - a) * (x.double() - torch.sqrt(a) * mu) / (a * s * s + 1 - a)
    return den


def _run_tables(name, S, den, xT, eta=0.0, noise=None):
    """The device step of wsr_sampler_step / wsr_sampler_step_multistep in float64 on the folded tables (no clamp)."""
    tab, levels = sm.tables(name, ABAR, S, eta)
    x = xT.double().clone()
    hist = torch.full_like(x, float("nan"))
    for c in range(S - 1, -1, -1):
        eps = den(x, torch.full((x.shape[0], 1), float(levels[c]), dtype=torch.float64))
        x0 = tab[0, c] * x - tab[1, c] * eps
        out = tab[2, c] * x0 + tab[3, c] * x
        if name == "ddim" and c > 0 and np.isfinite(tab[4, c]):
            out = out + np.exp(0.5 * tab[4, c]) * noise[S - c].double()
        if name == "dpmpp2m":
            if tab[4, c] != 0.0:
                out = out + tab[4, c] * hist
            hist = x0
        x = out
    return x


def test_tables_match_the_paper_form_chains():
    den = _gaussian(0.2, 0.5)
    g = torch.Generator().manual_seed(3)
    for S in (1, 2, 3, 7, 25):
        noise = torch.randn((S + 1, 4, 1, 8), generator=g, dtype=torch.float64)
        ref = dpmpp2m_chain(den, ABAR, S, noise, clip=False)
        assert (_run_tables("dpmpp2m", S, den, noise[0]) - ref).abs().max() < 1e-6, S
        for eta in (0.0, 0.5, 1.0):
            ref = ddim_chain(den, ABAR, S, noise, eta=eta, clip=False)
            assert (_run_tables("ddim", S, den, noise[0], eta, noise) - ref).abs().max() < 1e-6, (S, eta)


def test_gaussian_convergence_to_the_probability_flow_endpoint():
    """Data N(mu, s^2): the probability-flow ODE maps x_T to the same quantile of every marginal, so the exact output (x0_hat at
    tau = 0) is mu + sqrt(abar_0) s^2 z / sd_0 with z = (x_T - sqrt(abar_T) mu) / sd_T.  Both samplers converge to it as S grows, and
    DPM-Solver++(2M) at 40 steps is more accurate than DDIM at 80."""
    mu, s = 0.0, 0.5
    den = _gaussian(mu, s)
    xT = torch.randn((1, 20000), generator=torch.Generator().manual_seed(0), dtype=torch.float64)
    sd = lambda a: np.sqrt(a * s * s + 1 - a)                      # noqa: E731
    z = (xT - np.sqrt(ABAR[-1]) * mu) / sd(ABAR[-1])
    exact = mu + np.sqrt(ABAR[0]) * s * s * z / sd(ABAR[0])
    err = {}
    for name in ("ddim", "dpmpp2m"):
        for S in (10, 20, 40, 80, 160, 1000):
            err[name, S] = float((_run_tables(name, S, den, xT) - exact).norm() / exact.norm())
    print("\n[samplers] rel-L2 to the exact endpoint: " + " ".join("%s-%d %.2e" % (n, S, e) for (n, S), e in err.items()))
    for name in ("ddim", "dpmpp2m"):
        seq = [err[name, S] for S in (10, 20, 40, 80, 160, 1000)]
        assert all(b < a for a, b in zip(seq, seq[1:])), (name, seq)
    assert err["ddim", 1000] < 5e-3 and err["dpmpp2m", 1000] < 1e-3
    assert err["dpmpp2m", 40] < err["ddim", 80]                   # measured here: 6.3e-3 against 2.5e-2


def test_argument_validation():
    T = 8
    assert sm.check("ddpm", None, None, T) == ("ddpm", 8, 0.0)
    assert sm.check("ddim", 4, 0.5, T) == ("ddim", 4, 0.5)
    assert sm.check("dpmpp2m", None, None, T) == ("dpmpp2m", 8, 0.0)
    assert sm.check("ddpm", 8, None, T) == ("ddpm", 8, 0.0)
    for args in (("euler", None, None), ("ddim", 0, None), ("ddim", 9, None), ("ddim", 4, -0.1), ("ddim", 4, float("nan")),
                 ("dpmpp2m", 4, 0.0), ("ddpm", 4, None), ("ddpm", None, 1.0)):
        with pytest.raises(ValueError):
            sm.check(*args, T)


def test_set_sampler_on_the_diffusion():
    """set_sampler validates against the schedule and keeps p_sample's DDPM tables and the 12 schedule buffers unchanged."""
    D = wsr.sub("models.diffusion_models.diffusion").GaussianDiffusion
    diff = D(torch.nn.Identity())
    with pytest.raises(ValueError):
        diff.set_sampler("ddim", 4)                               # no schedule yet
    diff.set_new_noise_schedule(short_schedule(8), "cpu")
    names = [n for n, _ in diff.named_buffers()]
    assert len(names) == 12
    with pytest.raises(ValueError):
        diff.set_sampler("ddim", 9)
    with pytest.raises(ValueError):
        diff.set_sampler("dpmpp2m", 4, eta=0.0)
    diff.set_sampler("ddim", 4, eta=0.5)
    tab, levels = diff._tables_dev()
    assert tuple(tab.shape) == (5, 4) and tab.dtype == torch.float32 and tuple(levels.shape) == (4,)
    ref, _ = sm.ddim_tables(alphas_cumprod(short_schedule(8)), 4, 0.5)
    np.testing.assert_allclose(tab.numpy(), ref.astype(np.float32), rtol=0)
    assert tuple(diff._ddpm_tables_dev()[0].shape) == (5, 8)
    diff.set_sampler("dpmpp2m")
    assert tuple(diff._tables_dev()[0].shape) == (5, 8)
    diff.set_new_noise_schedule(short_schedule(6), "cpu")         # tables follow a new schedule
    assert tuple(diff._tables_dev()[0].shape) == (5, 6)
    assert [n for n, _ in diff.named_buffers()] == names
    diff.set_sampler()
    assert diff._tables_dev()[0] is diff._ddpm_tables_dev()[0]


def test_sample_py_flags():
    sample = wsr.sub("sample")
    base = ["-c", "cfg.json", "-o", "out"]
    a = sample.parse_args(base)
    assert sample.sampler_options(a) is None                     # the default DDPM loop is left untouched
    a = sample.parse_args(base + ["--sampler", "ddim", "--steps", "50", "--eta", "0.5"])
    assert sample.sampler_options(a) == dict(name="ddim", steps=50, eta=0.5)
    a = sample.parse_args(base + ["--sampler", "dpmpp2m", "--steps", "20", "--ensemble", "16", "--seed", "3"])
    assert sample.sampler_options(a) == dict(name="dpmpp2m", steps=20, eta=None) and a.ensemble == 16
    assert sample.sampler_options(sample.parse_args(base + ["--steps", "20"])) == dict(name="ddpm", steps=20, eta=None)
    with pytest.raises(SystemExit):
        sample.parse_args(base + ["--sampler", "euler"])
