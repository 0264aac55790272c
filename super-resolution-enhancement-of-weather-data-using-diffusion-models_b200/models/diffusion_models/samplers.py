"""Fewer-step samplers over a subset of the trained schedule: DDIM(eta) (Song et al. 2021) and DPM-Solver++(2M) (Lu et al. 2022,
data prediction), both with the reference's x0 clamp.  Host maths in float64; the device runs them from [5][S] fp32 tables.

Timesteps: tau_0 = T-1 > ... > tau_{S-1} = 0, ``round(linspace(T-1, 0, S))``.  Tables and the level vector are stored with row r = the
step whose network timestep is tau_{S-1-r}, so the device step counter runs S-1 -> 0 exactly as the DDPM loop's does (for S = T, row r is
timestep r).  Level row r = sqrt(alphas_cumprod[tau]), the value DDPM feeds at that timestep.

  ddim     (c_recip, c_recipm1, coef1, coef2, logvar): x0 = clamp(c_recip x - c_recipm1 eps), x' = coef1 x0 + coef2 x + exp(logvar / 2) z.
           Linear in (x0, x), so it is the DDPM table form and runs on the DDPM kernels.  eta = 1 is the respaced ancestral sampler.
  dpmpp2m  (c_recip, c_recipm1, c_x0, c_x, c_prev): x' = c_x0 x0 + c_x x + c_prev x0_prev, deterministic, with the previous step's x0
           held on the device (wsr_sampler_step_multistep).  First order on the first step and on the step into tau = 0.

The last row (counter 0) of both outputs x0 (coefficients (1, 0, 0)), as DDPM does."""
import numpy as np

SAMPLERS = ("ddpm", "ddim", "dpmpp2m")


def timesteps(T, S):
    """The S network timesteps of an S-step sampler on a T-step schedule, descending: round(linspace(T-1, 0, S)), unique for S <= T."""
    T, S = int(T), int(S)
    if not 1 <= S <= T:
        raise ValueError("steps must be in [1, %d], got %d" % (T, S))
    return np.rint(np.linspace(T - 1, 0, S)).astype(np.int64)


def check(name, steps, eta, T):
    """Validated (name, S, eta) of ``GaussianDiffusion.set_sampler``; steps=None is every timestep, eta=None is 0 (DDIM only)."""
    if name not in SAMPLERS:
        raise ValueError("unknown sampler %r (choose from %s)" % (name, ", ".join(SAMPLERS)))
    S = int(T) if steps is None else int(steps)
    timesteps(T, S)
    if name == "ddpm" and S != int(T):
        raise ValueError("ddpm runs every timestep (steps=%d given, T=%d); use ddim with eta=1 for a respaced ancestral sampler" % (S, T))
    if eta is not None and name != "ddim":
        raise ValueError("eta applies to ddim only")
    eta = 0.0 if eta is None else float(eta)
    if not eta >= 0.0:
        raise ValueError("eta must be >= 0, got %r" % eta)
    return name, S, eta


def _rows(abar, S):
    """alphas_cumprod at each row's timestep and at the next timestep of the chain (1 after the last), in row order."""
    abar = np.asarray(abar, dtype=np.float64)
    tau = timesteps(abar.shape[0], S)
    a = abar[tau]
    a_next = np.append(a[1:], 1.0)
    return tau[::-1], a[::-1], a_next[::-1]


def ddim_tables(abar, S, eta=0.0):
    """[5][S] float64 (c_recip, c_recipm1, coef1, coef2, logvar) and the S levels, rows in counter order."""
    tau, a, a1 = _rows(abar, S)
    with np.errstate(divide="ignore"):
        var = eta ** 2 * (1.0 - a1) / (1.0 - a) * (1.0 - a / a1)
        k = np.sqrt(np.maximum(1.0 - a1 - var, 0.0))
        tab = np.stack([np.sqrt(1.0 / a), np.sqrt(1.0 / a - 1.0), np.sqrt(a1) - k * np.sqrt(a) / np.sqrt(1.0 - a),
                        k / np.sqrt(1.0 - a), np.log(var)])
    return tab, np.sqrt(a)


def dpmpp2m_tables(abar, S):
    """[5][S] float64 (c_recip, c_recipm1, c_x0, c_x, c_prev) and the S levels, rows in counter order."""
    tau, a, a1 = _rows(abar, S)
    tab = np.zeros((5, S))
    tab[0], tab[1] = np.sqrt(1.0 / a), np.sqrt(1.0 / a - 1.0)
    lam = 0.5 * np.log(a / (1.0 - a))                    # log(alpha / sigma)
    for r in range(S):
        if r == 0:                                       # at tau_{S-1}: output x0
            tab[2, r] = 1.0
            continue
        h = lam[r - 1] - lam[r]                          # row r - 1 is the next step
        base = np.sqrt(a1[r]) * -np.expm1(-h)            # -alpha' (e^-h - 1)
        tab[3, r] = np.sqrt((1.0 - a1[r]) / (1.0 - a[r]))
        if r == S - 1 or r == 1:                         # first step, and the step into tau_{S-1} (lower order final)
            tab[2, r] = base
        else:
            q = (lam[r] - lam[r + 1]) / h                # r = h_prev / h
            tab[2, r] = base * (1.0 + 0.5 / q)
            tab[4, r] = -base * 0.5 / q
    return tab, np.sqrt(a)


def tables(name, abar, S, eta=0.0):
    """The device tables of a non-DDPM sampler: (tab [5][S], levels [S]), float64."""
    return ddim_tables(abar, S, eta) if name == "ddim" else dpmpp2m_tables(abar, S)
