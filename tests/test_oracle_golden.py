"""CPU tests: the oracle (oracle/) against the fixtures produced by the REAL reference (oracle/make_golden.py).
This is what pins the oracle; the CUDA parity tests (-m gpu) then compare against the same fixtures and the oracle.
Tolerance: fp32 restatement of fp32 code on the same CPU -> rel-L2 <= 1e-5 (reduction order differs slightly)."""
import numpy as np
import pytest
import torch

from conftest import load_golden, manifest, rel_l2
from oracle import nets, process, schedule
from oracle.cases import CASES, LINEAR_1000, short_schedule
from oracle.weights import seeded_state_dict

TOL = 1e-5


def _sd(tag, seed, cfg=None):
    if cfg is not None and cfg.get("inner_channel", 64) != 64:
        from conftest import module_manifest
        return seeded_state_dict(module_manifest(tag, cfg), seed)
    return seeded_state_dict(manifest(tag, cfg), seed)


def _wsum(sd):
    return np.array([float(sum(v.double().sum() for v in sd.values())), float(sum(v.double().abs().sum() for v in sd.values()))])


def test_schedule_tables_match_reference():
    g = load_golden("schedule")
    opts = {
        "linear1000": LINEAR_1000, "linear50": short_schedule(50),
        "quad20": {"schedule": "quad", "n_timestep": 20, "linear_start": 1e-4, "linear_end": 2e-2},
        "cosine20": {"schedule": "cosine", "n_timestep": 20, "linear_start": 1e-4, "linear_end": 2e-2},
        "warmup10_40": {"schedule": "warmup10", "n_timestep": 40, "linear_start": 1e-4, "linear_end": 2e-2},
        "warmup50_40": {"schedule": "warmup50", "n_timestep": 40, "linear_start": 1e-4, "linear_end": 2e-2},
        "const20": {"schedule": "const", "n_timestep": 20, "linear_start": 1e-4, "linear_end": 2e-2},
        "jsd20": {"schedule": "jsd", "n_timestep": 20, "linear_start": 1e-4, "linear_end": 2e-2},
    }
    for tag, opt in opts.items():
        with np.errstate(divide="ignore", invalid="ignore"):
            tabs, sap = schedule.ddpm_tables(opt)
        for n in schedule.BUFFER_NAMES:
            ref = g["%s.%s" % (tag, n)].numpy()
            np.testing.assert_array_equal(np.isfinite(tabs[n]), np.isfinite(ref), err_msg=tag + n)
            fin = np.isfinite(ref)
            np.testing.assert_allclose(tabs[n][fin], ref[fin], rtol=2e-6, atol=1e-30, err_msg=tag + "." + n)
        np.testing.assert_allclose(sap, g["%s.sqrt_alphas_cumprod_prev" % tag].numpy(), rtol=1e-12)
    # known answers quoted in SURVEY.md 8(a.1)
    tabs, sap = schedule.ddpm_tables(LINEAR_1000)
    assert abs(sap[1000] - 0.08138) < 1e-4
    assert abs(tabs["posterior_log_variance_clipped"][0] + 46.05) < 1e-2
    assert tabs["posterior_mean_coef1"][0] == 1.0 and tabs["posterior_mean_coef2"][0] == 0.0


def test_haar_known_answer():
    x = torch.tensor([[1.0, 2.0], [3.0, 4.0]]).view(1, 1, 2, 2)
    assert float(nets.haar_detail_sums(x, 1)[0]) == pytest.approx(-2 - 1 + 0)


@pytest.mark.parametrize("name", ["resdiff_step_small", "resdiff_step_full_b1", "resdiff_step_full_b2", "resdiff_step_c3_wide"])
def test_resdiff_step(name):
    g, spec = load_golden(name), CASES[name]
    sd = _sd("resdiff", spec["seed"], spec["cfg"])
    np.testing.assert_allclose(_wsum(sd), g["wsum"].numpy(), rtol=1e-9)
    with torch.no_grad():
        eps = nets.resdiff_unet(sd, torch.cat([g["cond"], g["x_t"]], 1), g["level"], spec["cfg"])
    assert rel_l2(eps, g["eps"]) < TOL


@pytest.mark.parametrize("name", ["resdiff_chain_small", "resdiff_chain_full_b1"])
def test_resdiff_chain(name):
    g, spec = load_golden(name), CASES[name]
    sd = _sd("resdiff", spec["seed"], spec["cfg"])
    with torch.no_grad():
        out = process.resdiff_chain(sd, spec["cfg"], short_schedule(spec["T"]), g["cond"], g["noise"])
    assert rel_l2(out, g["sr_out"]) < TOL


def test_resdiff_loss():
    g, spec = load_golden("resdiff_loss_small"), CASES["resdiff_loss_small"]
    sd = _sd("resdiff", spec["seed"], spec["cfg"])
    with torch.no_grad():
        loss, _ = process.resdiff_p_losses(sd, spec["cfg"], g["hr"], g["sr"], g["level"], g["noise"])
    assert abs(float(loss) - float(g["loss"])) / float(g["loss"]) < TOL


def test_simple_cnn():
    g, spec = load_golden("simple_cnn"), CASES["simple_cnn"]
    with torch.no_grad():
        out = nets.simple_cnn(_sd("simple_cnn", spec["seed"]), g["lr"])
    assert rel_l2(out, g["out"]) < TOL


def test_rrdb():
    g, spec = load_golden("rrdb_small"), CASES["rrdb_small"]
    with torch.no_grad():
        sr_img, feas = nets.rrdb_net(_sd("rrdb", spec["seed"]), g["lr"])
    assert rel_l2(sr_img, g["sr_img"]) < TOL
    assert rel_l2(torch.stack(feas, 0), g["feas"]) < TOL


def test_srdiff_step():
    g, spec = load_golden("srdiff_step_small"), CASES["srdiff_step_small"]
    with torch.no_grad():
        _, feas = nets.rrdb_net(_sd("rrdb", spec["seed"] + 1), g["lr"])
        eps = nets.srdiff_unet(_sd("srdiff", spec["seed"], spec["cfg"]), feas, g["x_t"], g["level"], spec["cfg"])
    assert rel_l2(eps, g["eps"]) < TOL


@pytest.mark.parametrize("name", ["sr3_step_small", "phydiff_step_small", "phydiff_step_full_b1", "phydiff_step_c3_small"])
def test_sr3_phydiff_step(name):
    """SURVEY 8f N1: the SR3 and PhyDiff ('ResDiff+Physics') denoisers against the real reference."""
    g, spec = load_golden(name), CASES[name]
    arch = name.split("_")[0]
    sd = _sd(arch, spec["seed"], spec["cfg"])
    np.testing.assert_allclose(_wsum(sd), g["wsum"].numpy(), rtol=1e-9)
    fn = nets.sr3_unet if arch == "sr3" else nets.phydiff_unet
    with torch.no_grad():
        eps = fn(sd, torch.cat([g["cond"], g["x_t"]], 1), g["level"], spec["cfg"])
    assert rel_l2(eps, g["eps"]) < TOL


@pytest.mark.parametrize("name", ["sr3_chain_small", "phydiff_chain_small"])
def test_sr3_phydiff_chain(name):
    g, spec = load_golden(name), CASES[name]
    arch = name.split("_")[0]
    sd = _sd(arch, spec["seed"], spec["cfg"])
    fn = nets.sr3_unet if arch == "sr3" else nets.phydiff_unet
    with torch.no_grad():
        out = process.cond_chain(fn, sd, spec["cfg"], short_schedule(spec["T"]), g["cond"], g["noise"], add_cond=(arch == "phydiff"))
    assert rel_l2(out, g["sr_out"]) < TOL


def test_phy_stencils_known_answer():
    """Reflect padding: on a horizontal ramp the x-difference is 1 inside and -1 in the last column (x[W] := x[W-2])."""
    x = torch.arange(8, dtype=torch.float32).view(1, 1, 1, 8).repeat(1, 1, 4, 1)
    st = nets.phy_stencils(x)
    assert torch.equal(st[0, 0, :, :-1], torch.ones(4, 7)) and torch.equal(st[0, 0, :, -1], -torch.ones(4))
    assert torch.equal(st[0, 1], torch.zeros(4, 8))
    assert float(st[0, 2, 1, 0]) == 2.0 and float(st[0, 2, 1, 7]) == -2.0 and float(st[0, 2, 1, 3]) == 0.0


@pytest.mark.parametrize("name", ["resdiff_grad_small", "resdiff_grad_full_b4"])
def test_resdiff_param_grads_match_reference(name):
    """Oracle autograd vs the gradient summaries of the real reference's training step (model.py:61-68); the second case is the
    BASELINE configs[2] shape itself (Cfg-A at 128x256, batch 4)."""
    from oracle.cases import grad_inputs, grad_summary
    g, spec = grad_inputs(name, load_golden(name)), CASES[name]
    sd = _sd("resdiff", spec["seed"], spec["cfg"])
    np.testing.assert_allclose(_wsum(sd), g["wsum"].numpy(), rtol=1e-9)
    loss, grads = process.resdiff_param_grads(sd, spec["cfg"], g["hr"], g["sr"], g["level"], g["noise"])
    assert abs(float(loss) - float(g["loss"])) / float(g["loss"]) < 1e-5
    names = [str(n) for n in g["names"]]
    assert sorted(names) == sorted(grads.keys())
    summ = grad_summary([(n, grads[n]) for n in names], spec["seed"])
    # the FFT-branch parameters of FD_Info_Spliter must be live in this case (non-zero reference gradient)
    for n in ("fd_spliter.sigma_resSE.fc.0.weight", "fd_spliter.HF_guided_resSE.fc.2.weight", "fd_spliter.channel_transform.weight"):
        assert float(g["norm/" + n]) > 0
    for n in names:
        ref_norm = float(g["norm/" + n])
        assert abs(float(summ["norm/" + n]) - ref_norm) <= 1e-4 * ref_norm + 1e-12, n
        assert abs(float(summ["dot/" + n]) - float(g["dot/" + n])) <= 2e-4 * ref_norm * np.sqrt(grads[n].numel()) + 1e-12, n
        if "full/" + n in g:
            assert rel_l2(grads[n], g["full/" + n]) < 1e-4 or ref_norm < 1e-12, n


@pytest.mark.parametrize("name", ["phydiff_grad_small", "sr3_grad_small"])
def test_phydiff_sr3_param_grads_match_reference(name):
    """Oracle autograd vs the gradient summaries of the real reference's PhyDiff / SR3 training step."""
    from oracle.cases import grad_summary
    g, spec = load_golden(name), CASES[name]
    arch = name.split("_")[0]
    sd = _sd(arch, spec["seed"], spec["cfg"])
    np.testing.assert_allclose(_wsum(sd), g["wsum"].numpy(), rtol=1e-9)
    loss, grads = process.arch_param_grads(arch, sd, spec["cfg"], g["hr"], g["sr"], g["level"], g["noise"])
    assert abs(float(loss) - float(g["loss"])) / float(g["loss"]) < 1e-5
    names = [str(n) for n in g["names"]]
    assert sorted(names) == sorted(grads.keys())
    summ = grad_summary([(n, grads[n]) for n in names], spec["seed"])
    for n in names:
        ref_norm = float(g["norm/" + n])
        assert abs(float(summ["norm/" + n]) - ref_norm) <= 1e-4 * ref_norm + 1e-12, n
        if "full/" + n in g:
            assert rel_l2(grads[n], g["full/" + n]) < 1e-4 or ref_norm < 1e-12, n


def test_srdiff_param_grads_match_reference():
    """SRDiff training step with the frozen RRDB encoder: oracle autograd vs the real reference's gradient summaries."""
    from oracle.cases import grad_summary
    g, spec = load_golden("srdiff_grad_small"), CASES["srdiff_grad_small"]
    sd = _sd("srdiff", spec["seed"], spec["cfg"])
    loss, grads = process.srdiff_param_grads(sd, _sd("rrdb", spec["seed"] + 1), spec["cfg"], g["lr"], g["hr"], g["sr"], g["level"], g["noise"])
    assert abs(float(loss) - float(g["loss"])) / float(g["loss"]) < 1e-5
    names = [str(n) for n in g["names"]]
    assert sorted(names) == sorted(grads.keys()) and "cond_proj.weight" in names
    summ = grad_summary([(n, grads[n]) for n in names], spec["seed"])
    assert float(g["norm/cond_proj.weight"]) > 0
    for n in names:
        ref_norm = float(g["norm/" + n])
        assert abs(float(summ["norm/" + n]) - ref_norm) <= 1e-4 * ref_norm + 1e-12, n


def test_srdiff_chain():
    """The oracle's SRDiff sampling loop (encoder + T reverse steps) against the real reference's run."""
    g, spec = load_golden("srdiff_chain_small"), CASES["srdiff_chain_small"]
    with torch.no_grad():
        out = process.srdiff_chain(_sd("srdiff", spec["seed"], spec["cfg"]), _sd("rrdb", spec["seed"] + 1), spec["cfg"],
                                   short_schedule(spec["T"]), g["lr"], g["cond"], g["noise"])
    assert rel_l2(out, g["sr_out"]) < TOL


def test_oracle_at_benchmark_shape_config4_vs_reference_probe():
    """The oracle restatement at a BENCHMARK shape against the real reference's output (probe fixture made by
    oracle/make_golden.py: strided sub-grid of eps_hat + per-sample norms): BASELINE configs[4], 3 variables, inner 128,
    128x256, the fixture's full batch of 8 (the ResDiff FFT couples the batch; ~40 s on 8 cores)."""
    from oracle.cases import fields, probe_levels, probe_summary
    from oracle.weights import seeded_randn
    name = "resdiff_step_c5_full_b8"
    g, spec = load_golden(name), CASES[name]
    cfg, b, seed = spec["cfg"], spec["batch"], spec["seed"]
    lr, sr, _ = fields(name, b, cfg["image_channels"], cfg["image_height"], cfg["image_width"], seed, scale=spec["scale"])
    x_t = seeded_randn(name + ".xt", sr.shape, seed)
    assert torch.equal(lr[:2, :, :2, :8], g["lr_head"]) and torch.equal(x_t[:2, :, :2, :8], g["xt_head"])
    level = torch.tensor(probe_levels(b), dtype=torch.float32).view(b, 1)
    sd = _sd("resdiff", seed, cfg)
    with torch.no_grad():
        eps = nets.resdiff_unet(sd, torch.cat([sr, x_t], 1), level, cfg)
    s = probe_summary(eps)
    assert rel_l2(s["eps_probe"], g["eps_probe"]) < TOL
    assert float(((s["eps_norm"] - g["eps_norm"]).abs() / g["eps_norm"]).max()) < TOL
