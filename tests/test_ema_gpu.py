"""EMA weights on the GPU: the fused Adam + EMA launch (``wsr_adam_step_ema``) against ``wsr_adam_step`` and torch, the EMA of a
small model against a torch restatement of the schedule, the raw trajectory left untouched, resume, the swap of
``DDPM.ema_weights()``, SRDiff's jointly trained encoder, and the ``--ema`` entry points.

Where two runs must agree bit for bit, the optimizer is fed seeded synthetic gradients (``_grad_step``): the hand-written
backward accumulates some weight gradients with float atomics, so two real backward passes may differ in the last bits whatever
the EMA does."""
import argparse
import json
import math
import os
import random

import numpy as np
import pytest
import torch

import wsr
from conftest import ROOT

pytestmark = pytest.mark.gpu

nat = wsr.pkg.native


# ----------------------------------------------------------------------------------------------------------------
# the kernel
# ----------------------------------------------------------------------------------------------------------------
def _adam_args(step, wd):
    return (1e-3, 0.9, 0.999, 1e-8, wd, step)


def _buffers(n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    p = torch.randn(n, device="cuda", generator=g)
    grad = torch.randn(n, device="cuda", generator=g)
    m = 0.1 * torch.randn(n, device="cuda", generator=g)
    v = torch.rand(n, device="cuda", generator=g) * 0.01 + 1e-4
    ema = torch.randn(n, device="cuda", generator=g)
    return p, grad, m, v, ema


def _stream():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("wd", [0.0, 0.01])
@pytest.mark.parametrize("step", [1, 7])
def test_adam_step_ema_matches_adam_and_torch(wd, step):
    n = 1_000_003                                           # not a multiple of the block or of any vector width
    p, g, m, v, ema = _buffers(n, 11 + step)
    ref = [t.clone() for t in (p, m, v)]
    nat.call("wsr_adam_step", ref[0].data_ptr(), g.data_ptr(), ref[1].data_ptr(), ref[2].data_ptr(), n, *_adam_args(step, wd), _stream())
    for d in (0.9, 0.9999, 0.5):
        pe, me, ve, ee = p.clone(), m.clone(), v.clone(), ema.clone()
        nat.call("wsr_adam_step_ema", pe.data_ptr(), g.data_ptr(), me.data_ptr(), ve.data_ptr(), ee.data_ptr(), n, *_adam_args(step, wd), d,
                 _stream())
        assert torch.equal(pe, ref[0]) and torch.equal(me, ref[1]) and torch.equal(ve, ref[2])
        assert torch.equal(ee, ema * d + (1 - d) * ref[0]), d
        assert not torch.equal(ee, ref[0])
    # d = 0 is an exact copy, whatever the EMA held
    pe, me, ve = p.clone(), m.clone(), v.clone()
    ee = torch.full_like(ema, float("nan"))
    nat.call("wsr_adam_step_ema", pe.data_ptr(), g.data_ptr(), me.data_ptr(), ve.data_ptr(), ee.data_ptr(), n, *_adam_args(step, wd), 0.0,
             _stream())
    assert torch.equal(pe, ref[0]) and torch.equal(ee, ref[0])


def test_adam_step_ema_rejects_bad_arguments_and_writes_nothing():
    n = 4099
    p, g, m, v, ema = _buffers(n, 3)
    big = torch.zeros(2 * n, device="cuda")
    before = [t.clone() for t in (p, g, m, v, ema, big)]
    P = lambda t: t.data_ptr()                               # noqa: E731
    good = dict(p=P(p), g=P(g), m=P(m), v=P(v), ema=P(ema), n=n, step=3, d=0.99)
    bad = [dict(p=0), dict(g=0), dict(m=0), dict(v=0), dict(ema=0), dict(n=0), dict(n=-5), dict(step=0), dict(step=-1),
           dict(d=1.0), dict(d=-0.25), dict(d=float("nan")), dict(d=2.0),
           dict(ema=P(p)), dict(ema=P(g)), dict(ema=P(m)), dict(ema=P(v)),
           dict(ema=P(big), p=P(big) + 4 * (n - 1)),            # the last element of ema is the first of p
           dict(ema=P(big) + 4 * (n - 1), m=P(big))]            # and the other way round
    for change in bad:
        a = dict(good, **change)
        with pytest.raises(nat.WsrError, match="adam_step_ema"):
            nat.call("wsr_adam_step_ema", a["p"], a["g"], a["m"], a["v"], a["ema"], a["n"], 1e-3, 0.9, 0.999, 1e-8, 0.0, a["step"], a["d"],
                     _stream())
        assert "adam_step_ema" in nat.last_error()
    torch.cuda.synchronize()
    for t, b in zip((p, g, m, v, ema, big), before):
        assert torch.equal(t, b)
    # the adjacent, non-overlapping layout is accepted
    nat.call("wsr_adam_step_ema", P(big) + 4 * n, P(g), P(m), P(v), P(big), n, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1, 0.5, _stream())


# ----------------------------------------------------------------------------------------------------------------
# models
# ----------------------------------------------------------------------------------------------------------------
def _opt(tmp_path, arch="sr3", in_channel=2, phase="train", resume=None, lock_weights=True, sched=None):
    cfgmod = wsr.sub("configs.config")
    opt = json.loads(cfgmod.strip_comments(open(os.path.join(ROOT, "configs_examples", "resdiff_eval_b200.json")).read()))
    opt["name"] = "t_ema_" + arch
    opt["model"]["architecture"] = arch
    opt["model"]["unet"].update(in_channel=in_channel, attn_res=[4])
    opt["model"]["diffusion"].update(image_height=32, image_width=64)
    for ph in ("train", "val"):
        opt["model"]["beta_schedule"][ph]["n_timestep"] = 4
    if arch == "srdiff":
        opt["model"]["pretrained_model"].update(model_path="", lock_weights=lock_weights)      # random-init encoder
    opt["data"].update(batch_size=2, val_batch_size=2, height=32)
    opt["train"].update(n_iter=2, print_freq=1, save_checkpoint_freq=2, val_freq=0)
    if sched is not None:
        opt["train"]["ema_scheduler"] = dict(zip(("step_start_ema", "update_ema_every", "ema_decay"), sched))
    for k in ("log", "tb_logger", "results", "checkpoint"):
        opt["path"][k] = str(tmp_path / k)
    os.makedirs(opt["path"]["checkpoint"], exist_ok=True)
    opt["path"]["resume_state"] = resume
    cfg = tmp_path / ("%s_%s.json" % (arch, phase))
    cfg.write_text(json.dumps(opt))
    return str(cfg), cfgmod.Config(argparse.Namespace(config=str(cfg), phase=phase, gpu_ids="0"), experiment=False).params


def _model(opt, seed=0):
    torch.manual_seed(seed)
    return wsr.sub("models.base_model").create_model(opt, None)


def _batch(arch, seed=1234):
    data = wsr.sub("data_synthetic")
    return next(data.synthetic_batches(1, 2, 1, 32, 64, seed=seed))[0]


def _seed_all(s):
    random.seed(s); np.random.seed(s); torch.manual_seed(s)


def _stepped(model):
    """[(name, parameter)] of the parameters the optimizer steps."""
    ids = {id(p) for grp in model.optG.param_groups for p in grp["params"] if p.requires_grad}
    return [(n, p) for n, p in model._net().named_parameters() if id(p) in ids]


def _grad_step(model, step, flat=True):
    """One optimizer step on seeded synthetic gradients (the same values for the flat launch and the per-parameter path)."""
    if flat:
        model._attach_flat(2)
        plan = model._net().denoise_fn.train_plan(2, model.device)
        gview = {id(p): g for p, g in plan.param_grads()}
    gen = torch.Generator(device="cuda").manual_seed(1000 + step)
    for name, p in _stepped(model):
        g = 1e-2 * torch.randn(p.shape, device="cuda", generator=gen)
        if flat and id(p) in gview:
            gview[id(p)].copy_(g)
            p.grad = gview[id(p)]
        else:
            p.grad = g
    model.optG.step()


def _state(model):
    return {k: v.detach().clone() for k, v in model._net().state_dict().items()}


def _ema_by_name(model):
    return {n: model.optG.ema[p].detach().clone() for n, p in _stepped(model)}


def _restate(ema, params, step, sched):
    """The schedule in plain torch: ema after the optimizer's step-th step, given the parameters after that step."""
    start, every, d = sched
    k = step - 1
    if k % every != 0:
        return ema
    if k < start:
        return {n: p.clone() for n, p in params.items()}
    return {n: ema[n] * d + (1 - d) * params[n] for n in ema}


SCHED = (3, 2, 0.9)


def test_ema_of_training_equals_the_torch_restatement(tmp_path):
    _, opt = _opt(tmp_path)
    model = _model(opt)
    model.enable_ema(SCHED)
    ref = {n: p.detach().clone() for n, p in _stepped(model)}
    batch = _batch("sr3")
    for s in range(1, 10):
        _seed_all(s)
        model.feed_data((batch, [1, 1]))
        model.optimize_parameters()
        assert model.optG._flat is not None and model.optG._flat["ema"] is not None      # the one-launch flat path
        ref = _restate(ref, {n: p.detach() for n, p in _stepped(model)}, s, SCHED)
        got = _ema_by_name(model)
        for n in ref:
            assert torch.equal(got[n], ref[n]), (s, n)
    assert any(not torch.equal(got[n], p.detach()) for n, p in _stepped(model))


def test_flat_launch_and_per_parameter_path_give_the_same_ema(tmp_path):
    _, opt = _opt(tmp_path)
    flat, each = _model(opt), _model(opt)
    for m in (flat, each):
        m.enable_ema(SCHED)
    ref = {n: p.detach().clone() for n, p in _stepped(each)}
    for s in range(1, 10):
        _grad_step(flat, s, flat=True)
        _grad_step(each, s, flat=False)
        ref = _restate(ref, {n: p.detach() for n, p in _stepped(each)}, s, SCHED)
    assert flat.optG._flat is not None and each.optG._flat is None
    a, b = _ema_by_name(flat), _ema_by_name(each)
    for n in a:
        assert torch.equal(a[n], b[n]) and torch.equal(b[n], ref[n]), n
    sa, sb = _state(flat), _state(each)
    assert all(torch.equal(sa[k], sb[k]) for k in sa)


def test_ema_leaves_the_raw_trajectory_unchanged(tmp_path):
    _, opt = _opt(tmp_path)
    plain, with_ema = _model(opt), _model(opt)
    with_ema.enable_ema((2, 1, 0.9))
    for s in range(1, 6):
        _grad_step(plain, s)
        _grad_step(with_ema, s)
    sa, sb = _state(plain), _state(with_ema)
    assert all(torch.equal(sa[k], sb[k]) for k in sa)
    oa, ob = plain.optG.state_dict()["state"], with_ema.optG.state_dict()["state"]
    for i in oa:
        for k in ("exp_avg", "exp_avg_sq", "step"):
            assert torch.equal(oa[i][k], ob[i][k]), (i, k)
    # the same forward on the same weights: the same loss
    batch = _batch("sr3")
    losses = []
    for m in (plain, with_ema):
        _seed_all(7)
        m.feed_data((batch, [1, 1]))
        m.optimize_parameters()
        losses.append(m.get_current_log()["l_pix"])
    assert losses[0] == losses[1]


def _ckpt_files(ck, it, ep):
    return {w: torch.load(os.path.join(ck, "I%d_E%d_%s.pth" % (it, ep, w)), map_location="cpu") for w in ("gen", "ema")}


def test_resume_continues_the_ema(tmp_path):
    straight_dir, split_dir = tmp_path / "a", tmp_path / "b"
    _, opt_a = _opt(straight_dir)
    a = _model(opt_a)
    a.enable_ema(SCHED)
    for s in range(1, 5):
        _grad_step(a, s)
    a.save_network(1, 4)
    _, opt_b = _opt(split_dir)
    b = _model(opt_b)
    b.enable_ema(SCHED)
    for s in range(1, 3):
        _grad_step(b, s)
    b.save_network(1, 2)
    ck_b = opt_b["path"]["checkpoint"]
    assert sorted(os.listdir(ck_b)) == ["I2_E1_ema.pth", "I2_E1_gen.pth", "I2_E1_opt.pth"]
    _, opt_c = _opt(split_dir, resume=os.path.join(ck_b, "I2_E1"))
    c = _model(opt_c, seed=99)
    c.enable_ema(SCHED)
    for s in range(3, 5):
        _grad_step(c, s)
    c.save_network(1, 4)
    fa, fc = _ckpt_files(opt_a["path"]["checkpoint"], 4, 1), _ckpt_files(ck_b, 4, 1)
    for w in ("gen", "ema"):
        assert fa[w].keys() == fc[w].keys()
        for k in fa[w]:
            assert torch.equal(fa[w][k], fc[w][k]), (w, k)
    assert any(not torch.equal(fa["ema"][k], fa["gen"][k]) for k in fa["gen"])
    # a checkpoint without an EMA file: the EMA starts from the loaded weights
    os.remove(os.path.join(ck_b, "I2_E1_ema.pth"))
    d = _model(opt_c, seed=98)
    d.enable_ema(SCHED)
    gen2 = torch.load(os.path.join(ck_b, "I2_E1_gen.pth"), map_location="cpu")
    for n, e in _ema_by_name(d).items():
        assert torch.equal(e.cpu(), gen2[n]), n


def _loss(model, batch, seed):
    """The training forward (the train plan's packed weights) on a fixed batch, without a backward pass or a step; no dropout,
    whose mask stream advances with every forward."""
    _seed_all(seed)
    model.feed_data((batch, [1, 1]))
    model._attach_flat(2)
    net = model._net().denoise_fn
    net.eval()
    try:
        return model.netG(model.data).detach().sum().item()
    finally:
        net.train()


def _sample(model, batch):
    model.prepare_to_eval()
    model.feed_data((batch, [1, 1]))
    model._net().sample_seed = 5
    model.generate_sr(False)
    model.prepare_to_train()
    return model.SR.clone()


def test_ema_weights_swap_is_exact_and_matches_the_ema_file(tmp_path):
    _, opt = _opt(tmp_path)
    with_val, without = _model(opt), _model(opt)
    for m in (with_val, without):
        m.enable_ema(SCHED)
    batch = _batch("sr3")
    for s in range(1, 6):
        for m in (with_val, without):
            _grad_step(m, s)
    assert _loss(with_val, batch, 3) == _loss(without, batch, 3)        # both plans have packed the trained weights
    before = _state(with_val)
    with with_val.ema_weights():                                # train.py's validation: generate_sr on the EMA
        ema = _ema_by_name(with_val)
        for n, p in _stepped(with_val):
            assert torch.equal(p.detach(), ema[n]), n
        sr_ema = _sample(with_val, batch)
        with pytest.raises(RuntimeError, match="ema_weights"):         # a training forward on the EMA is refused
            _loss(with_val, batch, 3)
    assert not torch.equal(sr_ema, _sample(without, batch))
    after = _state(with_val)
    assert all(torch.equal(before[k], after[k]) for k in before)
    for s in range(6, 9):
        for m in (with_val, without):
            _grad_step(m, s)
    sv, sw = _state(with_val), _state(without)
    assert all(torch.equal(sv[k], sw[k]) for k in sv)
    assert _loss(with_val, batch, 4) == _loss(without, batch, 4)
    assert torch.equal(_sample(with_val, batch), _sample(without, batch))
    # sampling under ema_weights() == sampling a fresh model loaded from the EMA file
    with_val.save_network(1, 8)
    _, opt_v = _opt(tmp_path, phase="val")
    fresh = _model(opt_v, seed=42)
    fresh.load_network(os.path.join(opt["path"]["checkpoint"], "I8_E1"), weights="ema")
    with with_val.ema_weights():
        again = _sample(with_val, batch)
    assert torch.isfinite(again).all() and not torch.equal(again, sr_ema)
    assert torch.equal(_sample(fresh, batch), again)


@pytest.mark.parametrize("lock_weights", [False, True])
def test_srdiff_encoder_in_the_ema_file(tmp_path, lock_weights):
    _, opt = _opt(tmp_path, arch="srdiff", in_channel=1, lock_weights=lock_weights)
    model = _model(opt)
    model.enable_ema((0, 1, 0.5))
    for s in range(1, 4):
        _grad_step(model, s)
    model.save_network(1, 3)
    f = _ckpt_files(opt["path"]["checkpoint"], 3, 1)
    ema = _ema_by_name(model)
    enc = ["rrdb_encoder." + n for n, _ in model._net().rrdb_encoder.named_parameters()]
    assert enc and f["ema"].keys() == f["gen"].keys()
    if lock_weights:
        assert not any(n in ema for n in enc)                 # a locked prior is not stepped: copied as it is
    else:
        assert all(n in ema for n in enc)
        assert any(not torch.equal(f["ema"][n], f["gen"][n]) for n in enc)
    for k in f["gen"]:
        if k in ema:
            assert torch.equal(f["ema"][k], ema[k].cpu()), k
        else:
            assert torch.equal(f["ema"][k], f["gen"][k]), k
    # sampling under ema_weights() runs the encoder on its EMA too: the same as a fresh model loaded from the EMA file, after the
    # encoder plan has packed the trained weights
    batch = _batch("srdiff")
    sr_trained = _sample(model, batch)
    with model.ema_weights():
        sr_ema = _sample(model, batch)
    assert torch.equal(_sample(model, batch), sr_trained)
    _, opt_v = _opt(tmp_path / "fresh", arch="srdiff", in_channel=1, phase="val", lock_weights=lock_weights)
    fresh = _model(opt_v, seed=42)
    fresh.load_network(os.path.join(opt["path"]["checkpoint"], "I3_E1"), weights="ema")
    assert torch.isfinite(sr_ema).all() and not torch.equal(sr_ema, sr_trained)
    assert torch.equal(_sample(fresh, batch), sr_ema)


def test_entry_points_with_ema(tmp_path, caplog):
    import logging
    cfg, _ = _opt(tmp_path, sched=(1, 1, 0.5))                # step 1 copies, step 2 blends: EMA != last iterate
    opt = json.loads(open(cfg).read())
    opt["train"].update(val_freq=2, full_val_freq=1000)
    open(cfg, "w").write(json.dumps(opt))
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        train, sample = wsr.sub("train"), wsr.sub("sample")
        with caplog.at_level(logging.INFO, logger="base"):
            assert train.main(["-c", cfg, "-p", "train", "-gpu", "0", "--ema"]) == (2, 1)
        assert "validation with the EMA weights" in caplog.text
        ck = opt["path"]["checkpoint"]
        assert sorted(os.listdir(ck)) == ["I2_E1_ema.pth", "I2_E1_gen.pth", "I2_E1_opt.pth"]
        gen = torch.load(os.path.join(ck, "I2_E1_gen.pth"), map_location="cpu")
        ema = torch.load(os.path.join(ck, "I2_E1_ema.pth"), map_location="cpu")
        assert gen.keys() == ema.keys() and all(gen[k].shape == ema[k].shape and gen[k].dtype == ema[k].dtype for k in gen)
        assert any(not torch.equal(gen[k], ema[k]) for k in gen)
        _, opt_v = _opt(tmp_path / "fresh", phase="val")
        _model(opt_v)._net().load_state_dict(ema, strict=True)
        # -p val --ema validates the EMA file
        opt["path"]["resume_state"] = os.path.join(ck, "I2_E1")
        open(cfg, "w").write(json.dumps(opt))
        m_ema, _ = train.main(["-c", cfg, "-p", "val", "-gpu", "0", "--ema"])
        m_gen, _ = train.main(["-c", cfg, "-p", "val", "-gpu", "0"])
        m_ema, m_gen = ({k: float(v) for k, v in m.items()} for m in (m_ema, m_gen))
        assert all(math.isfinite(v) for v in m_ema.values()) and m_ema != m_gen
        # sample.py --ema, plain and as a fewer-step ensemble
        for extra, name in (([], "sr.npy"), (["--ensemble", "2", "--sampler", "ddim", "--steps", "4"], "ensemble.npy")):
            outs = []
            for flag in (["--ema"], []):
                out = tmp_path / ("out_%s_%d" % (name, len(flag)))
                sample.main(["-c", cfg, "-o", str(out), "-gpu", "0", "-p", os.path.join(ck, "I2_E1"), "--seed", "77"] + flag + extra)
                outs.append(np.load(out / name))
            assert np.isfinite(outs[0]).all() and outs[0].shape == outs[1].shape
            assert not np.array_equal(outs[0], outs[1]), name
    finally:
        os.chdir(cwd)
