"""Host side of the EMA weights (train.py --ema, sample.py --ema): the update schedule of ``train.ema_scheduler`` and the
validation of the config and the command lines."""
import json
import os

import pytest

import wsr
from conftest import ROOT

glue = wsr.sub("autograd_glue")


def _actions(start, every, n=20):
    return "".join({"copy": "c", "blend": "b", "skip": "."}[glue.ema_action(s, start, every)] for s in range(1, n + 1))


def test_schedule_copy_blend_skip_over_steps_1_to_20():
    # step s uses k = s - 1: skip unless k % every == 0, copy while k < start, blend afterwards
    assert _actions(0, 1) == "b" * 20
    assert _actions(5, 1) == "ccccc" + "b" * 15
    assert _actions(3, 2) == "c.c.b.b.b.b.b.b.b.b."
    assert _actions(0, 3) == "b..b..b..b..b..b..b."
    assert _actions(4, 3) == "c..c..b..b..b..b..b."
    assert _actions(5000, 1) == "c" * 20
    assert _actions(7, 4) == "c...c...b...b...b..."


def test_schedule_from_config():
    assert glue.check_ema_schedule({"step_start_ema": 5000, "update_ema_every": 1, "ema_decay": 0.9999}) == (5000, 1, 0.9999)
    assert glue.check_ema_schedule({"step_start_ema": 0, "update_ema_every": 3, "ema_decay": 0.0}) == (0, 3, 0.0)
    bad = [None, {}, {"update_ema_every": 1, "ema_decay": 0.9},
           {"step_start_ema": 0, "update_ema_every": 0, "ema_decay": 0.9},
           {"step_start_ema": -1, "update_ema_every": 1, "ema_decay": 0.9},
           {"step_start_ema": 0, "update_ema_every": 1, "ema_decay": 1.0},
           {"step_start_ema": 0, "update_ema_every": 1, "ema_decay": -0.1},
           {"step_start_ema": 0, "update_ema_every": 1, "ema_decay": float("nan")}]
    for sched in bad:
        with pytest.raises(ValueError):
            glue.check_ema_schedule(sched)


def _config(tmp_path, sched):
    cfgmod = wsr.sub("configs.config")
    opt = json.loads(cfgmod.strip_comments(open(os.path.join(ROOT, "configs_examples", "resdiff_eval_b200.json")).read()))
    opt["name"] = "t_ema"
    if sched is None:
        del opt["train"]["ema_scheduler"]
    else:
        opt["train"]["ema_scheduler"] = sched
    p = tmp_path / "ema.json"
    p.write_text(json.dumps(opt))
    return str(p)


@pytest.mark.parametrize("sched,msg", [
    (None, "ema_scheduler"),
    ({"step_start_ema": 0, "update_ema_every": 1, "ema_decay": 1.5}, "ema_decay"),
    ({"step_start_ema": 0, "update_ema_every": 0, "ema_decay": 0.999}, "update_ema_every"),
])
def test_train_ema_rejects_a_missing_or_bad_schedule_before_building_the_model(tmp_path, monkeypatch, sched, msg):
    monkeypatch.chdir(tmp_path)
    monkeypatch.delenv("CUDA_VISIBLE_DEVICES", raising=False)      # restored after the test (Config sets it)
    train = wsr.sub("train")
    with pytest.raises(SystemExit, match=msg):
        train.main(["-c", _config(tmp_path, sched), "-p", "train", "--ema"])


def test_val_ema_needs_the_ema_file(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    monkeypatch.delenv("CUDA_VISIBLE_DEVICES", raising=False)
    train = wsr.sub("train")
    with pytest.raises(SystemExit, match="_ema.pth"):
        train.main(["-c", _config(tmp_path, None), "-p", "val", "--ema"])


def test_sample_ema_needs_a_model_path(tmp_path, capsys):
    sample = wsr.sub("sample")
    with pytest.raises(SystemExit):
        sample.parse_args(["-c", "x.json", "-o", str(tmp_path), "--ema"])
    assert "--ema needs -p" in capsys.readouterr().err
    args = sample.parse_args(["-c", "x.json", "-o", str(tmp_path), "-p", "ck/I4_E2", "--ema", "--ensemble", "2", "--sampler", "ddim",
                              "--steps", "4"])
    assert args.ema and args.model_path == "ck/I4_E2"
