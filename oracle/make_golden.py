"""TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

Generates tests/golden/*.npz by running the REAL reference (imported from /root/reference through
oracle/ref_shims.py) on the seeded cases of oracle/cases.py.  Run in the build container:

    python -m oracle.make_golden            # all cases
    python -m oracle.make_golden NAME ...   # selected cases

The fixtures store inputs and reference outputs (small fields only); weights are re-derived from the seed
(oracle/weights.py), with a checksum stored to detect RNG drift.
"""
import os
import sys

import numpy as np
import torch
import torch.nn.functional as F

from . import ref_shims
from .cases import CASES, LINEAR_1000, fields, short_schedule
from .schedule import BUFFER_NAMES
from .weights import fill_module, seeded_randn

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def _checksum(module):
    with torch.no_grad():
        return np.array([float(sum(p.double().sum() for p in module.parameters())),
                         float(sum(p.double().abs().sum() for p in module.parameters()))])


def _unet(ref, cfg, srdiff=False, arch=None):
    cls = ref.SRDiffUNet if srdiff else ref.ResDiffUNet
    extra = {}
    if arch == "sr3":
        cls = ref.SR3UNet
    elif arch == "phydiff":
        cls, extra = ref.PhyDiffUNet, {"device": "cpu"}
    net = cls(**extra, in_channel=cfg["in_channel"], out_channel=cfg["out_channel"], norm_groups=cfg["norm_groups"],
              inner_channel=cfg["inner_channel"], channel_mults=cfg["channel_mults"], attn_res=cfg["attn_res"],
              res_blocks=cfg["res_blocks"], dropout=cfg["dropout"], image_height=cfg["image_height"],
              image_width=cfg["image_width"], image_channels=cfg["image_channels"])
    return net.eval()


class _InjectedNoise:
    """Replaces torch.randn / torch.randn_like by an iterator over a pre-generated tensor (SURVEY 8c)."""

    def __init__(self, noise):
        self.noise, self.i = noise, 0

    def __enter__(self):
        self._randn, self._randn_like = torch.randn, torch.randn_like

        def nxt(*a, **k):
            out = self.noise[self.i].clone()
            self.i += 1
            return out

        torch.randn, torch.randn_like = nxt, nxt
        return self

    def __exit__(self, *exc):
        torch.randn, torch.randn_like = self._randn, self._randn_like


def run_grad_case(ref, name, spec):
    """The reference's training step up to the optimizer (model.py:61-68): p_losses -> sum / numel -> backward, with the
    random draws (t, continuous level, noise) injected and dropout = 0."""
    from .cases import grad_summary
    seed, b, cfg, t = spec["seed"], spec["batch"], spec["cfg"], spec["t"]
    arch = spec["kind"].split("_")[0]
    net = fill_module(_unet(ref, cfg, arch=arch, srdiff=(arch == "srdiff")), seed).train()
    D = {"resdiff": ref.ResDiffDiffusion, "phydiff": ref.PhyDiffDiffusion, "sr3": ref.SR3Diffusion, "srdiff": ref.SRDiffDiffusion}[arch]
    diff = D(net, image_height=cfg["image_height"], image_width=cfg["image_width"],
                                channels=cfg["image_channels"], conditional=True)
    diff.set_new_noise_schedule(LINEAR_1000, "cpu")
    diff.set_loss("cpu")
    lr, sr, hr = fields(name, b, cfg["image_channels"], cfg["image_height"], cfg["image_width"], seed)
    if arch == "srdiff" and spec.get("joint"):
        # trainable encoder (lock_weights=False): the loss gains l1(rrdb_sr, HR) and the encoder gets gradients (srdiff_diffusion.py:212-214)
        from .cases import calibrate_rrdb_head
        diff.rrdb_encoder = calibrate_rrdb_head(fill_module(ref.RRDBNet(1, 1, 64, 17, 32).train(), seed + 1))
        diff.lock_weights = False
    elif arch == "srdiff":
        # frozen encoder, as init_rrdb_encoder(lock_weights=True) leaves it (srdiff_diffusion.py:59-75)
        diff.rrdb_encoder = fill_module(ref.RRDBNet(1, 1, 64, 17, 32).eval(), seed + 1)
        for p_ in diff.rrdb_encoder.parameters():
            p_.requires_grad_(False)
    noise = seeded_randn(name + ".noise", sr.shape, seed)
    sap = diff.sqrt_alphas_cumprod_prev
    u = np.random.RandomState(seed).uniform(sap[t - 1], sap[t], size=b)
    _ri, _un = np.random.randint, np.random.uniform
    np.random.randint = lambda *a, **k: t
    np.random.uniform = lambda *a, **k: u
    try:
        loss = diff.p_losses({"HR": hr, "SR": sr, "LR": lr}, noise=noise)
    finally:
        np.random.randint, np.random.uniform = _ri, _un
    l_pix = loss.sum() / int(hr.numel())
    l_pix.backward()
    out = dict(level=torch.FloatTensor(u), loss=loss.detach().reshape(1), wsum=_checksum(net))
    inputs = dict(hr=hr, sr=sr, lr=lr, noise=noise)
    if spec.get("regenerate_inputs"):
        # 128x256 fields: the tests regenerate them from the seed (cases.grad_inputs); the heads detect RNG drift
        inputs = {k + "_head": v[:, :, :2, :8].clone() for k, v in inputs.items()}
    out.update(inputs)
    named = [(n, p.grad) for n, p in net.named_parameters() if p.grad is not None]
    if spec.get("joint"):
        named += [("rrdb_encoder." + n, p.grad) for n, p in diff.rrdb_encoder.named_parameters() if p.grad is not None]
    out["names"] = np.array([n for n, _ in named])
    out.update(grad_summary(named, seed, full_below=128 if spec.get("joint") else 4096))
    return {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in out.items()}


class _PerSampleHFCA:
    """Runs the reference's HF_guided_CA.forward (guided_cross_attention.py:24-44) one sample at a time: the module is
    per-sample independent (GroupNorm, 1x1 convolutions, softmax over that sample's keys), but at level 0 it materialises a
    (B, 8192, 8192) fp32 matrix several times over -- 17 GB each at the benchmark batch of 64, more than this container holds.
    The reference's own code runs unmodified on each batch slice."""

    def __enter__(self):
        import models.diffusion_models.resdiff.guided_cross_attention as m
        self.cls, self.orig = m.HF_guided_CA, m.HF_guided_CA.forward
        orig = self.orig

        def forward(mod, input, quary):
            return torch.cat([orig(mod, input[i:i + 1], quary[i:i + 1]) for i in range(input.shape[0])], 0)

        self.cls.forward = forward
        return self

    def __exit__(self, *exc):
        self.cls.forward = self.orig


def run_probe_case(ref, name, spec):
    """One denoiser call at a benchmark shape; keeps a probe of the output (cases.probe_summary)."""
    from .cases import probe_levels, probe_summary
    seed, b, cfg, arch = spec["seed"], spec["batch"], spec["cfg"], spec["arch"]
    c, H, W = cfg["image_channels"], cfg["image_height"], cfg["image_width"]
    lr, sr, _ = fields(name, b, c, H, W, seed, scale=spec["scale"])
    x_t = seeded_randn(name + ".xt", sr.shape, seed)
    level = torch.tensor(probe_levels(b), dtype=torch.float32).view(b, 1)
    with torch.no_grad():
        if arch == "srdiff":
            net = fill_module(_unet(ref, cfg, srdiff=True), seed)
            rrdb = fill_module(ref.RRDBNet(1, 1, 64, 17, 32).eval(), seed + 1)
            _, feas = rrdb(lr, True)
            eps = net((feas, x_t), level)
        else:
            net = fill_module(_unet(ref, cfg), seed)
            with _PerSampleHFCA():
                eps = net(torch.cat([sr, x_t], 1), level)
    out = dict(level=level, lr_head=lr[:2, :, :2, :8].clone(), xt_head=x_t[:2, :, :2, :8].clone(), wsum=_checksum(net))
    out.update(probe_summary(eps))
    return {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in out.items()}


def run_case(ref, name, spec):
    kind, seed, b = spec["kind"], spec["seed"], spec["batch"]
    if kind == "step_probe":
        return run_probe_case(ref, name, spec)
    if kind in ("resdiff_grad", "phydiff_grad", "sr3_grad", "srdiff_grad"):
        return run_grad_case(ref, name, spec)
    out = {}
    with torch.no_grad():
        if kind == "resdiff_step":
            cfg = spec["cfg"]
            net = fill_module(_unet(ref, cfg), seed)
            _, sr, _ = fields(name, b, cfg["image_channels"], cfg["image_height"], cfg["image_width"], seed)
            x_t = seeded_randn(name + ".xt", sr.shape, seed)
            level = torch.tensor(spec["level"], dtype=torch.float32).view(b, 1)
            out.update(cond=sr, x_t=x_t, level=level, eps=net(torch.cat([sr, x_t], 1), level), wsum=_checksum(net))
        elif kind == "resdiff_chain":
            cfg, T = spec["cfg"], spec["T"]
            net = fill_module(_unet(ref, cfg), seed)
            diff = ref.ResDiffDiffusion(net, image_height=cfg["image_height"], image_width=cfg["image_width"],
                                        channels=cfg["image_channels"], conditional=True)
            diff.set_new_noise_schedule(short_schedule(T), "cpu")
            _, sr, _ = fields(name, b, cfg["image_channels"], cfg["image_height"], cfg["image_width"], seed)
            noise = seeded_randn(name + ".noise", (T + 1,) + tuple(sr.shape), seed)
            with _InjectedNoise(noise) as inj:
                res = diff.super_resolution({"SR": sr})
                assert inj.i == T, inj.i          # 1 randn + (T-1) randn_like
            if spec.get("regenerate_noise"):
                # long chains: the noise is regenerated from its seed by the tests (same torch build on both machines), only the
                # condition and the reference's final field are stored
                out.update(cond=sr, sr_out=res, noise_head=noise[:2, :, :, :2, :8].clone(), wsum=_checksum(net))
            else:
                out.update(cond=sr, noise=noise, sr_out=res, wsum=_checksum(net))
        elif kind == "resdiff_loss":
            cfg, t = spec["cfg"], spec["t"]
            net = fill_module(_unet(ref, cfg), seed)
            diff = ref.ResDiffDiffusion(net, image_height=cfg["image_height"], image_width=cfg["image_width"],
                                        channels=cfg["image_channels"], conditional=True)
            diff.set_new_noise_schedule(LINEAR_1000, "cpu")
            diff.set_loss("cpu")
            _, sr, hr = fields(name, b, cfg["image_channels"], cfg["image_height"], cfg["image_width"], seed)
            noise = seeded_randn(name + ".noise", sr.shape, seed)
            sap = diff.sqrt_alphas_cumprod_prev
            u = np.random.RandomState(seed).uniform(sap[t - 1], sap[t], size=b)
            level = torch.FloatTensor(u)
            # inject t and the continuous level through numpy's global RNG entry points (resdiff_diffusion.py:128-135)
            _ri, _un = np.random.randint, np.random.uniform
            np.random.randint = lambda *a, **k: t
            np.random.uniform = lambda *a, **k: u
            try:
                loss = diff.p_losses({"HR": hr, "SR": sr}, noise=noise)
            finally:
                np.random.randint, np.random.uniform = _ri, _un
            out.update(hr=hr, sr=sr, noise=noise, level=level, loss=loss.reshape(1), wsum=_checksum(net))
        elif kind in ("sr3_step", "phydiff_step"):
            cfg, arch = spec["cfg"], kind.split("_")[0]
            net = fill_module(_unet(ref, cfg, arch=arch), seed)
            _, sr, _ = fields(name, b, cfg["image_channels"], cfg["image_height"], cfg["image_width"], seed)
            x_t = seeded_randn(name + ".xt", sr.shape, seed)
            level = torch.tensor(spec["level"], dtype=torch.float32).view(b, 1)
            out.update(cond=sr, x_t=x_t, level=level, eps=net(torch.cat([sr, x_t], 1), level), wsum=_checksum(net))
        elif kind in ("sr3_chain", "phydiff_chain"):
            cfg, T, arch = spec["cfg"], spec["T"], kind.split("_")[0]
            net = fill_module(_unet(ref, cfg, arch=arch), seed)
            D = ref.SR3Diffusion if arch == "sr3" else ref.PhyDiffDiffusion
            diff = D(net, image_height=cfg["image_height"], image_width=cfg["image_width"], channels=cfg["image_channels"], conditional=True)
            diff.set_new_noise_schedule(short_schedule(T), "cpu")
            _, sr, _ = fields(name, b, cfg["image_channels"], cfg["image_height"], cfg["image_width"], seed)
            noise = seeded_randn(name + ".noise", (T + 1,) + tuple(sr.shape), seed)
            with _InjectedNoise(noise) as inj:
                res = diff.super_resolution({"SR": sr})
                assert inj.i == T, inj.i
            out.update(cond=sr, noise=noise, sr_out=res, wsum=_checksum(net))
        elif kind == "simple_cnn":
            net = fill_module(ref.SimpleCNN(scale_factor=4, channels=1).eval(), seed)
            lr = seeded_randn(name + ".lr", (b, 1) + tuple(spec["lr_hw"]), seed)
            out.update(lr=lr, out=net(lr), wsum=_checksum(net))
        elif kind == "simple_cnn_pretrain":
            # SURVEY 8f N4: one pre-training step of the prior (pretrain.py:37-48): image_compare_loss and all parameter gradients
            from models.simple_cnn.loss import image_compare_loss, fft_mse_loss, dwt_mse_loss
            net = fill_module(ref.SimpleCNN(scale_factor=4, channels=1).train(), seed)
            lr, _, hr = fields(name, b, 1, 4 * spec["lr_hw"][0], 4 * spec["lr_hw"][1], seed)
            with torch.enable_grad():
                pred = net(lr)
                loss = image_compare_loss(pred, hr)
                loss.backward()
            pred, loss = pred.detach(), loss.detach()
            out.update(lr=lr, hr=hr, pred=pred, loss=loss.reshape(1), fft=fft_mse_loss(pred, hr).reshape(1), dwt=dwt_mse_loss(pred, hr).reshape(1))
            for n, prm in net.named_parameters():
                out["grad." + n] = prm.grad
        elif kind == "rrdb_pretrain":
            # SURVEY 8f N4: one pre-training step of the encoder (pretrain.py:37-48, criterion = F.l1_loss): all parameter gradients
            from .cases import grad_summary, calibrate_rrdb_head
            net = calibrate_rrdb_head(fill_module(ref.RRDBNet(1, 1, 64, spec["nb"], 32).train(), seed))
            lr, _, hr = fields(name, b, 1, 4 * spec["lr_hw"][0], 4 * spec["lr_hw"][1], seed)
            lr, hr = lr * 0.5, (hr * 0.25).clamp(-1, 1)
            with torch.enable_grad():
                pred = net(lr)
                loss = F.l1_loss(pred, hr)
                loss.backward()
            out.update(lr=lr, hr=hr, pred=pred.detach(), loss=loss.detach().reshape(1),
                       inside=torch.tensor([float(((pred > -1) & (pred < 1)).float().mean())]))
            named = [(n, prm.grad) for n, prm in net.named_parameters()]
            out["names"] = np.array([n for n, _ in named])
            out.update(grad_summary(named, seed, full_below=128))
        elif kind == "rrdb":
            net = fill_module(ref.RRDBNet(1, 1, 64, 17, 32).eval(), seed)
            lr = seeded_randn(name + ".lr", (b, 1) + tuple(spec["lr_hw"]), seed)
            sr_img, feas = net(lr, True)
            out.update(lr=lr, sr_img=sr_img, feas=torch.stack(feas, 0), wsum=_checksum(net))
        elif kind == "srdiff_step":
            cfg = spec["cfg"]
            net = fill_module(_unet(ref, cfg, srdiff=True), seed)
            rrdb = fill_module(ref.RRDBNet(1, 1, 64, 17, 32).eval(), seed + 1)
            lr, sr, _ = fields(name, b, 1, cfg["image_height"], cfg["image_width"], seed)
            _, feas = rrdb(lr, True)
            x_t = seeded_randn(name + ".xt", sr.shape, seed)
            level = torch.tensor(spec["level"], dtype=torch.float32).view(b, 1)
            out.update(lr=lr, x_t=x_t, level=level, eps=net((feas, x_t), level), wsum=_checksum(net))
        elif kind == "srdiff_chain":
            # the SRDiff sampling loop with its encoder (srdiff_diffusion.py:77-131): encode LR once, T reverse steps conditioned on
            # the features, + bicubic
            cfg, T = spec["cfg"], spec["T"]
            net = fill_module(_unet(ref, cfg, srdiff=True), seed)
            diff = ref.SRDiffDiffusion(net, image_height=cfg["image_height"], image_width=cfg["image_width"], channels=1, conditional=True)
            diff.rrdb_encoder = fill_module(ref.RRDBNet(1, 1, 64, 17, 32).eval(), seed + 1)
            diff.set_new_noise_schedule(short_schedule(T), "cpu")
            lr, sr, _ = fields(name, b, 1, cfg["image_height"], cfg["image_width"], seed)
            noise = seeded_randn(name + ".noise", (T + 1,) + tuple(sr.shape), seed)
            with _InjectedNoise(noise) as inj:
                res = diff.super_resolution({"SR": sr, "LR": lr})
                assert inj.i == T, inj.i
            out.update(lr=lr, cond=sr, noise=noise, sr_out=res, wsum=_checksum(net))
        else:
            raise KeyError(kind)
    return {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in out.items()}


def schedule_fixture(ref):
    """Reference schedule buffers for a handful of schedules (diffusion.py:49-96)."""
    out = {}
    dummy = torch.nn.Identity()
    for tag, opt in {
        "linear1000": LINEAR_1000, "linear50": short_schedule(50),
        "quad20": {"schedule": "quad", "n_timestep": 20, "linear_start": 1e-4, "linear_end": 2e-2},
        "cosine20": {"schedule": "cosine", "n_timestep": 20, "linear_start": 1e-4, "linear_end": 2e-2},
        "warmup10_40": {"schedule": "warmup10", "n_timestep": 40, "linear_start": 1e-4, "linear_end": 2e-2},
        "warmup50_40": {"schedule": "warmup50", "n_timestep": 40, "linear_start": 1e-4, "linear_end": 2e-2},
        "const20": {"schedule": "const", "n_timestep": 20, "linear_start": 1e-4, "linear_end": 2e-2},
        "jsd20": {"schedule": "jsd", "n_timestep": 20, "linear_start": 1e-4, "linear_end": 2e-2},
    }.items():
        diff = ref.ResDiffDiffusion(dummy, image_height=8, image_width=8, channels=1)
        diff.set_new_noise_schedule(opt, "cpu")
        for n in BUFFER_NAMES:
            out["%s.%s" % (tag, n)] = getattr(diff, n).numpy()
        out["%s.sqrt_alphas_cumprod_prev" % tag] = np.asarray(diff.sqrt_alphas_cumprod_prev)
    return out


def edge_fixture():
    """SURVEY 8f N2: collate interpolation, GlobalStandardScaling fit / transform / revert, MAE / MSE / RMSE / MR -- all through
    the reference's own classes (data/dataset_builder.py:374-380 is a bare F.interpolate call, reproduced verbatim)."""
    from torch.nn.functional import interpolate
    edge = ref_shims.import_reference_edge()
    out = {}
    lr = seeded_randn("edge.lr", (3, 2, 8, 16), 71)
    out["lr"] = lr
    out["sr"] = torch.cat([interpolate(lr[i:i + 1], scale_factor=4, mode="bicubic") for i in range(3)])
    # two months with different statistics, two fitting batches each
    stats = {}
    for month, (mu, sd) in {1: (270.0, 9.0), 7: (291.0, 5.5)}.items():
        t = edge.transforms.GlobalStandardScaling()
        batches = [seeded_randn("edge.fit%d.%d" % (month, k), (4, 1, 16, 32), 72) * sd + mu for k in range(2)]
        for bdata in batches:
            t._update_parameters(bdata)
        stats[month] = t
        out["fit%d" % month] = torch.stack(batches)
        out["mean%d" % month] = t._mean.reshape(1)
        out["std%d" % month] = t._std().reshape(1)
    x = seeded_randn("edge.x", (2, 1, 16, 32), 73) * 7.0 + 280.0
    out["x"] = x
    out["x_std1"] = stats[1].transform(x)
    out["x_back1"] = stats[1].revert(out["x_std1"])
    pred, target = seeded_randn("edge.pred", (4, 1, 16, 32), 74), seeded_randn("edge.target", (4, 1, 16, 32), 75)
    out["pred"], out["target"] = pred, target
    for name in ("MAE", "MSE", "RMSE", "MR"):
        m = getattr(edge.metrics, name)(device="cpu")
        m.update(pred[:2], target[:2])
        m.update(pred[2:], target[2:])
        out["metric_" + name] = torch.as_tensor(m.compute()).reshape(1).float()
    return {k: v.detach().cpu().numpy() for k, v in out.items()}


def store_fixture():
    """SURVEY 8f N3: the REAL reference DataHandler (npy_reader, datasets, transforms, dataset_builder) run on the synthetic
    store of oracle/store.py -- lengths, sample-index time stamps, fitted per-month statistics, the first validation batch,
    one training item, a batch fetched by date and its inverse transform."""
    import tempfile
    from . import store
    ref = ref_shims.import_reference_data()
    out = {}
    with tempfile.TemporaryDirectory() as root:
        store.write_store(root)
        spec = store.SPEC
        dh = ref.dataset_builder.DataHandler(root, list(store.VARIABLES), root, spec["months_subset"], spec["groups"],
                                             ref.transforms.GlobalStandardScaling, spec["train"][0], spec["train"][1],
                                             spec["val"][0], spec["val"][1], spec["val_batch_size"], spec["train_batch_size"], False, 0)
        train_loader, val_loader, metadata, transformer = dh.process_data()
        train_set, val_set = dh.get_datasets()
        out["train_len"], out["val_len"] = np.array(len(train_set)), np.array(len(val_set))
        first = list(train_set.data_groups["lr"].values())[0]
        probe = np.array([0, 1, 743, 744, 800, len(train_set) - 1])
        out["probe"] = probe
        out["probe_stamps"] = np.array([first._sample_index[int(i)] for i in probe]).astype("datetime64[h]").astype(np.int64)
        for v in store.VARIABLES:
            for kind in ("lr", "hr"):
                for month, t in transformer.transformation_dict[v][kind].items():
                    out["mean.%s.%s.%d" % (v, kind, month)] = t._mean.reshape(1).numpy()
                    out["std.%s.%s.%d" % (v, kind, month)] = t._std().reshape(1).numpy()
        batch, months = next(iter(val_loader))
        for k in ("HR", "LR", "SR"):
            out["val0." + k] = batch[k].numpy()
        out["val0.months"] = np.array(months)
        out["val_batches"] = np.array(len(val_loader))
        out["train_batches"] = np.array(len(train_loader))
        item = train_set[800]
        out["item800.lr"] = torch.cat([v[0] for v in item[0]], 1).numpy()
        out["item800.hr"] = torch.cat([v[0] for v in item[1]], 1).numpy()
        out["item800.month"] = np.array(item[0][0][2])
        by_date, bmonths = dh.get_data_by_date("2000-03-05-07")
        for k in ("HR", "LR", "SR"):
            out["date." + k] = by_date[k].numpy()
        out["date.months"] = np.array(bmonths)
        inv = transformer.inverse_transform(by_date, bmonths)
        for k in ("HR", "LR", "SR"):
            out["date_inv." + k] = inv[k].numpy()
        out["meta.hr_lat"] = np.asarray(metadata.hr_lat)
        out["channels.lr"] = np.array(int(train_set.get_channel_count("lr")))
    return out


def main(argv):
    if argv == ["edge"]:
        os.makedirs(GOLDEN_DIR, exist_ok=True)
        np.savez_compressed(os.path.join(GOLDEN_DIR, "edge.npz"), **edge_fixture())
        print("wrote edge.npz")
        return
    if argv == ["store"]:
        os.makedirs(GOLDEN_DIR, exist_ok=True)
        np.savez_compressed(os.path.join(GOLDEN_DIR, "store.npz"), **store_fixture())
        print("wrote store.npz")
        return
    ref = ref_shims.import_reference()
    os.makedirs(GOLDEN_DIR, exist_ok=True)
    names = argv or (list(CASES) + ["schedule", "manifest"])
    for name in names:
        if name == "schedule":
            data = schedule_fixture(ref)
        elif name == "manifest":
            # state_dict key/shape manifests: the drop-in contract for checkpoints (SURVEY 8b)
            from .cases import unet_cfg
            data = {}
            for tag, net in {"resdiff": _unet(ref, unet_cfg(128, 256)), "srdiff": _unet(ref, unet_cfg(128, 256, in_channel=1), srdiff=True),
                             "sr3": _unet(ref, unet_cfg(128, 256, in_channel=2), arch="sr3"),
                             "phydiff": _unet(ref, unet_cfg(128, 256), arch="phydiff"),
                             "rrdb": ref.RRDBNet(1, 1, 64, 17, 32), "simple_cnn": ref.SimpleCNN(4, 1)}.items():
                sd = net.state_dict()
                data[tag + ".keys"] = np.array(list(sd.keys()))
                data[tag + ".shapes"] = np.array([",".join(map(str, v.shape)) for v in sd.values()])
        else:
            data = run_case(ref, name, CASES[name])
        path = os.path.join(GOLDEN_DIR, name + ".npz")
        np.savez_compressed(path, **data)
        print("wrote", path, {k: v.shape for k, v in data.items() if hasattr(v, "shape")} if name not in ("schedule", "manifest") else "")


if __name__ == "__main__":
    torch.set_num_threads(os.cpu_count() or 1)
    main(sys.argv[1:])
