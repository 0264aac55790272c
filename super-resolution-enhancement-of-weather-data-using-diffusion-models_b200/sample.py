"""sample.py -- same command line as the reference's sample.py:26-39 for the accelerated path:

    python sample.py -c CONFIG.json -p MODEL_PATH -o OUT_DIR -gpu 0 [-n N]
    torchrun --nproc-per-node 8 sample.py -c CONFIG.json -o OUT_DIR -gpu 0,1,2,3,4,5,6,7     # batch-sharded
    python sample.py -c CONFIG.json -o OUT_DIR --ensemble 16 [--seed S]                      # 16 members per condition
    python sample.py -c CONFIG.json -o OUT_DIR --sampler dpmpp2m --steps 20                  # 20 network calls instead of T

Builds the model through the reference's registry path (Config -> create_model -> DDPM -> define_diffusion),
``prepare_to_eval``, ``feed_data``, ``generate_sr``; writes the super-resolved fields as ``sr.npy`` (the reference's
cartopy plots, training/visualization.py, are outside the accelerated path).  ``-p`` may be omitted to sample from
random-init weights (smoke / benchmarking).

``--ensemble N`` samples N members per condition instead (``DDPM.generate_ensemble``) and writes ``ensemble.npy`` (N, B, C, H, W),
``ensemble_mean.npy`` and ``ensemble_spread.npy`` (unbiased), their ``*_physical.npy`` versions with a store, and, when the batch
carries HR, ``ensemble_scores.json`` (training.metrics.EnsembleScores; physical units with a store).  Under torchrun the MEMBERS are
sharded (rank r runs a contiguous member range) and rank 0 gathers them; the condition batch is not split.  ``--seed S`` fixes the
Philox seed (member m uses member_key(S, m); member 0 is the plain run with seed S).

``--sampler {ddpm,ddim,dpmpp2m} --steps S --eta E`` selects the reverse loop (GaussianDiffusion.set_sampler): the reference's DDPM over
all T steps (default), DDIM(eta) or DPM-Solver++(2M) over S of the T trained timesteps.  It applies to plain, sharded and ensemble runs.

``--ema`` samples from the EMA weights ``{MODEL_PATH}_ema.pth`` written by ``train.py --ema`` instead of ``{MODEL_PATH}_gen.pth``; it needs
``-p`` and combines with every other option, since it only changes the weights."""
import argparse
import os
import sys

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(_HERE))
import wsr  # noqa: E402


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("-c", "--config", type=str, required=True, help="JSON file for configuration")
    ap.add_argument("-p", "--model_path", type=str, default=None, help="Path to trained model")
    ap.add_argument("-o", "--output_path", type=str, required=True, help="Path to save output")
    ap.add_argument("-gpu", "--gpu_ids", type=str, default=None, help="GPU ids to use")
    ap.add_argument("-n", "--number_of_samples", type=int, default=1)
    ap.add_argument("-t", "--image_types", nargs="+", default=["SR"], choices=["HR", "SR", "LR", "INTERPOLATED", "DELTA", "AE"])
    ap.add_argument("-m", "--color_map", type=str, default="coolwarm", choices=["coolwarm", "heat_muted"])
    ap.add_argument("-d", "--date", type=str, default=None)
    ap.add_argument("--ensemble", type=int, default=None, help="members per condition (ensemble sampling)")
    ap.add_argument("--seed", type=int, default=None, help="Philox seed of the sampler")
    ap.add_argument("--sampler", type=str, default=None, choices=["ddpm", "ddim", "dpmpp2m"],
                    help="reverse-loop sampler (default ddpm: every timestep of the schedule)")
    ap.add_argument("--steps", type=int, default=None, help="network calls of a ddim / dpmpp2m loop (default: every timestep)")
    ap.add_argument("--eta", type=float, default=None, help="DDIM noise scale (default 0: deterministic; 1: respaced ancestral)")
    ap.add_argument("--ema", action="store_true", help="load MODEL_PATH_ema.pth (EMA weights) instead of MODEL_PATH_gen.pth")
    args = ap.parse_args(argv)
    if args.ema and not args.model_path:
        ap.error("--ema needs -p MODEL_PATH")
    return args


def sampler_options(args):
    """set_sampler's keyword arguments from the command line, or None when no sampler flag was given (the default DDPM loop)."""
    if args.sampler is None and args.steps is None and args.eta is None:
        return None
    return dict(name=args.sampler or "ddpm", steps=args.steps, eta=args.eta)


def main(argv=None):
    args = parse_args(argv)

    Config = wsr.sub("configs.config").Config
    create_model = wsr.sub("models.base_model").create_model
    data = wsr.sub("data_synthetic")
    par = wsr.sub("parallel")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if world > 1:
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        torch.distributed.init_process_group("nccl")
    opt = Config(args, experiment=False).params
    opt["phase"] = "val"
    if args.ema:
        if not os.path.exists(args.model_path + "_ema.pth"):
            raise SystemExit("sample.py --ema: no EMA weights at %s_ema.pth" % args.model_path)
        opt["path"]["resume_state"] = None                 # the EMA file is loaded in place of the gen file
    elif args.model_path:
        opt["path"]["resume_state"] = args.model_path
    elif opt["path"].get("resume_state") and not os.path.exists(str(opt["path"]["resume_state"]) + "_gen.pth"):
        opt["path"]["resume_state"] = None                # config points at the authors' machine: random-init weights
    if opt["model"].get("pretrained_model", {}).get("model_path") and not os.path.exists(opt["model"]["pretrained_model"]["model_path"]):
        opt["model"]["pretrained_model"]["model_path"] = None
    model = create_model(opt, None)
    if args.ema:
        model.load_network(args.model_path, weights="ema")
    model.prepare_to_eval()
    handler = None
    if data.is_store(str(opt["data"].get("dataroot", ""))):
        # reference sample.py:45-56,76-79: -d DATE restricts the validation range to that hour and fetches it by date
        if args.date:
            from datetime import datetime, timedelta
            fmt = "%Y-%m-%d-%H"
            opt["data"]["months_subset"] = [datetime.strptime(args.date, fmt).month]
            opt["data"]["transform_groups"] = [opt["data"]["months_subset"]]
            opt["data"]["val_min_date"] = args.date
            opt["data"]["val_max_date"] = (datetime.strptime(args.date, fmt) + timedelta(hours=1)).strftime(fmt)
        handler = data.store_handler(opt, val_only=True)
    if handler is not None and args.date:
        batch, months = handler.get_data_by_date(args.date)
    else:
        batch, months = next(iter(data.batches_from_opt(opt, "val")))
    if args.seed is not None:
        model._net().sample_seed = args.seed
    opts = sampler_options(args)
    if opts is not None:
        try:
            model._net().set_sampler(**opts)
        except ValueError as e:
            raise SystemExit("sample.py: %s" % e)
    if args.ensemble is not None:
        _ensemble(args, model, batch, months, handler, par, rank, world)
        if world > 1:
            torch.distributed.destroy_process_group()
        return
    n_total = batch["SR"].shape[0]
    if world > 1:
        batch = par.shard_batch(batch, rank, world)
    model.feed_data((batch, months))
    model.generate_sr()
    sr = model.SR
    if world > 1:
        sr = par.gather_batch(sr, n_total)
    if rank == 0:
        os.makedirs(args.output_path, exist_ok=True)
        np.save(os.path.join(args.output_path, "sr.npy"), sr.float().cpu().numpy())
        print("saved %s %s" % (os.path.join(args.output_path, "sr.npy"), tuple(sr.shape)))
        if handler is not None:
            phys = handler.get_data_transformer().inverse_transform({"SR": sr}, months[:sr.shape[0]] if len(months) >= sr.shape[0] else months)
            np.save(os.path.join(args.output_path, "sr_physical.npy"), phys["SR"].float().cpu().numpy())
    if world > 1:
        torch.distributed.destroy_process_group()


def _ensemble(args, model, batch, months, handler, par, rank, world):
    n = int(args.ensemble)
    if n < 1:
        raise SystemExit("--ensemble needs at least one member")
    lo, hi = par.shard_bounds(n, rank, world)
    model.feed_data((batch, months))
    model.generate_ensemble(hi - lo, seed=args.seed, member_offset=lo)
    ens = model.ENS
    if world > 1:
        ens = par.gather_batch(ens, n)
    if rank != 0:
        return
    import json
    out = args.output_path
    os.makedirs(out, exist_ok=True)
    spread = ens.std(0, unbiased=True) if n > 1 else torch.zeros_like(ens[0])
    arrays = {"ensemble": ens, "ensemble_mean": ens.mean(0), "ensemble_spread": spread}
    hr = batch.get("HR") if isinstance(batch, dict) else None
    target = None if hr is None else hr.to(device=ens.device, dtype=torch.float32)
    if handler is not None:
        tr = handler.get_data_transformer()
        ms = months[:ens.shape[1]] if len(months) >= ens.shape[1] else months
        phys = torch.stack([tr.inverse_transform({"SR": m}, ms)["SR"].float() for m in ens], 0)
        arrays.update({"ensemble_physical": phys, "ensemble_mean_physical": phys.mean(0),
                       "ensemble_spread_physical": phys.std(0, unbiased=True) if n > 1 else torch.zeros_like(phys[0])})
        if target is not None:
            target = tr.inverse_transform({"HR": target}, ms)["HR"].float()
            ens = phys
    for name, a in arrays.items():
        np.save(os.path.join(out, name + ".npy"), a.float().cpu().numpy())
    print("saved %s %s" % (os.path.join(out, "ensemble.npy"), tuple(arrays["ensemble"].shape)))
    if target is not None and n > 1:
        scores = wsr.sub("training.metrics").EnsembleScores(ens.device)
        scores.update(ens, target)
        with open(os.path.join(out, "ensemble_scores.json"), "w") as fh:
            json.dump(scores.compute(), fh, indent=1)


if __name__ == "__main__":
    main()
