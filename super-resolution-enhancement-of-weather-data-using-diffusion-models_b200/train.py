"""train.py -- same command line as the reference's train.py:208-212 (``-c CONFIG -p {train,val} -gpu IDS``).

``-p val`` runs the validation loop (generate_sr per batch, MSE / RMSE / MAE / MR on device accumulators) on the CUDA path.
``-p train`` builds the optimiser and runs ``optimize_parameters`` (forward, hand-written backward, fused Adam).  Under
``torchrun`` (one process per GPU) the batch is sharded across ranks and the gradients are all-reduced in buckets
overlapped with the backward pass (parallel.FlatGradReducer); weights start identical on every rank (same seed).

``--ema`` keeps an exponential moving average of the weights on the schedule of the config's ``train.ema_scheduler``
(autograd_glue.ema_action), updated inside the Adam launch, saved as ``I{iter}_E{epoch}_ema.pth`` beside the gen / opt files at
every checkpoint, and used for the in-loop validation.  ``-p val --ema`` validates ``{resume_state}_ema.pth`` instead of the gen
file.  Every rank keeps its own EMA (the replicas are identical after the all-reduce); rank 0 writes the file.

``-p val --scores FILE`` also scores the whole validation loader with training.metrics.FieldScores (zonal power spectra per latitude
band, cos(latitude)-weighted and unweighted errors) for the model output and, as the baseline, the bicubic condition ``SR``, both
against HR, and writes them to FILE as JSON (sections ``model`` and ``bicubic``).  With a store the scores are in physical units (the
fitted mean and std of each sample's month); otherwise they are in standardised units (``units`` says which).  Under torchrun rank 0
writes the file."""
import argparse
import logging
import os
import sys

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(_HERE))
import wsr  # noqa: E402


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("-c", "--config", type=str, help="JSON file for configuration")
    ap.add_argument("-p", "--phase", type=str, choices=["train", "val"], default="train")
    ap.add_argument("-gpu", "--gpu_ids", type=str, default=None)
    ap.add_argument("--ema", action="store_true", help="train / validate EMA weights (config train.ema_scheduler)")
    ap.add_argument("--scores", type=str, default=None, metavar="FILE",
                    help="-p val: write spectral and latitude-weighted scores of the model and the bicubic baseline to FILE (JSON)")
    args = ap.parse_args(argv)
    if args.scores and args.phase != "val":
        ap.error("--scores needs -p val")
    return args


def main(argv=None):
    args = parse_args(argv)
    logging.basicConfig(level=logging.INFO)
    log = logging.getLogger("base")

    Config = wsr.sub("configs.config").Config
    create_model = wsr.sub("models.base_model").create_model
    data = wsr.sub("data_synthetic")
    import numpy as np
    import random
    random.seed(0); np.random.seed(0); torch.manual_seed(0)                 # training/utils.py:39-50
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
        dist.init_process_group("nccl")
        args.gpu_ids = os.environ.get("LOCAL_RANK", "0")
    opt = Config(args, experiment=True).params
    ema_schedule, ema_path = None, None
    if args.ema and args.phase == "train":
        try:
            ema_schedule = wsr.sub("autograd_glue").check_ema_schedule(opt["train"].get("ema_scheduler"))
        except ValueError as e:
            raise SystemExit("train.py --ema: %s" % e)
    if args.ema and args.phase == "val":
        ema_path = opt["path"].get("resume_state")
        if not ema_path or not os.path.exists(str(ema_path) + "_ema.pth"):
            raise SystemExit("train.py -p val --ema: no EMA weights at %s_ema.pth (path.resume_state)" % ema_path)
        opt["path"]["resume_state"] = None                 # the EMA file is loaded in place of the gen file
    for key in ("resume_state",):
        if opt["path"].get(key) and not os.path.exists(str(opt["path"][key]) + "_gen.pth"):
            opt["path"][key] = None
    pm = opt["model"].get("pretrained_model", {})
    if pm.get("model_path") and not os.path.exists(pm["model_path"]):
        pm["model_path"] = None
    model = create_model(opt, None)
    if ema_path is not None:
        model.load_network(ema_path, weights="ema")
    if ema_schedule is not None:
        model.enable_ema(ema_schedule)
    if world > 1:
        # weights were initialised under seed 0 on every rank (identical replicas); from here on each rank must draw its OWN
        # timestep, noise levels, noise and dropout masks (the reference's single process draws them once for the whole batch)
        random.seed(rank); np.random.seed(rank); torch.manual_seed(rank); torch.cuda.manual_seed(rank)
    if args.phase == "val":
        return validate(model, opt, data, log, scores_path=args.scores)
    # reference train.py:55-123: resume from the loaded iteration / epoch, stop at n_iter, validate every val_freq iterations,
    # checkpoints named by the REAL epoch and iteration
    curr_iter, curr_epoch = int(model.get_loaded_iter() or 0), int(model.get_loaded_epoch() or 0)
    n_iter = int(opt["train"]["n_iter"])
    val_freq = int(opt["train"].get("val_freq") or 0)
    full_val_freq = int(opt["train"].get("full_val_freq") or 0)
    par = wsr.sub("parallel")
    from_store = data.is_store(str(opt["data"].get("dataroot", "")))
    shard = (rank, world) if (world > 1 and from_store) else None        # the store loader reads only this rank's slice
    if curr_iter:
        log.info("resuming at iteration %d, epoch %d", curr_iter, curr_epoch)
    while curr_iter < n_iter:
        curr_epoch += 1
        served = 0
        for batch, months in data.epoch_batches(opt, n_iter - curr_iter, shard=shard):
            curr_iter += 1
            served += 1
            if world > 1 and shard is None:
                batch = par.shard_batch(batch, rank, world)
            model.feed_data((batch, months))
            model.optimize_parameters()
            if curr_iter % opt["train"]["print_freq"] == 0:
                log.info("epoch %d  iter %d  l_pix %.6f", curr_epoch, curr_iter, model.get_current_log()["l_pix"])
            if val_freq and curr_iter % val_freq == 0:
                # train.py:79-117: the first validation batch only, the whole loader every full_val_freq iterations
                model.prepare_to_eval()
                full = bool(full_val_freq) and curr_iter % full_val_freq == 0
                if ema_schedule is None:
                    validate(model, opt, data, log, max_batches=None if full else 1)
                else:
                    log.info("validation with the EMA weights")
                    with model.ema_weights():
                        validate(model, opt, data, log, max_batches=None if full else 1)
                model.prepare_to_train()
            if curr_iter % opt["train"]["save_checkpoint_freq"] == 0 and rank == 0:
                model.save_network(curr_epoch, curr_iter)
        if served == 0:
            break
    log.info("End of training.")
    return curr_iter, curr_epoch


def validate(model, opt, data, log, max_batches=None, scores_path=None):
    """reference train.py:132-196 (validate): generate_sr per batch, inverse transform, metric accumulators -- here the
    accumulators live on the device (training/metrics.py) and the inverse StandardScaling is folded into the same pass
    as a per-(sample, variable) scale, so nothing is copied to the host until the final compute.  ``scores_path``: also
    accumulate FieldScores of the model output and of the bicubic condition and write them there (rank 0)."""
    model.prepare_to_eval()
    metrics = wsr.sub("training.metrics")
    vm = metrics.ValidationMetrics(metrics.create_metric_dict(model.device))
    vm_k = metrics.ValidationMetrics(metrics.create_metric_dict(model.device))
    sigma_k = float(opt["data"].get("sigma_kelvin", 21.26))          # WeatherBench t2m std (synthetic data has no fitted transform)
    handler = data.store_handler(opt)                                # the reference's on-disk store, when dataroot is one
    fields, lat_source = None, None
    for i, (batch, months) in enumerate(data.batches_from_opt(opt, "val")):
        if max_batches is not None and i >= max_batches:
            break
        model.feed_data((batch, months))
        model.generate_sr(False)
        sr, hr = model.SR, model.data["HR"]
        vm.update(sr, hr)
        mean = std = None
        if handler is not None:
            # physical units = fitted std of each sample's month and variable (train.py:96-99 inverse_transform, folded in)
            mean, std = handler.get_data_transformer().batch_statistics("hr", months)
            vm_k.update(sr, hr, scale=std.reshape(-1))
        else:
            vm_k.update(sr, hr, scale=torch.full((sr.shape[0] * sr.shape[1],), sigma_k))
        if scores_path:
            if fields is None:
                variable = (opt["data"].get("variables") or [None])[0]
                lat, lat_source = metrics.field_latitudes(opt["data"].get("dataroot"), variable, hr.shape[2])
                lr_width = model.data["LR"].shape[-1] if "LR" in model.data else None
                fields = {name: metrics.FieldScores(model.device, lat, lr_width) for name in ("model", "bicubic")}
            fields["model"].update(sr, hr, std, mean)
            fields["bicubic"].update(model.data["SR"], hr, std, mean)      # the bicubic condition (the reference's INTERPOLATED)
    vm.compute_metrics(); vm_k.compute_metrics()
    log.info("validation (standardised units)%s", vm.metrics2str())
    if handler is not None:
        log.info("validation (physical units, fitted statistics)%s", vm_k.metrics2str())
    else:
        log.info("validation (x sigma = %.2f K)%s", sigma_k, vm_k.metrics2str())
    if fields is not None and int(os.environ.get("RANK", "0")) == 0:
        metrics.write_field_scores(scores_path, fields, "physical" if handler is not None else "standardised", lat_source,
                                   opt["data"].get("variables"))
        log.info("spectral and latitude-weighted scores written to %s", scores_path)
    return vm.metrics2dict(), vm_k.metrics2dict()


if __name__ == "__main__":
    main()
