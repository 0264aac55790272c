"""DDPM facade -- drop-in for the reference's models/diffusion_models/model.py:13-252 (same methods, same checkpoint
file names and contents: ``I{iter}_E{epoch}_gen.pth`` = netG.state_dict() on CPU, ``..._opt.pth`` = optimizer state)."""
import logging
import os
from collections import OrderedDict

import torch
import torch.nn as nn

from ..base_model import BaseModel
from . import networks

logger = logging.getLogger('base')


class DDPM(BaseModel):
    def __init__(self, opt):
        super().__init__(opt)
        if self.device.type != "cuda":
            raise RuntimeError("the B200-native path needs a CUDA device and '-gpu <ids>' (no CPU fallback); "
                               "the reference's quirk 'no -gpu flag => CPU' (config.py:65, base_model.py:17) does not apply")
        self.netG = self.set_device(networks.define_diffusion(opt))
        self.schedule_phase = None
        self.months = []
        self.set_loss()
        self.set_new_noise_schedule(opt['model']['beta_schedule']['train'], schedule_phase='train')
        if self.opt['phase'] == 'train':
            self.netG.train()
            if opt['model']['finetune_norm']:
                optim_params = []
                for k, v in self.netG.named_parameters():
                    v.requires_grad = False
                    if k.find('transformer') >= 0:
                        v.requires_grad = True
                        v.data.zero_()
                        optim_params.append(v)
            else:
                optim_params = list(self.netG.parameters())
            # torch.optim.Adam semantics and state layout, update done by wsr_adam_step (reference model.py:43-44)
            from ...autograd_glue import FusedAdam
            self.optG = FusedAdam(optim_params, lr=opt['train']["optimizer"]["lr"])
            self.log_dict = OrderedDict()
        self.load_network()
        self.print_network()

    def _net(self):
        return self.netG.module if isinstance(self.netG, nn.DataParallel) else self.netG

    def feed_data(self, data: tuple) -> None:
        self.data, self.months = self.set_device(data[0]), data[1]

    def optimize_parameters(self):
        """reference :61-69: zero_grad, loss / numel, backward, Adam step.  Under ``torch.distributed`` (one process per
        GPU) every rank holds a shard of the batch: the loss is divided by the GLOBAL element count and the gradients are
        SUM-all-reduced in buckets while the backward pass is still running (parallel.FlatGradReducer)."""
        import torch.distributed as dist
        world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        b, c, h, w = self.data['HR'].shape
        self._attach_flat(b)
        self.optG.zero_grad()
        reducer = self._grad_reducer(b) if world > 1 else None
        l_pix = self.netG(self.data)
        l_pix = l_pix.sum() / int(b * c * h * w * world)
        l_pix.backward()
        if reducer is not None:
            reducer.finish()
            self._reduce_outside_plan(reducer)
        self.optG.step()
        l_pix = l_pix.detach().clone()
        if world > 1:
            dist.all_reduce(l_pix)
        # the reference stores l_pix.item() here (model.py:69); the device->host read is deferred to get_current_log() so
        # that the launch queue is not drained after every optimizer step
        self.log_dict['l_pix'] = l_pix

    def _reduce_outside_plan(self, reducer):
        """Gradients of trainable parameters that are not part of the denoiser's flat buffer (a jointly trained RRDB encoder,
        ``lock_weights=False``): one coalesced SUM all-reduce after the backward pass."""
        import torch.distributed as dist
        in_plan = {id(p) for p in reducer.plan.param_order} if hasattr(reducer, "plan") else set()
        rest = [p for p in self._net().parameters() if p.requires_grad and p.grad is not None and id(p) not in in_plan]
        if not rest:
            return
        flat = torch.cat([p.grad.reshape(-1) for p in rest])
        dist.all_reduce(flat)
        off = 0
        for p in rest:
            p.grad.copy_(flat[off:off + p.numel()].view_as(p.grad))
            off += p.numel()

    def _attach_flat(self, batch):
        """The denoiser's parameters are flattened into the train plan's single buffer on the first step (after load_network), so
        that the optimizer update is ONE ``wsr_adam_step`` launch instead of one per parameter; a loaded optimizer state is
        carried over (FusedAdam.attach_flat)."""
        if getattr(self, "_flat_batch", None) == batch or self.opt['model']['finetune_norm']:
            return
        net = self._net().denoise_fn
        if not hasattr(net, "train_plan"):
            return
        self.optG.attach_flat(net.train_plan(batch, self.device))
        self._flat_batch = batch

    def _grad_reducer(self, batch):
        """FlatGradReducer bound to the denoiser's train plan for this local batch size (created once)."""
        from ...parallel import FlatGradReducer
        net = self._net().denoise_fn
        plan = net.train_plan(batch, self.device)
        red = getattr(plan, "_reducer", None)
        if red is None:
            red = plan._reducer = FlatGradReducer(plan)
        return red

    def generate_sr(self, continous=False):
        self.netG.eval()
        with torch.no_grad():
            self.SR = self._net().super_resolution(self.data, continous)
            self.SR = self.SR.unsqueeze(0) if len(self.SR.size()) == 3 else self.SR
        self.netG.train()

    def generate_ensemble(self, n_members, seed=None, member_offset=0):
        """self.ENS = (n_members, B, C, H, W): members member_offset .. member_offset + n_members - 1 of the ensemble of ``seed``
        for the fed batch (GaussianDiffusion.super_resolution_ensemble).  SR is left untouched."""
        self.netG.eval()
        with torch.no_grad():
            self.ENS = self._net().super_resolution_ensemble(self.data, n_members, seed=seed, member_offset=member_offset)
        self.netG.train()

    def sample(self, batch_size=1, continous=False):
        self.netG.eval()
        with torch.no_grad():
            self.SR = self._net().sample(batch_size, continous)
        self.netG.train()

    def set_loss(self):
        self._net().set_loss(self.device)

    def set_new_noise_schedule(self, schedule_opt, schedule_phase='train'):
        if self.schedule_phase is None or self.schedule_phase != schedule_phase:
            self.schedule_phase = schedule_phase
            self._net().set_new_noise_schedule(schedule_opt, self.device)

    def get_current_log(self):
        for k, v in list(self.log_dict.items()):
            if torch.is_tensor(v):
                self.log_dict[k] = v.item()
        return self.log_dict

    def get_images(self, need_LR=True, sample=False):
        out = OrderedDict()
        if sample:
            out['SAM'] = self.SR.detach().float().cpu()
        else:
            out['SR'] = self.SR.detach().float().cpu()
            out['INF'] = self.data['SR'].detach().float().cpu()
            out['HR'] = self.data['HR'].detach().float().cpu()
            if need_LR and 'LR' in self.data:
                out['LR'] = self.data['LR'].detach().float().cpu()
            else:
                out['LR'] = out['INF']
        return out

    def print_network(self):
        s, n = self.get_network_description(self.netG)
        logger.info('Network G structure: {}, with parameters: {:,d}'.format(self._net().__class__.__name__, n))
        logger.info(s)

    def save_network(self, epoch, iter_step):
        gen_path = os.path.join(self.opt['path']['checkpoint'], 'I{}_E{}_gen.pth'.format(iter_step, epoch))
        opt_path = os.path.join(self.opt['path']['checkpoint'], 'I{}_E{}_opt.pth'.format(iter_step, epoch))
        state = {k: v.cpu() for k, v in self._net().state_dict().items()}
        torch.save(state, gen_path)
        torch.save({'epoch': epoch, 'iter': iter_step, 'scheduler': None, 'optimizer': self.optG.state_dict()}, opt_path)
        logger.info('Saved model in [{:s}] ...'.format(gen_path))

    def load_network(self):
        load_path = self.opt['path']['resume_state']
        if load_path is None:
            return
        logger.info('Loading pretrained model for G [{:s}] ...'.format(load_path))
        self._net().load_state_dict(torch.load('{}_gen.pth'.format(load_path), map_location=self.device),
                                    strict=(not self.opt['model']['finetune_norm']))
        if self.opt['phase'] == 'train':
            # optimizer state: moments go to the device with load_state_dict; the per-parameter step counters stay on the host
            o = torch.load('{}_opt.pth'.format(load_path), map_location='cpu')
            self.optG.load_state_dict(o['optimizer'])
            self.begin_step = o['iter']
            self.begin_epoch = o['epoch']

    def prepare_to_train(self) -> None:
        self.set_new_noise_schedule(self.opt['model']['beta_schedule']['train'], schedule_phase='train')

    def prepare_to_eval(self) -> None:
        self.set_new_noise_schedule(self.opt['model']['beta_schedule']['val'], schedule_phase='val')

    def get_months(self) -> list:
        return self.months

    def get_loaded_iter(self):
        return self.begin_step

    def get_loaded_epoch(self):
        return self.begin_epoch
