"""Test infrastructure (NOT product code): a restatement of the parts of the reference's `Trainer` (model/runner.py)
that CALL the hot path, so that the drop-in can be exercised on the GPU box, where /root/reference does not exist
(and the build container, where it does, has no GPU - the real Trainer and the CUDA module can never meet here).

Pinned the same way as the oracle: tests/golden/make_golden.py runs the UNMODIFIED `Trainer.train_step` / `eval_step`
(with stubs for the third-party modules that are not installed: torch_ema, tensorboardX, imageio, open3d; chamfer -> a
CPU autograd restatement) on the reference model-on-shim on the CPU and stores their results together with every call
they made into the model (tests/golden/trainer_replay.npz); tests/test_trainer_dropin.py::
test_mirror_reproduces_reference_trainer replays those calls to this mirror and requires the same loss and predictions.

Restated (file:line into /root/reference):
  train_step         model/runner.py:166-377   (main loss :179-213, CD loss :215-220, flow loss :222-254)
  train iteration    model/runner.py:491-511   (zero_grad, autocast, GradScaler scale/step/update, scheduler)
  eval_step          model/runner.py:379-434
  EMA                torch_ema.ExponentialMovingAverage as used at runner.py:98-101,534-535,565-567,680
                     (update / store / copy_to / restore; copy_to and restore write `param.data.copy_`)
  checkpoints        model/runner.py:955-1073  (state keys: epoch, global_step, stats, model, optimizer, lr_scheduler,
                     scaler, ema)
  options            main_lidar4d.py:23-103 defaults
"""
from __future__ import annotations

import types

import numpy as np
import torch
import torch.nn.functional as F


def default_opt(**over):
    """The argparse defaults of main_lidar4d.py that the hot path's callers read (vars(opt) is splatted into render)."""
    o = dict(patch_size_lidar=1, raydrop_loss="mse", smooth_factor=0.2, alpha_d=1.0, alpha_i=0.1, alpha_r=0.01,
             scale=0.01, flow_loss=True, urf_loss=False, grad_loss=True, num_frames=51, num_steps=768, iters=30000,
             lr=1e-2, fp16=True, ema_decay=0.95, num_rays_lidar=1024, bound=1, near_lidar=1.0, far_lidar=81.0,
             sobel_grad=False, grad_norm_smooth=False, spatial_smooth=False, tv_loss=False, density_scale=1)
    o.update(over)
    return types.SimpleNamespace(**o)


def default_criterion():
    """main_lidar4d.py:185-207 with the default loss names (l1 depth, mse intensity / raydrop), reduction='none'."""
    return {"depth": torch.nn.L1Loss(reduction="none"), "raydrop": torch.nn.MSELoss(reduction="none"),
            "intensity": torch.nn.MSELoss(reduction="none"), "grad": torch.nn.L1Loss(reduction="none")}


class MirrorEMA:
    """torch_ema.ExponentialMovingAverage (decay, no num_updates warm-up when use_num_updates... the reference passes
    only `decay`, torch_ema's default use_num_updates=True): shadow = shadow - (1 - d) * (shadow - param),
    d = min(decay, (1 + n) / (10 + n))."""

    def __init__(self, parameters, decay):
        self.params = [p for p in parameters if p.requires_grad]
        self.decay, self.num_updates = decay, 0
        self.shadow = [p.detach().clone() for p in self.params]
        self.collected = None

    @torch.no_grad()
    def update(self):
        self.num_updates += 1
        d = min(self.decay, (1 + self.num_updates) / (10 + self.num_updates))
        for s, p in zip(self.shadow, self.params):
            s.sub_((1.0 - d) * (s - p))

    def store(self):
        self.collected = [p.detach().clone() for p in self.params]

    def copy_to(self):
        for s, p in zip(self.shadow, self.params):
            p.data.copy_(s.data)                      # what torch_ema does: no autograd version bump

    def restore(self):
        for c, p in zip(self.collected, self.params):
            p.data.copy_(c.data)
        self.collected = None

    def state_dict(self):
        return {"decay": self.decay, "num_updates": self.num_updates, "shadow_params": self.shadow}

    def load_state_dict(self, sd):
        self.decay, self.num_updates = sd["decay"], sd["num_updates"]
        self.shadow = [s.to(p.device) for s, p in zip(sd["shadow_params"], self.params)]


class MirrorTrainer:
    def __init__(self, opt, model, cham_fn, criterion=None, optimizer=None, lr_scheduler=None, ema_decay=None, fp16=False,
                 device=None, pc_list=None, pc_ground_list=None):
        self.opt, self.model, self.cham_fn = opt, model, cham_fn
        self.criterion = criterion or default_criterion()
        self.device = device or next(model.parameters()).device
        self.optimizer = optimizer(model) if optimizer is not None else None
        self.lr_scheduler = lr_scheduler(self.optimizer) if lr_scheduler is not None else None
        self.ema = MirrorEMA(model.parameters(), ema_decay) if ema_decay is not None else None
        self.fp16 = fp16
        self.scaler = torch.amp.GradScaler(self.device.type, enabled=fp16)
        self.pc_list, self.pc_ground_list = pc_list or {}, pc_ground_list or {}
        self.epoch, self.global_step, self.stats = 0, 0, {"loss": []}
        self.use_refine = False

    # ---- runner.py:166-254 ----------------------------------------------------------------------------------------
    def train_step(self, data):
        o = self.opt
        rays_o, rays_d, t, images = data["rays_o_lidar"], data["rays_d_lidar"], data["time"], data["images_lidar"]
        gt_raydrop = images[:, :, 0]
        gt_intensity = images[:, :, 1] * gt_raydrop
        gt_depth = images[:, :, 2] * gt_raydrop
        out = self.model.render(rays_o, rays_d, t, staged=False, perturb=True,
                                force_all_rays=False if o.patch_size_lidar == 1 else True, **vars(o))
        pred_raydrop = out["image_lidar"][:, :, 0]
        pred_intensity = out["image_lidar"][:, :, 1] * gt_raydrop
        pred_depth = out["depth_lidar"] * gt_raydrop
        if o.raydrop_loss == "bce":
            pred_raydrop = torch.sigmoid(pred_raydrop)
        gt_raydrop_smooth = gt_raydrop.clamp(o.smooth_factor, 1 - o.smooth_factor)
        lidar_loss = (o.alpha_d * self.criterion["depth"](pred_depth, gt_depth)
                      + o.alpha_r * self.criterion["raydrop"](pred_raydrop, gt_raydrop_smooth)
                      + o.alpha_i * self.criterion["intensity"](pred_intensity, gt_intensity))
        loss = lidar_loss.sum()
        pred_lidar = rays_d * pred_depth.unsqueeze(-1) / o.scale
        gt_lidar = rays_d * gt_depth.unsqueeze(-1) / o.scale
        d1, d2, _, _ = self.cham_fn(pred_lidar, gt_lidar)
        loss = loss + (d1 + d2).mean() * 0.5
        if o.flow_loss:
            frame_idx = int(t * (o.num_frames - 1))
            dev = rays_o.device
            pc = torch.from_numpy(self.pc_list[f"{frame_idx}"]).to(dev).float().contiguous()
            fl = self.model.flow(pc, t)
            for step in (1, 2):
                for sign, key in ((+1, "forward"), (-1, "backward")):
                    k = f"{frame_idx + sign * step}"
                    if k in self.pc_list:
                        pc_pred = pc + fl[key] * step
                        other = torch.from_numpy(self.pc_list[k]).to(dev).float().contiguous()
                        d1, d2, _, _ = self.cham_fn(pc_pred.unsqueeze(0), other.unsqueeze(0))
                        loss = loss + (d1.sum() + d2.sum()) * 0.5
            ground = torch.from_numpy(self.pc_ground_list[f"{frame_idx}"]).to(dev).float().contiguous()
            zero_flow = self.model.flow(ground, torch.rand(1).to(t))
            loss = loss + 0.001 * (zero_flow["forward"].abs().sum() + zero_flow["backward"].abs().sum())
        return pred_intensity.unsqueeze(-1), gt_intensity.unsqueeze(-1), pred_depth, gt_depth, loss

    # ---- runner.py:491-511,534-535 ------------------------------------------------------------------------------------
    def train_iteration(self, data):
        self.global_step += 1
        self.optimizer.zero_grad()
        with torch.autocast(self.device.type, dtype=torch.float16, enabled=self.fp16):
            *_, loss = self.train_step(data)
        self.scaler.scale(loss).backward()
        self.scaler.step(self.optimizer)
        self.scaler.update()
        if self.lr_scheduler is not None:
            self.lr_scheduler.step()
        return float(loss.item())

    def end_epoch(self):
        self.epoch += 1
        if self.ema is not None:
            self.ema.update()

    # ---- runner.py:379-434 ---------------------------------------------------------------------------------------------
    def eval_step(self, data):
        o = self.opt
        images = data["images_lidar"]
        H, W = data["H_lidar"], data["W_lidar"]
        gt_raydrop = images[:, :, :, 0]
        gt_intensity = images[:, :, :, 1] * gt_raydrop
        gt_depth = images[:, :, :, 2] * gt_raydrop
        out = self.model.render(data["rays_o_lidar"], data["rays_d_lidar"], data["time"], staged=True, perturb=False, **vars(o))
        pred = out["image_lidar"].reshape(-1, H, W, 2)
        pred_raydrop, pred_intensity = pred[:, :, :, 0], pred[:, :, :, 1]
        pred_depth = out["depth_lidar"].reshape(-1, H, W)
        if self.use_refine:
            x = torch.cat([pred_raydrop, pred_intensity, pred_depth], dim=0).unsqueeze(0)
            pred_raydrop = self.model.unet(x).squeeze(0)
        mask = torch.where(pred_raydrop > 0.5, 1, 0)
        loss = (o.alpha_d * self.criterion["depth"](pred_depth * mask, gt_depth).mean()
                + o.alpha_r * self.criterion["raydrop"](pred_raydrop, gt_raydrop).mean()
                + o.alpha_i * self.criterion["intensity"](pred_intensity * mask, gt_intensity).mean())
        return pred_intensity, pred_depth, pred_raydrop, gt_intensity, gt_depth, gt_raydrop, loss

    def evaluate(self, data):
        """runner.py:563-567,680: eval() -> ema.store()/copy_to() -> eval steps under no_grad -> ema.restore()."""
        self.model.eval()
        if self.ema is not None:
            self.ema.store()
            self.ema.copy_to()
        with torch.no_grad(), torch.autocast(self.device.type, dtype=torch.float16, enabled=self.fp16):
            res = self.eval_step(data)
        if self.ema is not None:
            self.ema.restore()
        self.model.train()
        return res

    # ---- runner.py:955-1073 --------------------------------------------------------------------------------------------
    def checkpoint(self):
        state = {"epoch": self.epoch, "global_step": self.global_step, "stats": self.stats,
                 "optimizer": self.optimizer.state_dict(), "scaler": self.scaler.state_dict(), "model": self.model.state_dict()}
        if self.lr_scheduler is not None:
            state["lr_scheduler"] = self.lr_scheduler.state_dict()
        if self.ema is not None:
            state["ema"] = self.ema.state_dict()
        return state

    def load_checkpoint(self, state):
        res = self.model.load_state_dict(state["model"], strict=False)
        if self.ema is not None and "ema" in state:
            self.ema.load_state_dict(state["ema"])
        self.epoch, self.global_step, self.stats = state["epoch"], state["global_step"], state["stats"]
        self.optimizer.load_state_dict(state["optimizer"])
        if self.lr_scheduler is not None and "lr_scheduler" in state:
            self.lr_scheduler.load_state_dict(state["lr_scheduler"])
        self.scaler.load_state_dict(state["scaler"])
        return res


def synthetic_batch(n_rays, frame=7, num_frames=51, seed=0, device="cpu", H=8, W=32):
    """A training batch / an eval image with the dataset's keys (kitti360_dataset.py:152-189): rays from the sensor
    model, GT image channels (raydrop, intensity, depth) synthetic."""
    from lidar4d_b200.rays import lidar_rays
    g = np.random.default_rng(seed)
    pose = np.eye(4, dtype=np.float32)
    pose[:3, 3] = [-0.25 + 0.5 * frame / (num_frames - 1), 0.0, 0.0]
    ro, rd = lidar_rays(pose, H, W)
    t = torch.tensor([[frame / (num_frames - 1)]], dtype=torch.float32, device=device)
    img = np.stack([(g.random(H * W) > 0.15).astype(np.float32), g.random(H * W).astype(np.float32) * 0.5,
                    (0.05 + 0.6 * g.random(H * W)).astype(np.float32)], -1)
    sel = g.choice(H * W, n_rays, replace=False)
    train = {"rays_o_lidar": torch.from_numpy(ro[sel])[None].to(device), "rays_d_lidar": torch.from_numpy(rd[sel])[None].to(device),
             "time": t, "images_lidar": torch.from_numpy(img[sel])[None].to(device)}
    ev = {"rays_o_lidar": torch.from_numpy(ro)[None].to(device), "rays_d_lidar": torch.from_numpy(rd)[None].to(device),
          "time": t, "images_lidar": torch.from_numpy(img.reshape(1, H, W, 3)).to(device), "H_lidar": H, "W_lidar": W}
    pcs = {str(k): (g.random((300 + 20 * k, 3)).astype(np.float32) * 1.6 - 0.8) for k in range(frame - 2, frame + 3)}
    ground = {str(frame): (g.random((150, 3)).astype(np.float32) * 1.6 - 0.8)}
    return train, ev, pcs, ground
