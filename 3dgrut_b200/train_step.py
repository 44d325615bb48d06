"""Thin view-parallel training step for the SH Gaussian model on the 3DGUT path (SURVEY.md section 8f row 1, without densification).

Replaces the render + backward + optimizer part of Trainer.run_train_iter (threedgrut/trainer.py:1119-1263) with the pieces of this
repository wired together -- no autograd graph, no per-parameter all-reduce, no separate activation backward:

    activations (sigmoid / exp / normalize, model.py:102-118)  ->  SplatRaster.trace
    -> loss gradient on the image (L1, trainer.py:698-704 + losses.py:20-21)  ->  SplatRaster.trace_bwd_compact
    -> CompactGradientExchange (all-reduce [N,12], all-gather [N,4], rebuild [N,48])  ->  FusedGaussianAdam.step
       (+ the opacity / scale regularisers of trainer.py:722-739, whose gradients the optimizer's launch adds once per step)

Every rank holds a replica of the parameters and renders its own camera of the step's batch; the loss is normalised by the global
batch (number of ranks), so the replicas stay identical.  The trainer, datasets, densification and logging of the reference stay out
of scope; this class exists so that the path can be run -- and tested -- as the training loop uses it."""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

import optimizers
import view_parallel
from threedgut_tracer.tracer import SplatRaster, _cfg_get


def loss_weights_from_conf(conf):
    """(lambda_l1, lambda_ssim, lambda_opacity, lambda_scale) from the reference's `loss` section (configs/base_gs.yaml:171-185;
    configs/base_mcmc.yaml turns on opacity and scale at 0.01 each).  A weight counts only when its use_* flag is true; missing keys take
    base_gs.yaml's values.  conf: a dict or an attribute-style config such as an OmegaConf object."""
    defaults = {"l1": (True, 0.8), "ssim": (True, 0.2), "opacity": (False, 0.0), "scale": (False, 0.0)}
    out = []
    for term, (use, weight) in defaults.items():
        on = bool(_cfg_get(conf, f"loss.use_{term}", use))
        out.append(float(_cfg_get(conf, f"loss.lambda_{term}", weight)) if on else 0.0)
    return tuple(out)


class GaussianTrainStep:
    def __init__(self, params: dict, lrs: dict, conf=None, sph_degree: int = 3, selective: bool = False, group=None, eps: float = 1e-15,
                 densify_conf=None, scene_extent: float = 1.0, lambda_l1: float = 1.0, lambda_ssim: float = 0.0, lambda_opacity: float = 0.0,
                 lambda_scale: float = 0.0):
        """params: raw leaf tensors for optimizers.GROUPS (positions, density, rotation, scale, features_albedo, features_specular).
        densify_conf: a densify.DensifyConfig (GS strategy: clone / split / prune / reset) or densify.MCMCConfig (relocate / add / perturb)
        turns on the replica-consistent strategy.  lambda_*: the reference's loss weights (loss_weights_from_conf maps its config)."""
        self.params = {k: params[k] for k in optimizers.GROUPS}  # ONE dict shared with the optimizer and the densifier
        self.device = self.params["positions"].device
        self.sph_degree = int(sph_degree)
        self.group = group
        self.world = dist.get_world_size(group) if dist.is_available() and dist.is_initialized() else 1
        self.raster = SplatRaster(conf if conf is not None else {"render": {}})
        self.optimizer = optimizers.FusedGaussianAdam(self.params, lrs, eps=eps, selective=selective)
        self.exchange = view_parallel.CompactGradientExchange(self.raster, self.n, self.device, group=group)
        self.frame = 0
        self.lambda_l1, self.lambda_ssim = float(lambda_l1), float(lambda_ssim)  # reference defaults: 0.8 / 0.2 (configs/base_gs.yaml:172-179)
        # reference's MCMC recipe: 0.01 / 0.01 (configs/base_mcmc.yaml:13-18); off in base_gs.yaml
        self.lambda_opacity, self.lambda_scale = float(lambda_opacity), float(lambda_scale)
        self._regularised = self.lambda_opacity != 0.0 or self.lambda_scale != 0.0
        self._reg_loss = torch.zeros(2, dtype=torch.float32, device=self.device)  # (mean sigmoid(density), mean exp(scale)), written by the step
        self._zero = torch.zeros((), dtype=torch.float32, device=self.device)
        self.last_losses = {}
        self.scene_extent = float(scene_extent)
        self.densifier = None
        if densify_conf is not None:
            import densify

            cls = densify.MCMCDensifier if isinstance(densify_conf, densify.MCMCConfig) else densify.GSDensifier
            self.densifier = cls(self.params, [self.optimizer.exp_avg, self.optimizer.exp_avg_sq], densify_conf, group=group)

    @property
    def n(self) -> int:
        return int(self.params["positions"].shape[0])

    @torch.no_grad()
    def activated(self):
        """[N,12] = pos3, sigmoid(density), normalize(rotation) (wxyz), exp(scale), 0 and [N,48] = cat(albedo, specular)
        (threedgut_tracer/tracer.py:176-178, model.py:94-118)"""
        p = self.params
        particles = torch.cat([p["positions"], torch.sigmoid(p["density"]), torch.nn.functional.normalize(p["rotation"]), torch.exp(p["scale"]),
                               torch.zeros_like(p["density"])], dim=1).contiguous()
        sph = torch.cat([p["features_albedo"], p["features_specular"]], dim=1).contiguous()
        return particles, sph

    @torch.no_grad()
    def render(self, rays_o, rays_d, sensor, pose):
        particles, sph = self.activated()
        rgba, dist_, hits, vis = self.raster.trace(self.frame, self.sph_degree, particles, sph, rays_o, rays_d, None, sensor, 0, 1, pose, pose)
        return rgba, dist_, hits, vis

    @torch.no_grad()
    def step(self, rays_o, rays_d, sensor, pose, target_rgb, all_sensor_positions=None):
        """One optimisation step on this rank's view.  target_rgb: [H,W,3].  all_sensor_positions: [world,3] sensor positions of every
        rank's view of this step in rank order (omit on a single GPU).  Returns this view's loss (a device scalar): the image loss, plus
        lambda_opacity mean sigmoid(density) + lambda_scale mean exp(scale) of the parameters before the update when those weights are
        set (the reference's total_loss).  last_losses holds the weighted terms under the reference's keys."""
        H, W = int(rays_o.shape[1]), int(rays_o.shape[2])
        particles, sph = self.activated()
        rgba, dst, hits, vis = self.raster.trace(self.frame, self.sph_degree, particles, sph, rays_o, rays_d, None, sensor, 0, 1, pose, pose)
        if self.lambda_ssim != 0.0:
            import losses

            # lambda_l1 L1 + lambda_ssim (1 - SSIM) and its image gradient in two launches (gut_loss.cu); global-batch normalisation
            loss, l1, ssim, d_rgba = losses.image_loss(rgba, target_rgb.contiguous(), self.lambda_l1 / self.world, self.lambda_ssim / self.world)
            loss = loss * self.world
            l1_loss, ssim_loss = self.lambda_l1 * l1, self.lambda_ssim * (1.0 - ssim)
        else:
            diff = rgba[..., :3] - target_rgb
            loss = self.lambda_l1 * diff.abs().mean()
            l1_loss, ssim_loss = loss, self._zero
            d_rgba = torch.zeros_like(rgba)
            d_rgba[..., :3] = self.lambda_l1 * torch.sign(diff) / (diff.numel() * self.world)  # d mean|.| / d rgb, global-batch normalisation
        d_dist = torch.zeros_like(dst)
        self.raster.trace_bwd_compact(self.frame, self.sph_degree, particles, sph, rays_o, rays_d, None, sensor, 0, 1, pose, pose, rgba, d_rgba,
                                      dst, d_dist, out=self.exchange.out())
        my_position = self.raster.sensor_position(sensor, pose, pose, W, H)
        if all_sensor_positions is None:
            if self.world != 1:
                raise RuntimeError("all_sensor_positions is required when more than one rank trains")
            all_sensor_positions = my_position[None]
        if self.densifier is not None:
            # this view's own position gradient, before the exchange (it is weighted by the distance to THIS view's sensor, gs.py:127-137);
            # x world undoes the global-batch normalisation so that the thresholds keep their per-view meaning
            self.densifier.update_gradient_buffer(self.exchange.d_particles[:, 0:3] * float(self.world), my_position)
        d_particles, d_sph = self.exchange.exchange(self.sph_degree, particles, np.asarray(all_sensor_positions, np.float32))
        if self.optimizer.selective and self.world > 1:
            dist.all_reduce(vis, op=dist.ReduceOp.MAX, group=self.group)  # visible in any view of the batch (SURVEY 8e)
        opacity_loss = scale_loss = self._zero
        if self._regularised:
            self.optimizer.step(d_particles, d_sph, visibility=vis if self.optimizer.selective else None, lambda_opacity=self.lambda_opacity,
                                lambda_scale=self.lambda_scale, reg_loss=self._reg_loss)
            opacity_loss, scale_loss = self.lambda_opacity * self._reg_loss[0], self.lambda_scale * self._reg_loss[1]
            loss = loss + opacity_loss + scale_loss
        else:
            self.optimizer.step(d_particles, d_sph, visibility=vis if self.optimizer.selective else None)
        self.last_losses = {"l1_loss": l1_loss, "ssim_loss": ssim_loss, "opacity_loss": opacity_loss, "scale_loss": scale_loss, "total_loss": loss}
        self.frame += 1
        if self.densifier is not None and self.densifier.post_optimizer_step(self.frame, self.scene_extent, positions_lr=self.optimizer.lrs["positions"]):
            # the number of Gaussians may have changed (identically on every rank): re-capacity the exchange buffers; the renderer's
            # scratch grows by itself
            if self.exchange.n != self.n:
                self.exchange = view_parallel.CompactGradientExchange(self.raster, self.n, self.device, group=self.group)
        return loss
