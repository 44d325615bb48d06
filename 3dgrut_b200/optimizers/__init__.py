"""Optimizer step of the Gaussian parameters on the B200 (SURVEY.md section 8f row 2).

`SelectiveAdam` mirrors threedgrut/optimizers/__init__.py:42-124 (same constructor, `step(visibility)`), backed by
gutb200_selective_adam_update instead of the reference's lib_optimizers_cc plugin.
`FusedGaussianAdam` (ours) takes the renderer's gradients directly -- [N,12] and [N,48] w.r.t. the activated values, e.g. straight out of
the view-parallel exchange -- and performs the activation chain rule and the Adam update of all six parameter tensors in one launch.
No CPU fallback: both raise if the tensors are not CUDA tensors or the library is missing."""
from __future__ import annotations

import ctypes as C

import torch

import b200_native as native

GROUPS = ("positions", "density", "rotation", "scale", "features_albedo", "features_specular")
WIDTHS = (3, 1, 4, 3, 3, 45)


def _lib():
    lib = native.load()
    if not getattr(lib, "_optim_bound", False):
        vp, i64, i32, f32 = C.c_void_p, C.c_int64, C.c_int32, C.c_float
        lib.gutb200_selective_adam_update.argtypes = [vp, vp, vp, vp, vp, vp, f32, f32, f32, f32, i64, i64]
        lib.gutb200_selective_adam_update.restype = C.c_int
        step_args = [vp, i64, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(f32), f32, f32, f32, i64, i32, vp, vp, vp]
        lib.gutb200_gaussian_adam_step.argtypes = step_args
        lib.gutb200_gaussian_adam_step.restype = C.c_int
        lib.gutb200_gaussian_adam_step_reg.argtypes = step_args + [f32, f32, vp]
        lib.gutb200_gaussian_adam_step_reg.restype = C.c_int
        lib._optim_bound = True
    return lib


def _check(t: torch.Tensor, what: str):
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()):
        raise RuntimeError(f"{what}: expected a contiguous float32 CUDA tensor (there is no CPU fallback)")


def selective_adam_update(param, param_grad, exp_avg, exp_avg_sq, visibility, lr, beta1, beta2, eps):
    """lib_optimizers_cc.selective_adam_update (threedgrut/optimizers/optimizers.cpp): in-place update of param / exp_avg / exp_avg_sq."""
    for t, w in ((param, "param"), (param_grad, "param_grad"), (exp_avg, "exp_avg"), (exp_avg_sq, "exp_avg_sq")):
        _check(t, w)
    n = int(param.shape[0]) if param.dim() > 0 else 0
    m = int(param.numel() // n) if n else 1
    vis = visibility.to(torch.bool).reshape(-1).contiguous()
    if vis.numel() != n:
        raise RuntimeError("visibility must have one entry per row of param")
    stream = torch.cuda.current_stream(param.device).cuda_stream
    with torch.cuda.device(param.device):
        rc = _lib().gutb200_selective_adam_update(stream, param.data_ptr(), param_grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                                                  vis.data_ptr(), float(lr), float(beta1), float(beta2), float(eps), n, m)
    if rc != 0:
        raise RuntimeError(f"gutb200_selective_adam_update failed ({rc})")


class SelectiveAdam(torch.optim.Adam):
    """threedgrut.optimizers.SelectiveAdam with the B200 kernel underneath (one tensor per parameter group, as in the reference)."""

    def __init__(self, params, lr=0.001, betas=(0.9, 0.999), eps=1e-08):
        super().__init__(params=params, lr=lr, eps=eps, betas=betas)
        _lib()  # fail now if the library is missing

    @torch.no_grad()
    def step(self, visibility):
        for group in self.param_groups:
            lr, eps = group["lr"], group["eps"]
            beta1, beta2 = group["betas"]
            assert len(group["params"]) == 1, "More than one tensor in group is not supported"
            param = group["params"][0]
            if param.grad is None:
                continue
            state = self.state[param]
            if len(state) == 0:
                state["step"] = torch.tensor(0.0, dtype=torch.float32)
                state["exp_avg"] = torch.zeros_like(param, memory_format=torch.preserve_format)
                state["exp_avg_sq"] = torch.zeros_like(param, memory_format=torch.preserve_format)
            if not param.is_contiguous() or not state["exp_avg"].is_contiguous():
                raise RuntimeError("SelectiveAdam: parameters and state must be contiguous (the update is in place)")
            selective_adam_update(param.data, param.grad.contiguous(), state["exp_avg"], state["exp_avg_sq"], visibility, lr, beta1, beta2, eps)


class FusedGaussianAdam:
    """One-launch optimizer step for the SH Gaussian model.

    params: dict name -> raw (pre-activation) leaf tensor for the six GROUPS; lrs: dict name -> learning rate (mutable: schedulers
    write `opt.lrs["positions"] = ...`).  step(d_particles, d_sph, visibility=None) consumes the renderer's gradients
    (Tracer / SplatRaster.trace_bwd outputs, or the view-parallel exchange's) -- no autograd pass over the activations is needed.
    step(..., lambda_opacity, lambda_scale) also applies the reference's opacity / scale regularisers (trainer.py:722-739) in the same
    launch; reg_loss, a float32 CUDA tensor of two elements, then receives their unweighted values (mean sigmoid(density), mean
    exp(scale)) before the update."""

    def __init__(self, params: dict, lrs: dict, betas=(0.9, 0.999), eps=1e-15, selective=False):
        # the dict itself is kept (not copied) when it holds exactly the six groups: densification replaces the tensors inside it
        self.params = params if set(params.keys()) == set(GROUPS) else {k: params[k] for k in GROUPS}
        self._validate()
        self.lrs = {k: float(lrs[k]) for k in GROUPS}
        self.betas, self.eps, self.selective = (float(betas[0]), float(betas[1])), float(eps), bool(selective)
        self.exp_avg = {k: torch.zeros_like(t.data) for k, t in self.params.items()}
        self.exp_avg_sq = {k: torch.zeros_like(t.data) for k, t in self.params.items()}
        self.steps = 0
        _lib()

    @property
    def n(self) -> int:
        return int(self.params["positions"].shape[0])

    def _validate(self):
        n = self.n
        for k, w in zip(GROUPS, WIDTHS):
            t = self.params[k]
            _check(t.data, k)
            if tuple(t.shape) != (n, w):
                raise RuntimeError(f"{k}: expected shape {(n, w)}, got {tuple(t.shape)}")

    def _array(self, tensors):
        arr = (C.c_void_p * 6)()
        for i, k in enumerate(GROUPS):
            arr[i] = tensors[k].data_ptr()
        return arr

    @torch.no_grad()
    def step(self, d_particles: torch.Tensor, d_sph: torch.Tensor, visibility: torch.Tensor | None = None, lambda_opacity: float = 0.0,
             lambda_scale: float = 0.0, reg_loss: torch.Tensor | None = None):
        _check(d_particles, "d_particles")
        _check(d_sph, "d_sph")
        self._validate()  # the tensors may have been replaced (densification); moments must have followed
        for k in GROUPS:
            if self.exp_avg[k].shape != self.params[k].shape or self.exp_avg_sq[k].shape != self.params[k].shape:
                raise RuntimeError(f"{k}: optimizer state does not match the parameter shape {tuple(self.params[k].shape)}")
        if tuple(d_particles.shape) != (self.n, 12) or tuple(d_sph.shape) != (self.n, 48):
            raise RuntimeError("gradient shapes must be [N,12] and [N,48]")
        vis_ptr = None
        if self.selective:
            if visibility is None:
                raise RuntimeError("selective mode needs the renderer's visibility")
            vis = visibility.reshape(-1)
            if vis.dtype != torch.float32:
                vis = vis.to(torch.float32)
            vis = vis.contiguous()
            _check(vis, "visibility")
            vis_ptr = vis.data_ptr()
        lambda_opacity, lambda_scale = float(lambda_opacity), float(lambda_scale)
        regularised = lambda_opacity != 0.0 or lambda_scale != 0.0 or reg_loss is not None
        if reg_loss is not None:
            _check(reg_loss, "reg_loss")
            if reg_loss.numel() < 2 or reg_loss.device != d_particles.device:
                raise RuntimeError("reg_loss must hold two floats on the gradients' device")
        self.steps += 1
        dev = d_particles.device
        lr = (C.c_float * 6)(*[self.lrs[k] for k in GROUPS])
        stream = torch.cuda.current_stream(dev).cuda_stream
        args = (stream, self.n, self._array({k: t.data for k, t in self.params.items()}), self._array(self.exp_avg), self._array(self.exp_avg_sq),
                lr, self.betas[0], self.betas[1], self.eps, self.steps, int(self.selective), d_particles.data_ptr(), d_sph.data_ptr(), vis_ptr)
        with torch.cuda.device(dev):
            if regularised:
                rc = _lib().gutb200_gaussian_adam_step_reg(*args, lambda_opacity, lambda_scale, None if reg_loss is None else reg_loss.data_ptr())
            else:
                rc = _lib().gutb200_gaussian_adam_step(*args)
        if rc != 0:
            raise RuntimeError(f"gutb200_gaussian_adam_step{'_reg' if regularised else ''} failed ({rc})")
