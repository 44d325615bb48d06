"""CPU restatement (numpy, float32) of the regularised optimizer step, gutb200_gaussian_adam_step_reg -- test infrastructure only.

Extends oracle/adam_oracle.py by the opacity and scale regularisers of the reference's loss (threedgrut/trainer.py:722-739):
    loss += lambda_opacity * mean|sigmoid(density)|  +  lambda_scale * mean|exp(scale)|          (means over [N,1] and [N,3])
Their gradients w.r.t. the ACTIVATED values, lambda_opacity / N * sign(sigmoid) and lambda_scale / (3N) * sign(exp), join the renderer's
d_particles columns 3 and 8..10 before the activation chain rule, which is where the kernel adds them too.
Pinned by tests/test_adam_reg_oracle.py against torch autograd of the reference's expression + torch.optim.Adam on the CPU."""
import numpy as np

from oracle import adam_oracle as ao

f32 = np.float32


def reg_coefficients(n, lambda_opacity, lambda_scale):
    """Per-element gradients of the two regularisers w.r.t. sigmoid(density) and exp(scale) (before the sign), as float32.
    Rounded as the kernel's entry point does (float weight, double division): where an image gradient nearly cancels the term, one ulp
    of difference here would be amplified by Adam's normalisation."""
    return f32(float(f32(lambda_opacity)) / n), f32(float(f32(lambda_scale)) / (3.0 * n))


def regularised_d_particles(params, d_particles, lambda_opacity, lambda_scale):
    """d_particles [N,12] with the regularisers' gradients added to the density and scale columns."""
    raw_d = np.asarray(params["density"], f32)
    raw_s = np.asarray(params["scale"], f32)
    c_o, c_s = reg_coefficients(raw_d.shape[0], lambda_opacity, lambda_scale)
    s = (f32(1) / (f32(1) + np.exp(-raw_d))).astype(f32)
    e = np.exp(raw_s).astype(f32)
    dp = np.array(d_particles, f32, copy=True)
    dp[:, 3:4] = (dp[:, 3:4] + c_o * np.sign(s)).astype(f32)
    dp[:, 8:11] = (dp[:, 8:11] + c_s * np.sign(e)).astype(f32)
    return dp


def reg_losses(params):
    """(mean sigmoid(density), mean exp(scale)) in float64: the unweighted loss values the step reports."""
    raw_d = np.asarray(params["density"], np.float64)
    raw_s = np.asarray(params["scale"], np.float64)
    return float(np.mean(1.0 / (1.0 + np.exp(-raw_d)))), float(np.mean(np.exp(raw_s)))


def gaussian_adam_step_reg(params, moments_m, moments_v, lrs, d_particles, d_sph, lambda_opacity, lambda_scale, **kw):
    """adam_oracle.gaussian_adam_step with the two regularisers; kw: b1, b2, eps, step, selective, visibility."""
    dp = regularised_d_particles(params, d_particles, lambda_opacity, lambda_scale)
    return ao.gaussian_adam_step(params, moments_m, moments_v, lrs, dp, d_sph, **kw)
