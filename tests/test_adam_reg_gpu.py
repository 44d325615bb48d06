"""GPU tests of the regularised optimizer step (gutb200_gaussian_adam_step_reg, 3dgrut_b200/csrc/gut_optim.cu) against
tests/adam_reg_oracle.py, and of the opacity / scale regularisers in GaussianTrainStep.
Bars, 2e-6 relative (fp32 FMA contraction and CUDA's expf differ from numpy's roundings by a few ulp):
  parameters: relative to 0.05 + the larger of |start| and |end|: a parameter keeps a few ulp of the largest value it held (density
              moves 0.16 per selective step at lr 0.05, e.g. 0.63 -> 0.035 in three);
  moments:    relative to the tensor's largest |x|: the density gradient dL/dsigmoid * s (1 - s) carries an absolute error of about an
              ulp of s times dL/dsigmoid (torch's sigmoid backward computes it the same way), which is large relative to a small
              (1 - s), and a moment that cancels to near zero keeps an absolute error of a few ulp of the terms that cancelled.
The groups the regularisers do not touch must also equal the plain step bit for bit.  Rotation is checked only that way: over the
1.2M rotation elements at N = 300001, Adam's normalisation turns fp32 rounding in the g - q (q . g) projection into relative errors
up to 4e-5 even between the numpy restatement and the same steps with float64 gradients (test_adam_gpu.py pins rotation at N = 4099)."""
import numpy as np
import pytest

import adam_reg_oracle as aro
import scenes
from oracle import adam_oracle as ao
from test_adam_oracle import LRS, _state

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _close(a, b, what, scale):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    err = np.abs(a - b) / scale
    assert err.max() <= 2e-6, f"{what}: max scaled error {err.max():.3e}"


def _param_scale(start, end):
    return 0.05 + np.maximum(np.abs(start), np.abs(end)).astype(np.float64)


def _moment_scale(b):
    return max(float(np.abs(np.asarray(b, np.float64)).max()), 1e-30)


@pytest.mark.parametrize("n", [1, 7, 300_001])
@pytest.mark.parametrize("selective", [False, True])
def test_regularised_step_matches_oracle(selective, n):
    import optimizers

    dev = torch.device("cuda", 0)
    lam_o, lam_s = 0.02, 0.005
    params, _, _ = _state(n=n, seed=3)
    rng = np.random.default_rng(11)
    k = 0.01 / n  # image gradients of the size of the regularisers' per-element gradients
    leaves = {name: torch.from_numpy(v.copy()).to(dev) for name, v in params.items()}
    opt = optimizers.FusedGaussianAdam(leaves, LRS, eps=1e-15, selective=selective)
    plain = optimizers.FusedGaussianAdam({name: torch.from_numpy(v.copy()).to(dev) for name, v in params.items()}, LRS, eps=1e-15,
                                         selective=selective)
    reg_loss = torch.full((2,), float("nan"), device=dev)
    p = {name: v.copy() for name, v in params.items()}
    m = {name: np.zeros_like(v) for name, v in params.items()}
    v = {name: np.zeros_like(vv) for name, vv in params.items()}
    for t in range(1, 4):
        dp = (k * rng.normal(size=(n, 12))).astype(np.float32)
        ds = (k * rng.normal(size=(n, 48))).astype(np.float32)
        vis_bits = (rng.uniform(size=n) > 0.3).astype(np.int32)  # the renderer writes int 1 into a float tensor
        vis = torch.from_numpy(vis_bits.view(np.float32).copy()).to(dev)
        want_losses = aro.reg_losses(p)
        tdp, tds = torch.from_numpy(dp).to(dev), torch.from_numpy(ds).to(dev)
        opt.step(tdp, tds, visibility=vis if selective else None, lambda_opacity=lam_o, lambda_scale=lam_s, reg_loss=reg_loss)
        plain.step(tdp, tds, visibility=vis if selective else None)
        got_losses = reg_loss.cpu().numpy().astype(np.float64)
        for got, want, what in zip(got_losses, want_losses, ("mean sigmoid(density)", "mean exp(scale)")):
            assert abs(got - want) <= 1e-5 * abs(want), f"step {t} {what}: {got} vs {want}"
        p, m, v = aro.gaussian_adam_step_reg(p, m, v, LRS, dp, ds, lam_o, lam_s, eps=1e-15, step=t, selective=selective,
                                             visibility=vis_bits != 0)
    torch.cuda.synchronize()
    for name in ao.GROUPS:
        if name in ("density", "scale"):
            assert not torch.equal(leaves[name], plain.params[name]), name
        else:
            assert torch.equal(leaves[name], plain.params[name]), name
            assert torch.equal(opt.exp_avg[name], plain.exp_avg[name]) and torch.equal(opt.exp_avg_sq[name], plain.exp_avg_sq[name]), name
        if name == "rotation":
            continue
        _close(leaves[name].cpu().numpy(), p[name], f"param {name}", _param_scale(params[name], p[name]))
        _close(opt.exp_avg[name].cpu().numpy(), m[name], f"exp_avg {name}", _moment_scale(m[name]))
        _close(opt.exp_avg_sq[name].cpu().numpy(), v[name], f"exp_avg_sq {name}", _moment_scale(v[name]))


@pytest.mark.parametrize("selective", [False, True])
def test_zero_weights_are_bit_identical_to_the_plain_step(selective):
    import optimizers

    dev = torch.device("cuda", 0)
    n = 4099
    params, _, _ = _state(n=n, seed=5)
    rng = np.random.default_rng(6)
    plain = optimizers.FusedGaussianAdam({k: torch.from_numpy(v.copy()).to(dev) for k, v in params.items()}, LRS, eps=1e-15, selective=selective)
    reg = optimizers.FusedGaussianAdam({k: torch.from_numpy(v.copy()).to(dev) for k, v in params.items()}, LRS, eps=1e-15, selective=selective)
    reg_loss = torch.zeros(2, device=dev)
    for _ in range(3):
        dp = torch.from_numpy(rng.normal(size=(n, 12)).astype(np.float32)).to(dev)
        ds = torch.from_numpy(rng.normal(size=(n, 48)).astype(np.float32)).to(dev)
        vis = torch.from_numpy((rng.uniform(size=n) > 0.3).astype(np.float32)).to(dev)
        plain.step(dp, ds, visibility=vis if selective else None)
        # reg_loss given: the regularised entry point runs with both weights at 0
        reg.step(dp, ds, visibility=vis if selective else None, lambda_opacity=0.0, lambda_scale=0.0, reg_loss=reg_loss)
    torch.cuda.synchronize()
    for k in ao.GROUPS:
        assert torch.equal(plain.params[k], reg.params[k]), k
        assert torch.equal(plain.exp_avg[k], reg.exp_avg[k]) and torch.equal(plain.exp_avg_sq[k], reg.exp_avg_sq[k]), k


def test_regularisers_alone_lower_density_and_scale_and_touch_nothing_else():
    import optimizers

    dev = torch.device("cuda", 0)
    n = 4099
    params, _, _ = _state(n=n, seed=8)
    leaves = {k: torch.from_numpy(v.copy()).to(dev) for k, v in params.items()}
    before = {k: t.clone() for k, t in leaves.items()}
    opt = optimizers.FusedGaussianAdam(leaves, LRS, eps=1e-15)
    opt.step(torch.zeros((n, 12), device=dev), torch.zeros((n, 48), device=dev), lambda_opacity=0.01, lambda_scale=0.01)
    torch.cuda.synchronize()
    assert bool((leaves["density"] < before["density"]).all())
    assert bool((leaves["scale"] < before["scale"]).all())
    for k in ("positions", "rotation", "features_albedo", "features_specular"):
        assert torch.equal(leaves[k], before[k]), k
        assert not opt.exp_avg[k].any() and not opt.exp_avg_sq[k].any(), k


def _mcmc_fit(lambda_opacity, lambda_scale):
    """The fit of test_train_step_gpu.py::test_fit_with_mcmc_strategy_runs_on_the_gpu, with the given regulariser weights."""
    import densify
    import train_step
    from threedgut_tracer.tracer import ShutterType, fromOpenCVPinholeCameraModelParameters

    dev = torch.device("cuda", 0)
    sc = scenes.scene_c1(n=600, width=96, height=96)
    W, H = sc.width, sc.height
    sensor = fromOpenCVPinholeCameraModelParameters(np.array([W, H]), ShutterType.GLOBAL, np.array([sc.cx, sc.cy], np.float32),
                                                    np.array([sc.fx, sc.fy], np.float32), np.zeros(6, np.float32), np.zeros(2, np.float32),
                                                    np.zeros(4, np.float32))
    ro, rd = sc.rays()
    rays_o, rays_d = torch.from_numpy(ro).to(dev), torch.from_numpy(rd).to(dev)
    P, S = torch.from_numpy(sc.particles).to(dev), torch.from_numpy(sc.sph).to(dev)

    def raw_from(particles, sph):
        dns = particles[:, 3:4].clamp(1e-4, 1 - 1e-4)
        return {"positions": particles[:, 0:3].clone(), "density": torch.log(dns / (1 - dns)), "rotation": particles[:, 4:8].clone(),
                "scale": torch.log(particles[:, 8:11]), "features_albedo": sph[:, 0:3].clone(), "features_specular": sph[:, 3:48].clone()}

    lrs = dict(positions=2e-3, density=0.05, rotation=1e-3, scale=5e-3, features_albedo=1e-2, features_specular=5e-4)
    truth = train_step.GaussianTrainStep(raw_from(P, S), lrs)
    views = [scenes.pose7_from_c2w(sc.camera(i, 6)) for i in range(6)]
    targets = [truth.render(rays_o, rays_d, sensor, p)[0][..., :3].clone() for p in views]
    gen = torch.Generator(device=dev).manual_seed(0)
    P2, S2 = P.clone(), S.clone()
    P2[:, 0:3] += 0.02 * torch.randn((sc.n, 3), device=dev, generator=gen)
    S2[:, 0:3] += 0.5 * torch.randn((sc.n, 3), device=dev, generator=gen)
    P2[::9, 3] = 0.001  # a few dead Gaussians for relocate()
    conf = densify.MCMCConfig(relocate_start=5, relocate_frequency=20, add_start=5, add_frequency=20, perturb_start=0, noise_lr=5e3, seed=2)
    fit = train_step.GaussianTrainStep(raw_from(P2, S2), lrs, densify_conf=conf, lambda_l1=0.8, lambda_ssim=0.2, lambda_opacity=lambda_opacity,
                                       lambda_scale=lambda_scale)

    def mean_loss():
        return float(np.mean([float((fit.render(rays_o, rays_d, sensor, p)[0][..., :3] - t).abs().mean()) for p, t in zip(views, targets)]))

    before = mean_loss()
    for it in range(90):
        loss = fit.step(rays_o, rays_d, sensor, views[it % 6], targets[it % 6])
    after = mean_loss()
    opacity = float(torch.sigmoid(fit.params["density"]).mean())
    return before, after, opacity, fit, loss


def test_mcmc_fit_with_regularisers_converges_with_lower_opacity():
    b0, a0, o0, _, _ = _mcmc_fit(0.0, 0.0)
    b1, a1, o1, fit, loss = _mcmc_fit(0.01, 0.01)  # configs/base_mcmc.yaml:13-18
    print(f"[train-step+mcmc] mean L1 {b0:.5f} -> {a0:.5f}, mean opacity {o0:.4f} without the regularisers; "
          f"{b1:.5f} -> {a1:.5f}, mean opacity {o1:.4f} with them")
    assert b1 == pytest.approx(b0, rel=1e-6)  # same start
    assert np.isfinite(a0) and a0 < 0.8 * b0
    assert np.isfinite(a1) and a1 < 0.8 * b1
    assert o1 < o0
    parts = fit.last_losses
    assert set(parts) == {"l1_loss", "ssim_loss", "opacity_loss", "scale_loss", "total_loss"} and parts["total_loss"] is loss
    total = sum(float(parts[k]) for k in ("l1_loss", "ssim_loss", "opacity_loss", "scale_loss"))
    assert float(loss) == pytest.approx(total, rel=1e-5)
    assert float(parts["opacity_loss"]) > 0 and float(parts["scale_loss"]) > 0
