"""Pins tests/adam_reg_oracle.py (the fused Adam step plus the opacity / scale regularisers) against the reference's own expression:
torch autograd of lambda_opacity |sigmoid(density)|.mean() + lambda_scale |exp(scale)|.mean() (threedgrut/trainer.py:722-739) through
the reference's activations, followed by torch.optim.Adam, or by the selective rule of threedgrut/optimizers/optimizers.cu:66-80.
Also maps the reference's loss configuration to the four weights of GaussianTrainStep."""
import types

import numpy as np
import pytest

torch = pytest.importorskip("torch")

import adam_reg_oracle as aro  # noqa: E402
from oracle import adam_oracle as ao  # noqa: E402
from test_adam_oracle import LRS, _state  # noqa: E402

# base_mcmc.yaml, configs/apps/*_mcmc_nht.yaml, and the scale term alone
LAMBDAS = [(0.01, 0.01), (0.02, 0.005), (0.0, 0.01)]


def _grad_scale(n):
    """Image gradients of the size of the regularisers' per-element gradients, so that neither hides the other."""
    return 0.01 / n


def _torch_gradients(leaves, dp, ds, lam_o, lam_s):
    """Gradients of the reference's loss w.r.t. the raw leaves: the renderer's gradients enter as a linear term."""
    for t in leaves.values():
        t.grad = None
    act = torch.cat([leaves["positions"], torch.sigmoid(leaves["density"]), torch.nn.functional.normalize(leaves["rotation"]),
                     torch.exp(leaves["scale"]), torch.zeros_like(leaves["density"])], 1)
    feat = torch.cat([leaves["features_albedo"], leaves["features_specular"]], 1)
    loss = (act * torch.tensor(dp)).sum() + (feat * torch.tensor(ds)).sum()
    loss = loss + lam_o * torch.abs(torch.sigmoid(leaves["density"])).mean() + lam_s * torch.abs(torch.exp(leaves["scale"])).mean()
    loss.backward()


def _sequence(n, seed, steps=3):
    rng = np.random.default_rng(seed)
    k = _grad_scale(n)
    return [((k * rng.normal(size=(n, 12))).astype(np.float32), (k * rng.normal(size=(n, 48))).astype(np.float32),
             rng.uniform(size=n) > 0.35) for _ in range(steps)]


@pytest.mark.parametrize("lambdas", LAMBDAS)
def test_regularised_chain_rule_matches_autograd(lambdas):
    n = 257
    params, _, _ = _state(n=n, seed=1)
    dp, ds, _ = _sequence(n, 7, 1)[0]
    leaves = {k: torch.tensor(v, requires_grad=True) for k, v in params.items()}
    _torch_gradients(leaves, dp, ds, *lambdas)
    got = ao.raw_gradients(params, aro.regularised_d_particles(params, dp, *lambdas), ds)
    k = _grad_scale(n)
    for name in ao.GROUPS:
        assert np.allclose(got[name], leaves[name].grad.numpy(), rtol=2e-6, atol=1e-7 * k), name
    # the regularisers are not lost in the image gradients: without them the density / scale gradients differ
    plain = ao.raw_gradients(params, dp, ds)
    if lambdas[0]:
        assert not np.allclose(plain["density"], got["density"], rtol=1e-2, atol=0)
    assert not np.allclose(plain["scale"], got["scale"], rtol=1e-2, atol=0)


@pytest.mark.parametrize("n", [257, 7])
@pytest.mark.parametrize("lambdas", LAMBDAS)
def test_three_regularised_adam_steps_match_torch_optim(lambdas, n):
    params, _, _ = _state(n=n, seed=2)
    seq = _sequence(n, 5)
    leaves = {k: torch.tensor(v, requires_grad=True) for k, v in params.items()}
    opt = torch.optim.Adam([{"params": [leaves[k]], "lr": LRS[k]} for k in ao.GROUPS], lr=0.0, eps=1e-15)
    p = {k: v.copy() for k, v in params.items()}
    m = {k: np.zeros_like(v) for k, v in params.items()}
    v = {k: np.zeros_like(vv) for k, vv in params.items()}
    for t, (dp, ds, _) in enumerate(seq, 1):
        _torch_gradients(leaves, dp, ds, *lambdas)
        opt.step()
        p, m, v = aro.gaussian_adam_step_reg(p, m, v, LRS, dp, ds, *lambdas, eps=1e-15, step=t)
    k = _grad_scale(n)
    for name in ao.GROUPS:
        st = opt.state[leaves[name]]
        assert np.allclose(p[name], leaves[name].detach().numpy(), rtol=1e-5, atol=1e-6), name
        assert np.allclose(m[name], st["exp_avg"].numpy(), rtol=1e-5, atol=1e-6 * k), name
        assert np.allclose(v[name], st["exp_avg_sq"].numpy(), rtol=1e-5, atol=1e-6 * k * k), name


@pytest.mark.parametrize("n", [257, 7])
@pytest.mark.parametrize("lambdas", LAMBDAS)
def test_three_selective_regularised_steps_match_the_plugin_rule(lambdas, n):
    """SelectiveAdam: param.grad holds the regularisers' gradient on every row, the plugin updates only the visible rows."""
    params, _, _ = _state(n=n, seed=3)
    seq = _sequence(n, 9)
    leaves = {k: torch.tensor(v, requires_grad=True) for k, v in params.items()}
    tm = {k: torch.zeros_like(t) for k, t in leaves.items()}
    tv = {k: torch.zeros_like(t) for k, t in leaves.items()}
    b1, b2, eps = torch.tensor(0.9), torch.tensor(0.999), torch.tensor(1e-15)
    p = {k: v.copy() for k, v in params.items()}
    m = {k: np.zeros_like(v) for k, v in params.items()}
    v = {k: np.zeros_like(vv) for k, vv in params.items()}
    for dp, ds, vis in seq:
        _torch_gradients(leaves, dp, ds, *lambdas)
        keep = torch.from_numpy(vis)[:, None]
        with torch.no_grad():
            for name, leaf in leaves.items():  # optimizers.cu:66-80, literally
                g = leaf.grad
                m_new = b1 * tm[name] + (1 - b1) * g
                v_new = b2 * tv[name] + (1 - b2) * g * g
                p_new = leaf - LRS[name] * m_new / (torch.sqrt(v_new) + eps)
                tm[name] = torch.where(keep, m_new, tm[name])
                tv[name] = torch.where(keep, v_new, tv[name])
                leaf.copy_(torch.where(keep, p_new, leaf))
        p, m, v = aro.gaussian_adam_step_reg(p, m, v, LRS, dp, ds, *lambdas, eps=1e-15, selective=True, visibility=vis)
    k = _grad_scale(n)
    never = ~np.logical_or.reduce([s[2] for s in seq])
    for name in ao.GROUPS:
        assert np.allclose(p[name], leaves[name].detach().numpy(), rtol=1e-5, atol=1e-6), name
        assert np.allclose(m[name], tm[name].numpy(), rtol=1e-5, atol=1e-6 * k), name
        assert np.allclose(v[name], tv[name].numpy(), rtol=1e-5, atol=1e-6 * k * k), name
        assert np.array_equal(p[name][never], params[name][never]) and not m[name][never].any(), name


def test_reported_losses_are_the_reference_terms():
    params, _, _ = _state(n=257, seed=4)
    want_o = torch.abs(torch.sigmoid(torch.tensor(params["density"], dtype=torch.float64))).mean().item()
    want_s = torch.abs(torch.exp(torch.tensor(params["scale"], dtype=torch.float64))).mean().item()
    got_o, got_s = aro.reg_losses(params)
    assert got_o == pytest.approx(want_o, rel=1e-12) and got_s == pytest.approx(want_s, rel=1e-12)


def _loss_conf(**loss):
    base = dict(use_l1=True, lambda_l1=0.8, use_l2=False, lambda_l2=1.0, use_ssim=True, lambda_ssim=0.2, use_opacity=False, lambda_opacity=0.0,
                use_scale=False, lambda_scale=0.0)  # configs/base_gs.yaml:171-185
    base.update(loss)
    return {"loss": base}


def test_loss_weights_from_conf():
    import train_step

    assert train_step.loss_weights_from_conf(_loss_conf()) == (0.8, 0.2, 0.0, 0.0)
    mcmc = _loss_conf(use_opacity=True, lambda_opacity=0.01, use_scale=True, lambda_scale=0.01)  # configs/base_mcmc.yaml:13-18
    assert train_step.loss_weights_from_conf(mcmc) == (0.8, 0.2, 0.01, 0.01)
    # a weight without its use_* flag does not count
    off = _loss_conf(use_l1=False, use_ssim=False, lambda_opacity=0.02, lambda_scale=0.005)
    assert train_step.loss_weights_from_conf(off) == (0.0, 0.0, 0.0, 0.0)
    # attribute-style configuration (as OmegaConf's DictConfig reads)
    ns = types.SimpleNamespace(loss=types.SimpleNamespace(**mcmc["loss"]))
    assert train_step.loss_weights_from_conf(ns) == (0.8, 0.2, 0.01, 0.01)
