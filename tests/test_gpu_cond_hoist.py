"""GPU parity of the hoisted conditioner projection: the per-call precompute (fd_wavenet_cond_term) against float64 on the
exact plane values, the denoiser with the hoisted term (gate GEMM over the three conv taps, term added in its epilogue)
against the four-segment gate GEMM, and the sampler with the hoist against the sampler with the byte budget at zero."""
import numpy as np
import pytest
import torch

from conftest import rel_l2
from fish_diffusion_b200 import DIFFUSIONS, WaveNet, synthetic
from fish_diffusion_b200 import _native as N
from fish_diffusion_b200 import diffusion as diffusion_mod
from gpu_util import dev, planes_to_f64

pytestmark = pytest.mark.gpu

WN_FULL = dict(mel_channels=128, d_encoder=256, residual_channels=512, residual_layers=20, use_linear_bias=True,
               dilation_cycle=4)
PRECISIONS = ["f16", "bf16", "f16x1"]


def make_net(cfg, seed, **kw):
    net = WaveNet(**cfg, **kw).to(dev())
    net.load_state_dict({k: torch.from_numpy(v) for k, v in synthetic.wavenet_weights(seed, **cfg).items()})
    return net.eval()


def operand_f64(planes, precision):
    """Exact operand values the GEMM multiplies: hi + lo, or the hi plane alone in the one-product modes."""
    pc = N.prec_code(precision)
    if precision.endswith("x1"):
        planes = torch.stack([planes[0], torch.zeros_like(planes[0])])
    return planes_to_f64(planes, pc)


@pytest.mark.parametrize("backend", ["simt", "tc"])
@pytest.mark.parametrize("precision", PRECISIONS)
def test_cond_term_vs_float64(precision, backend):
    cfg = dict(WN_FULL, residual_layers=3)
    net = make_net(cfg, 5, precision=precision, backend=backend)
    B, T, E, C, L = 2, 333, cfg["d_encoder"], cfg["residual_channels"], cfg["residual_layers"]
    g = torch.Generator().manual_seed(4)
    cond = torch.randn(B, T, E, generator=g).to(dev())
    mask = torch.zeros((B, T), dtype=torch.uint8, device=dev())
    mask[1, T - 40:] = 1
    cp = N.split_nwc(cond, N.prec_code(precision), mask=mask)
    out = torch.full((L, B, T, 2 * C), float("nan"), device=dev())
    net.cond_term(cp, out)
    torch.cuda.synchronize()
    pk = net._packed(dev())
    c64 = operand_f64(cp, precision)
    got = out.cpu().numpy()
    tol = 5e-5 if precision == "bf16" else 2e-6
    for l in range(L):
        w = operand_f64(net._pack_static["w1"][l], precision)[:, 3 * C:] * pk["w1_inv"][l]
        ref = c64 @ w.T                       # packed gate/filter column order, like the kernel's output
        e = rel_l2(got[l], ref)
        assert e < tol, (l, e)
        assert np.all(got[l, 1, T - 40:] == 0)   # rows the conditioner mask zeroed


@pytest.mark.parametrize("backend", ["simt", "tc"])
@pytest.mark.parametrize("precision", PRECISIONS)
def test_denoiser_with_and_without_cond_term(precision, backend):
    """Full width (C=512, E=256, L=20, cycle 4), ragged T, per-item steps (one gate-bias row per item), masks."""
    net = make_net(WN_FULL, 0, precision=precision, backend=backend)
    net.use_graph = False
    B, T, M, E = 3, 301, WN_FULL["mel_channels"], WN_FULL["d_encoder"]
    C, L = WN_FULL["residual_channels"], WN_FULL["residual_layers"]
    pc = N.prec_code(precision)
    g = torch.Generator().manual_seed(6)
    x = torch.randn(B, T, M, generator=g).to(dev())
    cond = torch.randn(B, T, E, generator=g).to(dev())
    mask = torch.zeros((B, T), dtype=torch.uint8, device=dev())
    mask[2, T - 57:] = 1
    steps = torch.tensor([3.0, 500.0, 977.0], device=dev())
    xp, cp = N.split_nwc(x, pc), N.split_nwc(cond, pc, mask=mask)
    plain = net.forward_cl(xp, steps, cp, x_mask=mask).clone()
    ct = net.cond_term(cp, torch.empty((L, B, T, 2 * C), device=dev()))
    hoisted = net.forward_cl(xp, steps, cp, x_mask=mask, cond_term=ct).clone()
    a, b = hoisted.cpu().numpy(), plain.cpu().numpy()
    e = rel_l2(a, b)
    print(f"denoiser [{precision},{backend}] hoisted vs four-segment gate GEMM: rel-L2 {e:.2e}, "
          f"max-abs {np.abs(a - b).max():.2e}")
    # the conditioner products are summed apart from the conv taps (fp32 reordering), and a reordering difference can
    # move the plane rounding of an activation that the next layer multiplies (in the one-product mode: the hi plane,
    # 11 bits).  Bounds: what tests/test_gpu_wavenet.py and test_gpu_single_product.py ask of each mode's denoiser.
    assert e < {"f16": 2e-5, "bf16": 3e-4, "f16x1": 2e-3}[precision], (e, np.abs(a - b).max())
    assert np.all(a[2, T - 57:] == 0)


def _diffusion(precision="f16"):
    cfg = dict(WN_FULL, residual_layers=4)
    diff = DIFFUSIONS.build(dict(type="GaussianDiffusion", denoiser=dict(type="WaveNetDenoiser", precision=precision, **cfg),
                                 mel_channels=128, sampler_interval=100, spec_min=[-5.0], spec_max=[0.0],
                                 noise_predictor="naive")).to(dev())
    diff.denoise_fn.load_state_dict({k: torch.from_numpy(v) for k, v in synthetic.wavenet_weights(3, **cfg).items()})
    return diff


@pytest.mark.parametrize("pred", ["naive", "unipc"])
def test_sampler_with_hoist_equals_budget_zero(monkeypatch, pred):
    g = torch.Generator().manual_seed(12)
    feats = torch.randn(2, 600, 256, generator=g).to(dev())
    hoisted_diff = _diffusion()
    hoisted = hoisted_diff(feats, noise_predictor=pred, seed=5)
    assert hoisted_diff._sws.get("cond_term") is not None
    monkeypatch.setattr(diffusion_mod, "COND_TERM_BUDGET_BYTES", 0)
    plain_diff = _diffusion()
    plain = plain_diff(feats, noise_predictor=pred, seed=5)
    assert plain_diff._sws.get("cond_term") is None
    e = rel_l2(hoisted.cpu().numpy(), plain.cpu().numpy())
    print(f"{pred} sampler, hoisted vs budget 0: rel-L2 {e:.2e}")
    assert torch.isfinite(hoisted).all() and e < 1e-5


def test_budget_decides_the_path(monkeypatch):
    diff = _diffusion()
    B, T, E = 1, 200, 256
    need = diff.denoise_fn.n_layers * B * T * 2 * diff.denoise_fn.residual_channels * 4
    feats = torch.randn(B, T, E, device=dev())
    calls = []
    orig = WaveNet.cond_term
    monkeypatch.setattr(WaveNet, "cond_term", lambda self, *a, **k: calls.append(1) or orig(self, *a, **k))
    monkeypatch.setattr(diffusion_mod, "COND_TERM_BUDGET_BYTES", need - 1)
    diff(feats, sampler_interval=500, seed=1)
    assert not calls and diff._sws.get("cond_term") is None
    monkeypatch.setattr(diffusion_mod, "COND_TERM_BUDGET_BYTES", need)
    diff(feats, sampler_interval=500, seed=1)
    assert calls == [1] and diff._sws["cond_term"].numel() * 4 == need
