"""CPU tests of the host logic: registries, state_dict compatibility with the reference classes, bit-exact schedule
buffers, sampler coefficient math, weight packing (all without touching the GPU)."""
import numpy as np
import pytest
import torch

from conftest import rel_l2
from fish_diffusion_b200 import (DENOISERS, DIFFUSIONS, VOCODERS, GaussianDiffusion, Generator, NsfHifiGAN, WaveNet)
from fish_diffusion_b200 import uni_pc as pu
from fish_diffusion_b200.mel import mel_filterbank
from fish_diffusion_b200.registry import _MiniRegistry
from oracle import sampler as osamp


def test_registry_api():
    r = _MiniRegistry("things")

    @r.register_module()
    class A:
        def __init__(self, x=1):
            self.x = x

    r.register_module(name="Bee", module=A)
    assert r.build(dict(type="A", x=3)).x == 3 and r.build(dict(type="Bee")).x == 1
    with pytest.raises(KeyError):
        r.register_module(name="A", module=A)
    r.register_module(name="A", module=A, force=True)
    with pytest.raises(KeyError):
        r.build(dict(type="Nope"))
    with pytest.raises(KeyError):
        r.build(dict(x=1))
    with pytest.raises(TypeError):
        r.build([1])
    assert "WaveNetDenoiser" in DENOISERS and "GaussianDiffusion" in DIFFUSIONS and "NsfHifiGAN" in VOCODERS
    assert DENOISERS.get("WaveNetDenoiser") is WaveNet


def test_wavenet_state_dict_keys_match_reference(golden_cfg):
    keys = golden_cfg["state_dict_keys"]
    net = WaveNet(**golden_cfg["WN_FULL"])
    mine = {k: list(v.shape) for k, v in net.state_dict().items()}
    assert mine == keys["wavenet_full"]
    assert sum(p.numel() for p in net.parameters()) == 54_994_560 + 0   # SURVEY.md C1: 54,994,560 params
    net = WaveNet(**golden_cfg["WN_NOBIAS"])
    assert {k: list(v.shape) for k, v in net.state_dict().items()} == keys["wavenet_nobias"]
    assert torch.count_nonzero(net.output_projection.conv.weight) == 0     # wavenet.py:192 zero init


def test_diffusion_state_dict_and_buffers(golden, golden_cfg):
    cfg = golden_cfg["WN_SMALL"]
    diff = DIFFUSIONS.build(dict(type="GaussianDiffusion", denoiser=dict(type="WaveNetDenoiser", **cfg),
                                 mel_channels=16, spec_min=[-5.0], spec_max=[0.0]))
    assert isinstance(diff, GaussianDiffusion)
    mine = {k: list(v.shape) for k, v in diff.state_dict().items()}
    assert mine == golden_cfg["state_dict_keys"]["diffusion_small"]
    assert diff.noise_predictor == "unipc" and diff.num_timesteps == 1000 and diff.sampler_interval == 10
    g = golden("schedules")
    for k, v in diff.naive_noise_predictor.state_dict().items():
        ref = g[f"sched_linear_naive_{k}"]
        assert np.array_equal(v.numpy().view(np.uint32), ref.view(np.uint32)), k       # bit exact
    assert np.array_equal(diff.plms_noise_predictor.alphas_cumprod.numpy().view(np.uint32),
                          g["sched_linear_plms_alphas_cumprod"].view(np.uint32))
    ns = diff.unipc_noise_predictor.noise_schedule
    assert np.array_equal(ns.t_array.view(np.uint32), g["sched_linear_unipc_t_array"].reshape(-1).view(np.uint32))
    assert np.array_equal(ns.log_alpha_array.view(np.uint32),
                          g["sched_linear_unipc_log_alpha_array"].reshape(-1).view(np.uint32))
    d1 = GaussianDiffusion(dict(type="WaveNetDenoiser", **cfg), mel_channels=16, sampler_interval=1, spec_min=[-5.0],
                           spec_max=[0.0])
    assert d1.noise_predictor == "naive"            # diffusion.py:115-116
    with pytest.raises(AssertionError):
        GaussianDiffusion(dict(type="WaveNetDenoiser", **cfg), mel_channels=16, spec_min=[-5.0])
    with pytest.raises(NotImplementedError):
        from fish_diffusion_b200.diffusion import get_noise_schedule_list
        get_noise_schedule_list("nope", 10)


def test_generator_state_dict_keys_match_reference(golden_cfg):
    import json, os
    keys = golden_cfg["state_dict_keys"]
    here = os.path.join(os.path.dirname(__file__), "golden", "nsf_configs")
    for name in ("config_v1", "config_v1_256"):
        with open(os.path.join(here, name + ".json")) as f:
            h = json.load(f)
        g = Generator(h)
        assert {k: list(v.shape) for k, v in g.state_dict().items()} == keys[f"generator_{name}_wn"]
        g.remove_weight_norm()
        assert {k: list(v.shape) for k, v in g.state_dict().items()} == keys[f"generator_{name}"]


def test_nsf_hifigan_wrapper_checkpoint_formats(tmp_path, golden_cfg):
    h = dict(golden_cfg["VOC_SMALL"], n_fft=2048, win_size=2048, fmin=40, fmax=16000)
    (tmp_path / "config.json").write_text(__import__("json").dumps(h))
    g = Generator(h)
    sd = g.state_dict()                                   # weight-norm format
    torch.save({"generator": sd}, tmp_path / "model")
    v = NsfHifiGAN(checkpoint_path=str(tmp_path / "model"), mel_channels=32)
    assert not any(k.endswith("weight_g") for k in v.model.state_dict())
    torch.save({"state_dict": {"generator." + k: t for k, t in sd.items()}}, tmp_path / "model2")
    v2 = NsfHifiGAN(checkpoint_path=str(tmp_path / "model2"), config_file=str(tmp_path / "config.json"))
    for (k1, a), (k2, b) in zip(v.model.state_dict().items(), v2.model.state_dict().items()):
        assert k1 == k2 and torch.equal(a, b)
    with pytest.raises(ValueError):
        NsfHifiGAN(checkpoint_path=str(tmp_path / "model"), num_mels=128)
    v.freeze()
    assert not any(p.requires_grad for p in v.parameters())
    assert v.device == torch.device("cpu")


def test_linspace_and_unipc_coefficients_vs_oracle():
    betas = osamp.get_noise_schedule_list("linear", 1000, 0.01)
    ns = pu.NoiseScheduleVP(betas)
    ons = osamp.NoiseScheduleVP(betas, dtype=np.float32)
    ts = pu.linspace_f32(1.0, 1e-3, 101)
    assert np.array_equal(ts.view(np.uint32), osamp.torch_linspace_f32(1.0, 1e-3, 101).view(np.uint32))
    for t in ts[::7]:
        assert ns.marginal_lambda(t) == pytest.approx(float(ons.marginal_lambda(t)), rel=1e-6)
    # closed-form update coefficients == the reference-ordered update applied to random tensors
    rng = np.random.RandomState(0)
    x, m0, m1, mt = (rng.randn(4, 5) for _ in range(4))
    t_prev, t = [ts[3], ts[4]], ts[5]
    A, base, pred, corr = pu._update_coefs(ns, t_prev, t, 2, True)
    lam = lambda q: float(ons.marginal_lambda(q))
    h = lam(t) - lam(t_prev[-1])
    rk = (lam(t_prev[-2]) - lam(t_prev[-1])) / h
    hh = -h
    h_phi_1 = np.expm1(hh); B_h = np.expm1(hh)
    h_phi_k = h_phi_1 / hh - 1
    b = [h_phi_k / B_h, (h_phi_k / hh - 0.5) * 2 / B_h]
    rc = np.linalg.solve(np.array([[1.0, 1.0], [rk, 1.0]]), np.array(b))
    alpha_t, sig_t, sig_p = float(ons.marginal_alpha(t)), float(ons.marginal_std(t)), float(ons.marginal_std(t_prev[-1]))
    x_t_ = sig_t / sig_p * x - alpha_t * h_phi_1 * m0
    D1 = (m1 - m0) / rk
    want_pred = x_t_ - alpha_t * B_h * 0.5 * D1
    want_corr = x_t_ - alpha_t * B_h * (rc[0] * D1 + rc[1] * (mt - m0))
    got_pred = A * x + (base + pred[0]) * m0 + pred[1] * m1
    got_corr = A * x + (base + corr[0]) * m0 + corr[1] * m1 + corr[2] * mt
    assert rel_l2(got_pred, want_pred) < 5e-6 and rel_l2(got_corr, want_corr) < 5e-6


def test_plms_coefficients_vs_oracle():
    betas = osamp.get_noise_schedule_list("linear", 1000, 0.01)
    tab = osamp.diffusion_tables(betas)
    from fish_diffusion_b200.diffusion import PLMSNoisePredictor
    p = PLMSNoisePredictor(betas)
    rng = np.random.RandomState(1)
    x, n = rng.randn(3, 4), rng.randn(3, 4)
    for t, tp in ((990, 980), (10, 0), (500, 400)):
        cx, cn = p.coefs(t, tp)
        assert rel_l2(cx * x + cn * n, osamp.plms_x_pred(tab, x, n, t, tp)) < 1e-5


def test_mel_filterbank_product_vs_oracle():
    from oracle import mel as omel
    a = mel_filterbank(44100, 2048, 128, 40, 16000)
    b = omel.slaney_mel_filterbank(44100, 2048, 128, 40, 16000)
    assert a.shape == (128, 1025) and np.max(np.abs(a - b)) < 1e-7


def test_transposed_conv_polyphase_packing_matches_definition():
    """Host-side check of Generator._pack_convt's tap table against the scatter definition of ConvTranspose1d."""
    from oracle.nsf_hifigan import conv_transpose1d
    rng = np.random.RandomState(2)
    for (u, k) in ((8, 16), (2, 8), (2, 2), (4, 8), (2, 4)):
        Ci, Co, T = 3, 2, 9
        p = (k - u) // 2
        w = rng.randn(Ci, Co, k)
        x = rng.randn(1, Ci, T)
        want = conv_transpose1d(x, w, np.zeros(Co), u, p)[0]                  # [Co, T*u]
        dmin, dmax = -((k - 1 - p) // u), (u - 1 + p) // u
        got = np.zeros((Co, T * u))
        for q in range(T):
            for r in range(u):
                for dl in range(dmin, dmax + 1):
                    kk = r + p - dl * u
                    if 0 <= kk < k and 0 <= q + dl < T:
                        got[:, q * u + r] += w[:, :, kk].T @ x[0, :, q + dl]
        assert np.allclose(got, want, atol=1e-12), (u, k)


def test_cosine_schedule_product_buffers_bit_exact(golden, golden_cfg):
    """noise_schedule="cosine" (diffusion.py:24-29: s=0.008, clip 0.999; the golden generator used max_beta=0.02, which the
    cosine branch ignores): every product buffer equals the reference's, bit for bit."""
    cfg = golden_cfg["WN_SMALL"]
    diff = DIFFUSIONS.build(dict(type="GaussianDiffusion", denoiser=dict(type="WaveNetDenoiser", **cfg), mel_channels=16,
                                 noise_schedule="cosine", max_beta=0.02, s=0.008, spec_min=[-5.0], spec_max=[0.0]))
    g = golden("schedules")
    for k, v in diff.naive_noise_predictor.state_dict().items():
        assert np.array_equal(v.numpy().view(np.uint32), g[f"sched_cosine_naive_{k}"].view(np.uint32)), k
    assert np.array_equal(diff.plms_noise_predictor.alphas_cumprod.numpy().view(np.uint32),
                          g["sched_cosine_plms_alphas_cumprod"].view(np.uint32))
    ns = diff.unipc_noise_predictor.noise_schedule
    assert np.array_equal(ns.t_array.view(np.uint32), g["sched_cosine_unipc_t_array"].reshape(-1).view(np.uint32))
    assert np.array_equal(ns.log_alpha_array.view(np.uint32),
                          g["sched_cosine_unipc_log_alpha_array"].reshape(-1).view(np.uint32))
    for name in ("betas", "alphas_cumprod", "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod"):
        assert getattr(diff, name).dtype == torch.float32 and getattr(diff, name).shape == (1000,)


def test_reference_written_checkpoint_loads_strictly(golden_cfg):
    """A checkpoint written by the reference classes (tests/golden/ref_ckpt_small.ckpt: Lightning layout, `model.` and
    `ema_model.` prefixes) loads key for key into the native GaussianDiffusion; the vocoder checkpoint with weight-norm
    keys loads through the reference's two-format rule (nsf_hifigan.py:38-52)."""
    import os
    from conftest import GOLDEN
    from fish_diffusion_b200 import formats
    cfg = golden_cfg["WN_SMALL"]
    ck = torch.load(os.path.join(GOLDEN, "ref_ckpt_small.ckpt"), map_location="cpu", weights_only=False)
    diff = DIFFUSIONS.build(dict(type="GaussianDiffusion", denoiser=dict(type="WaveNetDenoiser", **cfg), mel_channels=16,
                                 spec_min=[-5.0], spec_max=[0.0]))
    for part in ("model", "ema_model"):
        sd = formats.lightning_state_dict(ck, part)
        res = diff.load_state_dict({k[len("diffusion."):]: v for k, v in sd.items()}, strict=True)
        assert not res.missing_keys and not res.unexpected_keys
    gsd = torch.load(os.path.join(GOLDEN, "ref_generator_small.ckpt"), map_location="cpu", weights_only=False)["generator"]
    assert any(k.endswith("weight_g") or "parametrizations" in k for k in gsd)


def test_oracle_ref_copy_is_verbatim():
    """oracle/_ref (the files the CPU baseline runs, copied by build() where the reference is installed) is byte-identical
    to the reference release the golden vectors were made from (tests/golden/ref_sha256.json)."""
    import hashlib
    import json as _json
    import os
    from conftest import GOLDEN
    from oracle.ref_loader import REF_FILES
    here = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref")
    if not os.path.isdir(here):
        pytest.skip("oracle/_ref not built: the reference is not installed on this machine")
    with open(os.path.join(GOLDEN, "ref_sha256.json")) as f:
        want = _json.load(f)
    with open(os.path.join(here, "MANIFEST.json")) as f:
        man = _json.load(f)["sha256"]
    for rel in REF_FILES:
        assert man[rel] == want[rel], rel
        with open(os.path.join(here, rel), "rb") as f:
            assert hashlib.sha256(f.read()).hexdigest() == want[rel], rel


def test_step_vectors_batched_projection_matches_per_layer_definition():
    """WaveNet.step_vectors (host torch, differentiable): the batched per-layer diffusion projections equal the reference's
    per-layer Linear calls (wavenet.py:20-27,107,170-174), values and parameter gradients."""
    import math
    import torch.nn.functional as F
    torch.manual_seed(1234)        # the draws below set the magnitudes the float32 tolerances are judged at
    net = WaveNet(mel_channels=16, d_encoder=32, residual_channels=64, residual_layers=3, use_linear_bias=True, dilation_cycle=2)
    for p in net.parameters():
        torch.nn.init.normal_(p, std=0.3)
    t = torch.tensor([3.0, 250.0, 999.0])
    d = net.step_vectors(t)
    half = 32
    e = torch.exp(torch.arange(half) * -(math.log(10000) / (half - 1)))
    s = t[:, None] * e[None]
    s = torch.cat((s.sin(), s.cos()), dim=-1)
    s = net.mlp[0].linear(s)
    s = net.mlp[2].linear(s * torch.tanh(F.softplus(s)))
    want = torch.stack([blk.diffusion_projection.linear(s) for blk in net.residual_layers], dim=1)
    assert d.shape == (3, 3, 64) and torch.allclose(d, want, rtol=1e-4, atol=1e-4)
    g = torch.randn_like(d)
    params = [p for blk in net.residual_layers for p in blk.diffusion_projection.parameters()] + list(net.mlp.parameters())
    ga = torch.autograd.grad((d * g).sum(), params, retain_graph=True)
    gb = torch.autograd.grad((want * g).sum(), params)
    for a, b in zip(ga, gb):
        assert torch.allclose(a, b, rtol=1e-4, atol=1e-4 * float(b.abs().max()))
