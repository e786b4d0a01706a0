"""CPU tests of the vocoder training path (SURVEY.md section 8f, N4).

The arithmetic of the training nodes runs on CUDA kernels only; what is checked here, without a GPU, is everything else:
  * the HOST logic of fish_diffusion_b200/vocoder_train.py (tap shifts, transposed packs, time-folded weight gradients and
    their adjoint, polyphase ConvTranspose algebra, gradient scaling, the differentiable generator assembly) with the
    device primitives swapped for the emulation in tests/native_emu.py, against torch autograd and against golden vectors
    of the UNMODIFIED reference (tests/golden/make_golden_n4.py);
  * the torch-side modules of the training step (discriminators, losses) against the reference classes' stored outputs;
  * that the product refuses CPU tensors (no fallback).
"""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import n4_util as nu
from native_emu import emulated_native

HERE = os.path.dirname(os.path.abspath(__file__))


def rel(a, b):
    a, b = a.detach().double(), b.detach().double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def _load_ckpt_generator():
    return torch.load(os.path.join(HERE, "golden", "ref_generator_small.ckpt"), map_location="cpu")["generator"]


# ------------------------------------------------------------------------------------------------ algebra
def test_fold_and_polyphase_adjoints():
    """<fold(w), G> == <w, unfold(G)> and <polyphase(w), G> == <w, polyphase_grad(G)> for random tensors: the weight
    gradients of the folded / polyphase GEMMs map back to the conv weights by the exact adjoints of the forward packs."""
    from fish_diffusion_b200 import vocoder_train as VT
    from fish_diffusion_b200.nsf_hifigan import fold_conv_weight
    rng = torch.Generator().manual_seed(0)
    for Co, Ci, K, d, Fo in ((16, 16, 7, 3, 4), (32, 32, 11, 5, 2), (8, 8, 3, 1, 8), (24, 40, 3, 2, 8)):
        w = torch.randn(Co, Ci, K, generator=rng, dtype=torch.float64)
        wf, srows = fold_conv_weight(w, d, Fo)                       # [F*Co, S*F*Ci]
        G = torch.randn(Fo * Co, len(srows), Fo * Ci, generator=rng, dtype=torch.float64)
        offs = VT.conv_offsets(K, d)
        gw = VT.unfold_weight_grad(G, Co, Ci, offs, Fo, srows)       # [Co, K, Ci]
        lhs = float((wf.reshape(Fo * Co, len(srows), Fo * Ci) * G).sum())
        rhs = float((w.permute(0, 2, 1) * gw).sum())
        assert abs(lhs - rhs) < 1e-9 * max(1.0, abs(lhs))
    for Ci, Co, k, u in ((8, 4, 8, 4), (16, 8, 16, 8), (4, 4, 4, 2), (4, 2, 2, 2)):
        p = (k - u) // 2
        w = torch.randn(Ci, Co, k, generator=rng, dtype=torch.float64)
        W3, deltas = VT.polyphase_weight(w, u, p)
        G = torch.randn(*W3.shape, generator=rng, dtype=torch.float64)
        gw = VT.polyphase_weight_grad(G, Ci, Co, k, u, p)
        assert abs(float((W3 * G).sum()) - float((w * gw).sum())) < 1e-9
        # every kernel tap appears exactly once in the polyphase matrix
        ones, _ = VT.polyphase_weight(torch.ones(Ci, Co, k, dtype=torch.float64), u, p)
        assert float(ones.sum()) == Ci * Co * k


def test_fold_factor_rules():
    from fish_diffusion_b200 import vocoder_train as VT
    assert VT.fold_factor(128, 128, 100) == 1
    assert VT.fold_factor(32, 32, 100) == 2 and VT.fold_factor(32, 32, 101) == 0
    assert VT.fold_factor(16, 16, 64) == 4 and VT.fold_factor(8, 8, 64) == 8
    assert VT.fold_factor(128, 32, 16) == 2                     # conv_pre of the small config: (256, 64)
    assert VT.fold_factor(12, 12, 64) == 0


# ------------------------------------------------------------------------------------------------ nodes vs autograd
@pytest.mark.parametrize("C,K,dil,S", [(64, 3, (1, 3, 5), 64), (16, 7, (1, 3, 5), 128), (8, 11, (1, 3, 5), 256),
                                       (32, 3, (1, 3), 64)])
def test_resblock_node_host_logic(C, K, dil, S):
    from fish_diffusion_b200 import vocoder_train as VT
    torch.manual_seed(C + K)
    cfg = VT.TrainCfg("f16")
    B = 2
    x = torch.randn(B, S, C, requires_grad=True)
    wb = []
    for _ in range(2 * len(dil)):
        wb += [(torch.randn(C, C, K) * (0.9 / (C * K) ** 0.5)).requires_grad_(), (torch.randn(C) * 0.1).requires_grad_()]
    go = torch.randn(B, S, C) * 1e-4
    with emulated_native():
        y = VT.ResBlock1Fn.apply(cfg, dil, x, *wb)
        got = torch.autograd.grad(y, [x] + wb, go)
    xr = x.detach().double().transpose(1, 2).requires_grad_()
    wr = [w.detach().double().requires_grad_() for w in wb]
    h = xr
    for m, d in enumerate(dil):
        xt = F.conv1d(F.leaky_relu(h, 0.1), wr[4 * m], wr[4 * m + 1], dilation=d, padding=(K * d - d) // 2)
        xt = F.conv1d(F.leaky_relu(xt, 0.1), wr[4 * m + 2], wr[4 * m + 3], padding=(K - 1) // 2)
        h = xt + h
    want = torch.autograd.grad(h, [xr] + wr, go.double().transpose(1, 2))
    assert rel(y, h.transpose(1, 2)) < 1e-6
    assert rel(got[0], want[0].transpose(1, 2)) < 1e-6
    for a, b in zip(got[1:], want[1:]):
        assert a.shape == b.shape and rel(a, b) < 1e-6


@pytest.mark.parametrize("Ci,Co,k,u,L", [(128, 64, 8, 4, 16), (32, 16, 4, 2, 64), (16, 8, 4, 2, 64), (32, 16, 2, 2, 64)])
def test_conv_transpose_node_host_logic(Ci, Co, k, u, L):
    from fish_diffusion_b200 import vocoder_train as VT
    torch.manual_seed(Ci + k)
    cfg = VT.TrainCfg("f16")
    p = (k - u) // 2
    x = torch.randn(2, L, Ci, requires_grad=True)
    w = (torch.randn(Ci, Co, k) * 0.1).requires_grad_()
    b = torch.randn(Co).requires_grad_()
    with emulated_native():
        y = VT.ConvTranspose1dFn.apply(cfg, u, p, x, w, b)
        go = torch.randn_like(y) * 1e-3
        got = torch.autograd.grad(y, [x, w, b], go)
    xr, wr, br = (t.detach().double().requires_grad_() for t in (x.transpose(1, 2), w, b))
    h = F.conv_transpose1d(xr, wr, br, stride=u, padding=p)
    want = torch.autograd.grad(h, [xr, wr, br], go.double().transpose(1, 2))
    assert rel(y, h.transpose(1, 2)) < 1e-6 and rel(got[0], want[0].transpose(1, 2)) < 1e-6
    assert rel(got[1], want[1]) < 1e-6 and rel(got[2], want[2]) < 1e-6


def test_conv_node_host_logic_and_unsupported_shape():
    from fish_diffusion_b200 import _native as N
    from fish_diffusion_b200 import vocoder_train as VT
    cfg = VT.TrainCfg("f16")
    torch.manual_seed(3)
    x = torch.randn(2, 32, 32, requires_grad=True)
    w = (torch.randn(128, 32, 7) * 0.1).requires_grad_()
    b = torch.randn(128).requires_grad_()
    with emulated_native():
        y = VT.Conv1dFn.apply(cfg, 1, x, w, b)
        go = torch.randn_like(y) * 1e-3
        got = torch.autograd.grad(y, [x, w, b], go)
        # 16 channels need a time-fold of 4, which does not divide 66 steps: a loud error, not a silent fallback
        with pytest.raises(N.NativeError):
            y2 = VT.Conv1dFn.apply(cfg, 1, torch.randn(1, 66, 16, requires_grad=True),
                                   torch.randn(16, 16, 3).requires_grad_(), torch.zeros(16).requires_grad_())
            y2.sum().backward()
    xr, wr, br = (t.detach().double().requires_grad_() for t in (x.transpose(1, 2), w, b))
    h = F.conv1d(xr, wr, br, padding=3)
    want = torch.autograd.grad(h, [xr, wr, br], go.double().transpose(1, 2))
    assert rel(y, h.transpose(1, 2)) < 1e-6 and rel(got[0], want[0].transpose(1, 2)) < 1e-6
    assert rel(got[1], want[1]) < 1e-6 and rel(got[2], want[2]) < 1e-6


# ------------------------------------------------------------------------------------------------ vs the reference
def _draws(seed, shapes):
    rng = np.random.RandomState(seed)
    return [torch.from_numpy((rng.rand(*s) if i == 0 else rng.randn(*s)).astype(np.float32)) for i, s in enumerate(shapes)]


@pytest.mark.parametrize("name,wav_tol,worst_tol,median_tol", [("n4_gen_init", 1e-6, 5e-3, 1e-4), ("n4_gen", 1e-4, 1.5e-2, 4e-3)])
def test_generator_gradients_vs_reference_golden(golden, name, wav_tol, worst_tol, median_tol):
    """Host logic of the differentiable generator (emulated device primitives) against the float64 reference Generator's
    autograd under a smooth loss: every weight-norm parameter gradient.
      n4_gen_init  the reference's own initialisation (checkpoint / 3): well conditioned, the reference's float32 runs sit
                   7e-8 (audio) / 3.6e-6 worst gradient from float64 -- apart from single LeakyReLU mask flips of near-zero
                   activations, which move one conv's gradients by ~5e-4 (seen in the reference's 8-thread run as well);
      n4_gen       3x those weights: the final tanh saturates (rms 0.9998) and the gradient is chaotic -- the reference's own
                   float32 runs disagree with float64 by 9.9e-3 worst / 2.6e-3 median (8 threads), 1.4e-3 / 8.6e-4 (1)."""
    from fish_diffusion_b200 import Generator
    from fish_diffusion_b200 import vocoder_train as VT
    g = golden(name)
    gen = Generator(nu.train_config())
    gen.load_state_dict({k: v * float(g["weight_scale"]) for k, v in _load_ckpt_generator().items()}, strict=True)
    mel, f0 = torch.from_numpy(g["mels"]), torch.from_numpy(g["pitches"])
    B, S = mel.shape[0], mel.shape[2] * 64
    ri, nz = _draws(nu.SEED_DRAWS + 1, [(B, 9), (B, S, 9)])
    gw = torch.from_numpy(np.random.RandomState(int(g["gw_seed"])).randn(B, 1, S).astype(np.float32))
    with emulated_native():
        wav = VT.generator_forward_train(gen, mel, f0, VT.TrainCfg("f16"), rand_ini=ri, sine_noise=nz)
        (wav * gw).sum().backward()
    e_wav = rel(wav, torch.from_numpy(g["wav"]))
    print(f"[{name}] wav vs float64 reference {e_wav:.2e} (reference float32: {float(g['noise_f32_wav']):.2e})")
    assert e_wav < wav_tol
    nu.check_gradients(g, [(n, p.grad.numpy()) for n, p in gen.named_parameters()], "grad_", worst_tol, median_tol,
                       f"[{name}] generator gradients (emulated primitives) vs float64 reference")


def test_training_step_vs_reference_golden(golden):
    """One whole training step (discriminator update + generator update) against the reference's unmodified
    HSFHifiGAN.training_step: logged losses tightly; gradients loosely -- the L1 / max-pool losses make dL/d(audio) jump
    by ~6 % under a 1e-7 perturbation of the generated audio (measured on the reference)."""
    from fish_diffusion_b200.vocoder_gan import HifiGanTrainer
    g = golden("n4_train")
    tr = HifiGanTrainer(nu.train_config(), precision="f16")
    tr.generator.load_state_dict(_load_ckpt_generator(), strict=True)
    nu.fill_discriminators(tr.mpd, tr.msd)
    tr.train()
    batch = nu.make_batch()
    batch["mels"] = torch.from_numpy(g["mels"])
    B, S = batch["audio"].shape[0], batch["audio"].shape[2]
    ri, nz = _draws(nu.SEED_DRAWS, [(B, 9), (B, S, 9)])
    with emulated_native():
        out = tr.training_step(batch, rand_ini=ri, sine_noise=nz)
    assert abs(out["loss_disc"] - float(g["log_train_loss_disc"])) < 1e-4 * float(g["log_train_loss_disc"])
    assert abs(out["loss_gen"] - float(g["log_train_loss_gen"])) < 1e-4 * float(g["log_train_loss_gen"])
    assert abs(out["envelope"] - float(g["log_train_loss_g_envelope"])) < 1e-5
    for prefix, sub in (("generator", tr.generator), ("mpd", tr.mpd), ("msd", tr.msd)):
        nu.check_gradients(g, [(n, p.grad.numpy()) for n, p in sub.named_parameters()], f"grad_{prefix}.", 0.25, 0.05,
                           f"training-step gradients of {prefix} vs reference")
    # the optimisers moved the parameters
    sd0 = _load_ckpt_generator()
    assert any(not torch.equal(v, sd0[k]) for k, v in tr.generator.state_dict().items())


def test_discriminators_and_losses_match_reference_bit_for_bit(golden):
    """Same state_dict names and shapes as the reference discriminators, and the same logits, feature maps and losses on
    the same weights and inputs (tests/golden/n4_disc.npz).  Run side by side with the reference classes the outputs are
    bit-equal; against the stored outputs the bound is the float32 rounding that oneDNN's convolutions vary in between
    CPUs and thread counts (recorded next to the golden as noise_<tag>, 1e-6)."""
    from fish_diffusion_b200 import vocoder_gan as G
    g = golden("n4_disc")
    y, yh = (torch.from_numpy(a) for a in nu.disc_inputs())
    for tag, mine in (("mpd", G.MultiPeriodDiscriminator([3, 5])), ("msd", G.MultiScaleDiscriminator())):
        shapes = {k: tuple(int(n) for n in s if n) for k, s in zip(g[f"{tag}_keys"], g[f"{tag}_shapes"])}
        assert shapes == {k: tuple(v.shape) for k, v in mine.state_dict().items()}
        nu.fill_discriminators(mine)
        mine.train()
        d_r, d_g, f_r, f_g = mine(y, yh)
        for side, logits, fmaps in (("r", d_r, f_r), ("g", d_g, f_g)):
            assert len(logits) == len(fmaps) == len([k for k in g if k.startswith(f"{tag}_logit_{side}")])
            for i, t in enumerate(logits):
                assert rel(t, torch.from_numpy(g[f"{tag}_logit_{side}{i}"])) < 1e-5, (tag, side, i)
            for i, maps in enumerate(fmaps):
                assert len(maps) == len([k for k in g if k.startswith(f"{tag}_fmap_{side}{i}_") and k.endswith("_norm")])
                for j, t in enumerate(maps):
                    assert nu.summary_error(g, f"{tag}_fmap_{side}{i}_{j}", t.detach().numpy()) < 1e-5, (tag, side, i, j)
        for name, got in (("feature_loss", G.feature_loss(f_r, f_g)), ("discriminator_loss", G.discriminator_loss(d_r, d_g)[0]),
                          ("generator_loss", G.generator_loss(d_g)[0])):
            want = float(g[f"{tag}_{name}"])
            assert abs(float(got) - want) <= 1e-5 * abs(want), (tag, name, float(got), want)


def test_trainer_state_dict_layout():
    """`generator.*`, `mpd.*`, `msd.*` and nothing else: the loss-side mel transforms are not registered (the reference keeps
    them in a plain list, train.py:55-75), so the three networks of a reference Lightning checkpoint map key for key."""
    from fish_diffusion_b200.vocoder_gan import HifiGanTrainer
    tr = HifiGanTrainer(nu.train_config())
    keys = list(tr.state_dict().keys())
    assert all(k.split(".")[0] in ("generator", "mpd", "msd") for k in keys)
    assert {k[len("generator."):] for k in keys if k.startswith("generator.")} == set(_load_ckpt_generator().keys())
    assert len(tr.mpd.discriminators) == 2 and len(tr.msd.discriminators) == 3
    opts, scheds = tr.configure_optimizers()
    assert opts[0].defaults["lr"] == 0.0002 and opts[0].defaults["betas"] == (0.8, 0.99) and scheds[0].gamma == 0.999
    n_g = sum(p.numel() for g in opts[0].param_groups for p in g["params"])
    assert n_g == sum(p.numel() for p in tr.generator.parameters())


def test_training_nodes_refuse_cpu_tensors():
    """No CPU path: without the emulation the nodes raise on CPU tensors."""
    from fish_diffusion_b200 import Generator, _native
    from fish_diffusion_b200 import vocoder_train as VT
    gen = Generator(nu.train_config())
    with pytest.raises(_native.NativeError):
        VT.generator_forward_train(gen, torch.zeros(1, 32, 8), torch.zeros(1, 8))
    with pytest.raises(_native.NativeError):
        VT.ResBlock1Fn.apply(VT.TrainCfg(), (1,), torch.zeros(1, 8, 8), torch.zeros(8, 8, 3), torch.zeros(8),
                             torch.zeros(8, 8, 3), torch.zeros(8))


def test_generator_forward_train_argument_checks():
    """Loud errors of the differentiable generator (host logic): ResBlock2 generators have no native backward, and a
    config whose hop_size disagrees with its upsample rates is refused (models.py:411 relies on their equality)."""
    from fish_diffusion_b200 import Generator
    from fish_diffusion_b200 import vocoder_train as VT
    h = nu.train_config()
    mel, f0 = torch.zeros(1, 32, 4), torch.full((1, 4), 200.0)
    with emulated_native():
        gen2 = Generator(dict(h, resblock="2", resblock_dilation_sizes=[[1, 3]] * 3))
        with pytest.raises(NotImplementedError):
            VT.generator_forward_train(gen2, mel, f0)
        bad = Generator(dict(h, hop_size=128))
        with pytest.raises(ValueError):
            VT.generator_forward_train(bad, mel, f0)
        wav = VT.generator_forward_train(Generator(h), mel, f0[:, None])          # [B,1,T] pitches as the data loader gives
        assert wav.shape == (1, 1, 4 * 64) and wav.requires_grad
