"""CPU tests of fish_diffusion_b200/trainers.py: the host logic of the DiffSingerLightning role (schedule, EMA update,
optimizer wiring, checkpoint layout, batch plumbing).  The model call itself is the native path and has its own GPU parity
tests (tests/test_gpu_r2_golden.py::test_diffsinger_forward_features_and_train_step_vs_reference); here a small torch
stand-in with the same call contract takes its place."""
import json
import math

import pytest
import torch
from torch import nn

from fish_diffusion_b200.formats import lightning_state_dict
from fish_diffusion_b200.trainers import DiffSingerTrainer, WarmupCosine, ema_update


def test_warmup_cosine_matches_reference_class(golden):
    kw = dict(warm_up_steps=1000, val_final=2e-5, val_base=8e-4, val_start=1e-5, max_decay_steps=300000)
    mine = WarmupCosine(**kw)
    # closed-form anchors (configs/_base_/schedulers/warmup_cosine.py:5-11)
    assert mine(0) == 1e-5 and mine(1000) == pytest.approx(8e-4, rel=1e-12) and mine(300000) == pytest.approx(2e-5, rel=1e-9)
    assert mine(10 ** 7) == mine(300000) and mine(150500) == pytest.approx(2e-5 + 0.5 * (8e-4 - 2e-5), rel=1e-9)
    # the reference LambdaWarmUpCosineScheduler's values at the same settings (tests/golden/make_golden_r2.py)
    g = golden("r2_warmup_cosine")
    assert json.loads(str(g["kwargs"])) == kw
    mine = WarmupCosine(**kw)
    for n, lr, last_lr in zip(g["steps"].tolist(), g["lr"].tolist(), g["last_lr"].tolist()):
        assert mine(n) == lr, n                               # bit-equal floats
        assert mine.last_lr == last_lr


def test_ema_update_is_the_two_foreach_ops():
    torch.manual_seed(0)
    a, b = nn.Sequential(nn.Linear(4, 3), nn.BatchNorm1d(3)), nn.Sequential(nn.Linear(4, 3), nn.BatchNorm1d(3))
    b[1].running_mean.fill_(7.0)
    before = [p.detach().clone() for p in b.parameters()]
    ema_update(b, a, 0.9)
    for p_new, p_old, p_src in zip(b.parameters(), before, a.parameters()):
        assert torch.allclose(p_new, 0.9 * p_old + 0.1 * p_src, rtol=0, atol=1e-7)
    assert float(b[1].running_mean[0]) == 7.0                 # buffers are not averaged (diffsinger.py:388-400)


class _StubDiffusion(nn.Module):
    def forward(self, features, x_masks=None, cond_masks=None):
        return features * 2.0


class _StubModel(nn.Module):
    """Same call contract as DiffSinger.forward (diffsinger.py:136-179): keyword batch fields in, dict with loss out."""

    def __init__(self):
        super().__init__()
        self.text_encoder = nn.Linear(6, 5)
        self.diffusion = _StubDiffusion()
        self.seen = None

    def forward(self, speakers, contents, contents_lens, contents_max_len, mel=None, mel_lens=None, mel_max_len=None,
                pitches=None, pitch_shift=None, phones2mel=None, energy=None):
        self.seen = dict(speakers=speakers, pitches=pitches, pitch_shift=pitch_shift, energy=energy)
        f = self.text_encoder(contents)
        return dict(loss=((f - mel) ** 2).mean() * 1e4, features=f, x_masks=None, cond_masks=None,
                    x_lens=mel_lens, metrics={"aux": torch.tensor(3.0)})


def _batch():
    g = torch.Generator().manual_seed(5)
    return dict(contents=torch.randn(2, 7, 6, generator=g), contents_lens=torch.tensor([7, 5]), contents_max_len=7,
                mel=torch.randn(2, 7, 5, generator=g), mel_lens=torch.tensor([7, 5]), mel_max_len=7,
                speaker=torch.tensor([0, 1]), key_shift=torch.zeros(2, 1))


def test_trainer_wiring_schedule_clip_ema_and_layout():
    torch.manual_seed(1)
    model = _StubModel()
    seen = []
    tr = DiffSingerTrainer(model, vocoder=nn.Linear(2, 2), ema_momentum=0.5, reduce_grads=lambda ps: seen.append(len(ps)),
                           lr_lambda=WarmupCosine(warm_up_steps=4, max_decay_steps=10))
    # checkpoint layout of the reference: model.* / ema_model.* / vocoder.*
    keys = list(tr.state_dict().keys())
    assert {k.split(".")[0] for k in keys} == {"model", "ema_model", "vocoder"}
    assert set(lightning_state_dict({"state_dict": tr.state_dict()}, "ema_model")) == set(model.state_dict())
    assert not any(p.requires_grad for p in tr.ema_model.parameters()) and not tr.ema_model.training
    opts, sched = tr.configure_optimizers()
    n_opt = sum(p.numel() for g in opts[0].param_groups for p in g["params"])
    assert n_opt == sum(p.numel() for p in model.parameters())          # frozen EMA / vocoder weights are not optimised
    assert opts[0].defaults["betas"] == (0.9, 0.98) and opts[0].defaults["eps"] == 1e-9 and sched["interval"] == "step"
    assert opts[0].defaults["weight_decay"] == 1e-2

    w0 = model.text_encoder.weight.detach().clone()
    ema0 = tr.ema_model.text_encoder.weight.detach().clone()
    lam = WarmupCosine(warm_up_steps=4, max_decay_steps=10)
    for step in range(3):
        assert opts[0].param_groups[0]["lr"] == pytest.approx(lam(step), rel=1e-12)      # lr = 1.0 * lambda(step)
        loss = tr.training_step(_batch())
        gn = math.sqrt(sum(float(p.grad.pow(2).sum()) for p in model.parameters()))
        assert gn <= 0.5 * (1 + 1e-4)                                                      # clipped to 0.5 (norm)
        assert torch.isfinite(loss)
    assert seen == [2, 2, 2] and tr.global_step == 3 and "train_loss" in tr.logged and tr.logged["train_aux"] == 3.0
    assert model.seen["speakers"] is not None and model.seen["pitches"] is None and model.seen["pitch_shift"] is not None
    assert not torch.equal(model.text_encoder.weight, w0)
    assert not torch.equal(tr.ema_model.text_encoder.weight, ema0)
    # after one more step the EMA is momentum * previous + (1 - momentum) * new weights
    prev = tr.ema_model.text_encoder.weight.detach().clone()
    tr.training_step(_batch())
    assert torch.allclose(tr.ema_model.text_encoder.weight, 0.5 * prev + 0.5 * model.text_encoder.weight, atol=1e-7)

    # validation runs on the EMA weights and samples through model.diffusion
    with torch.no_grad():
        tr.ema_model.text_encoder.weight.zero_()
        tr.ema_model.text_encoder.bias.zero_()
    out = tr.validation_step(_batch())
    assert out["loss"] == pytest.approx(float((_batch()["mel"] ** 2).mean() * 1e4), rel=1e-5)
    assert torch.count_nonzero(out["mel"]) == 0 and out["mel"].shape == (2, 7, 5) and "valid_loss" in tr.logged


def test_trainer_without_ema_uses_the_model_for_validation():
    tr = DiffSingerTrainer(_StubModel(), ema_momentum=None, gradient_clip_val=None)
    assert not hasattr(tr, "ema_model") and {k.split(".")[0] for k in tr.state_dict()} == {"model"}
    tr.training_step(_batch())
    out = tr.validation_step(_batch())
    assert out["mel"].abs().sum() > 0 and "wavs" not in out
