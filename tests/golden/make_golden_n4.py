"""N4 golden vectors: ONE vocoder training step of the UNMODIFIED reference (tools/nsf_hifigan/train.py,
`HSFHifiGAN.training_step`, lines 114-231) on CPU.  Run in the build container:  python tests/golden/make_golden_n4.py

The file imports pytorch_lightning, wandb, matplotlib, mmengine and fish_diffusion package paths that do not exist in
this image; those NAMES are stubbed (a minimal LightningModule base with optimizers() / manual_backward() / log() /
lr_schedulers(), empty modules for the loggers and plotting) -- every executed line of the step, the generator, the
discriminators and the losses is the reference's own code (models.py, utils/audio.py loaded by file path).

  n4_train.npz   inputs (batch from tests/n4_util.make_batch, generator weights = ref_generator_small.ckpt, discriminator
                 weights = n4_util.fill_discriminators, random draws = RandomState(SEED_DRAWS) in call order),
                 the generator's input mel and output audio, the three logged losses, and norm + 256 sampled entries of
                 every gradient left on the generator and the discriminators after the step.
  n4_disc.npz    MultiPeriodDiscriminator([3, 5]) and MultiScaleDiscriminator() of the reference in train mode: state_dict
                 names and shapes, the logits, norm + 256 sampled entries of every feature map, and the three losses on
                 n4_util.disc_inputs() with n4_util.fill_discriminators weights.
"""
import json
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

import make_golden as mg  # noqa: E402
import n4_util as nu  # noqa: E402

REF = mg.REF


class _Any:
    def __getattr__(self, k):
        return _Any()

    def __call__(self, *a, **k):
        return _Any()


def _stub(name, **attrs):
    m = sys.modules.get(name) or types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


class FakeLightningModule(torch.nn.Module):
    """The five members of pl.LightningModule that training_step touches under manual optimisation."""

    def __init__(self):
        super().__init__()
        self.logged = {}
        self.trainer = types.SimpleNamespace(is_last_batch=False)
        self.logger = None
        self.global_step = 0
        self._opt = None

    def _conf(self):
        if self._opt is None:
            self._opt = self.configure_optimizers()
        return self._opt

    def optimizers(self):
        return self._conf()[0]

    def lr_schedulers(self):
        return self._conf()[1]

    def manual_backward(self, loss):
        loss.backward()

    def log(self, name, value, **kw):
        self.logged[name] = float(value)


class Cfg(dict):
    __getattr__ = dict.__getitem__


def load_reference_trainer():
    ref = mg.load_reference()
    _stub("matplotlib"); _stub("matplotlib.pyplot", close=lambda *a, **k: None)
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    pl = _stub("pytorch_lightning", LightningModule=FakeLightningModule, Trainer=_Any(), seed_everything=lambda *a, **k: None)
    _stub("pytorch_lightning.loggers", TensorBoardLogger=type("TensorBoardLogger", (), {}), WandbLogger=type("WandbLogger", (), {}))
    pl.loggers = sys.modules["pytorch_lightning.loggers"]
    _stub("wandb")
    _stub("mmengine", Config=_Any())
    for mod in ("librosa", "fish_audio_preprocess", "fish_audio_preprocess.utils"):
        _stub(mod)
    sys.modules["fish_audio_preprocess.utils"].loudness_norm = None
    sys.modules["fish_audio_preprocess.utils"].separate_audio = None
    au = mg._load("ref_audio_utils", f"{REF}/fish_diffusion/utils/audio.py")
    _stub("fish_diffusion"); _stub("fish_diffusion.datasets"); _stub("fish_diffusion.modules")
    _stub("fish_diffusion.datasets.utils", build_loader_from_config=_Any())
    _stub("fish_diffusion.modules.vocoders"); _stub("fish_diffusion.modules.vocoders.nsf_hifigan")
    sys.modules["fish_diffusion.modules.vocoders.nsf_hifigan.models"] = ref.nsf
    _stub("fish_diffusion.utils")
    sys.modules["fish_diffusion.utils.audio"] = au
    _stub("fish_diffusion.utils.viz", plot_mel=_Any())
    tr = mg._load("ref_nsf_train", f"{REF}/tools/nsf_hifigan/train.py")
    # train.py:28-29 switches float32 matmuls to "medium" (TF32 on GPUs; on CPU oneDNN's reduced-precision mode, which moved
    # the generator output by 1.4e-5 here).  The golden vectors are the reference's arithmetic in full fp32.
    torch.set_float32_matmul_precision("highest")
    return ref, tr


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)
    ref, tr = load_reference_trainer()
    h = nu.train_config()
    cfg_path = os.path.join(HERE, "n4_train_config.json")
    with open(cfg_path, "w") as f:
        json.dump(h, f)
    config = Cfg(model=Cfg(config=cfg_path), hop_length=h["hop_size"])
    mod = tr.HSFHifiGAN(config)
    sd = torch.load(os.path.join(HERE, "ref_generator_small.ckpt"), map_location="cpu")["generator"]
    print(mod.generator.load_state_dict(sd, strict=True))
    nu.fill_discriminators(mod.mpd, mod.msd)
    mod.train()
    batch = nu.make_batch()
    cap = {}
    mod.generator.register_forward_pre_hook(lambda m, a: cap.__setitem__("in", [t.detach().clone() for t in a]))
    calls = []
    mod.generator.register_forward_hook(lambda m, a, o: calls.append(o.detach().clone()))
    out = {}
    # validation_step (train.py:241-270) first, on the initial weights; its plotting / logging tail runs on stubs
    with mg.RecordedRandom(nu.SEED_DRAWS + 2), torch.no_grad():
        mod.validation_step(batch, 0)
    out["log_valid_loss"] = np.float64(mod.logged["valid_loss"])
    out["valid_wav"] = calls[-1].numpy()
    calls.clear()
    with mg.RecordedRandom(nu.SEED_DRAWS) as rr:
        mod.training_step(batch, 0)
    print("draws:", [(k, a.shape) for k, a in rr.log])
    out["draw_kinds"] = np.array([k for k, _ in rr.log])
    out["draw_shapes"] = np.array([list(a.shape) + [0] * (4 - a.ndim) for _, a in rr.log], dtype=np.int64)
    out["mels"], out["pitches"] = cap["in"][0].numpy(), cap["in"][1].numpy()
    out["wav"] = calls[0].numpy()
    for k, v in mod.logged.items():
        out["log_" + k] = np.float64(v)
    print(mod.logged)
    i = 0
    for prefix, sub in (("generator", mod.generator), ("mpd", mod.mpd), ("msd", mod.msd)):
        for n, p in sub.named_parameters():
            assert p.grad is not None, n
            nu.summarize(out, f"grad_{prefix}.{n}", p.grad.numpy(), 4300 + i)
            i += 1
    np.savez_compressed(os.path.join(HERE, "n4_train.npz"), **out)
    print("n4_train.npz:", os.path.getsize(os.path.join(HERE, "n4_train.npz")) // 1024, "KiB,", i, "gradients")
    gold_generator_grads(ref, sd, out["mels"], out["pitches"], 1.0, "n4_gen.npz")
    # the checkpoint holds 3x the reference's initial weights (round-2 golden: audible output), which saturates the final
    # tanh (rms 0.9998); a third of it is the reference's own initialisation -- a well-conditioned operating point
    gold_generator_grads(ref, {k: v / 3 for k, v in sd.items()}, out["mels"], out["pitches"], 1.0 / 3, "n4_gen_init.npz")
    gold_discriminators(ref)


def gold_discriminators(ref):
    """n4_disc.npz: the reference discriminators' forward in float32 (8 threads).  oneDNN's grouped convolutions of the
    multi-scale discriminator round differently with the thread count, so the same module on the same CPU moves in the
    last bits; the largest such move over 1, 3 and 8 threads is stored as `noise_<tag>`."""
    out = {}
    y, yh = (torch.from_numpy(a) for a in nu.disc_inputs())
    for tag, make in (("mpd", lambda: ref.nsf.MultiPeriodDiscriminator([3, 5])), ("msd", ref.nsf.MultiScaleDiscriminator)):
        runs = {}
        for nt in (1, 3, 8):
            torch.set_num_threads(nt)
            m = make()
            nu.fill_discriminators(m)
            m.train()
            with torch.no_grad():
                runs[nt] = m(y, yh)
        sd = m.state_dict()
        out[f"{tag}_keys"] = np.array(list(sd))
        out[f"{tag}_shapes"] = np.array([list(v.shape) + [0] * (4 - v.dim()) for v in sd.values()], dtype=np.int64)
        d_r, d_g, f_r, f_g = runs[8]
        noise = 0.0
        for side, logits, fmaps in (("r", d_r, f_r), ("g", d_g, f_g)):
            for i, t in enumerate(logits):
                out[f"{tag}_logit_{side}{i}"] = t.numpy()
                for nt in (1, 3):
                    o = runs[nt][0 if side == "r" else 1][i]
                    noise = max(noise, float((o - t).norm() / t.norm()))
            for i, maps in enumerate(fmaps):
                for j, t in enumerate(maps):
                    nu.summarize(out, f"{tag}_fmap_{side}{i}_{j}", t.numpy(), 4600 + 10 * i + j)
                    for nt in (1, 3):
                        o = runs[nt][2 if side == "r" else 3][i][j]
                        noise = max(noise, float((o - t).norm() / t.norm()))
        out[f"noise_{tag}"] = np.float64(noise)
        out[f"{tag}_feature_loss"] = np.float64(float(ref.nsf.feature_loss(f_r, f_g)))
        out[f"{tag}_discriminator_loss"] = np.float64(float(ref.nsf.discriminator_loss(d_r, d_g)[0]))
        out[f"{tag}_generator_loss"] = np.float64(float(ref.nsf.generator_loss(d_g)[0]))
        print(f"  {tag}: thread-count noise {noise:.2e}")
    torch.set_num_threads(8)
    np.savez_compressed(os.path.join(HERE, "n4_disc.npz"), **out)
    print("n4_disc.npz:", os.path.getsize(os.path.join(HERE, "n4_disc.npz")) // 1024, "KiB")


def gold_generator_grads(ref, sd, mels, pitches, scale, fname):
    """n4_gen.npz: gradients of the reference Generator (weight-norm parameters) under a SMOOTH loss sum(wav * gw), from
    the reference module in FLOAT64 (the arbiter, SURVEY.md section 8c).  Why float64 and why loose tolerances downstream:
    at this operating point the gradient is ill-conditioned -- LeakyReLU masks of near-zero activations flip under 1e-7
    forward noise -- and the reference's own float32 runs disagree with each other (1 thread vs 8 threads of oneDNN: 2e-5 on
    the audio, 1.1e-2 on the worst parameter gradient, 2.6e-3 median) and with float64 (1-thread float32: 1.4e-3 worst,
    9e-4 median).  The stored `noise_*` keys record that floor.  That is the 3x-initialisation checkpoint, whose output
    saturates the final tanh; at the reference's own initialisation (weights / 3, `n4_gen_init.npz`) the same comparison is
    well conditioned (float32 vs float64: 7e-8 on the audio, 3.5e-6 worst gradient) and pins the backward tightly.  The training losses proper (L1 / max-pool terms) are
    even less smooth: dL/d(audio) moves by ~6 % under a 1e-7 perturbation of the generated audio."""
    h = nu.train_config()
    out = {"mels": mels, "pitches": pitches, "gw_seed": np.array(4400), "weight_scale": np.float64(scale)}
    gw = np.random.RandomState(4400).randn(mels.shape[0], 1, mels.shape[2] * h["hop_size"])
    runs = {}
    for tag, dt, nt in (("f64", torch.float64, 8), ("f32", torch.float32, 8), ("f32_1t", torch.float32, 1)):
        torch.set_num_threads(nt)
        gen = ref.nsf.Generator(ref.nsf.AttrDict(h))
        gen.load_state_dict(sd, strict=True)
        gen = gen.to(dt).train()
        with mg.RecordedRandom(nu.SEED_DRAWS + 1) as rr:
            wav = gen(torch.from_numpy(mels).to(dt), torch.from_numpy(pitches).to(dt))
        (wav * torch.from_numpy(gw).to(dt)).sum().backward()
        runs[tag] = (wav.detach().double().numpy(), [(n, p.grad.double().numpy()) for n, p in gen.named_parameters()])
    torch.set_num_threads(8)
    wav64, grads64 = runs["f64"]
    out["wav"] = wav64.astype(np.float32)
    out["draw_shapes"] = np.array([list(a.shape) + [0] * (4 - a.ndim) for _, a in rr.log], dtype=np.int64)
    for i, (n, gr) in enumerate(grads64):
        nu.summarize(out, f"grad_{n}", gr, 4500 + i)
    for tag in ("f32", "f32_1t"):
        w, gs = runs[tag]
        errs = sorted(np.linalg.norm(a - b) / np.linalg.norm(b) for (_, a), (_, b) in zip(gs, grads64))
        out[f"noise_{tag}_wav"] = np.float64(np.linalg.norm(w - wav64) / np.linalg.norm(wav64))
        out[f"noise_{tag}_grad_worst"], out[f"noise_{tag}_grad_median"] = np.float64(errs[-1]), np.float64(errs[len(errs) // 2])
        print(f"  reference {tag} vs f64: wav {out[f'noise_{tag}_wav']:.2e}, grads worst {errs[-1]:.2e} median {errs[len(errs) // 2]:.2e}")
    out["wav_rms"] = np.float64(np.sqrt(np.mean(wav64 ** 2)))
    np.savez_compressed(os.path.join(HERE, fname), **out)
    print(f"{fname}: {os.path.getsize(os.path.join(HERE, fname)) // 1024} KiB, wav rms {out['wav_rms']:.4f}")


if __name__ == "__main__":
    main()
