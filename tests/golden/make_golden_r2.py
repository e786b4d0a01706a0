"""Round-2 golden vectors, again from the UNMODIFIED reference imported by file path (see make_golden.py for the loader
and the recorded-random machinery).  Run in the build container:  python tests/golden/make_golden_r2.py

  r2_traj.npz        100-step naive (DDPM) and UniPC sampler trajectories (sampler_interval=10, the BASELINE configs[1]
                     schedule) at a tensor-core-eligible width (WN_TC).  Noise is NOT stored: every draw of the reference
                     is served from np.random.RandomState(seed) in call order, and the test re-draws the same stream.
  r2_train_full.npz  full-width (M=128, E=256, C=512, L=20) training-step gradients through the reference's autograd at
                     B=1, T=128: per parameter the L2 norm and 256 seeded sample entries (the full set is 220 MB).
  r2_train_masked.npz  WaveNet.forward with x_masks / cond_masks under grad (wavenet.py:217-221,233-234): output and the
                     gradients w.r.t. x, the conditioner and every parameter (WN_TC width; norm + samples).
  r2_voc.npz         Generator(config_v1.json) and Generator(config_v1_256.json) at B=1, T=128 (config #3's training
                     segment); SineGen noise by seed as above.
  r2_voc_resblock2.npz  a small Generator with `resblock: "2"` (ResBlock2, models.py:119-158).
  r2_audio.npz       utils/audio.py get_mel_transform / get_mel_from_audio / dynamic_range_compression (torchaudio
                     MelSpectrogram variant used by the training losses); librosa / fish_audio_preprocess are stubbed,
                     the executed code path touches neither.
  r2_diffsinger.npz  archs/diffsinger/diffsinger.py DiffSinger.forward_features / forward (+ NaiveProjectionEncoder,
                     pitch_to_scale) with the un-importable Lightning-side names stubbed: features, masks, loss, encoder grads.
  r2_warmup_cosine.npz  schedulers/warmup_cosine_scheduler.py: the learning-rate multiplier over a set of steps.
  ref_ckpt_small.ckpt / ref_generator_small.ckpt   checkpoints WRITTEN by the reference classes (state_dict of the
                     reference GaussianDiffusion under Lightning's `model.diffusion.` prefix with an `ema_model.` copy; the
                     reference Generator with weight-norm keys as {"generator": ...}) plus the reference outputs.
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

import make_golden as mg  # noqa: E402
from oracle import nsf_hifigan as ovoc  # noqa: E402

REF = mg.REF
SAMPLES = 256


def summarize(out, key, arr, seed):
    """norm + SAMPLES seeded entries of a gradient tensor (flat indices from RandomState(seed))."""
    a = np.asarray(arr, dtype=np.float32).reshape(-1)
    idx = np.random.RandomState(seed).randint(0, a.size, size=min(SAMPLES, a.size))
    out[key + "_norm"] = np.float64(np.linalg.norm(a.astype(np.float64)))
    out[key + "_idx"] = idx.astype(np.int64)
    out[key + "_val"] = a[idx]


def gold_traj(ref, out):
    cfg = mg.WN_TC
    sd = mg.wn_weights(61, cfg)
    B, T, M, E = 1, 64, cfg["mel_channels"], cfg["d_encoder"]
    feats = np.random.RandomState(62).randn(B, T, E).astype(np.float32)
    out["traj_features"] = feats
    for pred, seed in (("naive", 2001), ("unipc", 2002)):
        diff = ref.diffusion.GaussianDiffusion(
            denoiser=dict(type="WaveNetDenoiser", **cfg), mel_channels=M, noise_schedule="linear", timesteps=1000,
            max_beta=0.01, noise_loss="smoothed-l1", sampler_interval=10, spec_min=[-5.0], spec_max=[0.0],
            noise_predictor=pred)
        diff.denoise_fn.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
        diff.eval()
        with mg.RecordedRandom(seed) as rr, torch.no_grad():
            y = diff(torch.from_numpy(feats), sampler_interval=10, noise_predictor=pred)
        out[f"traj_{pred}_mel"] = y.numpy()
        out[f"traj_{pred}_seed"] = np.array(seed)
        out[f"traj_{pred}_draws"] = np.array([list(a.shape) + [0] * (4 - a.ndim) for _, a in rr.log], dtype=np.int64)
        out[f"traj_{pred}_kinds"] = np.array([k for k, _ in rr.log])
        print(f"  traj {pred}: {len(rr.log)} draws, mel range [{y.min():.3f}, {y.max():.3f}]")


def gold_train_full(ref, out):
    cfg = mg.WN_FULL
    M, E = cfg["mel_channels"], cfg["d_encoder"]
    sd = mg.wn_weights(71, cfg)
    diff = ref.diffusion.GaussianDiffusion(
        denoiser=dict(type="WaveNetDenoiser", **cfg), mel_channels=M, noise_loss="smoothed-l1", sampler_interval=10,
        spec_min=[-5.0], spec_max=[0.0])
    diff.denoise_fn.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    B, T = 1, 128
    rng = np.random.RandomState(72)
    feats = torch.from_numpy(rng.randn(B, T, E).astype(np.float32)).requires_grad_(True)
    mel = (rng.rand(B, T, M).astype(np.float32) * 5 - 5)
    t = torch.tensor([321], dtype=torch.long)
    noise = rng.randn(B, M, T).astype(np.float32)
    x = diff.norm_spec(torch.from_numpy(mel)).transpose(1, 2)
    noised, eps, loss = diff.p_losses(x, t, feats.transpose(1, 2), noise=torch.from_numpy(noise))
    loss.backward()
    out["tf_features"], out["tf_mel"], out["tf_t"], out["tf_noise"] = feats.detach().numpy(), mel, t.numpy(), noise
    out["tf_loss"] = loss.detach().numpy()
    out["tf_eps"] = eps.detach().numpy()
    out["tf_gfeatures"] = feats.grad.numpy()
    for i, (k, p) in enumerate(diff.denoise_fn.named_parameters()):
        summarize(out, f"tf_g_{k}", p.grad.numpy(), 7000 + i)
    # float64 arbiter of the same gradients (bounds the fp32 accumulation-order noise of either implementation)
    diff64 = ref.diffusion.GaussianDiffusion(
        denoiser=dict(type="WaveNetDenoiser", **cfg), mel_channels=M, noise_loss="smoothed-l1", sampler_interval=10,
        spec_min=[-5.0], spec_max=[0.0]).double()
    diff64.denoise_fn.load_state_dict({k: torch.from_numpy(v).double() for k, v in sd.items()})
    f64 = feats.detach().double().requires_grad_(True)
    x64 = diff64.norm_spec(torch.from_numpy(mel).double()).transpose(1, 2)
    # p_losses (diffusion.py:129-151) restated for the arbiter only: DiffusionEmbedding needs a float64 step to stay in
    # float64 (SURVEY 8c), while q_sample's gather needs the long one
    n64 = torch.from_numpy(noise).double()
    x_t = diff64.q_sample(x_start=x64, t=t, noise=n64)
    eps64 = diff64.denoise_fn(x_t, t.double(), f64.transpose(1, 2))
    loss64 = torch.nn.functional.smooth_l1_loss(n64, eps64)
    loss64.backward()
    for i, (k, p) in enumerate(diff64.denoise_fn.named_parameters()):
        summarize(out, f"tf64_g_{k}", p.grad.numpy().astype(np.float32), 7000 + i)
    print(f"  train_full: loss {float(loss):.6f} / f64 {float(loss64):.6f}")


def gold_train_masked(ref, out):
    cfg = mg.WN_TC
    sd = mg.wn_weights(81, cfg)
    net = ref.wavenet.WaveNet(**cfg)
    net.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    B, T = 2, 200
    rng = np.random.RandomState(82)
    x = torch.from_numpy(rng.randn(B, cfg["mel_channels"], T).astype(np.float32)).requires_grad_(True)
    c = torch.from_numpy(rng.randn(B, cfg["d_encoder"], T).astype(np.float32)).requires_grad_(True)
    masks = np.zeros((B, T), dtype=bool)
    masks[0, T - 31:] = True
    masks[1, T - 3:] = True
    steps = torch.tensor([12, 777], dtype=torch.long)
    y = net(x, steps, c, x_masks=torch.from_numpy(masks), cond_masks=torch.from_numpy(masks))
    w = torch.from_numpy(rng.randn(*y.shape).astype(np.float32))
    loss = (y * w).sum() / y.numel()
    loss.backward()
    out["tm_x"], out["tm_c"], out["tm_masks"], out["tm_steps"], out["tm_w"] = (x.detach().numpy(), c.detach().numpy(), masks,
                                                                              steps.numpy(), w.numpy())
    out["tm_y"], out["tm_loss"] = y.detach().numpy(), loss.detach().numpy()
    out["tm_gx"], out["tm_gc"] = x.grad.numpy(), c.grad.numpy()
    for k, p in net.named_parameters():
        out[f"tm_g_{k}"] = p.grad.numpy()


def gold_voc(ref, out):
    for name, seed in (("config_v1", 91), ("config_v1_256", 92)):
        with open(f"{REF}/tools/nsf_hifigan/{name}.json") as f:
            hd = json.load(f)
        h = ref.nsf.AttrDict(hd)
        sd = ovoc.make_generator_weights(seed, hd)
        gen = ref.nsf.Generator(h)
        gen.remove_weight_norm()
        gen.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()}, strict=True)
        gen.eval()
        rng = np.random.RandomState(seed + 100)
        B, T = 1, 128
        mel = (rng.randn(B, h.num_mels, T) - 2.5).clip(-11.5, 2).astype(np.float32)
        f0 = mg.f0_contour(rng, B, T)
        with mg.RecordedRandom(seed + 200) as rr, torch.no_grad():
            wav = gen(torch.from_numpy(mel), torch.from_numpy(f0))
        kinds = [k for k, _ in rr.log]
        assert kinds == ["rand", "randn_like", "randn_like"], kinds
        out[f"voc_{name}_mel"], out[f"voc_{name}_f0"], out[f"voc_{name}_wav"] = mel, f0, wav.numpy()
        out[f"voc_{name}_wseed"], out[f"voc_{name}_rseed"] = np.array(seed), np.array(seed + 200)
        print(f"  voc {name}: wav {tuple(wav.shape)} rms {float(wav.pow(2).mean().sqrt()):.4f}")


def gold_voc_resblock2(ref, out):
    """Generator with `resblock: "2"` (ResBlock2, models.py:119-158: two dilated convs, one conv per residual) -- the variant
    the shipped JSON configs do not use."""
    hd = dict(mg.VOC_SMALL, resblock="2", resblock_dilation_sizes=[[1, 3], [1, 3], [1, 3]])
    h = ref.nsf.AttrDict(hd)
    torch.manual_seed(141)
    gen = ref.nsf.Generator(h)
    gen.remove_weight_norm()
    with torch.no_grad():
        for p in gen.parameters():
            p.mul_(3.0)
    gen.eval()
    for k, v in gen.state_dict().items():
        out["rb2_sd_" + k] = v.numpy()
    rng = np.random.RandomState(142)
    B, T = 2, 20
    mel = (rng.randn(B, h.num_mels, T) - 2.5).clip(-11.5, 2).astype(np.float32)
    f0 = mg.f0_contour(rng, B, T)
    with mg.RecordedRandom(143) as rr, torch.no_grad():
        wav = gen(torch.from_numpy(mel), torch.from_numpy(f0))
    out["rb2_cfg"] = np.array(json.dumps(hd))
    out["rb2_mel"], out["rb2_f0"], out["rb2_wav"], out["rb2_rseed"] = mel, f0, wav.numpy(), np.array(143)
    print(f"  resblock2: wav {tuple(wav.shape)} rms {float(wav.pow(2).mean().sqrt()):.4f}")


def gold_audio(ref, out):
    """fish_diffusion/utils/audio.py: the torchaudio mel used by training / validation losses."""
    for mod in ("librosa", "fish_audio_preprocess", "fish_audio_preprocess.utils"):
        if mod not in sys.modules:
            m = types.ModuleType(mod)
            sys.modules[mod] = m
    sys.modules["fish_audio_preprocess.utils"].loudness_norm = None
    sys.modules["fish_audio_preprocess.utils"].separate_audio = None
    sys.modules["fish_audio_preprocess"].utils = sys.modules["fish_audio_preprocess.utils"]
    au = mg._load("ref_audio_utils", f"{REF}/fish_diffusion/utils/audio.py")
    rng = np.random.RandomState(111)
    N = 44100 // 3
    wav = (rng.randn(1, N) * 0.05).astype(np.float32)
    tt = np.arange(N) / 44100.0
    wav[0] += 0.4 * np.sin(2 * np.pi * 220.0 * tt).astype(np.float32) * np.linspace(0, 1, N).astype(np.float32)
    out["au_wav"] = wav
    x = torch.from_numpy(wav)
    out["au_drc"] = au.dynamic_range_compression(x.abs() + 1e-7).numpy()
    for tag, kw in (("default", {}), ("hop256", dict(hop_length=256, win_length=1024, n_fft=1024, n_mels=80, f_min=0, f_max=8000))):
        tf = au.get_mel_transform(**kw)
        out[f"au_mel_{tag}"] = tf(x).numpy()
        out[f"au_from_audio_{tag}"] = au.get_mel_from_audio(x, **kw).numpy()
    out["au_kw_hop256"] = np.array(json.dumps(dict(hop_length=256, win_length=1024, n_fft=1024, n_mels=80, f_min=0, f_max=8000)))


def gold_ckpt(ref, out):
    """Checkpoints written by the reference classes (formats N3)."""
    cfg = mg.WN_SMALL
    torch.manual_seed(123)
    diff = ref.diffusion.GaussianDiffusion(
        denoiser=dict(type="WaveNetDenoiser", **cfg), mel_channels=cfg["mel_channels"], noise_schedule="linear",
        timesteps=1000, max_beta=0.01, noise_loss="smoothed-l1", sampler_interval=10, spec_min=[-5.0], spec_max=[0.0])
    torch.nn.init.kaiming_normal_(diff.denoise_fn.output_projection.conv.weight)
    sd = diff.state_dict()
    ema = {k: (v * 0.5 if v.dtype.is_floating_point and "denoise_fn" in k else v) for k, v in sd.items()}
    ckpt = {"state_dict": {**{"model.diffusion." + k: v for k, v in sd.items()},
                           **{"ema_model.diffusion." + k: v for k, v in ema.items()}},
            "epoch": 3, "global_step": 1234, "pytorch-lightning_version": "2.0.2"}
    torch.save(ckpt, os.path.join(HERE, "ref_ckpt_small.ckpt"))
    rng = np.random.RandomState(124)
    B, T = 2, 30
    x = rng.randn(B, cfg["mel_channels"], T).astype(np.float32)
    c = rng.randn(B, cfg["d_encoder"], T).astype(np.float32)
    with torch.no_grad():
        y = diff.denoise_fn.eval()(torch.from_numpy(x), torch.tensor([500], dtype=torch.long), torch.from_numpy(c))
    out["ck_x"], out["ck_c"], out["ck_y"] = x, c, y.numpy()
    # generator with weight norm, the {"generator": state_dict} format of the released vocoder checkpoints
    h = ref.nsf.AttrDict(mg.VOC_SMALL)
    gen = ref.nsf.Generator(h)
    with torch.no_grad():
        for p in gen.parameters():
            p.mul_(3.0)                     # init std 0.01 gives near-silent output; any deterministic weights do
    torch.save({"generator": gen.state_dict()}, os.path.join(HERE, "ref_generator_small.ckpt"))
    with open(os.path.join(HERE, "ref_generator_small.json"), "w") as f:
        json.dump(dict(mg.VOC_SMALL, n_fft=256, win_size=256, fmin=40, fmax=16000), f)   # + the mel front-end keys
    gen.eval()
    gen.remove_weight_norm()
    mel = (rng.randn(1, h.num_mels, 20) - 2.5).clip(-11.5, 2).astype(np.float32)
    f0 = mg.f0_contour(rng, 1, 20)
    with mg.RecordedRandom(125) as rr, torch.no_grad():
        wav = gen(torch.from_numpy(mel), torch.from_numpy(f0))
    out["ck_voc_mel"], out["ck_voc_f0"], out["ck_voc_wav"], out["ck_voc_rseed"] = mel, f0, wav.numpy(), np.array(125)


def gold_diffsinger(ref, out):
    """archs/diffsinger/diffsinger.py `DiffSinger` (UNMODIFIED file) with NaiveProjectionEncoder and pitch_to_scale.  The file
    needs loralib, matplotlib, pytorch_lightning, wandb, mmengine and package-level imports at import time only (for the
    Lightning wrapper class further down the same file): those names are stubbed; the executed code is the reference's
    `forward_features` / `forward`, its encoders (modules/encoders/naive_projection.py) and utils/pitch.py."""
    class _Any:
        def __getattr__(self, k):
            return _Any()

        def __call__(self, *a, **k):
            return _Any()

    def stub(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    class _LM(torch.nn.Module):
        pass

    stub("loralib")
    stub("matplotlib"); stub("matplotlib.pyplot")
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    stub("pytorch_lightning", LightningModule=_LM)
    stub("pytorch_lightning.loggers", TensorBoardLogger=_Any, WandbLogger=_Any)
    stub("wandb")
    stub("mmengine"); stub("mmengine.optim", OPTIMIZERS=_Any())
    enc_reg = mg._MiniRegistry("encoders")
    pkg = types.ModuleType("refenc2"); pkg.__path__ = [f"{REF}/fish_diffusion/modules/encoders"]; sys.modules["refenc2"] = pkg
    stub("refenc2.builder", ENCODERS=enc_reg)
    npj = mg._load("refenc2.naive_projection", f"{REF}/fish_diffusion/modules/encoders/naive_projection.py", "refenc2")
    pitch = mg._load("ref_pitch_utils", f"{REF}/fish_diffusion/utils/pitch.py")
    stub("fish_diffusion"); stub("fish_diffusion.modules")
    stub("fish_diffusion.modules.encoders", ENCODERS=enc_reg)
    stub("fish_diffusion.modules.vocoders", VOCODERS=_Any())
    stub("fish_diffusion.modules.vocoders.builder", VOCODERS=_Any())
    stub("fish_diffusion.schedulers", LR_SCHEUDLERS=_Any())
    stub("fish_diffusion.utils"); stub("fish_diffusion.utils.viz", viz_synth_sample=_Any())
    dpkg = types.ModuleType("refds"); dpkg.__path__ = [f"{REF}/fish_diffusion/archs/diffsinger"]; sys.modules["refds"] = dpkg
    diff_reg = mg._MiniRegistry("diffusions")
    diff_reg.register_module(name="GaussianDiffusion", module=ref.diffusion.GaussianDiffusion)
    stub("refds.diffusions", DIFFUSIONS=diff_reg)
    stub("refds.grad_tts", GradTTS=_Any)
    ds = mg._load("refds.diffsinger", f"{REF}/fish_diffusion/archs/diffsinger/diffsinger.py", "refds")

    class Cfg(dict):
        __getattr__ = dict.get

    wn = mg.WN_SMALL
    E, M = wn["d_encoder"], wn["mel_channels"]
    cfg = Cfg(text_encoder=dict(type="NaiveProjectionEncoder", input_size=24, output_size=E),
              speaker_encoder=dict(type="NaiveProjectionEncoder", input_size=5, output_size=E, use_embedding=True),
              pitch_encoder=dict(type="NaiveProjectionEncoder", input_size=1, output_size=E, preprocessing=pitch.pitch_to_scale),
              pitch_shift_encoder=dict(type="NaiveProjectionEncoder", input_size=1, output_size=E, use_neck=True, neck_size=4),
              energy_encoder=dict(type="NaiveProjectionEncoder", input_size=1, output_size=E),
              diffusion=dict(type="GaussianDiffusion", denoiser=dict(type="WaveNetDenoiser", **wn), mel_channels=M,
                             noise_loss="smoothed-l1", sampler_interval=10, spec_min=[-5.0], spec_max=[0.0]))
    torch.manual_seed(301)
    model = ds.DiffSinger(cfg)
    torch.nn.init.kaiming_normal_(model.diffusion.denoise_fn.output_projection.conv.weight)
    for k, v in model.state_dict().items():
        out["ds_sd_" + k] = v.numpy()
    rng = np.random.RandomState(302)
    B, T = 3, 37
    lens = torch.tensor([37, 20, 29])
    contents = torch.from_numpy(rng.randn(B, T, 24).astype(np.float32))
    pitches = torch.from_numpy((rng.rand(B, T).astype(np.float32) * 900 + 40))
    speakers = torch.tensor([0, 3, 4])
    pitch_shift = torch.from_numpy(rng.randn(B, 1).astype(np.float32))
    energy = torch.from_numpy(rng.rand(B, T, 1).astype(np.float32))
    with torch.no_grad():
        f = model.forward_features(speakers=speakers, contents=contents, contents_lens=lens, contents_max_len=T,
                                   mel_lens=lens, mel_max_len=T, pitches=pitches.clone(), pitch_shift=pitch_shift, energy=energy)
    out["ds_contents"], out["ds_pitches"], out["ds_speakers"], out["ds_lens"] = contents.numpy(), pitches.numpy(), speakers.numpy(), lens.numpy()
    out["ds_pitch_shift"], out["ds_energy"] = pitch_shift.numpy(), energy.numpy()
    out["ds_features"], out["ds_x_masks"] = f["features"].numpy(), f["x_masks"].numpy()
    mel = torch.from_numpy((rng.rand(B, T, M).astype(np.float32) * 5 - 5))
    with mg.RecordedRandom(303) as rr:
        torch.manual_seed(304)                      # randint(t) comes from torch's own generator
        o = model(speakers=speakers, contents=contents, contents_lens=lens, contents_max_len=T, mel=mel, mel_lens=lens,
                  mel_max_len=T, pitches=pitches.clone(), pitch_shift=pitch_shift, energy=energy)
    o["loss"].backward()
    out["ds_mel"], out["ds_t"], out["ds_loss"] = mel.numpy(), o["t"].numpy(), o["loss"].detach().numpy()
    out["ds_noise"] = rr.log[0][1]                  # randn_like(x) of train_step, [B, M, T]
    out["ds_g_text_w"] = model.text_encoder.projection.weight.grad.numpy()
    out["ds_g_pitch_w"] = model.pitch_encoder.projection.weight.grad.numpy()
    out["ds_g_spk_w"] = model.speaker_encoder.embedding.weight.grad.numpy()
    print(f"  diffsinger: features {tuple(f['features'].shape)}, loss {float(o['loss']):.5f}, draws {[k for k, _ in rr.log]}")


def gold_warmup_cosine(ref, out):
    """schedulers/warmup_cosine_scheduler.py LambdaWarmUpCosineScheduler with the warmup_cosine config's values: the
    multiplier and `last_lr` after each call, at every 7th step of the warm-up and around its ends."""
    sch = mg._load("ref_warmup_cosine", f"{REF}/fish_diffusion/schedulers/warmup_cosine_scheduler.py")
    out["kwargs"] = np.array(json.dumps(dict(warm_up_steps=1000, val_final=2e-5, val_base=8e-4, val_start=1e-5,
                                             max_decay_steps=300000)))
    s = sch.LambdaWarmUpCosineScheduler(**json.loads(str(out["kwargs"])))
    steps = list(range(0, 1200, 7)) + [999, 1000, 1001, 5000, 123456, 299999, 300000, 300001, 2_000_000]
    out["steps"] = np.array(steps, dtype=np.int64)
    vals, last = [], []
    for n in steps:
        vals.append(s(n))
        last.append(s.last_lr)
    out["lr"], out["last_lr"] = np.array(vals, dtype=np.float64), np.array(last, dtype=np.float64)


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)
    ref = mg.load_reference()
    groups = {"traj": gold_traj, "train_full": gold_train_full, "train_masked": gold_train_masked, "voc": gold_voc,
              "audio": gold_audio, "ckpt": gold_ckpt, "diffsinger": gold_diffsinger, "voc_resblock2": gold_voc_resblock2,
              "warmup_cosine": gold_warmup_cosine}
    only = sys.argv[1:]
    for name, fn in groups.items():
        if only and name not in only:
            continue
        out = {}
        fn(ref, out)
        path = os.path.join(HERE, f"r2_{name}.npz")
        np.savez_compressed(path, **out)
        print(f"{name}: {len(out)} arrays, {os.path.getsize(path) / 1e6:.2f} MB")


if __name__ == "__main__":
    main()
