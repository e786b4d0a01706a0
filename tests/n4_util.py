"""Shared by tests/golden/make_golden_n4.py and the N4 tests: the small vocoder-training configuration, deterministic
discriminator weights (too large to store: 46 M values) and the batch, all from numpy seeds."""
import json
import os

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))

# ref_generator_small.json (the VOC_SMALL generator, hop 64) + the training keys of tools/nsf_hifigan/config_v1_256.json
TRAIN_EXTRA = dict(learning_rate=0.0002, adam_b1=0.8, adam_b2=0.99, lr_decay=0.999, discriminator_periods=[2, 3],
                   segment_size=4096)
BATCH, SAMPLES_AUDIO = 2, 4096
SEED_DRAWS = 4101          # torch.rand / randn_like draws of the step (SineGen phases, noise), served from RandomState


def train_config():
    with open(os.path.join(HERE, "golden", "ref_generator_small.json")) as f:
        h = json.load(f)
    h.update(TRAIN_EXTRA)
    return h


def fill_discriminators(*modules, seed=4000):
    """Deterministic values for every parameter / buffer of the discriminators, in state_dict order.  Scales keep the
    logits O(1): weight-norm directions ~N(0,1) with gains that give each layer roughly unit variance, small biases,
    spectral-norm u / v as unit vectors."""
    i = 0
    for mod in modules:
        sd = mod.state_dict()
        new = {}
        for k, v in sd.items():
            rng = np.random.RandomState(seed + i)
            i += 1
            a = rng.standard_normal(tuple(v.shape)).astype(np.float32)
            if k.endswith("weight_g"):
                a = (1.0 + 0.25 * np.abs(a)).astype(np.float32)
            elif k.endswith("bias"):
                a *= 0.02
            elif k.endswith("weight_u") or (k.endswith("weight_v") and v.dim() == 1):
                a /= np.linalg.norm(a) + 1e-12                     # spectral-norm power-iteration vectors
            elif k.endswith("weight_orig"):
                fan_in = int(np.prod(v.shape[1:]))
                a *= 1.0 / np.sqrt(fan_in)
            new[k] = torch.from_numpy(a)
        mod.load_state_dict(new, strict=True)


def make_batch():
    rng = np.random.RandomState(4200)
    B, S = BATCH, SAMPLES_AUDIO
    hop = 64
    t = np.arange(S) / 44100.0
    f0 = np.zeros((B, S // hop), dtype=np.float32)
    audio = np.zeros((B, 1, S), dtype=np.float32)
    for b in range(B):
        base = 180.0 + 140.0 * b
        contour = base * 2 ** (0.2 * np.sin(np.arange(S // hop) / 9.0 + b))
        contour[rng.rand(S // hop) < 0.2] = 0.0
        f0[b] = contour
        audio[b, 0] = (0.35 * np.sin(2 * np.pi * base * t) + 0.15 * np.sin(2 * np.pi * 2.1 * base * t + 0.3)
                       + 0.05 * rng.randn(S)).astype(np.float32)
    return dict(pitches=torch.from_numpy(f0[:, None]), audio=torch.from_numpy(audio),
                audio_lens=torch.tensor([S, S - 3 * hop], dtype=torch.long))


def disc_inputs():
    """-> (y, y_hat) [2, 1, 2050] float32: real and generated audio for the discriminator comparison."""
    rng = np.random.RandomState(4250)
    return rng.randn(2, 1, 2050).astype(np.float32), rng.randn(2, 1, 2050).astype(np.float32)


def summarize(out, key, arr, seed, samples=256):
    a = np.asarray(arr, dtype=np.float32).reshape(-1)
    idx = np.random.RandomState(seed).randint(0, a.size, size=min(samples, a.size))
    out[key + "_norm"] = np.float64(np.linalg.norm(a.astype(np.float64)))
    out[key + "_idx"] = idx.astype(np.int64)
    out[key + "_val"] = a[idx]


def summary_error(g, key, arr):
    """-> max(norm error, sampled-entry error) of `arr` against the stored summary (relative)."""
    a = np.asarray(arr, dtype=np.float64).reshape(-1)
    n_ref = float(g[key + "_norm"])
    idx, val = g[key + "_idx"], g[key + "_val"].astype(np.float64)
    scale = max(n_ref, 1e-30)
    e_norm = abs(np.linalg.norm(a) - n_ref) / scale
    e_val = np.linalg.norm(a[idx] - val) / max(np.linalg.norm(val), scale * np.sqrt(len(idx) / a.size), 1e-30)
    return max(e_norm, e_val)


def check_gradients(g, named_grads, prefix, worst_tol, median_tol, what):
    """Every gradient against its stored summary: the worst and the median relative error must stay under the given
    tolerances (the reference's own float32 noise on these goldens is recorded next to them, see make_golden_n4.py)."""
    errs = sorted((summary_error(g, f"{prefix}{n}", a), n) for n, a in named_grads)
    worst, median = errs[-1], errs[len(errs) // 2]
    print(f"{what}: {len(errs)} gradients, worst {worst[0]:.2e} ({worst[1]}), median {median[0]:.2e}")
    assert worst[0] < worst_tol, f"{what}: worst gradient error {worst[0]:.2e} ({worst[1]}) >= {worst_tol:.1e}"
    assert median[0] < median_tol, f"{what}: median gradient error {median[0]:.2e} >= {median_tol:.1e}"
    return worst[0], median[0]
