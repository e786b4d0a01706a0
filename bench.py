#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native fish-diffusion hot path.

  python bench.py --gpus N --steps K --warmup W [--scaling weak|strong]   (N>1: torch.distributed.run, one rank / GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W          (the reference's own PyTorch-CPU path)
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR        (also writes the last timed step's mel to DIR)

Headline workload (BASELINE.json configs[1], svc_content_vec.py): the full 100-evaluation DDPM ("naive") sampler of the
WaveNet denoiser (M=128, E=256, C=512, L=20, dilation cycle 4, timesteps=1000, sampler_interval=10), B=32 items x
T=4000 mel frames per GPU, synthetic features, seeded random weights (no dataset / checkpoint is reachable offline).
One "step" = one complete sampler run over one batch; metric = mel-frames/s = (items over all ranks) * T / time.

Keys of the JSON line beyond the base contract:
  roofline      dominant kernel (WaveNet GEMM1), per-launch CUDA events in a separate pass of the same step
  cpu_baseline  the UNMODIFIED reference modules (oracle/_ref, torch CPU, physical cores) on a bounded sample
  vocoder       NSF-HiFiGAN config_v1 (hop 512) and config_v1_256: device time, RTF, roofline of its dominant kernel,
                e2e with host buffers, reference-CPU baseline
  train         BASELINE configs[3]: denoiser training step (fwd + bwd + NCCL gradient all-reduce + AdamW),
                per-GPU B=20 x T=1000, single-product (f16x1) headline and the three-product line
  unipc / single_product / strong   the reference's default predictor, the one-product arithmetic, and the
                B=32-sharded (strong-scaling) run next to the weak-scaling headline
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WN_CFG = dict(mel_channels=128, d_encoder=256, residual_channels=512, residual_layers=20, use_linear_bias=True,
              dilation_cycle=4)
TIMESTEPS, INTERVAL = 1000, 10
VOC_CFG_PATH = os.path.join(ROOT, "tests", "golden", "nsf_configs", "config_v1.json")
WORKLOAD = "svc_content_vec: WaveNet(128,256,512,L20) {evals}-eval DDPM (naive) sampler, timesteps=1000 interval={iv}"


def wn_block_flops(B, T, C=512, E=256):
    """Algorithmic FLOPs of one ResidualBlock (SURVEY.md 8d): B*T*(16C^2 + 4EC); GEMM1 / GEMM2 parts."""
    g1 = B * T * 2 * (3 * C + E) * 2 * C
    g2 = B * T * 2 * C * 2 * C
    return g1, g2


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(tflops=d["bf16_tflops"], tflops_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    hbm_gbs=d["hbm_gbs"], source="measured (MEASURED_PEAKS.json)")
    return dict(tflops=1590.0, tflops_sustained=1400.0, hbm_gbs=6650.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "200", "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(", ") for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, smax, reasons, power = [], [], set(), []
        for r in rows:
            try:
                sm.append(float(r[1])); smax.append(float(r[2])); power.append(float(r[3]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.strip().lower().startswith("active"):
                        reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(smax), "power_w_max": max(power),
                "samples": len(sm), "reasons": sorted(reasons)}


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, arrays):
    """Write each [B, T, ...] tensor as out_dir/<name>.npy in float32 so that two builds run with the same arguments can
    be compared output for output.  A tensor above the byte budget (shared evenly) keeps a sorted, seeded sample of its
    frames (axis 1), the same for every item and every run.  -> {name: description} for the JSON line."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    budget = DUMP_BYTES // len(arrays) - 4096          # room for the .npy header
    info = {}
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        desc = {"shape": list(a.shape), "dtype": "float32"}
        if a.nbytes > budget:
            per_frame = a.nbytes // a.shape[1]
            frames = np.sort(np.random.default_rng(0).choice(a.shape[1], budget // per_frame, replace=False))
            a = np.ascontiguousarray(a[:, frames])
            desc["sample"] = f"{len(frames)} of {desc['shape'][1]} frames (axis 1), np.random.default_rng(0).choice, sorted"
        np.save(os.path.join(out_dir, name + ".npy"), a)
        desc["file"] = name + ".npy"
        desc["saved_shape"] = list(a.shape)
        info[name] = desc
    return info


# ------------------------------------------------------------------------------------------ CPU arm: the reference itself
def cpu_info():
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or os.cpu_count()
    except Exception:  # noqa: BLE001
        phys = os.cpu_count()
    model = ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:  # noqa: BLE001
        pass
    return int(phys), os.cpu_count(), model


class ReferenceCPU:
    """The UNMODIFIED reference modules (fish_diffusion/modules/wavenet.py, archs/diffsinger/diffusions/{diffusion,
    noise_predictor,uni_pc}.py, modules/vocoders/nsf_hifigan/models.py) loaded by file path from /root/reference or its
    verbatim copy oracle/_ref (oracle/build_ref.py), run on torch CPU with one thread per physical core."""

    B, T = 4, 1000          # bounded sample of the workload: 4 items x 1000 frames, full network width

    def __init__(self):
        import torch
        from oracle.ref_loader import load_reference, reference_root
        self.torch = torch
        self.root = reference_root()
        if self.root is None:
            raise FileNotFoundError("neither /root/reference nor oracle/_ref present")
        self.ref = load_reference(self.root, with_mel=False)
        self.phys, self.logical, self.model = cpu_info()
        torch.set_num_threads(self.phys)
        torch.manual_seed(0)
        self.diff = self.ref.diffusion.GaussianDiffusion(
            denoiser=dict(type="WaveNetDenoiser", **WN_CFG), mel_channels=128, noise_schedule="linear", timesteps=TIMESTEPS,
            max_beta=0.01, sampler_interval=INTERVAL, spec_min=[-5.0], spec_max=[0.0], noise_predictor="naive").eval()
        torch.nn.init.kaiming_normal_(self.diff.denoise_fn.output_projection.conv.weight)   # zero-init otherwise (D8)
        self.feats = torch.randn(self.B, self.T, 256)
        self.evals = None

    def calibrate(self, budget_s=4.0):
        """Evaluations per step so that one step costs about `budget_s` seconds: the reference sampler is run with
        sampler_interval = 1000 // evals (every evaluation costs the same, diffusion.py:247-251)."""
        dt = self.step(2) / 2.0
        for ev in (10, 5, 4, 2):
            if ev * dt <= budget_s or ev == 2:
                self.evals = ev
                return ev, dt

    def step(self, evals=None):
        """One run of the reference GaussianDiffusion.forward with `evals` denoiser evaluations -> seconds."""
        torch = self.torch
        ev = evals or self.evals
        t0 = time.perf_counter()
        with torch.no_grad():
            self.diff(self.feats, sampler_interval=TIMESTEPS // ev)
        return time.perf_counter() - t0

    def frames_per_sec(self, dt, evals=None):
        """mel-frames/s of the 100-evaluation config = B*T / (100 evaluations' time)."""
        ev = evals or self.evals
        return self.B * self.T / (dt / ev * (TIMESTEPS // INTERVAL))

    def describe(self):
        return (f"unmodified reference GaussianDiffusion.forward (torch {self.torch.__version__} CPU, "
                f"{self.phys} threads = physical cores of {self.model}; files from {self.root}), B={self.B}, T={self.T}, "
                f"{self.evals} of the 100 evaluations per step (sampler_interval={TIMESTEPS // self.evals}); "
                f"value = B*T / (100 x mean evaluation time)")

    def vocoder(self, B=4, T=250, reps=2):
        """Reference Generator(config_v1).forward on CPU: audio-seconds per second (aggregate RTF)."""
        torch = self.torch
        with open(VOC_CFG_PATH) as f:
            h = json.load(f)
        gen = self.ref.nsf.Generator(self.ref.nsf.AttrDict(h)).eval()
        gen.remove_weight_norm()
        mel = torch.randn(B, 128, T) - 2.5
        f0 = torch.full((B, T), 220.0)
        ts = []
        with torch.no_grad():
            gen(mel, f0)
            for _ in range(reps):
                t0 = time.perf_counter()
                gen(mel, f0)
                ts.append(time.perf_counter() - t0)
        ts.sort()
        dt = ts[len(ts) // 2]
        audio_s = B * T * h["hop_size"] / h["sampling_rate"]
        return {"value": audio_s / dt, "unit": "audio-seconds/s (aggregate RTF)", "cores": self.phys, "kind": "reference",
                "sample": f"unmodified reference Generator(config_v1.json).forward, torch CPU, B={B}, T={T} frames, "
                          f"median of {reps}"}


def port_sample(warmup, steps, T_sample=1000):
    """Fallback when neither /root/reference nor oracle/_ref exists: the numpy oracle port (float32, BLAS threads) on
    one denoiser evaluation + DDPM update at B=1; frames/s = T / (100 x evaluation time)."""
    import numpy as np
    from oracle import sampler as osamp
    from oracle import wavenet as ownet
    sd = ownet.make_wavenet_weights(0, **{k: v for k, v in WN_CFG.items() if k != "dilation_cycle"})
    rng = np.random.RandomState(1)
    x = rng.randn(1, 128, T_sample).astype(np.float32)
    cond = rng.randn(1, 256, T_sample).astype(np.float32)
    tab = osamp.diffusion_tables(osamp.get_noise_schedule_list("linear", TIMESTEPS, 0.01))
    ts = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        eps = ownet.wavenet_forward(sd, x, np.array([990]), cond, dilation_cycle=4, dtype=np.float32)
        osamp.naive_step(tab, x, 990, eps, rng.randn(*x.shape).astype(np.float32))
        if i >= warmup:
            ts.append(time.perf_counter() - t0)
    ts.sort()
    dt = ts[len(ts) // 2]
    return (T_sample / (100.0 * dt), dt * 100, "numpy oracle port, 1 denoiser evaluation + DDPM update at B=1, "
            f"T={T_sample}, x100 evaluations", os.cpu_count(), 1, T_sample)


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores; rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import __graft_entry__ as ge
    try:
        ge.build_ref()
    except Exception:  # noqa: BLE001
        pass
    base = {"impl": "reference", "metric": "mel_frames_per_sec_100step_ddpm", "unit": "mel-frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "gpu_launches": 0}
    try:
        rc = ReferenceCPU()
        kind = "reference"
        evals, _ = rc.calibrate()
        for _ in range(max(0, args.warmup - 1)):       # calibrate() already ran the path twice
            rc.step()
        ts = sorted(rc.step() for _ in range(args.steps))
        dt = ts[len(ts) // 2]
        v = rc.frames_per_sec(dt)
        sample, cores, B, T = rc.describe(), rc.phys, rc.B, rc.T
    except FileNotFoundError as ex:   # no reference files on this box: time the numpy restatement instead
        v, dt, sample, cores, B, T = port_sample(args.warmup, args.steps)
        kind = "port"
        sample += f" [{ex}]"
    line = dict(base, value=v, ms_per_step=dt * 1e3,
                config={"workload": WORKLOAD.format(evals=100, iv=INTERVAL), "global_batch": B, "seq_len": T,
                        "sample": sample},
                cpu_baseline={"value": v, "unit": "mel-frames/s", "cores": cores, "kind": kind, "sample": sample},
                e2e={"value": v, "unit": "mel-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0})
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------ GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch items per GPU (headline); strong: --batch items in total, sharded over the ranks")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--frames", type=int, default=4000)
    ap.add_argument("--evals", type=int, default=100, help="denoiser evaluations per sampler run (100 = the config)")
    ap.add_argument("--backend", default="auto")
    ap.add_argument("--precision", default="f16")
    ap.add_argument("--no-vocoder", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-train", action="store_true")
    ap.add_argument("--no-voc-train", action="store_true", help="skip the vocoder-training side measurement (N4)")
    ap.add_argument("--no-extras", action="store_true", help="skip unipc / single-product / strong-scaling side runs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the mel [B, T, M] that the last timed step returned on rank 0 as "
                         "DIR/mel.npy (float32; at most 64 MB: a seeded sample of frames when larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import __graft_entry__ as ge
    ge.build()
    from fish_diffusion_b200 import DIFFUSIONS, Generator, _native as N
    from fish_diffusion_b200.dist import init_process_group, max_over_ranks, shard_range
    from fish_diffusion_b200 import synthetic

    rank, world, local = init_process_group()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    T, M, E = args.frames, WN_CFG["mel_channels"], WN_CFG["d_encoder"]
    if args.scaling == "strong":
        lo, hi = shard_range(args.batch, rank, world)
        B, first_item, global_B = hi - lo, lo, args.batch
    else:
        B, first_item, global_B = args.batch, rank * args.batch, world * args.batch
    interval = TIMESTEPS // args.evals

    def build_diffusion(precision):
        d = DIFFUSIONS.build(dict(
            type="GaussianDiffusion", denoiser=dict(type="WaveNetDenoiser", backend=args.backend, precision=precision,
                                                    **WN_CFG),
            mel_channels=M, noise_schedule="linear", timesteps=TIMESTEPS, max_beta=0.01, sampler_interval=interval,
            spec_min=[-5.0], spec_max=[0.0], noise_predictor="naive")).to(dev).eval()
        d.denoise_fn.load_state_dict({k: torch.from_numpy(v) for k, v in synthetic.wavenet_weights(0, **WN_CFG).items()})
        return d

    diff = build_diffusion(args.precision)
    if args.scaling == "strong":      # every rank draws the same global batch and keeps its slice
        feats_host = torch.randn(global_B, T, E, generator=torch.Generator().manual_seed(1))[first_item:first_item + B]
    else:
        feats_host = torch.randn(B, T, E, generator=torch.Generator().manual_seed(1 + rank))
    feats_host = feats_host.contiguous().pin_memory()
    feats = feats_host.to(dev)
    torch.manual_seed(2)          # one seed for all ranks: the Philox draws are indexed by the global item (first_item)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(fn, reps):
        """barrier + sync, `reps` calls between two events on the current stream, barrier + sync; max over ranks."""
        barrier()
        ev0.record()
        for _ in range(reps):
            fn()
        ev1.record()
        barrier()
        return max_over_ranks(ev0.elapsed_time(ev1), dev) / reps

    def sampler_step(d=None, feats_=None, predictor="naive", seed=None):
        return (d or diff)(feats if feats_ is None else feats_, sampler_interval=interval, noise_predictor=predictor,
                           first_item=first_item, seed=seed)

    # ---- device-resident timing: W warm-up steps, then exactly K steps (CUDA-graph replay of the denoiser is on)
    for _ in range(args.warmup):
        sampler_step()
    clocks = ClockSampler(local)
    clocks.start()
    launches0 = N.launch_count()
    last = {}

    def timed_step():
        last["mel"] = sampler_step()

    ms_per_step = timed(timed_step, args.steps)
    launches = N.launch_count() - launches0
    clk = clocks.stop()
    value = global_B * T / (ms_per_step * 1e-3)
    dumped = dump_outputs(args.dump_outputs, {"mel": last.pop("mel")}) if args.dump_outputs and rank == 0 else None
    # the graph replays launch the same kernels without passing the library's launch counter: count them from one
    # eager evaluation (identical launch sequence) -- kernels per sampler run, all of this repo's own
    diff.denoise_fn.use_graph = False
    c0 = N.launch_count()
    sampler_step()
    launches_per_step = N.launch_count() - c0

    # ---- roofline of the dominant kernel (WaveNet GEMM1): the same step once more with per-launch CUDA events
    #      on the launching stream (graphs off: events inside a captured graph cannot be timed)
    N.prof_enable(True)
    sampler_step()
    prof, overflow = N.prof_collect()
    N.prof_enable(False)
    diff.denoise_fn.use_graph = True
    pk = peaks()
    g1_flops, g2_flops = wn_block_flops(B, T)
    backend_name = "tc" if diff.denoise_fn._packed(dev)["backend"] == N.BACKEND_TC else "simt"
    single = args.precision.lower().endswith("x1")
    roof = None
    k1, k2 = f"gate/{backend_name}", f"res_skip/{backend_name}"
    if k1 in prof and prof[k1][1] > 0:
        t1 = prof[k1][0] / prof[k1][1] * 1e-3
        t2 = prof[k2][0] / prof[k2][1] * 1e-3 if k2 in prof else float("nan")
        ach = g1_flops / t1 / 1e12
        roof = {"bound": "tensor", "kernel": f"fd_tapgemm_{backend_name}<gate> (WaveNet GEMM1)", "achieved": ach,
                "peak": pk["tflops_sustained"], "unit": "TFLOP/s", "frac": ach / pk["tflops_sustained"],
                "peak_source": pk["source"] + ", sustained bf16 figure (kernel timed inside a long step)",
                "timed_in": "a separate pass of the same sampler step with a CUDA-event pair around every tap-GEMM launch "
                            "(graph replay off), right after the timed region",
                # dram__bytes_read.sum + dram__bytes_write.sum of ONE launch from the committed `ncu --set full` capture
                # (profiles/r01b_ncu_full_summary.json: 402.2 + 228.6 MB); only valid for the shape it was taken on
                "traffic": 630806528 if (B, T, args.precision, backend_name) == (32, 4000, "f16", "tc") else None,
                "traffic_unit": "bytes per launch (ncu, profiles/r01b_ncu_full_summary.json)",
                "algorithmic_bytes_per_launch": 4 * B * T * (512 + 256 + 512),
                "algorithmic_flops_per_launch": g1_flops, "avg_launch_ms": t1 * 1e3, "launches_timed": prof[k1][1],
                "mma_flops_per_launch": (1 if single else 3) * g1_flops if backend_name == "tc" else None,
                "note": "fp32 parity is emulated with 3 fp16 tensor-core products per algorithmic product; "
                        "tensor-pipe utilisation is ~3x frac",
                "block": {"gemm2_avg_launch_ms": t2 * 1e3, "block_tflops": (g1_flops + g2_flops) / (t1 + t2) / 1e12,
                          "block_hbm_gbs_algorithmic": 4 * B * T * (3 * 512 + 256) / (t1 + t2) / 1e9,
                          "hbm_peak_gbs": pk["hbm_gbs"]},
                "tapgemm_share_of_step": sum(v[0] for v in prof.values()) / ms_per_step, "prof_overflow": overflow}

    # ---- end-to-end through the public API with host buffers (H2D of features, D2H of the mel every step)
    e2e = None
    if not args.no_e2e:
        out_host = torch.empty((B, T, M), dtype=torch.float32).pin_memory()

        def e2e_step():
            f = feats_host.to(dev, non_blocking=True)
            mel = diff(f, sampler_interval=interval, noise_predictor="naive", first_item=first_item)
            out_host.copy_(mel, non_blocking=True)

        e2e_step()
        e_ms = timed(e2e_step, args.steps)
        e2e = {"value": global_B * T / (e_ms * 1e-3), "unit": "mel-frames/s", "ms_per_step": e_ms,
               "h2d_bytes_per_step": feats_host.numel() * 4, "d2h_bytes_per_step": out_host.numel() * 4}

    # ---- vocoder (BASELINE metric "RTF@44.1kHz NSF-HiFiGAN"): config_v1 (hop 512), B=32 x T=4000 frames per GPU
    voc = None
    if not args.no_vocoder:
        try:
            voc = bench_vocoder(args, torch, N, Generator, synthetic, dev, B, T, world, timed, barrier, pk, rank,
                                diff, feats, interval, first_item)
        except Exception as ex:  # noqa: BLE001
            voc = {"error": repr(ex)[:400]}

    extras = {}
    if not args.no_extras:
        # the reference's DEFAULT predictor for interval != 1 is UniPC (SURVEY D4): same 100 denoiser evaluations
        try:
            sampler_step(predictor="unipc")
            u_ms = timed(lambda: sampler_step(predictor="unipc"), 1)
            extras["unipc"] = {"ms_per_step": u_ms, "mel_frames_per_sec": global_B * T / (u_ms * 1e-3)}
        except Exception as ex:  # noqa: BLE001
            extras["unipc"] = {"error": repr(ex)[:300]}
        # single-product GEMM mode (hi planes only: half-precision operands, fp32 accumulation): same sampler, same
        # Philox seed; its output deviation from the headline (22-bit) path is reported
        if not single:
            try:
                d2 = build_diffusion(args.precision + "x1")
                ref_mel = sampler_step(seed=77)
                sampler_step(d2, seed=77)
                holder = {}
                x_ms = timed(lambda: holder.__setitem__("m", sampler_step(d2, seed=77)), 1)
                x1_mel = holder["m"]
                num = float((x1_mel - ref_mel).double().norm()); den = float(ref_mel.double().norm())
                extras["single_product"] = {
                    "precision": args.precision + "x1", "ms_per_step": x_ms,
                    "mel_frames_per_sec": global_B * T / (x_ms * 1e-3), "sampler_output_rel_l2_vs_headline": num / den,
                    "sampler_output_max_abs_diff": float((x1_mel - ref_mel).abs().max()),
                    "what": "same sampler, same Philox seed, one tensor-core product per k-step (11-bit operand mantissa)"}
                del d2, ref_mel, x1_mel, holder
            except Exception as ex:  # noqa: BLE001
                extras["single_product"] = {"error": repr(ex)[:300]}
        # strong scaling (SURVEY 8e row 1): the SAME global batch of 32 items sharded over the ranks (4 items per GPU
        # at N=8); per-rank items, ms and aggregate frames/s next to the weak-scaling headline
        if args.scaling == "weak":
            try:
                lo, hi = shard_range(args.batch, rank, world)
                fs = feats[: hi - lo].contiguous()

                def strong_step():
                    return diff(fs, sampler_interval=interval, noise_predictor="naive", first_item=lo)

                strong_step(); strong_step()            # second call captures the graph for this shape
                s_ms = timed(strong_step, 2)
                extras["strong"] = {"global_batch": args.batch, "items_per_gpu": hi - lo, "ms_per_step": s_ms,
                                    "mel_frames_per_sec": args.batch * T / (s_ms * 1e-3),
                                    "what": "B=32 sharded over the ranks, no data-path collective; at N=1 identical to "
                                            "the headline; efficiency(N) = value(N) / (N * value(1)), limited by tile "
                                            "quantisation (B*T/128 position tiles x 4 column tiles over 148 SMs) and "
                                            "per-launch latency of ~45 launches per evaluation inside one graph"}
                del fs
            except Exception as ex:  # noqa: BLE001
                extras["strong"] = {"error": repr(ex)[:300]}

    # ---- BASELINE configs[3]: denoiser training step under DDP (fwd + bwd + NCCL all-reduce + AdamW)
    train = None
    if not args.no_train:
        del diff, feats
        torch.cuda.empty_cache()
        try:
            train = bench_train(torch, N, dev, rank, world, timed, pk)
        except Exception as ex:  # noqa: BLE001
            train = {"error": repr(ex)[:400]}

    # ---- SURVEY 8f N4: vocoder training (config_v1_256, batch 20 x 32768 samples as configs/vocoder_nsf_hifigan.py):
    #      generator forward + backward on the native nodes next to the reference class under cuDNN autograd on the same
    #      GPU and on the host cores, and one whole GAN step (tools/bench_voc_train.py)
    voc_train = None
    if rank == 0 and world == 1 and not args.no_voc_train:
        torch.cuda.empty_cache()
        try:
            import importlib.util
            import types as _types
            spec = importlib.util.spec_from_file_location(
                "bench_voc_train", os.path.join(os.path.dirname(os.path.abspath(__file__)), "tools", "bench_voc_train.py"))
            bvt = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(bvt)
            voc_train = bvt.measure(_types.SimpleNamespace(batch=20, frames=128, steps=3, cpu=not args.no_cpu_baseline,
                                                           no_step=False))
        except Exception as ex:  # noqa: BLE001
            voc_train = {"error": repr(ex)[:400]}
        torch.cuda.empty_cache()

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            rc = ReferenceCPU()
            rc.calibrate()
            rc.step()
            ts = sorted(rc.step() for _ in range(5))
            cpu = {"value": rc.frames_per_sec(ts[2]), "unit": "mel-frames/s", "cores": rc.phys, "kind": "reference",
                   "sample": rc.describe() + "; median of 5 steps after 2 warm-up runs",
                   "spread": [rc.frames_per_sec(ts[-1]), rc.frames_per_sec(ts[0])]}
            if voc is not None and "error" not in voc:
                voc["cpu_baseline"] = rc.vocoder()
        except Exception as ex:  # noqa: BLE001
            cpu = {"value": None, "unit": "mel-frames/s", "cores": os.cpu_count(), "kind": "reference",
                   "sample": f"unavailable: {ex!r}"[:300]}

    if rank == 0:
        line = {
            "metric": "mel_frames_per_sec_100step_ddpm", "value": value, "unit": "mel-frames/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None,
            "dtype": ("f16 operands, fp32 accumulate (single tcgen05 product)" if single else
                      "f32 (3x fp16 split-product tcgen05, fp32 accumulate)") if backend_name == "tc" else "f32 (SIMT)",
            "data": "synthetic",
            "config": {"workload": WORKLOAD.format(evals=args.evals, iv=interval),
                       "global_batch": global_B, "per_gpu_batch": B, "seq_len": T,
                       "parallelism": f"batch-shard x{world} ({args.scaling}), no data-path collective",
                       "backend": backend_name, "precision": args.precision,
                       "l2": "inputs (features 131 MB + weights 420 MB + 1 GB activations per layer) larger than L2"},
            "clocks": clk, "e2e": e2e,
            "gpu_launches": launches_per_step * args.steps,
            "gpu_launches_note": f"{launches_per_step} kernels of this library per sampler run (counted on an eager run); "
                                 f"inside the timed region {launches} went through the launch counter, the rest were "
                                 f"replayed from CUDA graphs of the same launch sequence",
            "roofline": roof, "cpu_baseline": cpu, "vocoder": voc, "train": train, "voc_train": voc_train,
            "kernel_ms": {k: {"total_ms": v[0], "launches": v[1]} for k, v in prof.items()},
        }
        line.update(extras)
        if dumped is not None:
            line["dump_outputs"] = dumped
        print(json.dumps(line))
    if world > 1:
        torch.distributed.destroy_process_group()


def bench_vocoder(args, torch, N, Generator, synthetic, dev, B, T, world, timed, barrier, pk, rank, diff, feats,
                  interval, first_item):
    """NSF-HiFiGAN generator: device-resident time, RTF, roofline of the dominant kernel, e2e with host buffers."""
    g = torch.Generator().manual_seed(5 + rank)
    with open(VOC_CFG_PATH) as f:
        h = json.load(f)
    gen = Generator(h, backend=args.backend, precision=args.precision).to(dev)
    gen.remove_weight_norm()
    gen.load_state_dict({k: torch.from_numpy(v) for k, v in synthetic.generator_weights(3, h).items()})
    mel_host = (torch.randn(B, 128, T, generator=g) - 2.5).clamp(-11.5, 2).pin_memory()
    f0_host = (220.0 * 2 ** (0.3 * torch.sin(torch.arange(T) / 50.0))).repeat(B, 1)
    f0_host[:, ::5] = 0
    f0_host = f0_host.pin_memory()
    mel, f0 = mel_host.to(dev), f0_host.to(dev)
    hop = h["hop_size"]
    audio_s = T * hop / h["sampling_rate"]
    gen(mel, f0, seed=1)
    v_ms = timed(lambda: gen(mel, f0, seed=1), 2)
    voc = {"config": "config_v1.json (hop 512)", "B": B, "T": T, "ms": v_ms,
           "rtf_agg": world * B * audio_s / (v_ms * 1e-3), "rtf_stream": audio_s / (v_ms * 1e-3),
           "tflops": world * B * T * 652.1e6 / (v_ms * 1e-3) / 1e12,
           "fused_resblock_pairs": bool(gen.fused)}
    # roofline of the dominant kernel class: the fused ResBlock pair kernel at C=128 (stage 1: 18 launches per pass);
    # algorithmic FLOPs 2*C*C*(k1+k2) per position, bytes 8*C per position (4 in + 4 out)
    N.prof_enable(True)
    gen(mel, f0, seed=1)
    prof, _ = N.prof_collect()
    N.prof_enable(False)
    if "respair/128" in prof:
        tot_ms, n = prof["respair/128"]
        up = 1
        for i, r in enumerate(h["upsample_rates"]):   # positions per frame at the stage whose channel count is 128
            up *= r
            if h["upsample_initial_channel"] // (2 ** (i + 1)) == 128:
                break
        rows = B * T * up
        C = 128
        taps = sum(2 * k for k in h["resblock_kernel_sizes"]) * len(h["resblock_dilation_sizes"][0])
        fl = 2.0 * rows * C * C * taps               # all 9 pairs of the stage
        by = 8.0 * rows * C * (n)
        ach = fl / (tot_ms * 1e-3) / 1e12
        voc["roofline"] = {"bound": "tensor", "kernel": "fd_respair_tc<128> (fused ResBlock1 pair, stage 1)",
                           "achieved": ach, "peak": pk["tflops_sustained"], "unit": "TFLOP/s",
                           "frac": ach / pk["tflops_sustained"], "peak_source": pk["source"] + ", sustained bf16",
                           "avg_launch_ms": tot_ms / n, "launches_timed": n,
                           "algorithmic_flops_per_pass": fl, "algorithmic_bytes_per_pass": by,
                           "hbm_gbs_algorithmic": by / (tot_ms * 1e-3) / 1e9, "hbm_peak_gbs": pk["hbm_gbs"],
                           "traffic": 8380000000, "traffic_unit": "bytes per launch (ncu dram read+write, "
                                                                  "profiles/r02a_respair_c128k11.json; algorithmic 8.39e9)",
                           "share_of_pass": tot_ms / v_ms,
                           "kernel_ms": {k: {"total_ms": v[0], "launches": v[1]} for k, v in prof.items()}}
    # e2e: mel + f0 in pinned host memory -> H2D, generator, wav -> D2H, every step
    wav_host = torch.empty((B, 1, T * hop), dtype=torch.float32).pin_memory()

    def voc_e2e():
        m = mel_host.to(dev, non_blocking=True)
        f = f0_host.to(dev, non_blocking=True)
        wav_host.copy_(gen(m, f, seed=1), non_blocking=True)

    voc_e2e()
    e_ms = timed(voc_e2e, 2)
    voc["e2e"] = {"value": world * B * audio_s / (e_ms * 1e-3), "unit": "audio-seconds/s (aggregate RTF)", "ms": e_ms,
                  "rtf_stream": audio_s / (e_ms * 1e-3),
                  "h2d_bytes_per_step": (mel_host.numel() + f0_host.numel()) * 4, "d2h_bytes_per_step": wav_host.numel() * 4}
    del wav_host
    # config #5 flavour: sampler + vocoder back to back on one batch (B=16, T=4000), audio-seconds/s
    Bs5 = min(16, B)
    f5, f0_5 = feats[:Bs5].contiguous(), f0[:Bs5].contiguous()

    def synth_step():
        m5 = diff(f5, sampler_interval=interval, noise_predictor="naive", first_item=first_item)   # [B,T,M] ln-mel
        return gen(m5.transpose(1, 2).contiguous(), f0_5, seed=1)

    synth_step()
    s_ms = timed(synth_step, 1)
    voc["synth_e2e"] = {"B": Bs5, "T": T, "ms": s_ms, "audio_seconds_per_sec": world * Bs5 * audio_s / (s_ms * 1e-3),
                        "what": "100-eval DDPM sampler + NSF-HiFiGAN (hop 512) per batch, device resident"}
    del gen, f5
    # the config the reference's vocoder recipe trains (configs/vocoder_nsf_hifigan.py:31): hop 256
    try:
        with open(VOC_CFG_PATH.replace("config_v1.json", "config_v1_256.json")) as f:
            h2 = json.load(f)
        gen2 = Generator(h2, backend=args.backend, precision=args.precision).to(dev)
        gen2.remove_weight_norm()
        gen2.load_state_dict({k: torch.from_numpy(v) for k, v in synthetic.generator_weights(4, h2).items()})
        gen2(mel, f0, seed=1)
        h_ms = timed(lambda: gen2(mel, f0, seed=1), 1)
        audio2 = T * h2["hop_size"] / h2["sampling_rate"]
        voc["hop256"] = {"config": "config_v1_256.json (hop 256)", "B": B, "T": T, "ms": h_ms,
                         "rtf_agg": world * B * audio2 / (h_ms * 1e-3), "rtf_stream": audio2 / (h_ms * 1e-3)}
        del gen2
    except Exception as ex:  # noqa: BLE001
        voc["hop256"] = {"error": repr(ex)[:300]}
    torch.cuda.empty_cache()
    return voc


def bench_train(torch, N, dev, rank, world, timed, pk, B=20, T=1000, steps=5, warmup=3):
    """BASELINE configs[3] (svc_hifisinger_v2.py): GaussianDiffusion.train_step on the v2 WaveNet, per-GPU batch 20 x
    1000 frames (configs/_base_/datasets/naive_svc.py:16), smoothed-l1, AdamW + clip 0.5, gradient all-reduce over NCCL
    when world > 1.  Headline arithmetic: one tensor-core product (f16 operands, fp32 accumulate) -- the config asks for
    16-bit mixed precision; the three-product (fp32-faithful) line is reported beside it."""
    from fish_diffusion_b200 import DIFFUSIONS, synthetic
    from fish_diffusion_b200.train import DenoiserTrainer
    M, E = WN_CFG["mel_channels"], WN_CFG["d_encoder"]
    g = torch.Generator().manual_seed(100 + rank)
    feats = torch.randn(B, T, E, generator=g).to(dev)
    mel = (torch.rand(B, T, M, generator=g) * 5 - 5).to(dev)
    out = {"config": "svc_hifisinger_v2-class denoiser train step: WaveNet(128,256,512,L20), smoothed-l1, AdamW(8e-4, "
                     "wd 1e-2, betas (0.9,0.98), eps 1e-9), clip 0.5",
           "per_gpu_batch": B, "frames": T, "n_gpus": world, "global_batch": world * B}
    flops = 3 * 95.159e6 * B * T            # fwd + 2x bwd, algorithmic (SURVEY 8d: 95.159 MFLOP / position forward)
    for precision in ("f16x1", "f16"):
        diff = DIFFUSIONS.build(dict(type="GaussianDiffusion", denoiser=dict(type="WaveNetDenoiser", precision=precision, **WN_CFG),
                                     mel_channels=M, noise_loss="smoothed-l1", sampler_interval=10, spec_min=[-5.0],
                                     spec_max=[0.0])).to(dev).train()
        diff.denoise_fn.load_state_dict({k: torch.from_numpy(v) for k, v in synthetic.wavenet_weights(0, **WN_CFG).items()})
        tr = DenoiserTrainer(diff, device=dev)
        for _ in range(warmup):
            tr.step(feats, mel)
        ms = timed(lambda: tr.step(feats, mel), steps)
        tr.step(feats, mel, timing=True)
        tr.step(feats, mel, timing=True)        # fills last_split_ms with the split of the previous step
        ent = {"ms_per_step": ms, "samples_per_sec": world * B / (ms * 1e-3),
               "mel_frames_per_sec": world * B * T / (ms * 1e-3),
               "algorithmic_tflops_per_gpu": flops / (ms * 1e-3) / 1e12,
               "frac_of_peak_algorithmic": flops / (ms * 1e-3) / 1e12 / pk["tflops_sustained"]}
        split = getattr(tr, "last_split_ms", None)
        if split:
            ent["split_ms"] = split
        if precision == "f16x1":
            if world > 1:      # the same step without any gradient reduction: what the all-reduce costs on top
                tr0 = DenoiserTrainer(diff, device=dev, sync="none")
                for _ in range(warmup):
                    tr0.step(feats, mel)
                ent["ms_per_step_without_allreduce"] = timed(lambda: tr0.step(feats, mel), steps)
                ent["allreduce_exposed_ms"] = ms - ent["ms_per_step_without_allreduce"]
                del tr0
            with torch.no_grad():
                diff.train_step(feats, mel)
                ent["fwd_only_ms"] = timed(lambda: diff.train_step(feats, mel), steps)
        out[precision] = ent
        del tr, diff
        torch.cuda.empty_cache()
    out["headline"] = "f16x1"
    out["ddp"] = getattr(DenoiserTrainer, "SYNC_DESCRIPTION", "torch DDP over NCCL") if world > 1 else "single process"
    return out


if __name__ == "__main__":
    main()
