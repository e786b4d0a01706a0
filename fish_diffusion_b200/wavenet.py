"""B200-native WaveNet denoiser: drop-in for the reference ``fish_diffusion/modules/wavenet.py``.

Same constructor arguments, same ``state_dict`` keys and the same ``forward`` contract as the reference class
(wavenet.py:157-236, SURVEY.md section 8b), registered as ``DENOISERS["WaveNetDenoiser"]``.  The arithmetic runs in
the hand-written sm_100a kernels of libfishdiff_b200.so; there is no PyTorch/CPU fallback.

Data flow of one call (all activations channels-last split planes, see csrc/fd_common.cuh):
  step mlp (3 tiny kernels) -> gate-bias tables (2 kernels) -> head tap-GEMM (input_projection + ReLU + mask)
  -> L x [GEMM1: dilated conv + conditioner + gate | GEMM2: output projection + residual/skip]
  -> tail tap-GEMMs (skip_projection + ReLU, output_projection + mask).
"""
from __future__ import annotations

import ctypes
import math
import os

import torch
from torch import nn

from . import _native as N
from .registry import DENOISERS


class Mish(nn.Module):
    """Parameter-free placeholder so that ``mlp`` keeps the reference indices 0/2 (wavenet.py:8-10,170-174)."""

    def forward(self, x):  # pragma: no cover - never executed: the MLP runs in fd_wavenet_step_mlp
        raise RuntimeError("fish_diffusion_b200.WaveNet runs its MLP natively")


class DiffusionEmbedding(nn.Module):
    def __init__(self, d_denoiser):
        super().__init__()
        self.dim = d_denoiser


class LinearNorm(nn.Module):
    """Parameter holder with the reference's key names and initialiser (wavenet.py:30-43)."""

    def __init__(self, in_features, out_features, bias=False):
        super().__init__()
        self.linear = nn.Linear(in_features, out_features, bias)
        nn.init.xavier_uniform_(self.linear.weight)
        if bias:
            nn.init.constant_(self.linear.bias, 0.0)


class ConvNorm(nn.Module):
    """Parameter holder with the reference's key names and initialiser (wavenet.py:46-80)."""

    def __init__(self, in_channels, out_channels, kernel_size=1, stride=1, padding=None, dilation=1, bias=True):
        super().__init__()
        if padding is None:
            assert kernel_size % 2 == 1
            padding = int(dilation * (kernel_size - 1) / 2)
        self.conv = nn.Conv1d(in_channels, out_channels, kernel_size=kernel_size, stride=stride, padding=padding,
                              dilation=dilation, bias=bias)
        nn.init.kaiming_normal_(self.conv.weight)


class ResidualBlock(nn.Module):
    """Parameter holder for one block (wavenet.py:83-104); computed by fd_wavenet_block_fwd."""

    def __init__(self, d_encoder, residual_channels, use_linear_bias=False, dilation=1):
        super().__init__()
        self.dilation = dilation
        self.conv_layer = ConvNorm(residual_channels, 2 * residual_channels, kernel_size=3, stride=1,
                                   padding=dilation, dilation=dilation)
        self.diffusion_projection = LinearNorm(residual_channels, residual_channels, use_linear_bias)
        self.conditioner_projection = ConvNorm(d_encoder, 2 * residual_channels, kernel_size=1)
        self.output_projection = ConvNorm(residual_channels, 2 * residual_channels, kernel_size=1)


def _gate_half(C: int) -> int:
    for g in (128, 64, 16):
        if C % g == 0:
            return g
    raise ValueError(f"residual_channels={C} must be a multiple of 16")


class WaveNet(nn.Module):
    """WaveNet denoiser (reference wavenet.py:151-236) on sm_100a kernels.

    Extra keyword arguments (not in the reference, defaults keep reference configs working):
      precision: "f16" (22-bit split planes, fp32-faithful) or "bf16" (16-bit split planes, fp32 range); "f16x1" /
        "bf16x1" keep that storage but multiply the hi planes only (one tensor-core product, half-precision operands)
      backend:   "auto" (tcgen05 when the shape has a tensor-core instantiation, else the SIMT twin), "tc", "simt"
    """

    def __init__(self, mel_channels=128, d_encoder=256, residual_channels=512, residual_layers=20,
                 use_linear_bias=False, dilation_cycle=None, precision="f16", backend="auto"):
        super().__init__()
        self.mel_channels, self.d_encoder = mel_channels, d_encoder
        self.residual_channels, self.n_layers = residual_channels, residual_layers
        self.input_projection = ConvNorm(mel_channels, residual_channels, kernel_size=1)
        self.diffusion_embedding = DiffusionEmbedding(residual_channels)
        self.mlp = nn.Sequential(
            LinearNorm(residual_channels, residual_channels * 4, use_linear_bias),
            Mish(),
            LinearNorm(residual_channels * 4, residual_channels, use_linear_bias),
        )
        self.residual_layers = nn.ModuleList([
            ResidualBlock(d_encoder, residual_channels, use_linear_bias=use_linear_bias,
                          dilation=2 ** (i % dilation_cycle) if dilation_cycle else 1)
            for i in range(residual_layers)
        ])
        self.skip_projection = ConvNorm(residual_channels, residual_channels, kernel_size=1)
        self.output_projection = ConvNorm(residual_channels, mel_channels, kernel_size=1)
        nn.init.zeros_(self.output_projection.conv.weight)   # wavenet.py:192

        self.precision = precision
        self.backend = os.environ.get("FD_BACKEND", backend)
        self._pack = None
        self._pack_key = None
        self._pack_static = None
        self._scale_state = None
        self.register_load_state_dict_post_hook(lambda module, incompatible: setattr(module, "_scale_state", None))
        self._ws = {}
        self._graphs = {}
        # CUDA-graph replay of repeated evaluations on the same buffers (the sampler loop); FD_GRAPH=0 disables it
        self.use_graph = os.environ.get("FD_GRAPH", "1") != "0"

    # ------------------------------------------------------------------------------------ packing
    def _resolve_backend(self) -> int:
        if self.backend != "auto":
            return N.backend_code(self.backend)
        C, E, M = self.residual_channels, self.d_encoder, self.mel_channels
        ok = (C % 64 == 0 and E % 64 == 0 and M % 64 == 0 and _gate_half(C) in (128, 64))
        return N.BACKEND_TC if ok else N.BACKEND_SIMT

    def _scales(self, device, lag_ok=False):
        """Power-of-two prescales of every packed matrix (max |w| * s in [32, 64)); they need max |w| on the host.
        Inference repacks are rare and read it synchronously.  A training loop repacks every step: there (`lag_ok`) the
        maxima are fetched asynchronously into pinned memory and consumed by the NEXT repack, so no step waits for a
        device->host round trip; the one-step lag is harmless (fp16 planes saturate at 65504 = 2^10 above the target
        range) and load_state_dict() drops the lagged values."""
        L = self.n_layers
        raw = [self.input_projection.conv.weight, self.skip_projection.conv.weight, self.output_projection.conv.weight]
        for blk in self.residual_layers:
            raw += [blk.conv_layer.conv.weight, blk.conditioner_projection.conv.weight, blk.output_projection.conv.weight]

        def amax_dev():
            return torch.stack(torch._foreach_norm([w.detach() for w in raw], float("inf"))).to(torch.float32)

        st = self._scale_state
        pending = st.get("pending") if (lag_ok and st is not None and st["device"] == str(device)) else None
        if pending is not None:
            pending[0].synchronize()
            amax = pending[1].tolist()
        else:
            amax = amax_dev().tolist()

        def p2(m):
            return 1.0 if m == 0.0 or m != m else float(2.0 ** math.floor(math.log2(64.0 / m)))

        s1 = [p2(max(amax[3 + 3 * l], amax[4 + 3 * l])) for l in range(L)]
        s2 = [p2(amax[5 + 3 * l]) for l in range(L)]
        new = {"device": str(device), "s_in": p2(amax[0]), "s_skip": p2(amax[1]), "s_out": p2(amax[2]), "s1": s1, "s2": s2}
        if st is not None and st["device"] == str(device) and st["s1"] == s1 and st["s2"] == s2:
            new["dev"] = st["dev"]
        else:
            new["dev"] = torch.tensor(s1 + s2, dtype=torch.float32, device=device)
        if lag_ok and device.type == "cuda":
            host = st["pending"][1] if pending is not None else torch.empty(len(raw), dtype=torch.float32).pin_memory()
            host.copy_(amax_dev(), non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(torch.cuda.current_stream(device))
            new["pending"] = (ev, host)
        self._scale_state = new
        return new

    def _packed(self, device, want_bwd=False):
        """Packed weights for `device`, rebuilt whenever a parameter changed (version counters).  All residual layers
        are packed by ONE batched native call (fd_wavenet_pack_layers) that reads the parameters in place; with
        `want_bwd` the transposed packs of the data-gradient GEMMs are produced by the same launches."""
        key = (str(device), self.precision, tuple(p._version for p in self.parameters()),
               tuple(p.data_ptr() for p in self.parameters()))
        if self._pack is not None and self._pack_key == key and (self._pack["has_bwd"] or not want_bwd):
            return self._pack
        prec = N.prec_code(self.precision)
        C, E, M, L = self.residual_channels, self.d_encoder, self.mel_channels, self.n_layers
        KT = 3 * C + E
        half = _gate_half(C)
        gate_tile = 2 * half
        f32 = lambda t: t.detach().to(device=device, dtype=torch.float32)
        sc = self._scales(device, lag_ok=want_bwd)
        s_in, s_skip, s_out, s1, s2 = sc["s_in"], sc["s_skip"], sc["s_out"], sc["s1"], sc["s2"]

        # persistent buffers + parameter pointer tables (rebuilt only when a parameter moved)
        stat = self._pack_static
        has_bwd = bool(want_bwd or (stat is not None and stat["has_bwd"]))
        ptr_key = (str(device), self.precision, has_bwd)
        if stat is None or stat["key"] != ptr_key:
            i16 = dict(dtype=torch.int16, device=device)
            idx = torch.arange(C, device=device).view(C // half, half)
            stat = {"key": ptr_key, "has_bwd": has_bwd,
                    # gate/filter row interleave per column tile: tile q holds gates [q*half,(q+1)*half) then filters
                    "perm": torch.cat([idx, idx + C], dim=1).reshape(-1),
                    "w1p_f32": torch.empty((L, 2 * C, KT), dtype=torch.float32, device=device),
                    "w1": torch.empty((L, 2, 2 * C, KT), **i16), "w2": torch.empty((L, 2, 2 * C, C), **i16),
                    "w1t": torch.empty((L, 2, C, 6 * C), **i16) if has_bwd else None,
                    "wct": torch.empty((L, 2, E, 2 * C), **i16) if has_bwd else None,
                    "w2t": torch.empty((L, 2, C, 2 * C), **i16) if has_bwd else None}
            self._pack_static = stat
        srcs = [[f32(b.conv_layer.conv.weight).contiguous() for b in self.residual_layers],
                [f32(b.conditioner_projection.conv.weight).contiguous() for b in self.residual_layers],
                [f32(b.output_projection.conv.weight).contiguous() for b in self.residual_layers]]
        src_ptrs = tuple(t.data_ptr() for grp in srcs for t in grp)
        if stat.get("src_ptrs") != src_ptrs:
            stat["src_ptrs"] = src_ptrs
            stat["ptr_table"] = torch.tensor(src_ptrs, dtype=torch.int64).view(3, L).to(device)
        tab = stat["ptr_table"]
        N.check(N.lib().fd_wavenet_pack_layers(
            N.ptr(tab[0]), N.ptr(tab[1]), N.ptr(tab[2]), N.ptr(sc["dev"]), N.ptr(stat["w1p_f32"]), N.ptr(stat["w1"]),
            N.ptr(stat["w2"]), N.ptr(stat["w1t"]), N.ptr(stat["wct"]), N.ptr(stat["w2t"]), L, C, E, half, prec,
            N.stream_ptr(device)), "fd_wavenet_pack_layers")

        def pack(w2d, scale):
            return N.pack_weight(w2d, prec, scale), 1.0 / scale

        pk = {"prec": prec, "mma": N.mma_code(self.precision), "gate_tile": gate_tile,
              "backend": self._resolve_backend(), "perm": stat["perm"], "has_bwd": stat["has_bwd"],
              "s_in": s_in, "s_skip": s_skip, "s_out": s_out, "s1": s1, "s2": s2, "_srcs": srcs}
        pk["w_in"], pk["w_in_inv"] = pack(f32(self.input_projection.conv.weight)[:, :, 0], s_in)
        pk["b_in"] = f32(self.input_projection.conv.bias).contiguous()
        pk["mlp_w0"] = f32(self.mlp[0].linear.weight).contiguous()
        pk["mlp_b0"] = f32(self.mlp[0].linear.bias).contiguous() if self.mlp[0].linear.bias is not None else None
        pk["mlp_w1"] = f32(self.mlp[2].linear.weight).contiguous()
        pk["mlp_b1"] = f32(self.mlp[2].linear.bias).contiguous() if self.mlp[2].linear.bias is not None else None
        blocks = list(self.residual_layers)
        pk["w1p_f32"] = stat["w1p_f32"]
        pk["bias_sum"] = (torch.stack([f32(b.conv_layer.conv.bias) for b in blocks]) +
                          torch.stack([f32(b.conditioner_projection.conv.bias) for b in blocks]))[:, stat["perm"]].contiguous()
        pk["w1"], pk["w1_inv"] = [stat["w1"][l] for l in range(L)], [1.0 / v for v in s1]
        pk["w2"], pk["w2_inv"] = [stat["w2"][l] for l in range(L)], [1.0 / v for v in s2]
        pk["b2"] = torch.stack([f32(b.output_projection.conv.bias) for b in blocks]).contiguous()
        pk["wd"] = torch.stack([f32(b.diffusion_projection.linear.weight) for b in blocks]).contiguous()
        pk["bd"] = (torch.stack([f32(b.diffusion_projection.linear.bias) for b in blocks]).contiguous()
                    if blocks[0].diffusion_projection.linear.bias is not None else None)
        pk["dil"] = [b.dilation for b in blocks]
        pk["w_skip"], pk["w_skip_inv"] = pack(f32(self.skip_projection.conv.weight)[:, :, 0], s_skip)
        pk["b_skip"] = f32(self.skip_projection.conv.bias).contiguous()
        pk["w_out"], pk["w_out_inv"] = pack(f32(self.output_projection.conv.weight)[:, :, 0], s_out)
        pk["b_out"] = f32(self.output_projection.conv.bias).contiguous()
        if stat["has_bwd"]:
            bw = {"w1t": [stat["w1t"][l] for l in range(L)], "w1t_inv": pk["w1_inv"],
                  "wct": [stat["wct"][l] for l in range(L)], "wct_inv": pk["w1_inv"],
                  "w2t": [stat["w2t"][l] for l in range(L)], "w2t_inv": pk["w2_inv"]}
            bw["wot"], bw["wot_inv"] = pack(f32(self.output_projection.conv.weight)[:, :, 0].t().contiguous(), s_out)
            bw["wst"], bw["wst_inv"] = pack(f32(self.skip_projection.conv.weight)[:, :, 0].t().contiguous(), s_skip)
            bw["wit"], bw["wit_inv"] = pack(f32(self.input_projection.conv.weight)[:, :, 0].t().contiguous(), s_in)
            pk["_bwd"] = bw
        self._pack, self._pack_key = pk, key
        return pk

    def _workspace(self, device, B, T, Bs):
        key = (str(device), B, T, Bs)
        ws = self._ws.get(key)
        if ws is None:
            C, M, L = self.residual_channels, self.mel_channels, self.n_layers
            i16 = dict(dtype=torch.int16, device=device)
            f32 = dict(dtype=torch.float32, device=device)
            ws = {
                "xr": torch.empty((2, B, T, C), **i16), "z": torch.empty((2, B, T, C), **i16),
                "skip_planes": torch.empty((2, B, T, C), **i16), "skip_f32": torch.empty((B, T, C), **f32),
                "s": torch.empty((Bs, C), **f32), "mlp_ws": torch.empty((Bs * 5 * C,), **f32),
                "gb": torch.empty((3, L, Bs, 2 * C), **f32), "gb_ws": torch.empty((L * Bs * C,), **f32),
                "steps": torch.empty((Bs,), **f32),
            }
            self._ws = {key: ws}   # keep one shape resident
            self._graphs = {}      # captured evaluations reference the old workspace
        return ws

    # ------------------------------------------------------------------------------------ training path
    def train_param_list(self):
        """Conv parameters handed to WaveNetTrainFn, in the order of train_param_keys()."""
        ps = [self.input_projection.conv.weight, self.input_projection.conv.bias]
        for blk in self.residual_layers:
            ps += [blk.conv_layer.conv.weight, blk.conv_layer.conv.bias, blk.conditioner_projection.conv.weight,
                   blk.conditioner_projection.conv.bias, blk.output_projection.conv.weight,
                   blk.output_projection.conv.bias]
        ps += [self.skip_projection.conv.weight, self.skip_projection.conv.bias, self.output_projection.conv.weight,
               self.output_projection.conv.bias]
        return ps

    def train_param_keys(self):
        keys = [("w1x1", "input_projection.w"), ("b", "input_projection.b")]
        for l in range(self.n_layers):
            keys += [("w3", f"l{l}.w1"), ("b", f"l{l}.b1"), ("w1x1", f"l{l}.wc"), ("b", f"l{l}.b1"),
                     ("w1x1", f"l{l}.w2"), ("b", f"l{l}.b2")]
        keys += [("w1x1", "skip_projection.w"), ("b", "skip_projection.b"), ("w1x1", "output_projection.w"),
                 ("b", "output_projection.b")]
        return keys

    def step_vectors(self, diffusion_step):
        """d [Bs, L, C]: DiffusionEmbedding -> mlp -> per-layer diffusion_projection (wavenet.py:20-27,170-174,107)
        with ordinary torch ops on [Bs, C]-sized tensors, so autograd covers these (tiny) parameters."""
        import torch.nn.functional as F
        C = self.residual_channels
        half = C // 2
        emb = math.log(10000) / (half - 1)
        emb = torch.exp(torch.arange(half, device=diffusion_step.device) * -emb)
        emb = diffusion_step[:, None] * emb[None, :]
        s = torch.cat((emb.sin(), emb.cos()), dim=-1)
        s = self.mlp[0].linear(s)
        s = s * torch.tanh(F.softplus(s))
        s = self.mlp[2].linear(s)
        # the L per-layer projections as ONE batched product (same parameters, 3 ops instead of L addmm's and, in the
        # backward, 3 L more): the training step is within a few ms of being bound by host-side launches
        lin = [blk.diffusion_projection.linear for blk in self.residual_layers]
        d = torch.einsum("bc,lkc->blk", s, torch.stack([m.weight for m in lin]))
        if lin[0].bias is not None:
            d = d + torch.stack([m.bias for m in lin])[None]
        return d

    def forward_train_cl(self, x_cl, diffusion_step, cond_cl, x_mask=None, cond_mask=None):
        """Differentiable channels-last forward: x_cl [B,T,M], diffusion_step [B] or [1], cond_cl [B,T,E] -> eps [B,T,M].
        Gradients flow to every parameter, to x_cl, to cond_cl and (through d) to the step-embedding path.  Masks
        ([B,T] bool, True = masked) act where the reference's masked_fill calls do (wavenet.py:217-221,233-234); the
        reference's own training passes none (diffusion.py:134, SURVEY.md D10).
        Memory: the backward needs the residual stream, pre-activations and gated output of every layer as split
        planes: L * 16 * C bytes per position (164 KB at C=512, L=20; 21 GB at B=32, T=4000) -- run inference under
        torch.no_grad() (the registry classes' sampler does)."""
        from .wavenet_train import WaveNetTrainFn
        d = self.step_vectors(diffusion_step)
        masks = None
        if x_mask is not None or cond_mask is not None:
            u8 = lambda m: None if m is None else m.to(device=x_cl.device, dtype=torch.uint8).contiguous()
            masks = (u8(x_mask), u8(cond_mask))
        return WaveNetTrainFn.apply(self, masks, x_cl.contiguous(), cond_cl.contiguous(), d, *self.train_param_list())

    # ------------------------------------------------------------------------------------ native forward
    @torch.no_grad()
    def cond_term(self, cond_planes, out):
        """W_cond . cond of every residual layer (fd_wavenet_cond_term) -> out fp32 [L,B,T,2C] (packed gate/filter column
        order, no bias).  cond is the same for every evaluation of a sampler call, so the sampler computes this once and
        hands it to forward_cl(cond_term=...), whose gate GEMMs then multiply only the three conv taps."""
        dev = cond_planes.device
        N.require_cuda(cond_planes, "cond_planes")
        _, B, T, E = cond_planes.shape
        C, L = self.residual_channels, self.n_layers
        assert E == self.d_encoder and tuple(out.shape) == (L, B, T, 2 * C) and out.dtype == torch.float32
        pk = self._packed(dev)
        w1s = self._pack_static["w1"]
        w1_inv = (ctypes.c_float * L)(*pk["w1_inv"])
        N.check(N.lib().fd_wavenet_cond_term(N.ptr(cond_planes), N.ptr(w1s), w1s.stride(0), w1_inv, N.ptr(out), L, B, T,
                                             C, E, pk["mma"], pk["backend"], N.stream_ptr(dev)), "fd_wavenet_cond_term")
        return out

    @torch.no_grad()
    def forward_cl(self, x_planes, steps, cond_planes, x_mask=None, out=None, cond_term=None):
        """Channels-last entry used by the fused sampler.

        x_planes [2,B,T,M] int16 split planes, steps float32 [1] or [B] (device), cond_planes [2,B,T,E],
        x_mask uint8/bool [B,T] or None (True = masked), cond_term: None or cond_term(cond_planes) computed with the
        current weights.  Returns eps fp32 [B,T,M]."""
        dev = x_planes.device
        N.require_cuda(x_planes, "x_planes")
        _, B, T, M = x_planes.shape
        C, E, L = self.residual_channels, self.d_encoder, self.n_layers
        assert M == self.mel_channels and tuple(cond_planes.shape) == (2, B, T, E)
        pk = self._packed(dev)
        mma, backend = pk["mma"], pk["backend"]
        steps = steps.to(device=dev, dtype=torch.float32).reshape(-1).contiguous()
        Bs = steps.numel()
        if Bs not in (1, B):
            raise ValueError(f"diffusion_step must have 1 or B={B} entries, got {Bs}")
        ws = self._workspace(dev, B, T, Bs)
        st = N.stream_ptr(dev)
        lib = N.lib()
        if x_mask is not None:
            x_mask = x_mask.to(device=dev, dtype=torch.uint8).contiguous()
        if out is None:
            out = torch.empty((B, T, M), dtype=torch.float32, device=dev)

        # ONE native call per evaluation (fd_wavenet_fwd issues the ~45 launches back to back); when the same buffers
        # come back (the sampler loop) the call is captured into a CUDA graph on its second use and replayed afterwards,
        # which also removes the per-launch tensor-map encodes from the host path.
        steps_buf = ws["steps"]
        steps_buf.copy_(steps, non_blocking=True)
        if cond_term is not None:
            assert tuple(cond_term.shape) == (L, B, T, 2 * C) and cond_term.dtype == torch.float32
        d = self._fwd_desc(pk, ws, x_planes, cond_planes, steps_buf, x_mask, out, B, T, Bs)
        d.cond_term = N.ptr(cond_term)
        use_graph = self.use_graph and not N.prof_is_on()
        if not use_graph:
            N.check(lib.fd_wavenet_fwd(ctypes.byref(d), st), "fd_wavenet_fwd")
            return out
        key = (x_planes.data_ptr(), cond_planes.data_ptr(), 0 if cond_term is None else cond_term.data_ptr(),
               out.data_ptr(), 0 if x_mask is None else x_mask.data_ptr(), B, T, Bs, self._pack_key, id(ws))
        ent = self._graphs.get(key)
        if ent is None:                      # first sight of these buffers: run eagerly (lazy inits happen here)
            if len(self._graphs) >= 4:
                self._graphs.clear()
            self._graphs[key] = {"graph": None, "keep": (x_planes, cond_planes, cond_term, out, x_mask, pk)}
            N.check(lib.fd_wavenet_fwd(ctypes.byref(d), st), "fd_wavenet_fwd")
            return out
        if ent["graph"] is None:
            # capture on a side stream without torch.cuda.graph()'s device synchronise + empty_cache (the call sits in
            # the middle of a sampler loop); nothing inside allocates
            g = torch.cuda.CUDAGraph()
            cur = torch.cuda.current_stream(dev)
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(cur)
            with torch.cuda.stream(side):
                g.capture_begin()
                try:
                    N.check(lib.fd_wavenet_fwd(ctypes.byref(d), N.stream_ptr(dev)), "fd_wavenet_fwd")
                finally:
                    g.capture_end()
            cur.wait_stream(side)
            ent["graph"] = g
        ent["graph"].replay()
        return out

    def _fwd_desc(self, pk, ws, x_planes, cond_planes, steps, x_mask, out, B, T, Bs):
        C, E, M, L = self.residual_channels, self.d_encoder, self.mel_channels, self.n_layers
        if L > 64:
            raise ValueError("fd_wavenet_fwd supports up to 64 residual layers")
        d = N.WaveNetFwdDesc()
        d.x_planes, d.cond_planes, d.steps, d.x_mask, d.out = (N.ptr(x_planes), N.ptr(cond_planes), N.ptr(steps),
                                                               N.ptr(x_mask), N.ptr(out))
        d.w_in, d.b_in, d.w_in_inv = N.ptr(pk["w_in"]), N.ptr(pk["b_in"]), pk["w_in_inv"]
        d.mlp_w0, d.mlp_b0, d.mlp_w1, d.mlp_b1 = (N.ptr(pk["mlp_w0"]), N.ptr(pk["mlp_b0"]), N.ptr(pk["mlp_w1"]),
                                                  N.ptr(pk["mlp_b1"]))
        d.wd, d.bd, d.w1p_f32, d.bias_sum = N.ptr(pk["wd"]), N.ptr(pk["bd"]), N.ptr(pk["w1p_f32"]), N.ptr(pk["bias_sum"])
        w1s, w2s = self._pack_static["w1"], self._pack_static["w2"]
        d.w1, d.w1_lstride = N.ptr(w1s), w1s.stride(0)
        d.w2, d.w2_lstride = N.ptr(w2s), w2s.stride(0)
        d.b2, d.b2_lstride = N.ptr(pk["b2"]), pk["b2"].stride(0)
        d.w_skip, d.b_skip, d.w_skip_inv = N.ptr(pk["w_skip"]), N.ptr(pk["b_skip"]), pk["w_skip_inv"]
        d.w_out, d.b_out, d.w_out_inv = N.ptr(pk["w_out"]), N.ptr(pk["b_out"]), pk["w_out_inv"]
        for l in range(L):
            d.w1_inv[l], d.w2_inv[l], d.dilation[l] = pk["w1_inv"][l], pk["w2_inv"][l], pk["dil"][l]
        d.xr, d.z, d.skip_planes, d.skip_f32 = N.ptr(ws["xr"]), N.ptr(ws["z"]), N.ptr(ws["skip_planes"]), N.ptr(ws["skip_f32"])
        d.s, d.mlp_ws, d.gb, d.gb_ws = N.ptr(ws["s"]), N.ptr(ws["mlp_ws"]), N.ptr(ws["gb"]), N.ptr(ws["gb_ws"])
        d.B, d.T, d.M, d.C, d.E, d.L, d.Bs = B, T, M, C, E, L, Bs
        d.gate_tile, d.prec, d.backend = pk["gate_tile"], pk["mma"], pk["backend"]
        return d

    def forward(self, x, diffusion_step, conditioner, x_masks=None, cond_masks=None):
        """Reference contract (wavenet.py:194-236): x [B,M,T] (or [B,1,M,T]), diffusion_step [B] or [1] (int64 or
        float), conditioner [B,E,T], masks [B,T] bool -> [B,M,T] (4-D in -> 4-D out)."""
        if torch.is_grad_enabled() and (x.requires_grad or conditioner.requires_grad or
                                        any(p.requires_grad for p in self.parameters())):
            x3 = x[:, 0] if x.dim() == 4 else x
            eps = self.forward_train_cl(x3.transpose(1, 2), diffusion_step, conditioner.transpose(1, 2),
                                        x_mask=x_masks, cond_mask=cond_masks).transpose(1, 2)
            return eps[:, None] if x.dim() == 4 else eps
        use_4_dim = x.dim() == 4
        if use_4_dim:
            x = x[:, 0]
        assert x.dim() == 3, f"mel must be 3 dim tensor, but got {x.dim()}"
        N.require_cuda(x, "x")
        prec = N.prec_code(self.precision)
        B, M, T = x.shape
        x_planes = N.split_ncw(x.to(torch.float32), prec)
        cmask = None if cond_masks is None else cond_masks.to(torch.uint8).contiguous()
        cond_planes = N.split_ncw(conditioner.to(torch.float32), prec, mask=cmask)
        eps = self.forward_cl(x_planes, diffusion_step.to(torch.float32), cond_planes, x_mask=x_masks)
        out = torch.empty((B, M, T), dtype=torch.float32, device=x.device)
        N.check(N.lib().fd_transpose_nwc_to_ncw(N.ptr(eps), N.ptr(out), B, T, M, N.stream_ptr(x.device)),
                "fd_transpose_nwc_to_ncw")
        return out[:, None] if use_4_dim else out


DENOISERS.register_module(name="WaveNetDenoiser", module=WaveNet, force=True)
DENOISERS.register_module(name="B200WaveNetDenoiser", module=WaveNet, force=True)
