"""Host side of the fused maxdim-2 LGAE path: parameter flattening, the C descriptor, and the autograd
Functions that call the whole-model C entry points (include/lgae_b200.h).

The parameters keep the reference's state-dict names and shapes (SURVEY.md appendix A.9); the kernels read
them from one flat fp64 buffer ``theta`` in which every ``nn.Parameter`` is a view, and write the gradient to a
flat ``gtheta`` with the same offsets.
"""
from __future__ import annotations

import ctypes as C
from collections import OrderedDict
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import ACTIVATIONS, LATENT_MODES, LgaeModelDesc, check, ptr

GET_REAL_MODES = {"real": 0, "imag": 1, "sum": 2, "mean": 3, "norm": 4}


def get_real_mode(method: str) -> int:
    """utils/utils.py:194-207: an unknown method logs a warning and means 'real'."""
    m = str(method).lower()
    if m not in GET_REAL_MODES:
        import logging
        logging.warning(f"Invalid method of get_real: {method}. Using 'real' instead.")
        return 0
    return GET_REAL_MODES[m]


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


class FusedPlan:
    """Geometry + parameter offsets of one model (encoder or decoder) for the C library."""

    def __init__(self, kind: str, shapes: "OrderedDict[str, Tuple[int, ...]]", *, n_particles: int, channels: Sequence[int],
                 num_basis_fn: int = 10, mlp: bool = True, mlp_depth: int = 6, mlp_width: int = 6, latent_mode: str = "mean",
                 tau_s: int = 1, tau_v: int = 1, input_scale: float = 1.0, activation: str = "leakyrelu", maxdim: int = 2):
        assert kind in ("encoder", "decoder")
        self.kind = kind
        self.names: List[str] = list(shapes)
        self.offsets: Dict[str, Tuple[int, int, Tuple[int, ...]]] = OrderedDict()
        off = 0
        for name, shape in shapes.items():
            n = 1
            for s in shape:
                n *= int(s)
            self.offsets[name] = (off, n, tuple(int(s) for s in shape))
            off += n
        self.n_params = off
        self._sizes = [n for (_, n, _) in self.offsets.values()]
        self._shapes = [shp for (_, _, shp) in self.offsets.values()]
        self.n_particles = int(n_particles)
        self.channels = [int(c) for c in channels]
        self.n_levels = len(self.channels) - 1
        self.latent_mode = latent_mode
        self.tau_s, self.tau_v = int(tau_s), int(tau_v)
        if int(maxdim) not in (2, 3):
            raise NotImplementedError(f"maxdim {maxdim} is not implemented by the fused B200 path (2, or 3 forward only)")
        self.maxdim = int(maxdim)
        d = LgaeModelDesc()
        d.maxdim = self.maxdim
        d.is_decoder = 1 if kind == "decoder" else 0
        d.n_levels = self.n_levels
        d.n_particles = self.n_particles
        d.n_basis = 2 * int(num_basis_fn)
        for i, c in enumerate(self.channels):
            d.channels[i] = c
        d.has_mlp = 1 if mlp else 0
        d.mlp_hidden = int(mlp_depth)
        if activation.lower() not in ACTIVATIONS:
            raise ValueError(f"Activation function {activation} not implemented!")
        d.mlp_activation = ACTIVATIONS[activation.lower()]
        d.tau_s, d.tau_v = self.tau_s, self.tau_v
        d.n_params = self.n_params
        d.input_scale = float(input_scale)   # encoder: p4 * scale (lgn_encoder.py:371), applied inside the library
        mode = latent_mode.lower()
        if kind == "encoder":
            if mode not in LATENT_MODES:
                raise NotImplementedError(f"map_to_latent={latent_mode!r} is not implemented by the fused B200 path")
            d.latent_mode = LATENT_MODES[mode]

        def o(name):
            if name not in self.offsets:
                raise KeyError(f"parameter {name!r} missing from the {kind} state dict")
            return self.offsets[name][0]

        d.off_in00, d.off_in11 = o("input_func_node.weights.(0, 0)"), o("input_func_node.weights.(1, 1)")
        for l in range(self.n_levels):
            pre = f"rad_funcs.rad_funcs.{l}"
            d.off_rad_a[l], d.off_rad_b[l], d.off_rad_c[l] = o(pre + ".a"), o(pre + ".b"), o(pre + ".c")
            d.off_rad_w0[l], d.off_rad_b0[l] = o(pre + ".linear.0.weight"), o(pre + ".linear.0.bias")
            d.off_rad_w1[l], d.off_rad_b1[l] = o(pre + ".linear.1.weight"), o(pre + ".linear.1.bias")
            mixp = f"lgn_cg.node_levels.{l}.cat_mix.mix_reps.weights."
            d.off_mix00[l], d.off_mix11[l] = o(mixp + "(0, 0)"), o(mixp + "(1, 1)")
            if self.maxdim == 3:
                d.off_mix20[l], d.off_mix02[l], d.off_mix22[l] = o(mixp + "(2, 0)"), o(mixp + "(0, 2)"), o(mixp + "(2, 2)")
            if mlp:
                d.mlp_width[l] = int(mlp_width) * 2 * self.channels[l + 1]
                for i in range(int(mlp_depth) + 1):
                    d.off_mlp_w[l][i] = o(f"lgn_cg.mlp_levels.{l}.linear.{i}.weight")
                    d.off_mlp_b[l][i] = o(f"lgn_cg.mlp_levels.{l}.linear.{i}.bias")
        if kind == "encoder":
            d.off_lat00, d.off_lat11 = o("mix_reps.weights.(0, 0)"), o("mix_reps.weights.(1, 1)")
        else:
            d.off_graph00, d.off_graph11 = o("latent_to_graph.weights.(0, 0)"), o("latent_to_graph.weights.(1, 1)")
            d.off_out00, d.off_out11 = o("mix_to_output.weights.(0, 0)"), o("mix_to_output.weights.(1, 1)")
        self.desc = d
        self._lib = _lib.load()

    # -- parameter plumbing -------------------------------------------------------------------------------
    def flatten(self, tensors: Dict[str, torch.Tensor], device) -> torch.Tensor:
        theta = torch.empty(self.n_params, dtype=torch.float64, device=device)
        for name, (off, n, _) in self.offsets.items():
            theta[off:off + n].copy_(tensors[name].detach().reshape(-1))
        return theta

    def views(self, flat: torch.Tensor) -> "OrderedDict[str, torch.Tensor]":
        return OrderedDict((name, flat[off:off + n].view(shape)) for name, (off, n, shape) in self.offsets.items())

    # -- geometry ---------------------------------------------------------------------------------------------
    def latent_taus(self) -> Tuple[int, int]:
        mult = 2 if self.latent_mode.lower() == "min&max" else 1
        return self.tau_s * mult, self.tau_v * mult

    def workspace(self, batch: int, device) -> torch.Tensor:
        n = self._lib.lgae_workspace_doubles(C.byref(self.desc), batch)
        if n < 0:
            raise NotImplementedError("configuration not supported by the fused B200 path")
        return torch.empty(max(int(n), 1), dtype=torch.float64, device=device)

    def forward_supported(self) -> bool:
        """True if the library's forward entry points take this descriptor (no GPU needed)."""
        return self._lib.lgae_workspace_doubles(C.byref(self.desc), 1) >= 0

    def partials(self, batch: int, device) -> torch.Tensor:
        n = self._lib.lgae_partials_doubles(C.byref(self.desc), batch)
        return torch.empty(max(int(n), 1), dtype=torch.float64, device=device)

    def tiled_scratch(self, batch: int, device) -> torch.Tensor:
        """Scratch of the tiled adjoint (any N) for ``batch`` jets."""
        n = self._lib.lgae_backward_tiled_scratch_doubles(C.byref(self.desc), batch)
        if n < 0:
            raise NotImplementedError(f"configuration not supported by the tiled fused adjoint: {self.tiled_reason()}")
        return torch.empty(max(int(n), 1), dtype=torch.float64, device=device)

    def tiled_reason(self) -> Optional[str]:
        """None if the tiled adjoint runs this model, else the reason (no GPU needed)."""
        n = self._lib.lgae_backward_tiled_scratch_doubles(C.byref(self.desc), 1)
        if n >= 0:
            return None
        return ("a latent / input-map adjoint or a level adjoint whose shared memory does not fit at "
                f"{self.n_particles} particles")

    def ws_tensor(self, ws: torch.Tensor, batch: int, kind: int, level: int, shape) -> torch.Tensor:
        off = self._lib.lgae_workspace_offset(C.byref(self.desc), batch, kind, level)
        if off < 0:
            raise ValueError((kind, level))
        n = 1
        for s in shape:
            n *= s
        return ws[off:off + n].view(shape)

    def node_features(self, ws: torch.Tensor, batch: int, level: int, mlp: bool = True) -> Dict[Tuple[int, int], torch.Tensor]:
        """Planar (2,B,N,C,d) copies of the node features entering level ``level`` (level == n_levels: the
        output of the last level), in the reference's GVec part order: [(1,1), (0,0)] at maxdim 2; at maxdim 3 the order
        of md3_layout.node_order (the MixReps set order, with (0,0) last after a scalar MLP, ``mlp``)."""
        n, c = self.n_particles, self.channels[level]
        s = self.ws_tensor(ws, batch, 0, level, (batch, n, c, 2))
        v = self.ws_tensor(ws, batch, 1, level, (batch, n, c, 4, 2))
        parts = {(1, 1): v.permute(4, 0, 1, 2, 3).contiguous(), (0, 0): s.permute(3, 0, 1, 2).unsqueeze(-1).contiguous()}
        if self.maxdim == 2 or level == 0:
            return OrderedDict([((1, 1), parts[(1, 1)]), ((0, 0), parts[(0, 0)])])
        from . import md3_layout
        h = self.ws_tensor(ws, batch, 9, level, (batch, n, c, 15, 2)).permute(4, 0, 1, 2, 3)
        for key, lo, hi in (((2, 0), 0, 3), ((0, 2), 3, 6), ((2, 2), 6, 15)):
            parts[key] = h[..., lo:hi].contiguous()
        return OrderedDict((k, parts[k]) for k in md3_layout.node_order("mlp" if mlp else "nomlp"))


# -----------------------------------------------------------------------------------------------------------
# raw calls (no autograd)
# -----------------------------------------------------------------------------------------------------------
def encoder_forward_raw(plan: FusedPlan, theta, p4, node_mask):
    lib = plan._lib
    b = p4.shape[0]
    ts, tv = plan.latent_taus()
    dev = p4.device
    ws = plan.workspace(b, dev)
    lat00 = torch.empty((2, b, 1, ts, 1), dtype=torch.float64, device=dev)
    lat11 = torch.empty((2, b, 1, tv, 4), dtype=torch.float64, device=dev)
    tmax = max(plan.tau_s, plan.tau_v)
    sel = torch.empty((4, 2, b, tmax), dtype=torch.int32, device=dev)
    check(lib.lgae_encoder_forward(C.byref(plan.desc), ptr(theta), ptr(p4), ptr(node_mask), b, ptr(ws), ptr(lat00), ptr(lat11),
                                   ptr(sel), _stream()), "encoder_forward")
    return lat00, lat11, ws, sel


def encoder_backward_raw(plan: FusedPlan, theta, p4, node_mask, ws, sel, g00, g11):
    lib = plan._lib
    dev = p4.device
    gtheta = torch.empty(plan.n_params, dtype=torch.float64, device=dev)
    part = plan.partials(p4.shape[0], dev)
    check(lib.lgae_encoder_backward(C.byref(plan.desc), ptr(theta), ptr(p4), ptr(node_mask), p4.shape[0], ptr(ws), ptr(sel),
                                    ptr(g00), ptr(g11), ptr(gtheta), ptr(part), 0.0, None, _stream()), "encoder_backward")
    return gtheta


def encoder_backward_tiled_raw(plan: FusedPlan, theta, p4, node_mask, ws, sel, g00, g11):
    """encoder_backward_raw for any N: the tiled adjoint (lgae_encoder_backward_tiled)."""
    lib = plan._lib
    dev = p4.device
    gtheta = torch.empty(plan.n_params, dtype=torch.float64, device=dev)
    scratch = plan.tiled_scratch(p4.shape[0], dev)
    check(lib.lgae_encoder_backward_tiled(C.byref(plan.desc), ptr(theta), ptr(p4), ptr(node_mask), p4.shape[0], ptr(ws), ptr(sel),
                                          ptr(g00), ptr(g11), ptr(gtheta), ptr(scratch), 0.0, None, _stream()), "encoder_backward_tiled")
    return gtheta


def encoder_backward_p4_raw(plan: FusedPlan, theta, p4, node_mask, ws, sel, g00, g11, tiled: bool):
    """The encoder adjoint with the gradient with respect to p4 (lgae_encoder_backward_p4 / _tiled_p4) -> (gtheta, g_p4)."""
    lib = plan._lib
    dev = p4.device
    b = p4.shape[0]
    gtheta = torch.empty(plan.n_params, dtype=torch.float64, device=dev)
    g_p4 = torch.empty_like(p4)
    n = lib.lgae_encoder_input_grad_scratch_doubles(C.byref(plan.desc), b)
    if n < 0:
        raise NotImplementedError("input gradient not supported by the fused B200 path for this configuration")
    gp = torch.empty(max(int(n), 1), dtype=torch.float64, device=dev)
    if tiled:
        scratch = plan.tiled_scratch(b, dev)
        check(lib.lgae_encoder_backward_tiled_p4(C.byref(plan.desc), ptr(theta), ptr(p4), ptr(node_mask), b, ptr(ws), ptr(sel), ptr(g00),
                                                 ptr(g11), ptr(gtheta), ptr(scratch), 0.0, None, ptr(g_p4), ptr(gp), _stream()),
              "encoder_backward_tiled_p4")
    else:
        part = plan.partials(b, dev)
        check(lib.lgae_encoder_backward_p4(C.byref(plan.desc), ptr(theta), ptr(p4), ptr(node_mask), b, ptr(ws), ptr(sel), ptr(g00),
                                           ptr(g11), ptr(gtheta), ptr(part), 0.0, None, ptr(g_p4), ptr(gp), _stream()), "encoder_backward_p4")
    return gtheta, g_p4


def decoder_forward_raw(plan: FusedPlan, theta, lat11, want_gen00: bool = False):
    lib = plan._lib
    b = lat11.shape[1]
    dev = lat11.device
    ws = plan.workspace(b, dev)
    recon = torch.empty((2, b, plan.n_particles, 4), dtype=torch.float64, device=dev)
    gen00 = torch.empty((2, b, plan.n_particles, 1, 1), dtype=torch.float64, device=dev) if want_gen00 else None
    check(lib.lgae_decoder_forward(C.byref(plan.desc), ptr(theta), ptr(lat11), b, ptr(ws), ptr(recon), ptr(gen00), _stream()),
          "decoder_forward")
    return recon, gen00, ws


def decoder_backward_raw(plan: FusedPlan, theta, lat11, ws, g_recon, g_gen00):
    lib = plan._lib
    dev = lat11.device
    b = lat11.shape[1]
    gtheta = torch.empty(plan.n_params, dtype=torch.float64, device=dev)
    g_lat11 = torch.empty_like(lat11)
    part = plan.partials(b, dev)
    check(lib.lgae_decoder_backward(C.byref(plan.desc), ptr(theta), ptr(lat11), b, ptr(ws), ptr(g_recon), ptr(g_gen00), ptr(g_lat11),
                                    ptr(gtheta), ptr(part), 0.0, None, _stream()), "decoder_backward")
    return g_lat11, gtheta


def decoder_backward_tiled_raw(plan: FusedPlan, theta, lat11, ws, g_recon, g_gen00):
    """decoder_backward_raw for any N: the tiled adjoint (lgae_decoder_backward_tiled)."""
    lib = plan._lib
    dev = lat11.device
    b = lat11.shape[1]
    gtheta = torch.empty(plan.n_params, dtype=torch.float64, device=dev)
    g_lat11 = torch.empty_like(lat11)
    scratch = plan.tiled_scratch(b, dev)
    check(lib.lgae_decoder_backward_tiled(C.byref(plan.desc), ptr(theta), ptr(lat11), b, ptr(ws), ptr(g_recon), ptr(g_gen00), ptr(g_lat11),
                                          ptr(gtheta), ptr(scratch), 0.0, None, _stream()), "decoder_backward_tiled")
    return g_lat11, gtheta


# -----------------------------------------------------------------------------------------------------------
# autograd
# -----------------------------------------------------------------------------------------------------------
def _contig(t):
    return None if t is None else t.contiguous()


class _FlatParamsFn(torch.autograd.Function):
    """The flat parameter buffer as ONE differentiable tensor: forward returns the buffer every ``nn.Parameter`` of the model
    aliases; backward hands each parameter its slice of the flat gradient as a view (no kernel).  The model-level Functions
    below and the L1 / L2 norms take this tensor, so their gradients meet in a single flat add instead of one add per
    parameter tensor (~130 per model), and ``param.grad`` ends up as views of one flat bucket."""

    @staticmethod
    def forward(ctx, plan, theta, *params):
        ctx.plan = plan
        return theta.view(-1)

    @staticmethod
    def backward(ctx, g):
        plan = ctx.plan
        parts = torch.split(g.contiguous(), plan._sizes)     # one call: views of the flat gradient
        return (None, None) + tuple(p.view(shp) for p, shp in zip(parts, plan._shapes))


class _EncoderFn(torch.autograd.Function):
    """LGNEncoder.forward (lgn/models/lgn_encoder.py:255-336) as one autograd node; theta: the flat parameters
    (``_FlatParamsFn``), whose gradient comes back as one flat tensor."""

    @staticmethod
    def forward(ctx, plan, theta, p4, node_mask, holder):
        lat00, lat11, ws, sel = encoder_forward_raw(plan, theta, p4, node_mask)
        ctx.plan, ctx.theta, ctx.p4, ctx.node_mask, ctx.ws, ctx.sel = plan, theta, p4, node_mask, ws, sel
        if holder is not None:
            holder["ws"] = ws
        return lat00, lat11

    @staticmethod
    def backward(ctx, g00, g11):
        plan = ctx.plan
        if ctx.needs_input_grad[2]:
            gtheta, g_p4 = encoder_backward_p4_raw(plan, ctx.theta, ctx.p4, ctx.node_mask, ctx.ws, ctx.sel, _contig(g00), _contig(g11),
                                                   tiled=plan.n_particles > 32)
            return None, gtheta, g_p4, None, None
        bwd = encoder_backward_raw if plan.n_particles <= 32 else encoder_backward_tiled_raw   # one particle per lane, or tiled
        gtheta = bwd(plan, ctx.theta, ctx.p4, ctx.node_mask, ctx.ws, ctx.sel, _contig(g00), _contig(g11))
        return None, gtheta, None, None, None


class _DecoderFn(torch.autograd.Function):
    """LGNDecoder.forward (lgn/models/lgn_decoder.py:218-303) as one autograd node."""

    @staticmethod
    def forward(ctx, plan, theta, lat11, want_gen00, holder):
        lat11 = lat11.contiguous()
        recon, gen00, ws = decoder_forward_raw(plan, theta, lat11, want_gen00)
        ctx.plan, ctx.theta, ctx.lat11, ctx.ws = plan, theta, lat11, ws
        if holder is not None:
            holder["ws"] = ws
        if want_gen00:
            return recon, gen00
        return recon

    @staticmethod
    def backward(ctx, g_recon, g_gen00=None):
        plan = ctx.plan
        if g_recon is None:
            g_recon = torch.zeros((2, ctx.lat11.shape[1], plan.n_particles, 4), dtype=torch.float64, device=ctx.lat11.device)
        bwd = decoder_backward_raw if plan.n_particles <= 32 else decoder_backward_tiled_raw
        g_lat11, gtheta = bwd(plan, ctx.theta, ctx.lat11, ctx.ws, g_recon.contiguous(), _contig(g_gen00))
        return None, gtheta, g_lat11, None, None


class _ChamferFn(torch.autograd.Function):
    """ChamferLoss.forward (utils/losses/chamfer_loss/chamfer_loss.py:16-31) on the complex reconstruction with
    get_real(..., method) (utils/train.py:292) folded in; the gradient is produced by the same launch."""

    @staticmethod
    def forward(ctx, recon, target, mode):
        lib = _lib.load()
        recon = recon.contiguous()
        target = target.contiguous()
        b, n, m = recon.shape[1], recon.shape[2], target.shape[1]
        dev = recon.device
        loss = torch.empty((), dtype=torch.float64, device=dev)
        jet = torch.empty(b, dtype=torch.float64, device=dev)
        g = torch.empty_like(recon)
        check(lib.lgae_chamfer(ptr(recon), ptr(target), b, n, m, mode, ptr(loss), ptr(jet), None, ptr(g), _stream()), "chamfer")
        ctx.save_for_backward(g, recon, target)
        ctx.mode = mode
        return loss

    @staticmethod
    def backward(ctx, g_loss):
        g, recon, target = ctx.saved_tensors
        g_target = None
        if ctx.needs_input_grad[1]:
            g_loss = g_loss.contiguous()
            g_target = torch.empty_like(target)
            check(_lib.load().lgae_chamfer_target_grad(ptr(recon), ptr(target), recon.shape[1], recon.shape[2], target.shape[1], ctx.mode,
                                                       ptr(g_loss), ptr(g_target), _stream()), "chamfer_target_grad")
        return g * g_loss, g_target, None


def chamfer_loss(recon: torch.Tensor, target: torch.Tensor, get_real: str = "real") -> torch.Tensor:
    """Chamfer loss (summed over the batch) between ``get_real(recon, method)`` of the complex reconstruction (2,B,N,4) and
    ``target`` (B,M,4).  ``get_real``: 'real' (the reference's default, main.py:295-300), 'imag', 'sum', 'mean', 'norm'."""
    return _ChamferFn.apply(recon, target, get_real_mode(get_real))


def chamfer_per_jet(recon: torch.Tensor, target: torch.Tensor, get_real: str = "real") -> torch.Tensor:
    """Per-jet chamfer distance (anomaly score), no gradient."""
    lib = _lib.load()
    recon, target = recon.contiguous(), target.contiguous()
    b, n, m = recon.shape[1], recon.shape[2], target.shape[1]
    jet = torch.empty(b, dtype=torch.float64, device=recon.device)
    check(lib.lgae_chamfer(ptr(recon), ptr(target), b, n, m, get_real_mode(get_real), None, ptr(jet), None, None, _stream()), "chamfer")
    return jet


SCORE_NAMES = ("chamfer_particle_cartesian", "mse_particle_cartesian", "chamfer_particle_lorentz", "mse_particle_lorentz", "jet_cartesian",
               "jet_lorentz")


def anomaly_scores(recon: torch.Tensor, target: torch.Tensor, get_real: str = "real", factor: Optional[torch.Tensor] = None) -> Dict[str, torch.Tensor]:
    """Per-jet anomaly scores of the Cartesian family (utils/jet_analysis/anomaly_detection.py:251-419) in one launch:
    ``recon`` (2,B,N,4) complex reconstruction, ``target`` (B,N,4); ``factor`` (B,) optionally rescales both (the reference scores the
    un-normalised jets ``recons * norm_factor`` and the normalised ones).  Returns {name: (B,)} for SCORE_NAMES."""
    lib = _lib.load()
    recon, target = recon.contiguous(), target.contiguous()
    b, n = recon.shape[1], recon.shape[2]
    if target.shape[1] != n:
        raise ValueError("anomaly scores compare jets with the same number of particles")
    out = torch.empty((b, len(SCORE_NAMES)), dtype=torch.float64, device=recon.device)
    f = None if factor is None else factor.reshape(-1).to(torch.float64).contiguous()
    check(lib.lgae_anomaly_scores(ptr(recon), ptr(target), ptr(f), b, n, get_real_mode(get_real), ptr(out), _stream()), "anomaly_scores")
    return {name: out[:, i] for i, name in enumerate(SCORE_NAMES)}


class _NormalizeFn(torch.autograd.Function):
    """normalize_p4 'overall_max'; the adjoint routes the factor's gradient to the maxima as torch's amax does."""

    @staticmethod
    def forward(ctx, p4):
        lib = _lib.load()
        p4 = p4.contiguous()
        out = torch.empty_like(p4)
        f = torch.empty((p4.shape[0], 1, 1), dtype=torch.float64, device=p4.device)
        check(lib.lgae_normalize_p4(ptr(p4), p4.shape[0], p4.shape[1], ptr(out), ptr(f), _stream()), "normalize_p4")
        ctx.save_for_backward(p4)
        return out, f

    @staticmethod
    def backward(ctx, g_out, g_f):
        (p4,) = ctx.saved_tensors
        g_p4 = torch.empty_like(p4)
        check(_lib.load().lgae_normalize_p4_backward(ptr(p4), p4.shape[0], p4.shape[1], ptr(_contig(g_out)), ptr(_contig(g_f)), ptr(g_p4),
                                                     _stream()), "normalize_p4_backward")
        return g_p4


def normalize_p4(p4: torch.Tensor):
    """normalize_p4(p4, 'overall_max') (utils/normalize_p4.py:39-52) -> (normalised, factor (B,1,1)), differentiable in p4."""
    return _NormalizeFn.apply(p4)
