"""LGNEncoder (reference: lgn/models/lgn_encoder.py:20-583): jets -> latent GVec {(0,0), (1,1)}.

At maxdim 2 (all five configurations of BASELINE.json except the wide maxdim-3 model) the whole forward and the
hand-written backward run in the sm_100a library through ``fused._EncoderFn`` -- one autograd node, ~8 kernel
launches.  Other configurations use the generic layer-level composite built from the sub-modules."""
import logging
from typing import Dict, List, Tuple, Union

import numpy as np
import torch

from .. import fused
from ..cg_lib import CGDict, CGModule, ZonalFunctions, ZonalFunctionsRel, normsq4, rep_to_p
from ..g_lib import GTau, GVec
from ..nn import MixReps, RadialFilters
from .fused_module import FusedParamsMixin
from .lgn_cg import LGNCG
from .utils import adapt_var_list

IMPLEMENTED_AGGREGATIONS = ("sum", "mean", "average", "min", "max", "mix")


class LGNEncoder(FusedParamsMixin, CGModule):
    def __init__(self, num_input_particles: int, tau_input_scalars: int, tau_input_vectors: int, tau_latent_scalars: int,
                 tau_latent_vectors: int, maxdim, num_basis_fn: int, num_channels: List[int], max_zf, weight_init, level_gain,
                 activation: str = "leakyrelu", mlp: bool = True, mlp_depth: int = None, mlp_width: int = None, scale: float = 1.0,
                 jet_features: bool = False, map_to_latent: str = "mean", device=None, dtype=None, cg_dict: CGDict = None):
        if device is None:
            device = torch.device("cuda" if torch.cuda.is_available() else "cpu")
        if dtype is None:
            dtype = torch.float64
        num_cg_levels = len(num_channels) - 1
        level_gain = adapt_var_list(level_gain, num_cg_levels)
        maxdim = adapt_var_list(maxdim, num_cg_levels)
        max_zf = adapt_var_list(max_zf, num_cg_levels)
        super().__init__(maxdim=max(maxdim + max_zf), device=device, dtype=dtype, cg_dict=cg_dict)
        misc = {"dtype": self.dtype, "device": self.device}
        logging.info(f"Initializing encoder with device: {self.device} and dtype: {self.dtype}")
        self.num_input_particles = num_input_particles
        self.input_basis = "cartesian"
        self.num_cg_levels, self.num_basis_fn, self.max_zf, self.num_channels = num_cg_levels, num_basis_fn, max_zf, num_channels
        self.level_maxdim = maxdim
        self.jet_features, self.map_to_latent = jet_features, map_to_latent
        self.mlp, self.mlp_depth, self.mlp_width, self.activation = mlp, mlp_depth, mlp_width, activation
        self.tau_input_scalars, self.tau_input_vectors = tau_input_scalars, tau_input_vectors
        if jet_features:
            self.num_input_particles += 1
            tau_input_scalars += 1

        self.zonal_fns_in = ZonalFunctions(maxdim=max(max_zf), basis=self.input_basis, cg_dict=self.cg_dict, **misc)
        self.zonal_fns = ZonalFunctionsRel(maxdim=max(max_zf), basis=self.input_basis, cg_dict=self.cg_dict, **misc)
        self.rad_funcs = RadialFilters(max_zf=max_zf, num_basis_fn=num_basis_fn, num_channels_out=num_channels, num_levels=num_cg_levels, **misc)
        tau_pos = self.rad_funcs.tau

        tau_in = GTau({**{(0, 0): tau_input_scalars, (1, 1): tau_input_vectors}, **{(l, l): 1 for l in range(2, max_zf[0] + 1)}})
        self.tau_dict = {"input": tau_in}
        tau_out = GTau({(l, l): num_channels[0] for l in range(max_zf[0] + 1)})
        self.input_func_node = MixReps(tau_in, tau_out, **misc)
        self.lgn_cg = LGNCG(maxdim=maxdim, max_zf=max_zf, tau_in=self.input_func_node.tau, tau_pos=tau_pos, num_cg_levels=num_cg_levels,
                            num_channels=num_channels, level_gain=level_gain, weight_init=weight_init, mlp=mlp, mlp_depth=mlp_depth,
                            mlp_width=mlp_width, activation=activation, cg_dict=self.cg_dict, **misc)
        self.tau_cg_levels_node = self.lgn_cg.tau_levels_node
        self.tau_dict["cg_layers"] = self.tau_cg_levels_node.copy()
        if map_to_latent.lower() == "mix":
            self.tau_cg_levels_node[-1] = GTau({w: int(v * num_input_particles) for w, v in self.tau_cg_levels_node[-1].items()})
        self.tau_output = {w: 1 for w in self.tau_cg_levels_node[-1].keys()}
        self.tau_output[(0, 0)] = tau_latent_scalars
        self.tau_output[(1, 1)] = tau_latent_vectors
        self.tau_dict["latent"] = self.tau_output
        self.mix_reps = MixReps(self.tau_cg_levels_node[-1], self.tau_output, **misc)
        self.scale = scale
        self.tau_latent = self.tau_output
        self.num_learnable_parameters = sum(p.nelement() for p in self.parameters() if p.requires_grad)

        self._fused_reason = self._why_not_fused()
        self._forward_reason = self._why_not_fused(maxdims=(2, 3))   # forward-only calls: maxdim 3 too
        self._tiled_reason = None   # why autograd calls with N > 32 train through the composite (None: the tiled fused adjoint)
        if self._forward_reason is None:
            self._build_plan("encoder", n_particles=self.num_input_particles, channels=list(num_channels), num_basis_fn=num_basis_fn,
                             mlp=mlp, mlp_depth=mlp_depth if mlp else 0, mlp_width=mlp_width if mlp else 0,
                             latent_mode=map_to_latent, tau_s=tau_latent_scalars, tau_v=tau_latent_vectors, input_scale=scale,
                             activation=activation, maxdim=maxdim[0])
            if not self.fused and not self._plan.forward_supported():
                self._forward_reason = "maxdim-3 level kernels: shared memory does not fit this configuration"
            if self.fused and self.num_input_particles > 32:
                self._tiled_reason = self._plan.tiled_reason()

    # ---------------------------------------------------------------------------------------------------------
    def _why_not_fused(self, maxdims=(2,)):
        """None if the sm_100a fused path implements this configuration, else the reason.  ``maxdims``: the maxdim every level
        may have (2: training and forward; 3: the forward only, csrc/lgae_md3.cu)."""
        if not any(all(m == md for m in self.level_maxdim) for md in maxdims):
            return f"maxdim {self.level_maxdim} (fused path: {' or '.join(map(str, maxdims))})"
        if any(z != 1 for z in self.max_zf):
            return f"max_zf {self.max_zf} (fused path: 1)"
        if self.jet_features:
            return "jet_features"
        if self.tau_input_scalars != 1 or self.tau_input_vectors != 1:
            return "more than one input scalar / vector per particle"
        if self.map_to_latent.lower() not in fused.LATENT_MODES:
            return f"map_to_latent {self.map_to_latent!r}"
        if max(self.num_channels) > 8:
            return "more than 8 channels"
        if self.mlp and (not self.mlp_depth or self.mlp_depth < 1):
            return "MLP depth 0"
        if self.mlp and any(((self.mlp_width * 2 * c + 7) // 8) > 12 for c in self.num_channels[1:]):
            return "MLP hidden width above 96"
        if 2 * self.num_basis_fn > 32:
            return "more than 16 radial basis functions"
        return None

    @property
    def fused(self) -> bool:
        """Trains (and runs) on the fused path."""
        return self._fused_reason is None

    @property
    def fused_forward(self) -> bool:
        """Calls that need no gradient run on the fused path (maxdim 2, and maxdim 3 forward-only)."""
        return self._forward_reason is None

    # ---------------------------------------------------------------------------------------------------------
    def forward(self, data: Union[Dict[str, torch.Tensor], torch.Tensor, np.ndarray], covariance_test: bool = False
                ) -> Union[GVec, Tuple[GVec, List[GVec]]]:
        """data: dict with 'p4' (B,N,4) Cartesian (and optionally 'labels' (B,N), 'scalars'), or a bare array.
        Returns the latent GVec {(0,0): (2,B,1,T_s,1), (1,1): (2,B,1,T_v,4) Cartesian}; with covariance_test=True also
        the list of node GVecs after the input mix and after every level."""
        if not isinstance(data, dict):
            data = {"p4": torch.as_tensor(data)}
        p4 = torch.as_tensor(data["p4"]).to(self.device, self.dtype)
        if p4.device.type != "cuda":
            raise RuntimeError("lgn_autoencoder_b200 runs on CUDA devices only (no CPU fallback); construct the model with device='cuda'")
        # N > 32 trains on the tiled fused adjoint; a configuration it cannot run (_tiled_reason) trains through the
        # layer-level composite, whose autograd covers any N; forward-only calls keep the fused kernels
        needs_grad = torch.is_grad_enabled() and (p4.requires_grad or any(p.requires_grad for p in self.parameters()))
        if self.fused and "scalars" not in data and not (needs_grad and p4.shape[1] > 32 and self._tiled_reason is not None):
            return self._forward_fused(data, p4, covariance_test)
        # maxdim 3: the fused forward for calls that need no gradient (the adjoint is the composite's autograd)
        if self.fused_forward and not self.fused and "scalars" not in data and not needs_grad:
            return self._forward_fused(data, p4, covariance_test)
        return self._forward_generic(data, p4, covariance_test)

    @staticmethod
    def _mask_from(data):
        """The node mask the reference takes from the batch (lgn_encoder.py:387-398): 'labels', else 'masks', else 'mask';
        None means p4[..., 0] != 0."""
        for key in ("labels", "masks", "mask"):
            if key in data:
                return torch.as_tensor(data[key])
        return None

    def _forward_fused(self, data, p4, covariance_test):
        p4 = p4.contiguous()   # the input scale is applied inside the library (LgaeModelDesc.input_scale)
        mask = self._mask_from(data)
        if mask is not None:
            mask = (mask.to(self.device) != 0).to(torch.uint8).contiguous()
        holder = {} if covariance_test else None
        lat00, lat11 = fused._EncoderFn.apply(self._plan, self._theta_node(), p4, mask, holder)
        if self.map_to_latent.lower() == "sum":      # the reference's sum keeps a spurious extra axis (lgn_encoder.py:424)
            lat00, lat11 = lat00.unsqueeze(-3), lat11.unsqueeze(-3)
        latent = GVec({(0, 0): lat00, (1, 1): lat11}, ignore_check=True)
        if not covariance_test:
            return latent
        b = p4.shape[0]
        nodes_all = [GVec(self._plan.node_features(holder["ws"], b, l, mlp=self.mlp), ignore_check=True) for l in range(self.num_cg_levels + 1)]
        return latent, nodes_all

    # generic layer-level composite (any maxdim / pooling); follows the call sequence of lgn_encoder.py:255-412
    def _forward_generic(self, data, p4, covariance_test):
        node_scalars, node_ps, node_mask, edge_mask = self._prepare_input(data, p4)
        zf_in, _, _ = self.zonal_fns_in(node_ps)
        zf_in[(0, 0)] = torch.stack([node_scalars.unsqueeze(-1), torch.zeros_like(node_scalars.unsqueeze(-1))])
        zonal, norms, _ = self.zonal_fns(node_ps, node_ps)
        rad = self.rad_funcs(norms, edge_mask * (norms != 0).byte())
        node = self.input_func_node(zf_in)
        nodes_all = self.lgn_cg(node, node_mask, rad, zonal)
        feats = nodes_all[-1]
        if self.map_to_latent.lower() == "mix":
            feats = GVec({k: v.reshape(2, v.shape[1], 1, -1, v.shape[-1]) for k, v in feats.items()}, ignore_check=True)
        latent = self.mix_reps(feats)
        latent = GVec({w: latent[w] for w in [(0, 0), (1, 1)]}, ignore_check=True)
        latent[(1, 1)] = rep_to_p(latent[(1, 1)])
        latent = aggregate(self.map_to_latent, latent)
        return (latent, nodes_all) if covariance_test else latent

    def _prepare_input(self, data, p4):
        node_ps = p4 * self.scale
        scalars = normsq4(node_ps).abs().sqrt().unsqueeze(-1)
        if "scalars" in data:
            scalars = torch.cat([scalars, torch.as_tensor(data["scalars"]).to(self.device, self.dtype)], dim=-1)
        if self.jet_features:
            jet = node_ps.sum(1, keepdim=True)
            node_ps = torch.cat([node_ps, jet], 1)
            scalars = torch.cat([scalars, normsq4(jet).abs().sqrt().unsqueeze(-1).expand(-1, -1, scalars.shape[-1])], 1)
        given = self._mask_from(data)
        if given is not None:
            node_mask = given.to(self.device).to(torch.uint8)
            if self.jet_features:
                node_mask = torch.cat([node_mask, torch.ones_like(node_mask[:, :1])], 1)
        else:
            node_mask = (node_ps[..., 0] != 0).to(torch.uint8)
        edge_mask = node_mask.unsqueeze(1) * node_mask.unsqueeze(2)
        return scalars, node_ps, node_mask, edge_mask


# ---- latent pooling (reference lgn_encoder.py:419-583), generic path -------------------------------------------
def get_msq(p4):
    return p4[..., 0] ** 2 - torch.norm(p4[..., 1:], dim=-1) ** 2


def gather_righthand(src, index, check=True):
    index = index.unsqueeze(2).unsqueeze(-1).expand(-1, -1, 1, -1, src.shape[-1])
    return torch.gather(src, 2, index)


def get_min_features(feature):
    if feature.shape[-1] == 1:
        key = feature.min(dim=-1).values
    elif feature.shape[-1] == 4:
        key = get_msq(feature)
    else:
        raise NotImplementedError(f"min pooling of irreps of dimension {feature.shape[-1]}")
    return gather_righthand(feature, torch.min(key, dim=-2).indices)


def get_max_features(feature):
    if feature.shape[-1] not in (1, 4):
        raise NotImplementedError(f"max pooling of irreps of dimension {feature.shape[-1]}")
    return gather_righthand(feature, torch.max(get_msq(feature), dim=-2).indices)


def aggregate(method, latent):
    m = method.lower()
    wrap = lambda d: GVec(d, ignore_check=True)
    if m == "sum":
        return wrap({k: v.sum(dim=-3, keepdim=True).unsqueeze(-3) for k, v in latent.items()})
    if m in ("mean", "average"):
        return wrap({k: v.mean(dim=-3, keepdim=True) for k, v in latent.items()})
    if m == "max":
        return wrap({k: get_max_features(v) for k, v in latent.items()})
    if m == "min":
        return wrap({k: get_min_features(v) for k, v in latent.items()})
    if m == "mix":
        return latent
    if "+" in m:
        parts = [aggregate(x, latent) for x in method.split("+")]
        return wrap({k: sum(p[k] for p in parts) / len(parts) for k in latent.keys()})
    if "&" in m:
        parts = [aggregate(x, latent) for x in method.split("&")]
        return wrap({k: torch.cat([p[k] for p in parts], dim=3) for k in latent.keys()})
    raise NotImplementedError(f"map_to_latent={method!r}")
