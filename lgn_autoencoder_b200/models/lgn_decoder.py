"""LGNDecoder (reference: lgn/models/lgn_decoder.py:16-349): latent GVec -> complex Cartesian 4-momenta (2,B,N,4).

Reference behaviours kept on purpose (SURVEY.md appendix A.6): the decoder's node and edge masks are all zero, so the
radial functions reduce to their Linear biases; the zonal (0,0) function is 1+1j; the latent scalars never reach
the output."""
import logging

import torch

from .. import fused
from ..cg_lib import CGDict, CGModule, ZonalFunctions, ZonalFunctionsRel, cg_product, p_cplx_to_rep, rep_to_p
from ..g_lib import GTau, GVec
from ..nn import MixReps, RadialFilters
from .fused_module import FusedParamsMixin
from .lgn_cg import LGNCG
from .utils import adapt_var_list


class LGNDecoder(FusedParamsMixin, CGModule):
    def __init__(self, tau_latent_scalars, tau_latent_vectors, num_output_particles, tau_output_scalars, tau_output_vectors, maxdim,
                 num_basis_fn, num_channels, max_zf, weight_init, level_gain, activation="leakyrelu", mlp=True, mlp_depth=None,
                 mlp_width=None, device=None, dtype=None, cg_dict: CGDict = None):
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
        logging.info(f"Initializing decoder with device: {self.device} and dtype: {self.dtype}")
        self.input_basis = "canonical"
        self.tau_latent_scalars, self.tau_latent_vectors = tau_latent_scalars, tau_latent_vectors
        self.tau_output_scalars, self.tau_output_vectors = tau_output_scalars, tau_output_vectors
        self.tau_dict = {"input": GTau({(0, 0): tau_latent_scalars, (1, 1): tau_latent_vectors})}
        self.num_output_particles = num_output_particles
        self.num_cg_levels, self.num_basis_fn, self.max_zf, self.num_channels = num_cg_levels, num_basis_fn, max_zf, num_channels
        self.level_maxdim = maxdim
        self.mlp, self.mlp_depth, self.mlp_width, self.activation = mlp, mlp_depth, mlp_width, activation

        tau_graph = GTau({**{w: num_output_particles for w in [(0, 0), (1, 1)]}, **{(l, l): 1 for l in range(2, max_zf[0] + 1)}})
        self.latent_to_graph = MixReps(tau_in=self.tau_dict["input"], tau_out=tau_graph, **misc)
        self.input_func_node = MixReps(tau_in=GTau({w: 1 for w in [(0, 0), (1, 1)]}), tau_out=GTau({w: num_channels[0] for w in [(0, 0), (1, 1)]}), **misc)
        self.zonal_fns_in = ZonalFunctions(maxdim=max(max_zf), basis=self.input_basis, cg_dict=self.cg_dict, **misc)
        self.zonal_fns = ZonalFunctionsRel(maxdim=max(max_zf), basis=self.input_basis, cg_dict=self.cg_dict, **misc)
        self.rad_funcs = RadialFilters(max_zf=max_zf, num_basis_fn=num_basis_fn, num_channels_out=num_channels, num_levels=num_cg_levels,
                                       input_basis=self.input_basis, **misc)
        self.lgn_cg = LGNCG(maxdim=maxdim, max_zf=max_zf, tau_in=self.input_func_node.tau, tau_pos=self.rad_funcs.tau,
                            num_cg_levels=num_cg_levels, num_channels=num_channels, level_gain=level_gain, weight_init=weight_init,
                            mlp=mlp, mlp_depth=mlp_depth, mlp_width=mlp_width, activation=activation, cg_dict=self.cg_dict, **misc)
        self.tau_cg_levels_node = self.lgn_cg.tau_levels_node
        self.tau_dict["cg_layers"] = self.tau_cg_levels_node.copy()
        self.tau_output = {w: 1 for w in self.tau_cg_levels_node[-1].keys()}
        self.tau_output[(0, 0)] = tau_output_scalars
        self.tau_output[(1, 1)] = tau_output_vectors
        self.tau_dict["output"] = self.tau_output
        self.mix_to_output = MixReps(tau_in=self.tau_cg_levels_node[-1], tau_out=self.tau_output, **misc)
        self.num_learnable_parameters = sum(p.nelement() for p in self.parameters() if p.requires_grad)

        self._fused_reason = self._why_not_fused()
        self._tiled_reason = None   # why autograd calls with N > 32 train through the composite (None: the tiled fused adjoint)
        if self._fused_reason is None:
            self._build_plan("decoder", n_particles=num_output_particles, channels=list(num_channels), num_basis_fn=num_basis_fn, mlp=mlp,
                             mlp_depth=mlp_depth if mlp else 0, mlp_width=mlp_width if mlp else 0, tau_s=tau_latent_scalars,
                             tau_v=tau_latent_vectors, activation=activation)
            if num_output_particles > 32:
                self._tiled_reason = self._plan.tiled_reason()

    def _why_not_fused(self):
        if any(m != 2 for m in self.level_maxdim):
            return f"maxdim {self.level_maxdim} (fused path: 2)"
        if any(z != 1 for z in self.max_zf):
            return f"max_zf {self.max_zf} (fused path: 1)"
        if self.tau_output_scalars != 1 or self.tau_output_vectors != 1:
            return "more than one output scalar / vector per particle"
        if max(self.num_channels) > 8:
            return "more than 8 channels"
        if self.mlp and (not self.mlp_depth or self.mlp_depth < 1):
            return "MLP depth 0"
        if self.mlp and any(((self.mlp_width * 2 * c + 7) // 8) > 12 for c in self.num_channels[1:]):
            return "MLP hidden width above 96"
        return None

    @property
    def fused(self) -> bool:
        return self._fused_reason is None

    def forward(self, latent_features, covariance_test=False, nodes_all=None):
        """latent GVec {(0,0): (2,B,1,T_s,1), (1,1): (2,B,1,T_v,4)} -> (2,B,N,4) complex Cartesian momenta.  With
        covariance_test=True returns (generated GVec in the canonical basis, nodes_all + decoder node GVecs)."""
        if covariance_test and nodes_all is None:
            raise ValueError("covariance_test is set to True, but the list nodes_all is not provided!")
        lat11 = latent_features[(1, 1)]
        if lat11.device.type != "cuda":
            raise RuntimeError("lgn_autoencoder_b200 runs on CUDA devices only (no CPU fallback)")
        # N > 32 trains on the tiled fused adjoint unless it cannot run this configuration (_tiled_reason)
        needs_grad = torch.is_grad_enabled() and (lat11.requires_grad or any(p.requires_grad for p in self.parameters()))
        if self.fused and not (needs_grad and self.num_output_particles > 32 and self._tiled_reason is not None):
            return self._forward_fused(lat11, covariance_test, nodes_all)
        return self._forward_generic(latent_features, covariance_test, nodes_all)

    def _forward_fused(self, lat11, covariance_test, nodes_all):
        b = lat11.shape[1]
        lat11 = lat11.to(self.device, self.dtype).reshape(2, b, 1, self.tau_latent_vectors, 4)
        holder = {} if covariance_test else None
        out = fused._DecoderFn.apply(self._plan, self._theta_node(), lat11, covariance_test, holder)
        if not covariance_test:
            return out
        recon, gen00 = out
        gen = GVec({(0, 0): gen00, (1, 1): p_cplx_to_rep(recon)[(1, 1)].unsqueeze(-2)}, ignore_check=True)
        for l in range(self.num_cg_levels + 1):
            nodes_all.append(GVec(self._plan.node_features(holder["ws"], b, l), ignore_check=True))
        nodes_all.append(gen)
        return gen, nodes_all

    # generic composite, call sequence of lgn_decoder.py:218-345
    def _forward_generic(self, latent_features, covariance_test, nodes_all):
        graph = self.latent_to_graph(latent_features)
        graph = GVec({k: v.squeeze(-3) for k, v in graph.items()}, ignore_check=True)
        node_ps = p_cplx_to_rep(graph[(1, 1)])[(1, 1)]
        zf_in, _, _ = self.zonal_fns_in(node_ps)
        node = self.input_func_node(zf_in)
        dec_nodes = [node]
        if any(z != 1 for z in self.max_zf):
            # the reference's O(N^2) form: pairwise zonal functions, (masked-out) radial functions, edge features, aggregation
            b, n = node_ps.shape[1], node_ps.shape[2]
            node_mask = torch.zeros(2, b, n, dtype=torch.float32, device=node_ps.device)     # lgn_decoder.py:335-340
            zonal, norms, _ = self.zonal_fns(node_ps, node_ps)
            rad = self.rad_funcs.forward_masked_out(norms.shape)
            dec_nodes = self.lgn_cg(node, node_mask, rad, zonal)
        else:
            for idx, lvl in enumerate(self.lgn_cg.node_levels):
                node = self._level_closed_form(lvl, self.rad_funcs.rad_funcs[idx], node, zf_in[(1, 1)])
                if self.lgn_cg.mlp:
                    node = self.lgn_cg.mlp_levels[idx](node)
                dec_nodes.append(node)
        gen = self.mix_to_output(dec_nodes[-1])
        gen = GVec({w: gen[w] for w in [(0, 0), (1, 1)]}, ignore_check=True)
        if not covariance_test:
            return rep_to_p(gen[(1, 1)].clone()).squeeze(-2)
        for node in dec_nodes:
            nodes_all.append(node)
        nodes_all.append(gen)
        return gen, nodes_all

    def _level_closed_form(self, lvl, rad, node, y):
        """One LGN level of the decoder (lgn_levels.py:96-121) in O(N).  The decoder's edge mask is identically zero
        (lgn_decoder.py:335-340), so the radial weights are the constants R^l[c] = bias_l[c] (1+i) and the edge features are
        e^(0,0)_ij = R^0 (1+i), e^(1,1)_ij = R^1 (y_i - y_j).  The CG product is bilinear, hence
            sum_j CG(node_j (x) e_ij) = CG(M (x) E_i) - sum_j CG(node_j (x) E'_j),
        M = sum_j node_j,  E_i = {(0,0): R^0 (1+i), (1,1): R^1 y_i},  E'_j = {(0,0): 0, (1,1): R^1 y_j}:
        two point-wise products over the N particles instead of one over the N^2 edges; no (2,B,N,N,C,d) tensor exists.
        y: (2,B,N,1,4) canonical momenta of the nodes.  Same pair order / channel layout as the aggregated product."""
        b0, b1 = rad.linear[0].bias, rad.linear[1].bias          # (C,)
        some = next(iter(node.values()))
        B, N = some.shape[1], some.shape[2]
        zero = torch.zeros_like(b0)
        e00 = torch.stack((zero, 2.0 * b0)).view(2, 1, 1, -1, 1).expand(2, B, N, -1, 1)          # b0 (1+i)(1+i) = 2i b0
        yr, yi = y[0], y[1]                                                                       # (B,N,1,4)
        b1v = b1.view(1, 1, -1, 1)
        e11 = torch.stack((b1v * yr - b1v * yi, b1v * yi + b1v * yr))                             # b1 (1+i) y
        mom = GVec({k: v.sum(dim=2, keepdim=True).expand(-1, -1, N, -1, -1) for k, v in node.items()}, ignore_check=True)
        edge = GVec({(0, 0): e00, (1, 1): e11}, ignore_check=True)
        edge1 = GVec({(0, 0): torch.zeros_like(e00), (1, 1): e11}, ignore_check=True)
        a = cg_product(self.cg_dict, mom, edge, maxdim=lvl.maxdim)
        bj = cg_product(self.cg_dict, node, edge1, maxdim=lvl.maxdim)
        reps_ag = GVec({k: a[k] - bj[k].sum(dim=2, keepdim=True) for k in a.keys()}, ignore_check=True)
        reps_sq = lvl.cg_power(node, node)
        return lvl.cat_mix([reps_ag, node, reps_sq])
