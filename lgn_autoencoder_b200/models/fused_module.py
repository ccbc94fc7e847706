"""Mixin that keeps all parameters of a model as views of one flat fp64 buffer (what the kernels read) while
preserving the reference's per-tensor ``nn.Parameter`` names and shapes (SURVEY.md appendix A.9)."""
from collections import OrderedDict

import torch

from .. import fused


import os

_PARAM_GRAPH = os.environ.get("LGAE_PARAM_GRAPH") == "1"


class FusedParamsMixin:
    _plan = None
    _theta = None
    _param_list = None
    _probes = None
    _theta_nodes = None
    _grad_flat = None
    _grad_views = None

    def _build_plan(self, kind, **geometry):
        shapes = OrderedDict((name, tuple(p.shape)) for name, p in self.named_parameters())
        self._plan_kind, self._plan_geometry = kind, geometry
        self._plan = fused.FusedPlan(kind, shapes, **geometry)
        self._theta = None

    def _flat_params(self):
        """The flat buffer, rebuilt (and the parameters re-pointed into it) whenever a parameter no longer aliases
        it, e.g. after ``.to(device)``; ``load_state_dict`` and optimizer steps write in place and keep the aliasing.
        The aliasing of every parameter is verified when the buffer is built; afterwards each call probes the first, a middle
        and the last parameter (module-wide moves such as ``.to()`` / ``.double()`` re-create all of them)."""
        theta = self._theta
        if theta is not None:
            base, ok = theta.data_ptr(), True
            for p, off in self._probes:
                if p.data_ptr() != base + 8 * off or p.device != theta.device:
                    ok = False
                    break
            if ok:
                return theta, self._param_list
        params = OrderedDict(self.named_parameters())
        device = next(iter(params.values())).device
        theta = self._plan.flatten({k: v.data for k, v in params.items()}, device)
        for name, view in self._plan.views(theta).items():
            params[name].data = view
        self._theta = theta
        self._param_list = list(params.values())
        names = list(self._plan.offsets)
        self._probes = [(params[n], self._plan.offsets[n][0]) for n in (names[0], names[len(names) // 2], names[-1])]
        self._theta_nodes = {}
        return theta, self._param_list

    def _theta_node(self):
        """The flat parameter buffer as ONE autograd leaf.  The model-level Functions and the L1 / L2 norms take this tensor, so
        autograd sees one input per model instead of ~130: their gradients meet in a single flat add, and after the backward a
        post-accumulate hook hands the result to the parameters -- ``param.grad`` of every parameter is a view of one persistent
        flat bucket, bound once and re-bound only after ``zero_grad(set_to_none=True)``.  (With LGAE_PARAM_GRAPH=1 the
        parameters themselves are the graph's leaves, through ``fused._FlatParamsFn``: needed only by callers that ask autograd
        for gradients with respect to individual parameters, e.g. ``torch.autograd.grad(loss, model.parameters())``.)"""
        theta, params = self._flat_params()
        if not torch.is_grad_enabled():
            return theta
        flags = tuple(p.requires_grad for p in params)
        if not any(flags):
            return theta
        if _PARAM_GRAPH:
            key = (True, flags)   # (freezing / unfreezing parameters makes a new node)
            node = self._theta_nodes.get(key)
            if node is None:
                node = fused._FlatParamsFn.apply(self._plan, theta, *params)
                self._theta_nodes[key] = node
            return node
        leaf = self._theta_nodes.get("leaf")
        if leaf is None:
            leaf = theta.detach().requires_grad_(True)          # aliases the flat buffer
            leaf.register_post_accumulate_grad_hook(self._scatter_grad)
            self._theta_nodes["leaf"] = leaf
            self._grad_flat = torch.zeros_like(theta)
            self._grad_views = list(self._plan.views(self._grad_flat).values())
        return leaf

    def _scatter_grad(self, leaf):
        """Post-accumulate hook of the flat leaf: move its gradient into the persistent bucket the parameters' ``.grad`` view."""
        g = leaf.grad
        leaf.grad = None
        if g is None:
            return
        params, views, flat = self._param_list, self._grad_views, self._grad_flat
        probes = (params[0], params[len(params) // 2], params[-1])
        pviews = (views[0], views[len(params) // 2], views[-1])
        if all(p.grad is None for p in probes):
            flat.copy_(g)                                        # fresh gradients (zero_grad(set_to_none=True), the default)
            for p, v in zip(params, views):
                if p.requires_grad:
                    p.grad = v
        elif all(p.grad is not None and p.grad.data_ptr() == v.data_ptr() for p, v in zip(probes, pviews)):
            flat.add_(g)                                         # accumulating into the bound bucket
            for p, v in zip(params, views):
                if p.requires_grad and p.grad is None:
                    p.grad = v
        else:                                                    # somebody else owns (some of) the .grad tensors: per parameter
            for p, gv in zip(params, self._plan.views(g.contiguous()).values()):
                if not p.requires_grad:
                    continue
                if p.grad is None:
                    p.grad = gv.clone()
                else:
                    p.grad.add_(gv)

    def l1_norm(self):
        """sum |p| over all parameters (lgn_encoder.py:249-250), evaluated on the flat buffer in one reduction."""
        if self._plan is None or not self.fused:   # models that train on the composite (maxdim 3) sum per tensor
            return sum(p.abs().sum() for p in self.parameters())
        return _FlatNormFn.apply(self._theta_node(), 1)

    def l2_norm(self):
        """sum p^2 over all parameters (lgn_encoder.py:252-253)."""
        if self._plan is None or not self.fused:
            return sum(torch.pow(p, 2).sum() for p in self.parameters())
        return _FlatNormFn.apply(self._theta_node(), 2)


class _FlatNormFn(torch.autograd.Function):
    """L1 / squared-L2 norm of all parameters through the flat buffer they alias: two launches instead of two per tensor."""

    @staticmethod
    def forward(ctx, theta, order):
        ctx.order = order
        ctx.save_for_backward(theta)
        return theta.abs().sum() if order == 1 else (theta * theta).sum()

    @staticmethod
    def backward(ctx, g):
        (theta,) = ctx.saved_tensors
        return (torch.sign(theta) * g if ctx.order == 1 else 2.0 * theta * g), None
